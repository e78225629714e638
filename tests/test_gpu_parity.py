"""GPU parity tests: every stage of the CUDA path against the CPU oracle, through the C ABI (libzkb200.so)."""
import ctypes as C
import random

import numpy as np
import pytest

import zk_stark_project_b200 as Z
from zk_stark_project_b200 import lib as L
from tests import common as T

pytestmark = pytest.mark.gpu
P = Z.P


def test_field_kat(gpu_ctx, oracle):
    rng = random.Random(11)
    edge = [0, 1, 2, P - 1, P - 2, 2**127, 2**64, 2**64 - 1, 45 * 2**40 - 1, 45 * 2**40, 2**96, P >> 1]
    a = edge * len(edge) + [rng.randrange(P) for _ in range(4000)]
    b = [y for y in edge for _ in edge] + [rng.randrange(P) for _ in range(4000)]
    n = len(a)
    ab = b"".join(L.fe_bytes(x) for x in a)
    bb = b"".join(L.fe_bytes(x) for x in b)
    outs = [C.create_string_buffer(16 * n) for _ in range(4)]
    gpu_ctx.check(gpu_ctx.lib.zkb_test_field(gpu_ctx.handle, ab, bb, C.c_uint32(n), *outs))
    mul, add, sub, inv = [[L.fe_int(o.raw[16 * i:16 * i + 16]) for i in range(n)] for o in outs]
    for i in range(n):
        assert mul[i] == a[i] * b[i] % P, (a[i], b[i])
        assert add[i] == (a[i] + b[i]) % P
        assert sub[i] == (a[i] - b[i]) % P
        assert inv[i] == (pow(a[i], P - 2, P) if a[i] else 0)
    # and against the oracle's field
    for i in range(0, n, 97):
        assert mul[i] == oracle.fe_op("mul", a[i], b[i])


@pytest.mark.parametrize("count", [1, 2, 3, 4, 5, 6, 7, 16, 60, 63, 64, 65, 120, 127, 128, 129, 192, 193, 240, 255])
def test_hash_elements(gpu_ctx, oracle, count):
    """Blake3_256::hash_elements for every leaf shape on the path (SURVEY Appendix C) and the chunk boundaries around them."""
    rows = 37
    data = T.random_felts(rows * count, 1000 + count).tobytes()
    out = C.create_string_buffer(32 * rows)
    gpu_ctx.check(gpu_ctx.lib.zkb_test_hash_elements(gpu_ctx.handle, data, C.c_uint32(count), C.c_uint32(rows), out))
    for r in range(rows):
        assert out.raw[32 * r:32 * r + 32] == oracle.blake3(data[r * count * 16:(r + 1) * count * 16]), (count, r)


@pytest.mark.parametrize("n", [2, 4, 64, 1024, 4096])
def test_merkle_root(gpu_ctx, oracle, n):
    leaves = np.random.default_rng(n).integers(0, 256, size=(n, 32), dtype=np.uint8)
    root = C.create_string_buffer(32)
    gpu_ctx.check(gpu_ctx.lib.zkb_test_merkle_root(gpu_ctx.handle, leaves.tobytes(), C.c_uint64(n), root))
    assert root.raw == oracle.merkle_root([leaves[i].tobytes() for i in range(n)])


LDE_CASES = [(512, 20, 4), (512, 50, 2), (256, 17, 16), (8, 1, 2), (8, 3, 8), (16, 5, 16), (32, 120, 16), (64, 17, 8), (128, 240, 16), (256, 16, 4), (512, 33, 2),
             (1024, 64, 8), (4096, 9, 16), (8192, 20, 8), (1 << 14, 2, 16), (1 << 16, 4, 4)]


@pytest.mark.parametrize("n,w,blowup", LDE_CASES)
def test_interpolate_and_lde(gpu_ctx, oracle, n, w, blowup):
    """K1 + K2 against winter-math's interpolate_poly / evaluate_poly_with_offset (oracle), every pass plan:
    single pass (n <= 2^8 with 16-column tiles), two passes, narrow-column tiles, ragged column tiles."""
    data = T.random_felts(w * n, 7 * n + w).reshape(w, n, 2)
    buf = np.ascontiguousarray(data)
    cols = (C.c_void_p * w)(*[buf.ctypes.data + j * n * 16 for j in range(w)])
    polys = C.create_string_buffer(16 * n * w)
    lde = C.create_string_buffer(16 * n * w * blowup)
    gpu_ctx.check(gpu_ctx.lib.zkb_test_lde(gpu_ctx.handle, cols, C.c_uint32(w), C.c_uint64(n), C.c_uint32(blowup), polys, lde))
    root, o_lde, o_polys = oracle.trace_commit(buf.tobytes(), n, w, blowup, want_lde=True, want_polys=True)
    # oracle polys are column-major [w][n]; the product keeps them row-major [n][w]
    got = np.frombuffer(polys.raw, dtype=np.uint64).reshape(n, w, 2).transpose(1, 0, 2)
    exp = np.frombuffer(o_polys, dtype=np.uint64).reshape(w, n, 2)
    assert np.array_equal(got, exp), "interpolated polynomials differ"
    assert lde.raw == o_lde, "LDE differs"


def _prove_both(gpu_ctx, oracle, air, trace):
    proof_o, ts_o, _ = oracle.prove(air, trace.to_bytes())
    data = np.ascontiguousarray(trace.data)
    proof_g, ts_g = gpu_ctx.prove_host(air, data.ctypes.data)
    diff = T.transcript_diff(ts_o, ts_g)
    assert diff is None, f"transcripts diverge at `{diff}`"
    assert proof_g == proof_o, "proof bytes differ although the transcript matches"
    oracle.verify(air, proof_g)
    assert Z.verify(proof_g, air)  # the product's own (Python) verifier
    return proof_g


@pytest.mark.parametrize("width,steps,blowup", [(1, 64, 8), (4, 64, 8), (64, 256, 8), (3, 1024, 16), (8, 1 << 14, 8),
                                                (64, 1 << 13, 8)])  # the last one takes the boundary-polynomial path
def test_mimc_proof_parity(gpu_ctx, oracle, width, steps, blowup):
    p = T.mimc_prover(width, steps, T.options(blowup=blowup))
    if steps <= 1024:
        trace = p.build_trace()
    else:
        raw = oracle.mimc_trace(p.seeds, steps, p.rc)
        trace = Z.TraceTable(np.frombuffer(raw, dtype=np.uint64).reshape(width, steps, 2))
    _prove_both(gpu_ctx, oracle, p.describe(trace), trace)


def test_mimc_device_trace(gpu_ctx, oracle):
    rc = Z.get_round_constants()
    seeds = [3, 5, 7]
    assert gpu_ctx.mimc_trace(seeds, 512, rc) == oracle.mimc_trace(seeds, 512, rc)


@pytest.mark.parametrize("updates", [1, 6, 16, 30])
def test_aggregation_proof_parity(gpu_ctx, oracle, updates):
    p = T.aggregation_prover(updates, T.options())
    trace = p.build_trace()
    _prove_both(gpu_ctx, oracle, p.describe(trace), trace)


@pytest.mark.parametrize("bs", [1, 2, 5])
def test_training_proof_parity(gpu_ctx, oracle, bs):
    p = T.training_prover(bs, T.options())
    trace = p.build_trace()
    _prove_both(gpu_ctx, oracle, p.describe(trace), trace)


def test_training_reference_options_bs1(gpu_ctx, oracle):
    """The exact ProofOptions of src/main.rs:98-107 (21-bit grinding): smallest-nonce PoW must match the oracle."""
    p = T.training_prover(1, Z.ProofOptions.reference())
    trace = p.build_trace()
    _prove_both(gpu_ctx, oracle, p.describe(trace), trace)


def test_training_synthetic_8192(gpu_ctx, oracle):
    """bs=50-sized trace (the largest the reference CLI reaches, src/main.rs:77): two-pass NTT, 2^17-row LDE."""
    n = 8192
    data = T.random_felts(240 * n, 0x5EED0400).reshape(240, n, 2)
    air = T.synthetic_training_air(n, T.options(), data)
    _prove_both(gpu_ctx, oracle, air, Z.TraceTable(data))


def test_python_prover_surface(gpu_ctx, oracle):
    """`prover.prove(trace)` as main.rs drives it, verified by the oracle's restatement of winterfell::verify."""
    p = T.aggregation_prover(16, T.options())
    trace = p.build_trace()
    proof = p.prove(trace)
    oracle.verify(p.describe(trace), proof.to_bytes())
    assert proof.transcript.n_positions > 0 and len(proof) == len(proof.to_bytes())


def test_invalid_inputs_rejected(gpu_ctx):
    """tests/integration_tests.rs:201-230 expects a panic on mismatched batch sizes; the C ABI returns ZKB_ERR_INVALID."""
    with pytest.raises(AssertionError):
        Z.TrainingUpdateProver(T.options(), [[0] * 9] * 6, [0] * 6, [[0] * 9] * 6, [0] * 6, [[0] * 9], [[0] * 9], [[0] * 6], 1, 1, 2)
    p = T.mimc_prover(2, 64, T.options(blowup=8))
    trace = p.build_trace()
    air = p.describe(trace)
    bad = dict(air)
    bad["options"] = dict(air["options"], blowup=4)  # below the degree-7 constraint blowup
    data = np.ascontiguousarray(trace.data)
    with pytest.raises(L.ZkbError) as e:
        gpu_ctx.prove_host(bad, data.ctypes.data)
    assert e.value.status == -1
    bad = dict(air, assertions=[(5, 0, 1)])  # column out of range
    with pytest.raises(L.ZkbError):
        gpu_ctx.prove_host(bad, data.ctypes.data)


def test_staged_api_matches_one_shot(gpu_ctx, oracle):
    """The staged surface (TraceLde / ConstraintEvaluator / ConstraintCommitment + DEEP/FRI stages) reproduces the oracle transcript."""
    p = T.aggregation_prover(16, T.options())
    trace = p.build_trace()
    air = p.describe(trace)
    _, ts, _ = oracle.prove(air, trace.to_bytes())
    lib, h = gpu_ctx.lib, gpu_ctx.handle
    d = L.make_desc(air)
    data = np.ascontiguousarray(trace.data)
    w, n = trace.width(), trace.length()
    cols = (C.c_void_p * w)(*[data.ctypes.data + j * n * 16 for j in range(w)])
    root = C.create_string_buffer(32)
    gpu_ctx.check(lib.zkb_begin(h, C.byref(d)))
    gpu_ctx.check(lib.zkb_trace_commit(h, cols, root))
    assert root.raw == bytes(ts.trace_root)
    # TraceLde::read_main_trace_frame_into
    cur, nxt = C.create_string_buffer(16 * w), C.create_string_buffer(16 * w)
    gpu_ctx.check(lib.zkb_trace_read_frame(h, C.c_uint64(0), cur, nxt))
    _, lde, _ = oracle.trace_commit(trace.to_bytes(), n, w, 16, want_lde=True)
    assert cur.raw == lde[:16 * w] and nxt.raw == lde[16 * 16 * w:17 * 16 * w]
    gpu_ctx.check(lib.zkb_constraints_eval(h, bytes(ts.constraint_alpha), None))
    gpu_ctx.check(lib.zkb_constraints_commit(h, root))
    assert root.raw == bytes(ts.constraint_root)
    # out-of-order call is refused
    assert lib.zkb_deep_compose(h, bytes(ts.deep_alpha)) == -3
    gpu_ctx.check(lib.zkb_ood_eval(h, bytes(ts.z), None, None, None))
    gpu_ctx.check(lib.zkb_deep_compose(h, bytes(ts.deep_alpha)))
    nl = C.c_uint32()
    gpu_ctx.check(lib.zkb_fri_num_layers(h, C.byref(nl)))
    assert nl.value == ts.n_fri_layers
    for l in range(nl.value):
        gpu_ctx.check(lib.zkb_fri_commit_layer(h, root))
        assert root.raw == bytes(ts.fri_roots[l])
        gpu_ctx.check(lib.zkb_fri_fold(h, bytes(ts.fri_alphas[l])))
    rem, cnt = C.create_string_buffer(16 * 64), C.c_uint64()
    gpu_ctx.check(lib.zkb_fri_remainder(h, rem, C.byref(cnt), root))
    assert root.raw == bytes(ts.remainder_commitment)


def test_column_sharded_proof_two_gpus():
    """SURVEY §8e / BASELINE configs[4]: a proof produced cooperatively by 2 GPUs (column-sharded LDE, NVLink all-to-all,
    row-sharded hashing, all-gather of subtree roots) is byte-identical to the single-GPU proof."""
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = __import__("os").path.dirname(__import__("os").path.dirname(__import__("os").path.abspath(__file__)))
    cases = '[["mimc", 64, 1024, 8], ["mimc", 16, 256, 8], ["training", 128, 512, 16], ["training", 240, 256, 16], ["mimc", 6, 128, 8]]'
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29611", "tests/mg_worker.py", cases], cwd=root, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "mg ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_column_sharded_proof_ranks_share_one_gpu():
    """The sharded path with 2 and 4 ranks on one GPU, the ranks talking over NCCL's socket transport: rows and authentication
    nodes owned by one rank, the cap levels of the trace paths, the all-reduce of the openings, the OOD frame reorder and, with
    more ranks than the blowup, the replicated composition commitment.  The proofs must equal the single-GPU proof."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0], NCCL_SOCKET_IFNAME="lo",
               GLOO_SOCKET_IFNAME="lo", NCCL_IB_DISABLE="1")
    for g, port, cases in ((2, 29613, '[["mimc", 64, 1024, 8], ["training", 128, 512, 16], ["mimc", 6, 128, 8]]'),
                           (4, 29615, '[["training", 128, 1024, 2], ["mimc", 16, 256, 8]]')):
        r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(g), "--master-addr", "127.0.0.1",
                            "--master-port", str(port), "tests/mg_worker.py", cases], cwd=root, env=env, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0 and "mg ok" in r.stdout, f"{g} ranks: " + r.stdout[-2000:] + r.stderr[-2000:]


def _training_shaped(oracle, gpu_ctx, w, n, opts, seed):
    data = T.random_felts(w * n, seed).reshape(w, n, 2)
    air = T.synthetic_training_air(n, opts, data)
    return _prove_both(gpu_ctx, oracle, air, Z.TraceTable(data))


@pytest.mark.parametrize("w,n,blowup", [(2, 8, 2), (2, 8, 16), (4, 16, 4), (254, 16, 8), (6, 32, 32), (10, 64, 64), (2, 8, 128), (30, 2048, 2)])
def test_edge_shapes_training_air(gpu_ctx, oracle, w, n, blowup):
    """Minimum trace length (TraceInfo: n >= 8), extreme widths, every blowup factor ProofOptions accepts (2..128),
    domains small enough that FRI has zero layers (N <= 128: the remainder is interpolated straight from the DEEP evaluations)."""
    _training_shaped(oracle, gpu_ctx, w, n, Z.ProofOptions(27, blowup, 6, Z.FieldExtension.NONE, 16, 7), 31 * w + n)


@pytest.mark.parametrize("queries,grinding,rem", [(1, 0, 7), (255, 3, 7), (40, 10, 0), (40, 4, 3), (40, 4, 15), (12, 32 - 16, 31)])
def test_option_extremes(gpu_ctx, oracle, queries, grinding, rem):
    """num_queries 1 and 255, no grinding, remainder degrees 0..31 (FRI depth changes with the remainder bound)."""
    opts = Z.ProofOptions(queries, 16, grinding, Z.FieldExtension.NONE, 16, rem)
    # with remainder degree 0 FRI folds all the way to a constant: the trace length must be a power of the folding factor
    # or the verifier reports degree truncation (as Winterfell's does)
    n = 4096 if rem == 0 else 1024
    _training_shaped(oracle, gpu_ctx, 8, n, opts, 77 + queries)


def test_mimc_width_255_like(gpu_ctx, oracle):
    """Widest MiMC trace that still fits TraceInfo (255 columns: 4 BLAKE3 chunks per leaf with a ragged tail)."""
    p = T.mimc_prover(255, 64, T.options(blowup=8))
    trace = p.build_trace()
    _prove_both(gpu_ctx, oracle, p.describe(trace), trace)


def test_repeated_proofs_reuse_context(gpu_ctx, oracle):
    """A context is reused across proofs of different shapes (buffers grow, tables are rebuilt); results stay exact."""
    for width, steps, blowup in [(4, 4096, 8), (2, 64, 16), (16, 512, 8), (4, 4096, 8)]:
        p = T.mimc_prover(width, steps, T.options(blowup=blowup))
        raw = oracle.mimc_trace(p.seeds, steps, p.rc)
        trace = Z.TraceTable(np.frombuffer(raw, dtype=np.uint64).reshape(width, steps, 2))
        _prove_both(gpu_ctx, oracle, p.describe(trace), trace)


def test_pageable_and_scattered_columns(gpu_ctx, oracle):
    """Columns handed over as separate, non-contiguous, pageable host buffers (what a Vec<Vec<Felt>> TraceTable looks like)."""
    p = T.aggregation_prover(16, T.options())
    trace = p.build_trace()
    air = p.describe(trace)
    w, n = trace.width(), trace.length()
    cols = [np.array(trace.data[j], copy=True) for j in reversed(range(w))][::-1]  # separately allocated
    ptrs = (C.c_void_p * w)(*[c.ctypes.data for c in cols])
    d = L.make_desc(air)
    out, ln, ts = C.c_void_p(), C.c_uint64(), L.Transcript()
    gpu_ctx.check(gpu_ctx.lib.zkb_prove(gpu_ctx.handle, C.byref(d), ptrs, C.c_uint64(0), C.byref(out), C.byref(ln), C.byref(ts)))
    proof = C.string_at(out, ln.value)
    gpu_ctx.lib.zkb_free(out)
    ref, _, _ = oracle.prove(air, trace.to_bytes())
    assert proof == ref


def test_mimc_helpers_batch(gpu_ctx):
    """GPU mimc_cipher / mimc_hash_matrix against the Python restatement of src/helper.rs:213-233 (benches/bench_mimc.rs shapes)."""
    rng = random.Random(5)
    xs = [rng.randrange(P) for _ in range(300)] + [0, P - 1]
    rcs = [rng.randrange(2**64) for _ in xs]
    zs = [0] * 100 + [rng.randrange(P) for _ in range(len(xs) - 100)]
    assert L.mimc_cipher_batch(gpu_ctx, xs, rcs, zs) == [Z.mimc_cipher(x, r, z) for x, r, z in zip(xs, rcs, zs)]
    rc = Z.get_round_constants()
    ws = [[[rng.randrange(P) for _ in range(9)] for _ in range(6)] for _ in range(40)]
    bs = [[rng.randrange(P) for _ in range(6)] for _ in range(40)]
    ws[0] = [[Z.f64_to_felt(42.0)] * 9 for _ in range(6)]  # the criterion bench's fixed input
    bs[0] = [Z.f64_to_felt(1.0)] * 6
    assert L.mimc_hash_matrix_batch(gpu_ctx, ws, bs, rc) == [Z.mimc_hash_matrix(w, b, rc) for w, b in zip(ws, bs)]


def test_full_size_training_proof(gpu_ctx, oracle):
    """BASELINE.json configs[1] at full size (2^16 x 240, blowup 16, the reference's exact options: 40 queries, 21-bit grinding):
    the CUDA proof equals the oracle's byte for byte and both verifier restatements accept it."""
    n = 1 << 16
    data = T.random_felts(240 * n, 0x5EED0002).reshape(240, n, 2)
    air = T.synthetic_training_air(n, Z.ProofOptions.reference(), data)
    proof, ts = gpu_ctx.prove_host(air, np.ascontiguousarray(data).ctypes.data)
    assert ts.n_fri_layers == 4 and ts.n_positions <= 40
    assert Z.verify(proof, air)
    oracle.verify(air, proof)
    ref, ts_o, _ = oracle.prove(air, data.tobytes())
    assert T.transcript_diff(ts_o, ts) is None and proof == ref


def test_large_mimc_proof_verifies(gpu_ctx, oracle):
    """MiMC 64 x 2^18 (three NTT passes, LDE 2 GiB), trace generated on the device: size-independent acceptance check
    (prove -> verify) with both verifiers, plus determinism of the proof."""
    w, n = 64, 1 << 18
    rc = Z.get_round_constants()
    raw = gpu_ctx.mimc_trace([j + 1 for j in range(w)], n, rc)
    data = np.frombuffer(raw, dtype=np.uint64).reshape(w, n, 2)
    get = lambda c, r: int(data[c, r, 0]) | (int(data[c, r, 1]) << 64)
    air = Z.MimcAir(w, n, Z.MimcInputs([get(j, 0) for j in range(w)], [get(j, n - 1) for j in range(w)]),
                    Z.ProofOptions(40, 8, 21, Z.FieldExtension.NONE, 16, 7)).describe()
    proof, ts = gpu_ctx.prove_host(air, np.ascontiguousarray(data).ctypes.data)
    assert ts.n_fri_layers == 4
    assert Z.verify(proof, air)
    oracle.verify(air, proof)
    again, _ = gpu_ctx.prove_host(air, np.ascontiguousarray(data).ctypes.data)
    assert again == proof
    # a wrong claimed result must be rejected
    bad = dict(air, assertions=air["assertions"][:-1] + [(air["assertions"][-1][0], air["assertions"][-1][1], 12345)])
    with pytest.raises(Z.VerifierError):
        Z.verify(proof, bad)


def test_prove_batch_single_rank(gpu_ctx, oracle):
    """multi_gpu.prove_batch (BASELINE configs[3]: a batch of independent proofs) on one rank: order preserved, all verify."""
    from zk_stark_project_b200 import multi_gpu as M
    jobs = []
    for i in range(4):
        p = Z.MimcProver(T.options(blowup=8, grinding=4), [50 * i + j + 1 for j in range(1 + i)], 128)
        jobs.append((p, p.build_trace()))
    proofs = M.prove_batch(jobs, gpu_ctx)
    assert len(proofs) == 4 and len({M.digest(p) for p in proofs}) == 4
    assert M.prove_batch(jobs, gpu_ctx, lanes=[L.Context(0, own_stream=True)]) == proofs  # same through zkb_prove_batch with two lanes
    for (p, tr), proof in zip(jobs, proofs):
        assert Z.verify(proof, p.describe(tr))
        assert proof == oracle.prove(p.describe(tr), tr.to_bytes())[0]


def test_randomized_shape_sweep(gpu_ctx, oracle):
    """Seeded sweep over trace shapes (length, width, blowup, AIR): every layout decision in the driver (pass plans, ragged
    column tiles, ingest groups, panel sizes, FRI depth) is shape dependent, so proofs of many odd shapes are compared byte
    for byte with the oracle."""
    rng = random.Random(0xB200)
    for case in range(36):
        kind = rng.choice(["training", "training", "mimc"])
        n = 1 << rng.randint(3, 12)
        if kind == "mimc":
            n = max(n, 64)
            w = rng.choice([1, 2, 3, 5, 8, 13, 16, 17, 31, 33, 48, 49, 64, 65, 80])
            blowup = rng.choice([8, 16, 32])
            p = Z.MimcProver(Z.ProofOptions(rng.randint(1, 60), blowup, rng.randint(0, 8), Z.FieldExtension.NONE, 16, rng.choice([3, 7, 15])),
                             [rng.randrange(P) for _ in range(w)], n)
            raw = oracle.mimc_trace(p.seeds, n, p.rc)
            trace = Z.TraceTable(np.frombuffer(raw, dtype=np.uint64).reshape(w, n, 2))
            air = p.describe(trace)
        else:
            w = 2 * rng.randint(1, 127)
            blowup = rng.choice([2, 4, 8, 16, 32, 64])
            opts = Z.ProofOptions(rng.randint(1, 60), blowup, rng.randint(0, 8), Z.FieldExtension.NONE, 16, rng.choice([3, 7, 15]))
            data = T.random_felts(w * n, 1000 + case).reshape(w, n, 2)
            air = T.synthetic_training_air(n, opts, data)
            trace = Z.TraceTable(data)
        try:
            _prove_both(gpu_ctx, oracle, air, trace)
        except RuntimeError as e:
            # the only legitimate verifier complaint for arbitrary option combinations (as in Winterfell): the remainder bound
            # does not divide the degree along the FRI layers
            assert "degree truncation" in str(e) or "remainder degree" in str(e), (case, kind, n, w, blowup, str(e))


def test_device_side_training_trace(gpu_ctx, oracle):
    """SURVEY §8f: the training trace built on the GPU equals its host reconstruction (same raw states, same ChaCha20 mask
    stream under the test's key) and proves / verifies like a host-built one; without a key the masks come from OS entropy."""
    p = T.training_prover(3, T.options())
    key = bytes(range(32))
    dt = p.build_trace_device(key=key, ctx=gpu_ctx)
    assert (dt.width(), dt.length()) == (240, 512)
    host = dt.to_host()
    states = p.raw_states()
    assert len(states) == 4
    for i in (0, 1, 2, 3, 4, 100, 511):
        raw = states[min(i, 3)]
        for j in (0, 1, 7, 8, 57, 119):
            mask = T.training_mask(key, i, j, 120)
            assert host.get(120 + j, i) == mask and host.get(j, i) == (raw[j] + mask) % P
    assert [dt.get(c, 0) for c in range(240)] == [host.get(c, 0) for c in range(240)]
    assert [dt.get(c, 511) for c in range(240)] == [host.get(c, 511) for c in range(240)]
    proof = p.prove(dt)
    air = p.describe(dt)
    assert Z.verify(proof, air)
    oracle.verify(air, proof.to_bytes())
    assert proof.to_bytes() == oracle.prove(air, host.to_bytes())[0]
    # default: a fresh OS-entropy key per call - two traces must not share their masks
    a = p.build_trace_device(ctx=gpu_ctx).to_host()
    b = p.build_trace_device(ctx=gpu_ctx).to_host()
    assert not np.array_equal(a.data[120:], b.data[120:])
    assert np.all(a.data[120:, :, 1] == 0)  # 64-bit masks (src/training/prover.rs:119-121)


def test_boundary_polynomial_path_forced():
    """The evaluator takes boundary numerators either as per-point sums or as polynomials combined in coefficient space and
    extended once; the library picks by cost.  ZKB_BOUNDARY_POLY=1 forces the polynomial path for every AIR and shape: the
    proof-parity tests must still produce the oracle's bytes (the env var is read once per process, hence the subprocess)."""
    import os
    import subprocess
    import sys
    env = dict(os.environ, ZKB_BOUNDARY_POLY="1")
    sel = "mimc_proof_parity or aggregation_proof_parity or training_proof_parity or edge_shapes or staged_api or randomized_shape_sweep"
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-m", "gpu", "-k", sel, "-p", "no:cacheprovider"],
                       env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]


def test_native_prove_batch(gpu_ctx, oracle):
    """zkb_prove_batch (BASELINE configs[3]): a mixed batch over three lanes returns, in order, exactly the proofs the one-shot
    call produces; a bad job fails the call with its status and leaves the other jobs' proofs intact."""
    lanes = [gpu_ctx, L.Context(0, own_stream=True), L.Context(0, own_stream=True)]
    jobs = []
    for i in range(7):
        p = T.mimc_prover(1 + i, 128, T.options(blowup=8, grinding=4)) if i % 2 else T.training_prover(1 + i // 2, T.options(grinding=4))
        tr = p.build_trace()
        jobs.append((p.describe(tr), np.ascontiguousarray(tr.data)))
    proofs = L.prove_batch(lanes, [a for a, _ in jobs], [d.ctypes.data for _, d in jobs])
    for (air, data), proof in zip(jobs, proofs):
        single, _ = gpu_ctx.prove_host(air, data.ctypes.data)
        assert proof == single
        oracle.verify(air, proof)
    assert L.prove_batch(lanes, [], []) == []
    bad = dict(jobs[1][0], options=dict(jobs[1][0]["options"], blowup=3))
    with pytest.raises(L.ZkbError) as e:
        L.prove_batch(lanes, [jobs[0][0], bad, jobs[2][0]], [jobs[0][1].ctypes.data, jobs[1][1].ctypes.data, jobs[2][1].ctypes.data])
    assert e.value.status == -1  # ZKB_ERR_INVALID
    # the lanes are still usable afterwards
    again, _ = lanes[1].prove_host(jobs[0][0], jobs[0][1].ctypes.data)
    assert again == proofs[0]
