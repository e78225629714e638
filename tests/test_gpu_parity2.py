"""GPU parity tests, part 2 (round 2): every BASELINE.json configuration at its exact size, the values the three Winterfell
associated types return through the C ABI (TraceLde / ConstraintEvaluator / ConstraintCommitment), and error paths added
in round 2.  Everything goes through libzkb200.so; the oracle is only the checker."""
import ctypes as C
import random

import numpy as np
import pytest

import zk_stark_project_b200 as Z
from zk_stark_project_b200 import lib as L
from zk_stark_project_b200.verifier import _Reader, _fold_positions
from tests import common as T

pytestmark = pytest.mark.gpu
P = Z.P


def _mimc_case(ctx, oracle, w, n, opts, check_trace=True):
    rc = Z.get_round_constants()
    seeds = [j + 1 for j in range(w)]
    raw = ctx.mimc_trace(seeds, n, rc)
    if check_trace:
        assert raw == oracle.mimc_trace(seeds, n, rc), "device-side MiMC trace differs from the oracle's"
    data = np.frombuffer(raw, dtype=np.uint64).reshape(w, n, 2)
    get = lambda c, r: int(data[c, r, 0]) | (int(data[c, r, 1]) << 64)
    air = Z.MimcAir(w, n, Z.MimcInputs([get(j, 0) for j in range(w)], [get(j, n - 1) for j in range(w)]), opts).describe()
    return air, data


def _parity(ctx, oracle, air, data):
    proof, ts = ctx.prove_host(air, np.ascontiguousarray(data).ctypes.data)
    ref, ts_o, _ = oracle.prove(air, data.tobytes())
    assert T.transcript_diff(ts_o, ts) is None, f"transcripts diverge at `{T.transcript_diff(ts_o, ts)}`"
    assert proof == ref
    oracle.verify(air, proof)
    return proof


def test_config0_mimc_2p14_exact(gpu_ctx, oracle):
    """BASELINE.json configs[0] exactly: MiMC 64 chains x 2^14 steps, blowup 8, the reference's other options
    (40 queries, 21-bit grinding, FRI folding 16, remainder degree <= 7; src/main.rs:98-107)."""
    air, data = _mimc_case(gpu_ctx, oracle, 64, 1 << 14, Z.ProofOptions(40, 8, 21, Z.FieldExtension.NONE, 16, 7))
    proof = _parity(gpu_ctx, oracle, air, data)
    assert Z.verify(proof, air)


def test_mimc_2p20_parity(gpu_ctx, oracle):
    """The headline shape (BASELINE.json metric: 2^20-row trace; configs[4] lower end): MiMC 64 x 2^20, blowup 8 (LDE 8 GiB),
    reference options — byte-identical to the oracle (three NTT passes, boundary-polynomial path, five FRI layers)."""
    air, data = _mimc_case(gpu_ctx, oracle, 64, 1 << 20, Z.ProofOptions(40, 8, 21, Z.FieldExtension.NONE, 16, 7))
    _parity(gpu_ctx, oracle, air, data)


def _parse_queries(proof, w, c):
    """trace / constraint Queries sections of Proof::to_bytes() (rows bytes, BatchMerkleProof bytes)."""
    r = _Reader(proof)
    r.take(4 + 2 + 1 + 16 + 8 + 2)
    r.u8()
    r.take(r.uint(2))
    t_rows, t_paths = r.take(r.usize()), r.take(r.usize())
    c_rows, c_paths = r.take(r.usize()), r.take(r.usize())
    return t_rows, t_paths, c_rows, c_paths


def _parse_fri_layers(proof):
    """FriProof layers of Proof::to_bytes(): (rows bytes, BatchMerkleProof bytes) per layer."""
    r = _Reader(proof)
    r.take(4 + 2 + 1 + 16 + 8 + 2)
    r.u8()
    r.take(r.uint(2))
    for _ in range(4):  # trace and constraint Queries
        r.take(r.usize())
    for _ in range(3):  # OOD trace frame, Lagrange kernel frame, OOD constraint evaluations
        r.take(r.uint(2))
    return [(r.take(r.uint(4)), r.take(r.uint(4))) for _ in range(r.u8())]


def _staged_values(ctx, oracle, air, data, ce):
    """What the Rust associated types would hand to Winterfell: trace polynomials (TracePolyTable), main-trace frames
    (read_main_trace_frame_into) incl. the wrap-around rows, CompositionPolyTrace, and both Queries."""
    lib, h = ctx.lib, ctx.handle
    w, n, beta = air["trace_width"], air["trace_len"], air["options"]["blowup"]
    N = n * beta
    d = L.make_desc(air)
    buf = np.ascontiguousarray(data)
    cols = (C.c_void_p * w)(*[buf.ctypes.data + j * n * 16 for j in range(w)])
    comp, ref_proof, ts = oracle.comp_trace(air, buf.tobytes(), ce)
    _, lde, polys = oracle.trace_commit(buf.tobytes(), n, w, beta, want_lde=True, want_polys=True)
    root = C.create_string_buffer(32)
    ctx.check(lib.zkb_begin(h, C.byref(d)))
    ctx.check(lib.zkb_trace_commit(h, cols, root))
    assert root.raw == bytes(ts.trace_root)
    # TracePolyTable: row-major [n][w] on our side, column-major [w][n] in the oracle
    out = C.create_string_buffer(16 * n * w)
    ctx.check(lib.zkb_trace_polys_read(h, out))
    got = np.frombuffer(out.raw, dtype=np.uint64).reshape(n, w, 2).transpose(1, 0, 2)
    assert np.array_equal(got, np.frombuffer(polys, dtype=np.uint64).reshape(w, n, 2)), "trace polynomials differ"
    # frames: first, last blowup rows (next wraps to the start), and random steps
    rng = random.Random(N + w)
    steps = [0, 1, beta, N - 1, N - beta, N - beta - 1, N - beta + 1] + [rng.randrange(N) for _ in range(24)]
    cur, nxt = C.create_string_buffer(16 * w), C.create_string_buffer(16 * w)
    row = lambda r: lde[r * 16 * w:(r + 1) * 16 * w]
    for s in steps:
        ctx.check(lib.zkb_trace_read_frame(h, C.c_uint64(s), cur, nxt))
        assert cur.raw == row(s) and nxt.raw == row((s + beta) % N), f"frame at LDE step {s} differs"
    assert lib.zkb_trace_read_frame(h, C.c_uint64(N), cur, nxt) == -1  # out of range
    # batched frame read: the same rows in one call
    k = len(steps)
    arr = (C.c_uint64 * k)(*steps)
    cur_b, nxt_b = C.create_string_buffer(16 * w * k), C.create_string_buffer(16 * w * k)
    ctx.check(lib.zkb_trace_read_frames(h, arr, C.c_uint32(k), cur_b, nxt_b))
    for i, s in enumerate(steps):
        assert cur_b.raw[i * 16 * w:(i + 1) * 16 * w] == row(s) and nxt_b.raw[i * 16 * w:(i + 1) * 16 * w] == row((s + beta) % N)
    # ConstraintEvaluator::evaluate -> CompositionPolyTrace
    ev = C.create_string_buffer(16 * n * ce)
    ctx.check(lib.zkb_constraints_eval(h, bytes(ts.constraint_alpha), ev))
    assert ev.raw == comp, "constraint evaluations differ"
    ctx.check(lib.zkb_constraints_commit(h, root))
    assert root.raw == bytes(ts.constraint_root)
    # TraceLde::query / ConstraintCommitment::query against the Queries sections of the oracle's proof — asked right after the
    # constraint commitment, as Winterfell's own generate_proof does when only the associated types are swapped (OOD, DEEP and
    # FRI then run on the host), and before this test drives the remaining device stages
    c = 6 if air["air_id"] == 3 else 1
    t_rows, t_paths, c_rows, c_paths = _parse_queries(ref_proof, w, c)
    pos = (C.c_uint32 * ts.n_positions)(*list(ts.positions)[:ts.n_positions])
    for which, width, want_rows, want_paths in ((0, w, t_rows, t_paths), (1, c, c_rows, c_paths)):
        rows = C.create_string_buffer(16 * width * ts.n_positions)
        po, ln = C.c_void_p(), C.c_uint64()
        ctx.check(lib.zkb_query(h, C.c_uint32(which), pos, C.c_uint32(ts.n_positions), rows, C.byref(po), C.byref(ln)))
        paths = C.string_at(po, ln.value)
        lib.zkb_free(po)
        assert rows.raw == want_rows, f"queried rows of commitment {which} differ"
        assert paths == want_paths, f"batch Merkle proof of commitment {which} differs"
    ctx.check(lib.zkb_ood_eval(h, bytes(ts.z), None, None, None))
    ctx.check(lib.zkb_deep_compose(h, bytes(ts.deep_alpha)))
    nl = C.c_uint32()
    ctx.check(lib.zkb_fri_num_layers(h, C.byref(nl)))
    for l in range(nl.value):
        ctx.check(lib.zkb_fri_commit_layer(h, root))
        assert root.raw == bytes(ts.fri_roots[l])
        ctx.check(lib.zkb_fri_fold(h, bytes(ts.fri_alphas[l])))
    rem, cnt = C.create_string_buffer(16 * 256), C.c_uint64()
    ctx.check(lib.zkb_fri_remainder(h, rem, C.byref(cnt), root))
    assert root.raw == bytes(ts.remainder_commitment)
    # FriProver::build_proof: every layer at the positions folded as winter-fri's fold_positions does
    layers = _parse_fri_layers(ref_proof)
    assert len(layers) == nl.value
    fpos, dom = list(ts.positions)[:ts.n_positions], N
    for l, (want_rows, want_paths) in enumerate(layers):
        fpos, dom = _fold_positions(fpos, dom, 16), dom // 16
        arr = (C.c_uint32 * len(fpos))(*fpos)
        rows = C.create_string_buffer(16 * 16 * len(fpos))
        po, ln = C.c_void_p(), C.c_uint64()
        ctx.check(lib.zkb_query(h, C.c_uint32(2 + l), arr, C.c_uint32(len(fpos)), rows, C.byref(po), C.byref(ln)))
        paths = C.string_at(po, ln.value)
        lib.zkb_free(po)
        assert rows.raw == want_rows, f"queried rows of FRI layer {l} differ"
        assert paths == want_paths, f"batch Merkle proof of FRI layer {l} differs"


def test_staged_values_aggregation(gpu_ctx, oracle):
    """BASELINE.json configs[2] (FedAvg over 16 updates, reference options) through the staged surface."""
    p = T.aggregation_prover(16, Z.ProofOptions.reference())
    trace = p.build_trace()
    _staged_values(gpu_ctx, oracle, p.describe(trace), np.ascontiguousarray(trace.data), 2)


def test_staged_values_training_2p16(gpu_ctx, oracle):
    """BASELINE.json configs[1] (2^16 x 240, reference options) through the staged surface."""
    n = 1 << 16
    data = T.random_felts(240 * n, 0x5EED0002).reshape(240, n, 2)
    air = T.synthetic_training_air(n, Z.ProofOptions.reference(), data)
    _staged_values(gpu_ctx, oracle, air, data, 2)


def test_staged_values_mimc(gpu_ctx, oracle):
    """MiMC (ce = beta = 8, six composition columns) through the staged surface, two NTT passes."""
    air, data = _mimc_case(gpu_ctx, oracle, 16, 1 << 12, T.options(blowup=8))
    _staged_values(gpu_ctx, oracle, air, data, 8)


def test_one_rank_sharded_proof(oracle):
    """A column-sharded proof on a one-rank communicator (row view of the LDE, Merkle cap, all-reduce of the openings) equals the
    single-GPU proof, and zkb_query refuses to open the commitments of a sharded proof."""
    ctx = L.Context(0)
    try:
        ctx.mg_init(0, 1, L.mg_unique_id())
        mimc = _mimc_case(ctx, oracle, 16, 1 << 10, T.options(blowup=8), check_trace=False)
        data = T.random_felts(32 * 512, 0x5EED0005).reshape(32, 512, 2)
        for air, trace in (mimc, (T.synthetic_training_air(512, T.options(blowup=16), data), data)):
            ptr = np.ascontiguousarray(trace).ctypes.data
            single, _ = ctx.prove_host(air, ptr)
            sharded, _ = ctx.mg_prove_host(air, ptr, 1)
            assert sharded == single
        pos = (C.c_uint32 * 1)(0)
        rows, po, ln = C.create_string_buffer(16 * 32), C.c_void_p(), C.c_uint64()
        assert ctx.lib.zkb_query(ctx.handle, C.c_uint32(0), pos, C.c_uint32(1), rows, C.byref(po), C.byref(ln)) == -3
    finally:
        ctx.close()


def test_non_canonical_trace_is_reduced(gpu_ctx, oracle):
    """Winterfell's BaseElement::new reduces a u128 >= p; trace cells handed over as raw u128 in [p, 2^128) must give the same
    proof as their canonical representatives (ADVICE r1: canonicalise on ingest)."""
    p = T.mimc_prover(4, 256, T.options(blowup=8))
    trace = p.build_trace()
    air = p.describe(trace)
    data = np.ascontiguousarray(trace.data).copy()
    ref, _ = gpu_ctx.prove_host(air, data.ctypes.data)
    # cells small enough that v + p < 2^128: the seeds in row 0 (and any other small cell)
    bumped = 0
    for j in range(4):
        for i in range(256):
            v = int(data[j, i, 0]) | (int(data[j, i, 1]) << 64)
            if v + P < 2**128:
                v += P
                data[j, i, 0], data[j, i, 1] = v & (2**64 - 1), v >> 64
                bumped += 1
    assert bumped >= 4
    got, _ = gpu_ctx.prove_host(air, data.ctypes.data)
    assert got == ref
    assert ref == oracle.prove(air, trace.to_bytes())[0]


def test_invalid_trace_reports_degree_failure(gpu_ctx, oracle):
    """A trace that violates the AIR: the composition polynomial does not fit its c*n coefficients.  The oracle flags it in the
    transcript (comp_degree_ok = 0); the library must do the same instead of silently truncating (ADVICE r1)."""
    p = T.mimc_prover(2, 128, T.options(blowup=8))
    trace = p.build_trace()
    air = p.describe(trace)
    data = np.ascontiguousarray(trace.data).copy()
    data[1, 77, 0] ^= 1  # break one transition
    _, ts_o, _ = oracle.prove(air, data.tobytes())
    assert ts_o.comp_degree_ok == 0
    _, ts = gpu_ctx.prove_host(air, data.ctypes.data)
    assert ts.comp_degree_ok == 0
    # and a valid trace keeps the flag set
    _, ts = gpu_ctx.prove_host(air, np.ascontiguousarray(trace.data).ctypes.data)
    assert ts.comp_degree_ok == 1


def test_graph_replay_small_proofs(oracle):
    """Small proofs are replayed from a CUDA graph from the third proof of a shape on (first eager, second captured): every
    replay must honour that proof's own trace, public inputs and assertion values.  Different seeds, same shape, each proof
    compared with the oracle; interleaved with a second shape so that both graphs stay valid side by side."""
    ctx = L.Context(0, own_stream=True)
    for rnd in range(5):
        p = T.aggregation_prover(16, Z.ProofOptions.reference(), seed=0x5EED0003 + rnd)
        tr = p.build_trace()
        air = p.describe(tr)
        got, ts = ctx.prove_host(air, np.ascontiguousarray(tr.data).ctypes.data)
        ref, ts_o, _ = oracle.prove(air, tr.to_bytes())
        assert T.transcript_diff(ts_o, ts) is None and got == ref, f"aggregation proof {rnd} differs"
        m = Z.MimcProver(T.options(blowup=8, grinding=5), [100 * rnd + j + 1 for j in range(4)], 256)
        mt = m.build_trace()
        mair = m.describe(mt)
        got, _ = ctx.prove_host(mair, np.ascontiguousarray(mt.data).ctypes.data)
        assert got == oracle.prove(mair, mt.to_bytes())[0], f"mimc proof {rnd} differs"
    # same shape, different round constants: the periodic column is baked into the evaluator tables, so this must not replay
    # the graph captured for the default constants
    for rnd in range(3):
        rc = [(7 * rnd + 3) * (i + 1) * 10**6 for i in range(64)]
        m = Z.MimcProver(T.options(blowup=8, grinding=5), [j + 1 for j in range(4)], 256, round_constants=rc)
        mt = m.build_trace()
        mair = m.describe(mt)
        got, _ = ctx.prove_host(mair, np.ascontiguousarray(mt.data).ctypes.data)
        assert got == oracle.prove(mair, mt.to_bytes())[0], f"mimc proof with custom round constants {rnd} differs"
    # a forced nonce takes the eager path and must still work on the same context
    p = T.aggregation_prover(16, T.options(grinding=0))
    tr = p.build_trace()
    air = p.describe(tr)
    got, ts = ctx.prove_host(air, np.ascontiguousarray(tr.data).ctypes.data, force_nonce=12345)
    assert ts.pow_nonce == 12345 and got == oracle.prove(air, tr.to_bytes(), force_nonce=12345)[0]
    ctx.close()


def test_training_2p18_parity(gpu_ctx, oracle):
    """Training shape 240 x 2^18, blowup 16 (LDE 15 GiB, three NTT passes with 128-row tiles — the pass plan of the 2^20-row
    headline), reference options: byte-identical to the oracle."""
    import bench
    n, w = 1 << 18, 240
    data = bench.counter_felts(w, n, 0x5EED1800)
    air = T.synthetic_training_air(n, Z.ProofOptions.reference(), data)
    _parity(gpu_ctx, oracle, air, data)


def test_training_2p20_proof_verifies(gpu_ctx, oracle):
    """The metric's own shape — a 2^20-row x 240-column trace, blowup 16, LDE 60 GiB — is too large for the CPU oracle to prove
    inside a test, so it is covered by size-independent properties: the CUDA proof is accepted by both verifier restatements
    (which recompute the whole transcript, the OOD consistency check, 40 Merkle openings per commitment and FRI), a proof with a
    tampered public input is rejected, and proving twice gives the same bytes.  (bench.py additionally checks that the proof
    sharded over N GPUs equals this single-GPU proof.)"""
    import bench
    n, w = 1 << 20, 240
    pin = L.PinnedBuffer(w * n * 16)
    arr = pin.view().view(np.uint64).reshape(w, n, 2)
    arr[:] = bench.counter_felts(w, n, 0x5EED2000)
    get = lambda c, r: int(arr[c, r, 0]) | (int(arr[c, r, 1]) << 64)
    opts = Z.ProofOptions.reference()
    air = bench.training_air_from_rows(n, w, opts, [get(j, 0) for j in range(w)], [get(j, n - 1) for j in range(w)])
    proof, ts = gpu_ctx.prove_host(air, pin.ptr)
    assert ts.n_fri_layers == 5 and ts.comp_degree_ok == 1
    oracle.verify(air, proof)
    assert Z.verify(proof, air)
    again, _ = gpu_ctx.prove_host(air, pin.ptr)
    assert again == proof
    bad = dict(air, assertions=[(air["assertions"][0][0], air["assertions"][0][1], 7)] + list(air["assertions"][1:]))
    with pytest.raises(RuntimeError):
        oracle.verify(bad, proof)
    pin.free()


@pytest.mark.parametrize("w", [65, 128, 129, 192, 193])
def test_small_domain_leaf_chunk_boundaries(gpu_ctx, oracle, w):
    """Small LDE domains hash a row's 1 KiB BLAKE3 chunks on separate lanes (k_hash_lde_rows_split) and give every
    constraint-evaluation point a warp: widths on both sides of the 2-, 3- and 4-chunk boundaries, training-shaped and MiMC AIRs."""
    n = 16
    opts = Z.ProofOptions(20, 8, 4, Z.FieldExtension.NONE, 16, 7)
    data = T.random_felts(w * n, 900 + w).reshape(w, n, 2)
    _parity(gpu_ctx, oracle, T.synthetic_training_air(n, opts, data), data)
    air, mdata = _mimc_case(gpu_ctx, oracle, w, 64, opts)
    _parity(gpu_ctx, oracle, air, mdata)
