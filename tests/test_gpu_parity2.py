"""GPU parity tests, part 2 (round 2): every BASELINE.json configuration at its exact size, the values the three Winterfell
associated types return through the C ABI (TraceLde / ConstraintEvaluator / ConstraintCommitment), and error paths added
in round 2.  Everything goes through libzkb200.so; the oracle is only the checker."""
import ctypes as C
import random

import numpy as np
import pytest

import zk_stark_project_b200 as Z
from zk_stark_project_b200 import lib as L
from zk_stark_project_b200.verifier import _fold_positions
from tests import common as T

pytestmark = pytest.mark.gpu
P = Z.P


def test_config0_mimc_2p14_exact(gpu_ctx, oracle):
    """BASELINE.json configs[0] exactly: MiMC 64 chains x 2^14 steps, blowup 8, the reference's other options
    (40 queries, 21-bit grinding, FRI folding 16, remainder degree <= 7; src/main.rs:98-107)."""
    air, data = T.mimc_case(oracle, 64, 1 << 14, Z.ProofOptions(40, 8, 21, Z.FieldExtension.NONE, 16, 7))
    seeds, rc = [j + 1 for j in range(64)], Z.get_round_constants()
    assert gpu_ctx.mimc_trace(seeds, 1 << 14, rc) == data.tobytes(), "device-side MiMC trace differs from the oracle's"
    T.prove_both(gpu_ctx, oracle, air, data)


def test_mimc_2p20_parity(gpu_ctx, oracle):
    """The headline shape (BASELINE.json metric: 2^20-row trace; configs[4] lower end): MiMC 64 x 2^20, blowup 8 (LDE 8 GiB),
    reference options — byte-identical to the oracle (three NTT passes, boundary-polynomial path, five FRI layers)."""
    air, data = T.mimc_case(oracle, 64, 1 << 20, Z.ProofOptions(40, 8, 21, Z.FieldExtension.NONE, 16, 7))
    seeds, rc = [j + 1 for j in range(64)], Z.get_round_constants()
    assert gpu_ctx.mimc_trace(seeds, 1 << 20, rc) == data.tobytes(), "device-side MiMC trace differs from the oracle's"
    T.prove_both(gpu_ctx, oracle, air, data)


def _staged_values(ctx, oracle, air, data, ce):
    """What the Rust associated types would hand to Winterfell: trace polynomials (TracePolyTable), main-trace frames
    (read_main_trace_frame_into) incl. the wrap-around rows, CompositionPolyTrace, and both Queries."""
    w, n, beta = air["trace_width"], air["trace_len"], air["options"]["blowup"]
    N = n * beta
    comp, ref_proof, ts = oracle.comp_trace(air, data.tobytes(), ce)
    _, lde, polys = oracle.trace_commit(data.tobytes(), n, w, beta, want_lde=True, want_polys=True)
    st = T.Staged(ctx, air)
    assert st.trace_commit(data) == bytes(ts.trace_root)
    # TracePolyTable: row-major [n][w] on our side, column-major [w][n] in the oracle
    got = np.frombuffer(st.trace_polys(), dtype=np.uint64).reshape(n, w, 2).transpose(1, 0, 2)
    assert np.array_equal(got, np.frombuffer(polys, dtype=np.uint64).reshape(w, n, 2)), "trace polynomials differ"
    # frames: first, last blowup rows (next wraps to the start), and random steps
    rng = random.Random(N + w)
    steps = [0, 1, beta, N - 1, N - beta, N - beta - 1, N - beta + 1] + [rng.randrange(N) for _ in range(24)]
    row = lambda r: lde[r * 16 * w:(r + 1) * 16 * w]
    for s in steps:
        cur, nxt = st.read_frame(s)
        assert cur == row(s) and nxt == row((s + beta) % N), f"frame at LDE step {s} differs"
    with pytest.raises(L.ZkbError) as e:  # out of range
        st.read_frame(N)
    assert e.value.status == -1
    # batched frame read: the same rows in one call
    cur_b, nxt_b = st.read_frames(steps)
    for i, s in enumerate(steps):
        assert cur_b[i * 16 * w:(i + 1) * 16 * w] == row(s) and nxt_b[i * 16 * w:(i + 1) * 16 * w] == row((s + beta) % N)
    # ConstraintEvaluator::evaluate -> CompositionPolyTrace
    assert st.constraints_eval(bytes(ts.constraint_alpha), ce) == comp, "constraint evaluations differ"
    assert st.constraints_commit() == bytes(ts.constraint_root)
    # TraceLde::query / ConstraintCommitment::query against the Queries sections of the oracle's proof — asked right after the
    # constraint commitment, as Winterfell's own generate_proof does when only the associated types are swapped (OOD, DEEP and
    # FRI then run on the host), and before this test drives the remaining device stages
    c = 6 if air["air_id"] == 3 else 1
    sec = T.proof_sections(ref_proof)
    pos = list(ts.positions)[:ts.n_positions]
    for which, width, name in ((0, w, "trace"), (1, c, "constraint")):
        rows, paths = st.query(which, pos, width)
        assert rows == ref_proof[sec[f"{name} rows"]], f"queried rows of commitment {which} differ"
        assert paths == ref_proof[sec[f"{name} paths"]], f"batch Merkle proof of commitment {which} differs"
    st.ood_eval(bytes(ts.z))
    st.deep_compose(bytes(ts.deep_alpha))
    nl = st.fri_num_layers()
    for l in range(nl):
        assert st.fri_commit_layer() == bytes(ts.fri_roots[l])
        st.fri_fold(bytes(ts.fri_alphas[l]))
    assert st.fri_remainder() == bytes(ts.remainder_commitment)
    # FriProver::build_proof: every layer at the positions folded as winter-fri's fold_positions does
    layers = T.fri_layers(ref_proof)
    assert len(layers) == nl
    fpos, dom = pos, N
    for l, (want_rows, want_paths) in enumerate(layers):
        fpos, dom = _fold_positions(fpos, dom, 16), dom // 16
        rows, paths = st.query(2 + l, fpos, 16)
        assert rows == want_rows, f"queried rows of FRI layer {l} differ"
        assert paths == want_paths, f"batch Merkle proof of FRI layer {l} differs"


def test_staged_values_aggregation(gpu_ctx, oracle):
    """BASELINE.json configs[2] (FedAvg over 16 updates, reference options) through the staged surface."""
    _staged_values(gpu_ctx, oracle, *T.prover_case(T.aggregation_prover(16, Z.ProofOptions.reference())), 2)


def test_staged_values_training_2p16(gpu_ctx, oracle):
    """BASELINE.json configs[1] (2^16 x 240, reference options) through the staged surface."""
    _staged_values(gpu_ctx, oracle, *T.training_case(240, 1 << 16, Z.ProofOptions.reference(), 0x5EED0002), 2)


def test_staged_values_mimc(gpu_ctx, oracle):
    """MiMC (ce = beta = 8, six composition columns) through the staged surface, two NTT passes."""
    air, data = T.mimc_case(oracle, 16, 1 << 12, T.options(blowup=8))
    seeds, rc = [j + 1 for j in range(16)], Z.get_round_constants()
    assert gpu_ctx.mimc_trace(seeds, 1 << 12, rc) == data.tobytes(), "device-side MiMC trace differs from the oracle's"
    _staged_values(gpu_ctx, oracle, air, data, 8)


def test_one_rank_sharded_proof(oracle):
    """A column-sharded proof on a one-rank communicator (row view of the LDE, Merkle cap, all-reduce of the openings) equals the
    single-GPU proof, and zkb_query refuses to open the commitments of a sharded proof."""
    ctx = L.Context(0)
    try:
        ctx.mg_init(0, 1, L.mg_unique_id())
        for air, data in (T.mimc_case(oracle, 16, 1 << 10, T.options(blowup=8)), T.training_case(32, 512, T.options(blowup=16), 0x5EED0005)):
            ptr = data.ctypes.data
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
    air, trace = T.prover_case(T.mimc_prover(4, 256, T.options(blowup=8)))
    data = trace.copy()
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
    assert ref == oracle.prove(air, trace.tobytes())[0]


def test_invalid_trace_reports_degree_failure(gpu_ctx, oracle):
    """A trace that violates the AIR: the composition polynomial does not fit its c*n coefficients.  The oracle flags it in the
    transcript (comp_degree_ok = 0); the library must do the same instead of silently truncating (ADVICE r1)."""
    air, trace = T.prover_case(T.mimc_prover(2, 128, T.options(blowup=8)))
    data = trace.copy()
    data[1, 77, 0] ^= 1  # break one transition
    _, ts_o, _ = oracle.prove(air, data.tobytes())
    assert ts_o.comp_degree_ok == 0
    _, ts = gpu_ctx.prove_host(air, data.ctypes.data)
    assert ts.comp_degree_ok == 0
    # and a valid trace keeps the flag set
    _, ts = gpu_ctx.prove_host(air, trace.ctypes.data)
    assert ts.comp_degree_ok == 1


def test_graph_replay_small_proofs(oracle):
    """Small proofs are replayed from a CUDA graph from the third proof of a shape on (first eager, second captured): every
    replay must honour that proof's own trace, public inputs and assertion values.  Different seeds, same shape, each proof
    compared with the oracle; interleaved with a second shape so that both graphs stay valid side by side."""
    ctx = L.Context(0, own_stream=True)
    for rnd in range(5):
        air, data = T.prover_case(T.aggregation_prover(16, Z.ProofOptions.reference(), seed=0x5EED0003 + rnd))
        got, ts = ctx.prove_host(air, data.ctypes.data)
        ref, ts_o, _ = oracle.prove(air, data.tobytes())
        assert T.transcript_diff(ts_o, ts) is None and got == ref, f"aggregation proof {rnd} differs"
        air, data = T.prover_case(Z.MimcProver(T.options(blowup=8, grinding=5), [100 * rnd + j + 1 for j in range(4)], 256))
        got, _ = ctx.prove_host(air, data.ctypes.data)
        assert got == oracle.prove(air, data.tobytes())[0], f"mimc proof {rnd} differs"
    # same shape, different round constants: the periodic column is baked into the evaluator tables, so this must not replay
    # the graph captured for the default constants
    for rnd in range(3):
        rc = [(7 * rnd + 3) * (i + 1) * 10**6 for i in range(64)]
        air, data = T.prover_case(Z.MimcProver(T.options(blowup=8, grinding=5), [j + 1 for j in range(4)], 256, round_constants=rc))
        got, _ = ctx.prove_host(air, data.ctypes.data)
        assert got == oracle.prove(air, data.tobytes())[0], f"mimc proof with custom round constants {rnd} differs"
    # a forced nonce takes the eager path and must still work on the same context
    air, data = T.prover_case(T.aggregation_prover(16, T.options(grinding=0)))
    got, ts = ctx.prove_host(air, data.ctypes.data, force_nonce=12345)
    assert ts.pow_nonce == 12345 and got == oracle.prove(air, data.tobytes(), force_nonce=12345)[0]
    ctx.close()


def test_training_2p18_parity(gpu_ctx, oracle):
    """Training shape 240 x 2^18, blowup 16 (LDE 15 GiB, three NTT passes with 128-row tiles — the pass plan of the 2^20-row
    headline), reference options: byte-identical to the oracle."""
    import bench
    n, w = 1 << 18, 240
    data = bench.counter_felts(w, n, 0x5EED1800)
    T.prove_both(gpu_ctx, oracle, T.synthetic_training_air(n, Z.ProofOptions.reference(), data), data)


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
    opts = Z.ProofOptions(20, 8, 4, Z.FieldExtension.NONE, 16, 7)
    T.prove_both(gpu_ctx, oracle, *T.training_case(w, 16, opts, 900 + w))
    seeds, rc = [j + 1 for j in range(w)], Z.get_round_constants()
    assert gpu_ctx.mimc_trace(seeds, 64, rc) == oracle.mimc_trace(seeds, 64, rc), "device-side MiMC trace differs from the oracle's"
    T.prove_both(gpu_ctx, oracle, *T.mimc_case(oracle, w, 64, opts))
