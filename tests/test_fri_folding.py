"""FRI folding factors 2, 4 and 8 (ProofOptions accepts 2, 4, 8 and 16): the CPU oracle and both verifiers without a GPU, and the
CUDA prover byte for byte against the oracle on the GPU (one-shot, graph replay, staged surface, column-sharded)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import zk_stark_project_b200 as Z
from zk_stark_project_b200 import lib as L
from zk_stark_project_b200.verifier import _Reader, _fold_positions
from tests import common as T
from tests.test_gpu_parity import _prove_both
from tests.test_gpu_parity2 import _parse_fri_layers

SMALL_FACTORS = [2, 4, 8]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _opts(folding, blowup=16, rem=7, queries=40, grinding=8):
    return Z.ProofOptions(queries, blowup, grinding, Z.FieldExtension.NONE, folding, rem)


def _training(w, n, opts, seed):
    data = T.random_felts(w * n, seed).reshape(w, n, 2)
    return T.synthetic_training_air(n, opts, data), data


def _mimc(oracle, w, n, opts):
    p = T.mimc_prover(w, n, opts)
    raw = oracle.mimc_trace(p.seeds, n, p.rc)
    trace = Z.TraceTable(np.frombuffer(raw, dtype=np.uint64).reshape(w, n, 2))
    return p.describe(trace), np.ascontiguousarray(trace.data)


def _commitments(proof):
    """The Commitments section of Proof::to_bytes(): trace root, constraint root, one root per FRI layer, remainder."""
    r = _Reader(proof)
    r.take(4 + 2 + 1 + 16 + 8 + 2)
    r.u8()
    blob = r.take(r.uint(2))
    return [blob[i:i + 32] for i in range(0, len(blob), 32)]


# ---- CPU: the oracle and both verifiers ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("folding", SMALL_FACTORS)
def test_oracle_proofs_verify(oracle, folding):
    """Training-shaped, MiMC and aggregation proofs at the folding factor are accepted by the oracle verifier and Z.verify."""
    air, data = _training(8, 1024, _opts(folding), 0xF01D + folding)
    mair, mdata = _mimc(oracle, 4, 256, _opts(folding, blowup=8))
    p = T.aggregation_prover(16, _opts(folding))
    tr = p.build_trace()
    for a, d in ((air, data), (mair, mdata), (p.describe(tr), np.ascontiguousarray(tr.data))):
        proof, ts, _ = oracle.prove(a, d.tobytes())
        assert ts.comp_degree_ok == 1 and ts.n_fri_layers >= 1
        assert len(_parse_fri_layers(proof)) == ts.n_fri_layers
        oracle.verify(a, proof)
        assert Z.verify(proof, a)


@pytest.mark.parametrize("folding", SMALL_FACTORS)
def test_tampered_fri_layer_rejected(oracle, folding):
    """A flipped byte inside one FRI layer's queried values fails both verifiers."""
    air, data = _training(8, 1024, _opts(folding), 0xF02D + folding)
    proof, _, _ = oracle.prove(air, data.tobytes())
    layers = _parse_fri_layers(proof)
    for rows, _ in (layers[0], layers[-1]):
        off = proof.find(rows)
        assert off > 0 and len(rows) % (16 * folding) == 0
        bad = bytearray(proof)
        bad[off + len(rows) // 2 - 16] ^= 1   # the low byte of an element in the middle of the values
        with pytest.raises(RuntimeError):
            oracle.verify(air, bytes(bad))
        with pytest.raises(Z.VerifierError):
            Z.verify(bytes(bad), air)


def test_degree_truncation_rejected(oracle):
    """Folding 8 down to a constant (remainder degree 0) from n = 256, not a power of 8: both verifiers report degree truncation,
    as Winterfell's does."""
    air, data = _training(8, 256, _opts(8, rem=0), 0xF03D)
    proof, _, _ = oracle.prove(air, data.tobytes())
    with pytest.raises(RuntimeError, match="FRI degree truncation"):
        oracle.verify(air, proof)
    with pytest.raises(Z.VerifierError, match="FRI degree truncation"):
        Z.verify(proof, air)


# ---- GPU: the CUDA prover against the oracle -------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_hash_elements_count_8(gpu_ctx, oracle):
    """Leaves of a folding-8 FRI layer: Blake3_256::hash_elements of 8 elements (128 bytes, two BLAKE3 blocks)."""
    rows = 37
    data = T.random_felts(rows * 8, 1008).tobytes()
    out = C.create_string_buffer(32 * rows)
    gpu_ctx.check(gpu_ctx.lib.zkb_test_hash_elements(gpu_ctx.handle, data, C.c_uint32(8), C.c_uint32(rows), out))
    for r in range(rows):
        assert out.raw[32 * r:32 * r + 32] == oracle.blake3(data[r * 128:(r + 1) * 128]), r


@pytest.mark.gpu
@pytest.mark.parametrize("folding", SMALL_FACTORS)
def test_training_shaped_parity(gpu_ctx, oracle, folding):
    air, data = _training(8, 1024, _opts(folding), 0xF04D + folding)
    _prove_both(gpu_ctx, oracle, air, Z.TraceTable(data))


@pytest.mark.gpu
@pytest.mark.parametrize("folding", SMALL_FACTORS)
def test_mimc_parity(gpu_ctx, oracle, folding):
    air, data = _mimc(oracle, 8, 1 << 14, _opts(folding, blowup=8))
    _prove_both(gpu_ctx, oracle, air, Z.TraceTable(data))


@pytest.mark.gpu
@pytest.mark.parametrize("folding", SMALL_FACTORS)
def test_aggregation_graph_replay(oracle, folding):
    """Aggregation over 16 updates proved three times on one context: eager, captured, replayed from the CUDA graph.  Each proof
    has its own inputs and must equal the oracle's."""
    ctx = L.Context(0, own_stream=True)
    try:
        for rnd in range(3):
            p = T.aggregation_prover(16, _opts(folding, grinding=21), seed=0x5EED0003 + rnd)
            tr = p.build_trace()
            air = p.describe(tr)
            got, ts = ctx.prove_host(air, np.ascontiguousarray(tr.data).ctypes.data)
            ref, ts_o, _ = oracle.prove(air, tr.to_bytes())
            assert T.transcript_diff(ts_o, ts) is None and got == ref, f"proof {rnd} differs"
            assert Z.verify(got, air)
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("folding", SMALL_FACTORS)
def test_zero_layer_domain(gpu_ctx, oracle, folding):
    """N = 128 <= (7 + 1) * 16: no FRI layer at all, whatever the folding factor."""
    air, data = _training(2, 8, _opts(folding), 0xF05D + folding)
    _prove_both(gpu_ctx, oracle, air, Z.TraceTable(data))


@pytest.mark.gpu
@pytest.mark.parametrize("folding", SMALL_FACTORS)
@pytest.mark.parametrize("rem", [0, 31])
def test_remainder_degrees(gpu_ctx, oracle, folding, rem):
    """Remainder degree 0 (folding down to a constant: n a power of the factor) and 31."""
    n = 4096 if (rem == 0 and folding == 8) else 1024
    air, data = _training(8, n, _opts(folding, rem=rem), 0xF06D + folding + rem)
    _prove_both(gpu_ctx, oracle, air, Z.TraceTable(data))


@pytest.mark.gpu
def test_config1_folding_8(gpu_ctx, oracle):
    """BASELINE.json configs[1] (240 x 2^16, blowup 16, reference options) with folding factor 8."""
    o = Z.ProofOptions.reference()
    air, data = _training(240, 1 << 16, _opts(8, grinding=o.grinding_factor), 0x5EED0002)
    _prove_both(gpu_ctx, oracle, air, Z.TraceTable(data))


def _seventeen_layers():
    """2 x 2^17, blowup 2, remainder degree 0, folding 2: 17 FRI layers, more than the transcript's 16 slots."""
    return _training(2, 1 << 17, _opts(2, blowup=2, rem=0), 0xF07D)


@pytest.mark.gpu
def test_more_than_16_layers(gpu_ctx, oracle):
    air, data = _seventeen_layers()
    proof, ts = gpu_ctx.prove_host(air, data.ctypes.data)
    ref, ts_o, _ = oracle.prove(air, data.tobytes())
    assert ts.n_fri_layers == 17 and ts_o.n_fri_layers == 17
    assert T.transcript_diff(ts_o, ts) is None and proof == ref
    roots = _commitments(proof)
    assert len(roots) == 2 + 17 + 1
    assert [bytes(ts.fri_roots[l]) for l in range(16)] == roots[2:18]
    oracle.verify(air, proof)
    assert Z.verify(proof, air)


def _staged_fri(ctx, oracle, air, data):
    """Every stage through the staged surface with the oracle's challenges, then each FRI layer opened with zkb_query(2 + l) at the
    positions folded by the folding factor, against the FriProof of the oracle's proof.  With more than 16 layers the last fold
    takes a stand-in challenge, so the remainder is not compared."""
    lib, h = ctx.lib, ctx.handle
    w, n, beta, folding = air["trace_width"], air["trace_len"], air["options"]["blowup"], air["options"]["folding"]
    ref, ts, _ = oracle.prove(air, data.tobytes())
    roots = _commitments(ref)
    d = L.make_desc(air)
    cols = (C.c_void_p * w)(*[data.ctypes.data + j * n * 16 for j in range(w)])
    root = C.create_string_buffer(32)
    ctx.check(lib.zkb_begin(h, C.byref(d)))
    ctx.check(lib.zkb_trace_commit(h, cols, root))
    assert root.raw == bytes(ts.trace_root)
    ctx.check(lib.zkb_constraints_eval(h, bytes(ts.constraint_alpha), None))
    ctx.check(lib.zkb_constraints_commit(h, root))
    ctx.check(lib.zkb_ood_eval(h, bytes(ts.z), None, None, None))
    ctx.check(lib.zkb_deep_compose(h, bytes(ts.deep_alpha)))
    nl = C.c_uint32()
    ctx.check(lib.zkb_fri_num_layers(h, C.byref(nl)))
    assert nl.value == ts.n_fri_layers
    for l in range(nl.value):
        ctx.check(lib.zkb_fri_commit_layer(h, root))
        assert root.raw == roots[2 + l], f"FRI layer {l} root differs"
        # the transcript holds the first 16 folding challenges; a later layer's root only depends on the earlier ones
        ctx.check(lib.zkb_fri_fold(h, bytes(ts.fri_alphas[l]) if l < 16 else bytes(16)))
    rem, cnt = C.create_string_buffer(16 * 256), C.c_uint64()
    ctx.check(lib.zkb_fri_remainder(h, rem, C.byref(cnt), root))
    if nl.value <= 16:
        assert root.raw == bytes(ts.remainder_commitment) == roots[-1]
    layers = _parse_fri_layers(ref)
    assert len(layers) == nl.value
    fpos, dom = list(ts.positions)[:ts.n_positions], n * beta
    for l, (want_rows, want_paths) in enumerate(layers):
        fpos, dom = _fold_positions(fpos, dom, folding), dom // folding
        arr = (C.c_uint32 * len(fpos))(*fpos)
        rows = C.create_string_buffer(16 * folding * len(fpos))
        po, ln = C.c_void_p(), C.c_uint64()
        ctx.check(lib.zkb_query(h, C.c_uint32(2 + l), arr, C.c_uint32(len(fpos)), rows, C.byref(po), C.byref(ln)))
        paths = C.string_at(po, ln.value)
        lib.zkb_free(po)
        assert rows.raw == want_rows, f"queried rows of FRI layer {l} differ"
        assert paths == want_paths, f"batch Merkle proof of FRI layer {l} differs"


@pytest.mark.gpu
def test_staged_surface_folding_4(gpu_ctx, oracle):
    p = T.aggregation_prover(16, _opts(4))
    tr = p.build_trace()
    _staged_fri(gpu_ctx, oracle, p.describe(tr), np.ascontiguousarray(tr.data))


@pytest.mark.gpu
def test_staged_surface_17_layers(gpu_ctx, oracle):
    """Layers past the transcript's 16 slots through the staged surface: all 17 roots and openings equal the oracle proof's."""
    air, data = _seventeen_layers()
    _staged_fri(gpu_ctx, oracle, air, data)


@pytest.mark.gpu
def test_invalid_folding_factors(gpu_ctx, oracle):
    """Folding factors 3 and 32 are refused with ZKB_ERR_INVALID; the context then proves a valid proof."""
    air, data = _training(8, 1024, _opts(4), 0xF08D)
    for bad in (3, 32):
        broken = dict(air, options=dict(air["options"], folding=bad))
        with pytest.raises(L.ZkbError, match="2, 4, 8, 16") as e:
            gpu_ctx.prove_host(broken, data.ctypes.data)
        assert e.value.status == -1
    _prove_both(gpu_ctx, oracle, air, Z.TraceTable(data))


@pytest.mark.gpu
def test_column_sharded_small_factors():
    """The column-sharded proof with 2 ranks on one GPU (NCCL socket transport): FRI runs replicated on each rank, so MiMC at
    folding 8 and a training shape at folding 2 must equal the single-GPU proof."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0], NCCL_SOCKET_IFNAME="lo",
               GLOO_SOCKET_IFNAME="lo", NCCL_IB_DISABLE="1")
    cases = '[["mimc", 64, 1024, 8, 8], ["training", 128, 512, 16, 2]]'
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29617", "tests/mg_folding_worker.py", cases], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "mg ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
