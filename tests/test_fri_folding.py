"""FRI folding factors 2, 4 and 8 (ProofOptions accepts 2, 4, 8 and 16): the CPU oracle and both verifiers without a GPU, and the
CUDA prover byte for byte against the oracle on the GPU (one-shot, graph replay, staged surface, column-sharded)."""
import ctypes as C

import pytest

import zk_stark_project_b200 as Z
from zk_stark_project_b200 import lib as L
from zk_stark_project_b200.verifier import _fold_positions
from tests import common as T

SMALL_FACTORS = [2, 4, 8]


# ---- CPU: the oracle and both verifiers ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("folding", SMALL_FACTORS)
def test_oracle_proofs_verify(oracle, folding):
    """Training-shaped, MiMC and aggregation proofs at the folding factor are accepted by the oracle verifier and Z.verify."""
    for a, d in (T.training_case(8, 1024, T.options(folding=folding), 0xF01D + folding),
                 T.mimc_case(oracle, 4, 256, T.options(blowup=8, folding=folding)),
                 T.prover_case(T.aggregation_prover(16, T.options(folding=folding)))):
        proof, ts, _ = oracle.prove(a, d.tobytes())
        assert ts.comp_degree_ok == 1 and ts.n_fri_layers >= 1
        assert len(T.fri_layers(proof)) == ts.n_fri_layers
        oracle.verify(a, proof)
        assert Z.verify(proof, a)


@pytest.mark.parametrize("folding", SMALL_FACTORS)
def test_tampered_fri_layer_rejected(oracle, folding):
    """A flipped byte inside one FRI layer's queried values fails both verifiers."""
    air, data = T.training_case(8, 1024, T.options(folding=folding), 0xF02D + folding)
    proof, _, _ = oracle.prove(air, data.tobytes())
    layers = T.fri_layers(proof)
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
    air, data = T.training_case(8, 256, T.options(folding=8, rem=0), 0xF03D)
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
    T.prove_both(gpu_ctx, oracle, *T.training_case(8, 1024, T.options(folding=folding), 0xF04D + folding))


@pytest.mark.gpu
@pytest.mark.parametrize("folding", SMALL_FACTORS)
def test_mimc_parity(gpu_ctx, oracle, folding):
    T.prove_both(gpu_ctx, oracle, *T.mimc_case(oracle, 8, 1 << 14, T.options(blowup=8, folding=folding)))


@pytest.mark.gpu
@pytest.mark.parametrize("folding", SMALL_FACTORS)
def test_aggregation_graph_replay(oracle, folding):
    """Aggregation over 16 updates proved three times on one context: eager, captured, replayed from the CUDA graph.  Each proof
    has its own inputs and must equal the oracle's."""
    ctx = L.Context(0, own_stream=True)
    try:
        for rnd in range(3):
            T.prove_both(ctx, oracle, *T.prover_case(T.aggregation_prover(16, T.options(grinding=21, folding=folding), seed=0x5EED0003 + rnd)))
    finally:
        ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("folding", SMALL_FACTORS)
def test_zero_layer_domain(gpu_ctx, oracle, folding):
    """N = 128 <= (7 + 1) * 16: no FRI layer at all, whatever the folding factor."""
    T.prove_both(gpu_ctx, oracle, *T.training_case(2, 8, T.options(folding=folding), 0xF05D + folding))


@pytest.mark.gpu
@pytest.mark.parametrize("folding", SMALL_FACTORS)
@pytest.mark.parametrize("rem", [0, 31])
def test_remainder_degrees(gpu_ctx, oracle, folding, rem):
    """Remainder degree 0 (folding down to a constant: n a power of the factor) and 31."""
    n = 4096 if (rem == 0 and folding == 8) else 1024
    T.prove_both(gpu_ctx, oracle, *T.training_case(8, n, T.options(folding=folding, rem=rem), 0xF06D + folding + rem))


@pytest.mark.gpu
def test_config1_folding_8(gpu_ctx, oracle):
    """BASELINE.json configs[1] (240 x 2^16, blowup 16, reference options) with folding factor 8."""
    o = Z.ProofOptions.reference()
    T.prove_both(gpu_ctx, oracle, *T.training_case(240, 1 << 16, T.options(grinding=o.grinding_factor, folding=8), 0x5EED0002))


def _seventeen_layers():
    """2 x 2^17, blowup 2, remainder degree 0, folding 2: 17 FRI layers, more than the transcript's 16 slots."""
    return T.training_case(2, 1 << 17, T.options(blowup=2, folding=2, rem=0), 0xF07D)


@pytest.mark.gpu
def test_more_than_16_layers(gpu_ctx, oracle):
    air, data = _seventeen_layers()
    proof = T.prove_both(gpu_ctx, oracle, air, data)
    roots = T.commitments(proof)
    assert len(roots) == 2 + 17 + 1
    # the transcripts hold the true layer count and the first 16 roots
    for ts in (gpu_ctx.prove_host(air, data.ctypes.data)[1], oracle.prove(air, data.tobytes())[1]):
        assert ts.n_fri_layers == 17 and [bytes(ts.fri_roots[l]) for l in range(16)] == roots[2:18]


def _staged_fri(ctx, oracle, air, data):
    """Every stage through the staged surface with the oracle's challenges, then each FRI layer opened with zkb_query(2 + l) at the
    positions folded by the folding factor, against the FriProof of the oracle's proof.  With more than 16 layers the last fold
    takes a stand-in challenge, so the remainder is not compared."""
    n, beta, folding = air["trace_len"], air["options"]["blowup"], air["options"]["folding"]
    ref, ts, _ = oracle.prove(air, data.tobytes())
    roots = T.commitments(ref)
    st = T.Staged(ctx, air)
    assert st.trace_commit(data) == bytes(ts.trace_root)
    st.constraints_eval(bytes(ts.constraint_alpha))
    st.constraints_commit()
    st.ood_eval(bytes(ts.z))
    st.deep_compose(bytes(ts.deep_alpha))
    nl = st.fri_num_layers()
    assert nl == ts.n_fri_layers
    for l in range(nl):
        assert st.fri_commit_layer() == roots[2 + l], f"FRI layer {l} root differs"
        # the transcript holds the first 16 folding challenges; a later layer's root only depends on the earlier ones
        st.fri_fold(bytes(ts.fri_alphas[l]) if l < 16 else bytes(16))
    remainder_root = st.fri_remainder()
    if nl <= 16:
        assert remainder_root == bytes(ts.remainder_commitment) == roots[-1]
    layers = T.fri_layers(ref)
    assert len(layers) == nl
    fpos, dom = list(ts.positions)[:ts.n_positions], n * beta
    for l, (want_rows, want_paths) in enumerate(layers):
        fpos, dom = _fold_positions(fpos, dom, folding), dom // folding
        rows, paths = st.query(2 + l, fpos, folding)
        assert rows == want_rows, f"queried rows of FRI layer {l} differ"
        assert paths == want_paths, f"batch Merkle proof of FRI layer {l} differs"


@pytest.mark.gpu
def test_staged_surface_folding_4(gpu_ctx, oracle):
    _staged_fri(gpu_ctx, oracle, *T.prover_case(T.aggregation_prover(16, T.options(folding=4))))


@pytest.mark.gpu
def test_staged_surface_17_layers(gpu_ctx, oracle):
    """Layers past the transcript's 16 slots through the staged surface: all 17 roots and openings equal the oracle proof's."""
    _staged_fri(gpu_ctx, oracle, *_seventeen_layers())


@pytest.mark.gpu
def test_invalid_folding_factors(gpu_ctx, oracle):
    """Folding factors 3 and 32 are refused with ZKB_ERR_INVALID; the context then proves a valid proof."""
    air, data = T.training_case(8, 1024, T.options(folding=4), 0xF08D)
    for bad in (3, 32):
        broken = dict(air, options=dict(air["options"], folding=bad))
        with pytest.raises(L.ZkbError, match="2, 4, 8, 16") as e:
            gpu_ctx.prove_host(broken, data.ctypes.data)
        assert e.value.status == -1
    T.prove_both(gpu_ctx, oracle, air, data)


@pytest.mark.gpu
def test_column_sharded_small_factors():
    """The column-sharded proof with 2 ranks on one GPU (NCCL socket transport): FRI runs replicated on each rank, so MiMC at
    folding 8 and a training shape at folding 2 must equal the single-GPU proof."""
    T.run_sharded(2, 29617, [["mimc", 64, 1024, 8, 8], ["training", 128, 512, 16, 2]], one_gpu=True)
