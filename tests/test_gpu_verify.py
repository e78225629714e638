"""zkb_verify_batch / Z.verify_batch: winterfell::verify for a batch of proofs on the GPU.  Every verdict is compared with the
CPU oracle's verifier (orc_verify) on the same bytes, and every accepted proof's re-derived transcript with the oracle's."""
import ctypes as C
import random

import pytest

import zk_stark_project_b200 as Z
from zk_stark_project_b200 import lib as L
from tests import common as T

OK, MALFORMED = 0, 1
# first words of the oracle verifier's failure messages -> zkb_verdict
ORACLE_CATEGORIES = [
    ("trace info mismatch", 2), ("unacceptable proof options", 3), ("wrong number of commitments", 4),
    ("wrong number of FRI layers", 4), ("bad OOD frame", 5), ("inconsistent OOD constraint evaluations", 6),
    ("query seed proof-of-work", 7), ("number of unique queries", 8), ("bad trace query values", 9),
    ("trace query did not match", 10), ("bad constraint query values", 11), ("constraint query did not match", 12),
    ("bad FRI layer values", 13), ("FRI layer query did not match", 14), ("invalid FRI layer folding", 15),
    ("FRI degree truncation", 16), ("FRI remainder degree mismatch", 17), ("FRI remainder commitment mismatch", 18),
    ("invalid FRI remainder folding", 19),
]


def oracle_verdict(oracle, air, proof):
    """(zkb_verdict, oracle transcript or None) of the CPU verifier on `proof`."""
    try:
        return OK, oracle.verify(air, proof)
    except RuntimeError as e:
        msg = str(e)
    for key, v in ORACLE_CATEGORIES:
        if key in msg:
            return v, None
    assert msg.startswith(("proof:", "reader:", "std::")) or "alloc" in msg, msg   # deserialization
    return MALFORMED, None


# ---- accepted proofs -----------------------------------------------------------------------------------------------------------

def accepted_cases(oracle):
    ref = Z.ProofOptions.reference()
    cases = {
        "training bs=1": T.prover_case(T.training_prover(1, ref)),
        "training bs=2": T.prover_case(T.training_prover(2, ref)),
        "configs[1] 2^16 x 240": T.training_case(240, 1 << 16, ref, 0x5EED0002),
        "aggregation 1": T.prover_case(T.aggregation_prover(1, ref)),
        "aggregation 6": T.prover_case(T.aggregation_prover(6, ref)),
        "aggregation 16": T.prover_case(T.aggregation_prover(16, ref)),
        "mimc 1x64": T.mimc_case(oracle, 1, 64, T.options(blowup=8)),
        "mimc 4x128": T.mimc_case(oracle, 4, 128, T.options(blowup=8)),
        "mimc 64x2^14": T.mimc_case(oracle, 64, 1 << 14, T.options(blowup=8)),
        "17 layers": T.training_case(2, 1 << 17, T.options(blowup=2, folding=2, rem=0), 0xF07D),
        "0 layers": T.training_case(2, 8, T.options(folding=4), 0xF05D),
        "remainder degree 0": T.training_case(8, 4096, T.options(folding=8, rem=0), 0xF06D),
        "remainder degree 31": T.training_case(8, 1024, T.options(folding=4, rem=31), 0xF06E),
        "1 query": T.training_case(8, 1024, T.options(queries=1), 0xF101),
        "255 queries": T.training_case(8, 1024, T.options(queries=255), 0xF102),
        "grinding 0": T.training_case(8, 1024, T.options(grinding=0), 0xF103),
        "grinding 21": T.training_case(8, 1024, T.options(grinding=21), 0xF104),
    }
    for f in (2, 4, 8, 16):
        cases[f"training folding {f}"] = T.training_case(8, 1024, T.options(folding=f), 0xF200 + f)
        cases[f"mimc folding {f}"] = T.mimc_case(oracle, 4, 256, T.options(blowup=8, folding=f))
    return cases


@pytest.mark.gpu
def test_accepted_proofs_and_transcripts(gpu_ctx, oracle):
    """Every accepted shape: GPU proofs (and oracle proofs of the small shapes) get ZKB_VERIFY_OK in one batch, with the
    transcript the oracle verifier re-derives."""
    airs, proofs, names = [], [], []
    for name, (air, data) in accepted_cases(oracle).items():
        airs.append(air); proofs.append(gpu_ctx.prove_host(air, data.ctypes.data)[0]); names.append(name + " (zkb_prove)")
        if data.size <= 2 * 8 * 4096 and air["options"]["grinding"] <= 8:
            airs.append(air); proofs.append(oracle.prove(air, data.tobytes())[0]); names.append(name + " (oracle)")
    verdicts, ts = gpu_ctx.verify_batch(airs, proofs)
    for name, air, proof, v, t in zip(names, airs, proofs, verdicts, ts):
        want, ts_o = oracle_verdict(oracle, air, proof)
        assert want == OK, name
        assert v == OK, f"{name}: verdict {v}"
        assert T.transcript_diff(ts_o, t) is None, f"{name}: transcript differs at {T.transcript_diff(ts_o, t)}"
    assert any("oracle" in n for n in names)


# ---- rejected proofs -----------------------------------------------------------------------------------------------------------

def flip_cases(gpu_ctx, oracle):
    """(air, proof) pairs whose sections get flipped: training, MiMC and aggregation, two folding factors"""
    out = []
    for air, data in (T.training_case(8, 1024, T.options(), 0xF301), T.training_case(8, 1024, T.options(queries=20, folding=4), 0xF302),
                      T.mimc_case(oracle, 4, 256, T.options(blowup=8)), T.prover_case(T.aggregation_prover(6, T.options()))):
        out.append((air, gpu_ctx.prove_host(air, data.ctypes.data)[0]))
    air, data = T.training_case(8, 512, T.options(folding=8), 0xF303)
    out.append((air, oracle.prove(air, data.tobytes())[0]))
    return out


@pytest.mark.gpu
def test_section_flips_match_oracle(gpu_ctx, oracle):
    """Seeded byte flips in every section of several proofs (>= 200 flips): the GPU verdict equals the oracle's category for
    every flip, including flips the oracle accepts."""
    rng = random.Random(0xF11F)
    airs, proofs, want = [], [], []
    for air, proof in flip_cases(gpu_ctx, oracle):
        for name, span in T.proof_sections(proof).items():
            a, b = span.start, span.stop
            if b <= a:
                continue
            for _ in range(5 if b - a > 64 else 3):
                bad = bytearray(proof)
                bad[rng.randrange(a, b)] ^= rng.randrange(1, 256)
                airs.append(air); proofs.append(bytes(bad)); want.append((name, oracle_verdict(oracle, air, bytes(bad))[0]))
    assert len(proofs) >= 200
    verdicts, _ = gpu_ctx.verify_batch(airs, proofs)
    bad = [(n, w, v) for (n, w), v in zip(want, verdicts) if w != v]
    assert not bad, f"{len(bad)} of {len(want)} verdicts differ from the oracle, e.g. {bad[:5]}"
    assert len({w for _, w in want}) >= 8   # the flips reach many different checks


@pytest.mark.gpu
def test_truncations_and_other_inputs_match_oracle(gpu_ctx, oracle):
    """Truncation at every section boundary, one trailing byte, changed public input / assertion value / options, and the proof
    of an AIR-violating trace: the GPU verdict equals the oracle's."""
    air, data = T.training_case(8, 1024, T.options(), 0xF401)
    proof = gpu_ctx.prove_host(air, data.ctypes.data)[0]
    cases = [(air, proof[:span.start]) for span in T.proof_sections(proof).values()] + [(air, proof + b"\0"), (air, b"")]
    pub = dict(air, pub_elems=list(air["pub_elems"]))
    pub["pub_elems"][0] = (pub["pub_elems"][0] + 1) % Z.P
    cases.append((pub, proof))
    av = dict(air, assertions=[tuple(a) for a in air["assertions"]])
    c0, s0, v0 = av["assertions"][0]
    av["assertions"][0] = (c0, s0, (v0 + 1) % Z.P)
    cases.append((av, proof))
    for k, v in (("num_queries", 41), ("folding", 8), ("blowup", 8)):
        cases.append((dict(air, options=dict(air["options"], **{k: v})), proof))
    mair, bad_trace = T.prover_case(T.mimc_prover(2, 128, T.options(blowup=8)))
    bad_trace[1, 77, 0] ^= 1
    bad_proof, ts = gpu_ctx.prove_host(mair, bad_trace.ctypes.data)
    assert ts.comp_degree_ok == 0
    cases.append((mair, bad_proof))
    verdicts, _ = gpu_ctx.verify_batch([a for a, _ in cases], [q for _, q in cases])
    want = [oracle_verdict(oracle, a, q)[0] for a, q in cases]
    assert verdicts == want
    assert want[-1] != OK and OK not in want


# ---- batches -------------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_mixed_batch_is_independent(gpu_ctx, oracle):
    """>= 64 proofs of the three AIRs, several shapes and options, valid and invalid interleaved: each gets the verdict it gets
    alone, and a permuted batch gives the permuted verdicts."""
    rng = random.Random(0xBA7C)
    base = [T.training_case(8, 1024, T.options(), 0xF501), T.training_case(16, 256, T.options(blowup=4, folding=2), 0xF502),
            T.mimc_case(oracle, 4, 256, T.options(blowup=8, folding=4)), T.prover_case(T.aggregation_prover(3, T.options())),
            T.training_case(2, 8, T.options(folding=8), 0xF503)]
    airs, proofs = [], []
    for i in range(72):
        air, data = base[i % len(base)]
        proof = gpu_ctx.prove_host(air, data.ctypes.data)[0] if i < len(base) else proofs[i % len(base)]
        if i % 3 == 1:
            bad = bytearray(proof)
            bad[rng.randrange(len(bad))] ^= 0x40
            proof = bytes(bad)
        airs.append(air); proofs.append(proof)
    together, _ = gpu_ctx.verify_batch(airs, proofs)
    alone = [gpu_ctx.verify_batch([a], [p])[0][0] for a, p in zip(airs, proofs)]
    assert together == alone
    assert together == [oracle_verdict(oracle, a, p)[0] for a, p in zip(airs, proofs)]
    assert OK in together and any(v != OK for v in together)
    perm = list(range(len(airs)))
    rng.shuffle(perm)
    permuted, _ = gpu_ctx.verify_batch([airs[i] for i in perm], [proofs[i] for i in perm])
    assert permuted == [together[i] for i in perm]


@pytest.mark.gpu
def test_256_proofs_in_one_call(gpu_ctx):
    """BASELINE configs[3]-sized round: 256 device proofs in one call are all accepted."""
    ref = Z.ProofOptions.reference()
    airs, proofs = [], []
    for k in range(4):
        air, data = T.prover_case(T.training_prover(1, ref, seed=0x5EED0100 + k))
        proof = gpu_ctx.prove_host(air, data.ctypes.data)[0]
        airs += [air] * 64
        proofs += [proof] * 64
    verdicts, _ = gpu_ctx.verify_batch(airs, proofs)
    assert verdicts == [OK] * 256


# ---- arguments and context reuse -----------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_arguments(gpu_ctx):
    lib = gpu_ctx.lib
    assert lib.zkb_verify_batch(gpu_ctx.handle, None, None, None, C.c_uint32(0), None, None) == 0
    air, data = T.training_case(8, 64, T.options(), 0xF601)
    proof = gpu_ctx.prove_host(air, data.ctypes.data)[0]
    d = L.make_desc(air)
    airs = (C.POINTER(L.AirDesc) * 1)(C.pointer(d))
    proofs = (C.c_char_p * 1)(proof)
    lens = (C.c_uint64 * 1)(len(proof))
    out = (C.c_int32 * 1)(-7)
    for args in ((None, proofs, lens, out), (airs, None, lens, out), (airs, proofs, None, out), (airs, proofs, lens, None)):
        assert lib.zkb_verify_batch(gpu_ctx.handle, *args[:3], C.c_uint32(1), args[3], None) == -1   # ZKB_ERR_INVALID
    assert lib.zkb_verify_batch(gpu_ctx.handle, airs, (C.c_char_p * 1)(None), lens, C.c_uint32(1), out, None) == -1
    bad = L.make_desc(dict(air, options=dict(air["options"], folding=3)))
    assert lib.zkb_verify_batch(gpu_ctx.handle, (C.POINTER(L.AirDesc) * 1)(C.pointer(bad)), proofs, lens, C.c_uint32(1), out, None) == -1
    assert b"folding" in lib.zkb_last_error(gpu_ctx.handle)
    b0 = gpu_ctx.h2d_bytes()
    assert lib.zkb_verify_batch(gpu_ctx.handle, airs, proofs, lens, C.c_uint32(1), out, None) == 0 and out[0] == OK
    assert gpu_ctx.h2d_bytes() - b0 >= len(proof)   # the staging copy holds every byte of the proof's sections
    assert Z.verify_batch([], []) == []
    res = Z.verify_batch([proof, proof[:-1]], [air, air], ctx=gpu_ctx)
    assert res[0] is None and isinstance(res[1], Z.VerifierError) and res[1].verdict == MALFORMED


@pytest.mark.gpu
def test_verify_prove_verify_matches_fresh_context(oracle):
    """Verify, prove, verify on one context: proofs are byte-identical to a fresh context's, including an aggregation proof
    replayed from a CUDA graph after the verifier's buffers grew."""
    ctx = L.Context(0)
    agg_air, agg = T.prover_case(T.aggregation_prover(16, Z.ProofOptions.reference()))
    big_air, big = T.training_case(240, 1 << 12, T.options(), 0xF701)
    first = [ctx.prove_host(agg_air, agg.ctypes.data)[0] for _ in range(3)]   # eager, capture, replay
    assert ctx.verify_batch([agg_air] * 3, first)[0] == [OK] * 3
    proofs = [ctx.prove_host(big_air, big.ctypes.data)[0]]
    v, _ = ctx.verify_batch([big_air] * 200, proofs * 200)    # grows the verifier's buffers
    assert v == [OK] * 200
    again = [ctx.prove_host(agg_air, agg.ctypes.data)[0] for _ in range(3)]
    fresh = L.Context(0)
    ref = fresh.prove_host(agg_air, agg.ctypes.data)[0]
    assert all(p == ref for p in first + again)
    assert ctx.prove_host(big_air, big.ctypes.data)[0] == fresh.prove_host(big_air, big.ctypes.data)[0] == proofs[0]
    assert ctx.verify_batch([agg_air, big_air], [again[-1], proofs[0]])[0] == [OK, OK]
    ctx.close(); fresh.close()


# ---- CPU: the wrapper checks its arguments before it reaches the library ---------------------------------------------------------

def test_verify_batch_argument_checks():
    air = {"air_id": 1}
    with pytest.raises(ValueError):
        Z.verify_batch([b"x", b"y"], [air])
    with pytest.raises(TypeError):
        Z.verify_batch(b"x", [air])
    with pytest.raises(TypeError):
        Z.verify_batch([123], [air])
    with pytest.raises(TypeError):
        Z.verify_batch([b"x"], ["not an air"])
    assert Z.verify_batch([], []) == []
