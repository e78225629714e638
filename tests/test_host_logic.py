"""CPU: the Python mirror of the reference's host-side code, following the reference's own unit tests
(src/helper.rs:414-689, tests/simple_check.rs) and its trace-shape rules."""
import math

import numpy as np
import pytest

import zk_stark_project_b200 as Z
from zk_stark_project_b200 import field as F
from zk_stark_project_b200.training import AC, FE
from tests import common as T

P = Z.P


def test_constants():
    """tests/simple_check.rs:33-41."""
    assert (AC, FE) == (6, 9)
    assert Z.f64_to_felt(1.5) == 1500000 and Z.f64_to_felt(0.0) == 0
    assert Z.get_round_constants()[0] == 10**6 and len(Z.get_round_constants()) == 64


def test_signed_ops_with_sign_zero_are_plain_field_ops():
    """src/helper.rs:425-467."""
    a, b = 123456789, 987654
    assert F.add(a, b, 0, 0) == ((a + b) % P, 0)
    assert F.multiply(a, b, 0, 0) == (a * b % P, 0)
    assert F.divide(a, b, 0, 0) == (a * pow(b, P - 2, P) % P, 0)
    # sub_generic(a, 0, b, 0) = add_generic(a, 0, b, 1): with exactly one negative operand the "wrapped" branch is not
    # taken (src/signed.rs:17-31), so the value is a + b and the sign bit s_a*s_b = 0
    assert F.subtract(a, b, 0, 0) == ((a + b) % P, 0)


def test_encode_signed_round_trip():
    v, s = F.encode_signed(5)
    assert (v, s) == (5, 0)
    v, s = F.encode_signed(-5)
    assert s == 1 and v == F.Felt((2**128 - 5) & (2**128 - 1))
    assert F.cleanse(v, s) == (F.MAX - v + 1) % P == 5  # cleanse recovers |x| for negative encodings


def test_f64_round_half_away_from_zero():
    assert F._rust_round(0.5) == 1 and F._rust_round(2.5) == 3 and F._rust_round(-0.5) == -1


def test_transpose_and_trace_table():
    """src/helper.rs:482-496 and TraceTable::init limits."""
    rows = [[r * 10 + c for c in range(3)] for r in range(8)]
    t = Z.TraceTable.from_rows(rows)
    assert (t.width(), t.length()) == (3, 8) and t.get(2, 5) == 52 and t.column(1) == [r * 10 + 1 for r in range(8)]
    with pytest.raises(ValueError):
        Z.TraceTable.from_rows([[1, 2]] * 6)  # length not a power of two
    with pytest.raises(ValueError):
        Z.TraceTable(np.zeros((256, 8, 2), dtype=np.uint64))  # too wide


def test_proof_options_validation():
    o = Z.ProofOptions.reference()
    assert (o.num_queries, o.blowup_factor, o.grinding_factor, o.fri_folding_factor, o.fri_remainder_max_degree) == (40, 16, 21, 16, 7)
    for bad in (dict(num_queries=0), dict(blowup_factor=3), dict(grinding_factor=33), dict(fri_folding_factor=5), dict(fri_remainder_max_degree=6)):
        kw = dict(num_queries=40, blowup_factor=16, grinding_factor=21, field_extension=1, fri_folding_factor=16, fri_remainder_max_degree=7)
        kw.update(bad)
        with pytest.raises(ValueError):
            Z.ProofOptions(**kw)


def test_training_trace_shape_and_public_inputs():
    """src/training/prover.rs:63-65,128-130,245-246; src/training/air.rs:75-89."""
    for bs, n in ((1, 128), (2, 256), (5, 1024)):
        p = T.training_prover(bs, T.options())
        assert p.trace_length == n
        tr = p.build_trace()
        assert (tr.width(), tr.length()) == (240, n)
        # masked = raw + mask: column j minus column j+120 is the raw state, constant once the batch is consumed
        raw_last = [(tr.get(j, n - 1) - tr.get(j + 120, n - 1)) % P for j in range(120)]
        raw_prev = [(tr.get(j, n - 2) - tr.get(j + 120, n - 2)) % P for j in range(120)]
        assert raw_last == raw_prev
        assert all(tr.get(j + 120, 5) < 2**64 for j in range(120))
        pub = p.get_pub_inputs(tr)
        assert len(pub.to_elements()) == 244 + 15 * bs  # SURVEY Appendix C
        assert pub.to_elements()[240] == Z.f64_to_felt(float(n - 1))
        air = p.describe(tr)
        assert len(air["assertions"]) == 240 and air["assertions"][120] == (0, n - 1, tr.get(0, n - 1))


def test_training_step_port_is_structurally_sound():
    """src/helper.rs:580-689 compares one SGD step with an f64 implementation.  That comparison cannot hold in general: the
    reference "divides" with field inverses (src/signed.rs:42-48), which only equals fixed-point division when the quotient
    is exact — so this test pins the port's structure (shapes, sign bits, field range) instead."""
    from zk_stark_project_b200.training import backward_propagation_layer, forward_propagation_layer, mse_prime
    pr, lr = Z.f64_to_felt(1e6), Z.f64_to_felt(0.01)  # pr = 1e12 as a felt, lr = 1e4
    wf = [[0.1 * (i + 1) - 0.05 * j for j in range(FE)] for i in range(AC)]
    bf = [0.01 * i for i in range(AC)]
    xf = [0.1 * j for j in range(FE)]
    yf = [1.0 if i == 2 else 0.0 for i in range(AC)]
    enc = lambda v: F.f64_to_signed_felt(v, 1e6)
    w, ws = [[enc(v)[0] for v in r] for r in wf], [[enc(v)[1] for v in r] for r in wf]
    b, bs = [enc(v)[0] for v in bf], [enc(v)[1] for v in bf]
    x, xs = [enc(v)[0] for v in xf], [enc(v)[1] for v in xf]
    y = [Z.f64_to_felt(v) for v in yf]
    out, out_s = forward_propagation_layer(w, b, x, ws, bs, xs, pr)
    dec = lambda v, s: (-(F.cleanse(v, s)) if s else v) / 1e6
    out_f = [sum(wf[i][j] * xf[j] for j in range(FE)) + bf[i] for i in range(AC)]
    # the reference divides by pr = f64_to_felt(1e6) = 1e12 in the field (exact division is not integer division), so only the
    # structure is checked here: signs are bits and outputs are field elements
    assert all(s in (0, 1) for s in out_s) and all(0 <= v < P for v in out)
    err, err_s = mse_prime(y, out, out_s, pr)
    w2, b2, ws2, bs2 = backward_propagation_layer([r[:] for r in w], b[:], x, err, lr, pr, [r[:] for r in ws], bs[:], xs, err_s)
    assert len(w2) == AC and len(w2[0]) == FE and all(s in (0, 1) for r in ws2 for s in r)
    assert isinstance(out_f[0], float) and not math.isnan(dec(out[0], out_s[0]))


def test_aggregation_trace_rules():
    """src/aggregation/prover.rs:63-64,98-154; src/aggregation/air.rs:110-115,135-145."""
    p = T.aggregation_prover(16, T.options())
    rows = p.compute_iterative_trace_augmented()
    assert len(rows) == 32 and len(rows[0]) == 120
    k = p.k
    for i in range(31):  # k*(next - cur) - next.update == 0 on every transition
        for c in range(60):
            assert (k * (rows[i + 1][c] - rows[i][c]) - rows[i + 1][c + 60]) % P == 0
    assert rows[17][60:] == [0] * 60 and rows[18] == rows[17] and rows[31] == rows[17]
    pub = p.get_pub_inputs()
    assert len(pub.to_elements()) == 123 and pub.steps == 18 and pub.to_elements()[-1] == 18
    air = p.describe(p.build_trace())
    assert len(air["assertions"]) == 120 and all(a[1] == 17 for a in air["assertions"])


def test_mimc_trace_matches_oracle(oracle):
    p = T.mimc_prover(3, 128, T.options(blowup=8))
    assert p.build_trace().to_bytes() == oracle.mimc_trace(p.seeds, 128, p.rc)
    assert Z.mimc_cipher(5, 10**6, 3) == oracle.mimc_cipher(5, 10**6, 3)


def test_invalid_inputs_panic():
    """tests/integration_tests.rs:201-230."""
    with pytest.raises(AssertionError):
        Z.TrainingUpdateProver(T.options(), [[0] * 9] * 6, [0] * 6, [[0] * 9] * 6, [0] * 6, [[0] * 9], [[0] * 9], [[0] * 6], 1, 1, 2)
    with pytest.raises(ValueError):
        Z.MimcProver(T.options(), [1], 100)


def test_device_field_constants_in_source():
    """Constants and the inversion addition chain hard-wired in csrc/f128.cuh, re-derived here (the GPU KAT checks the code;
    this guards the numbers against an edit on a machine without a GPU)."""
    import os
    import re
    src = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "zk_stark_project_b200", "csrc", "f128.cuh")).read()
    c = (1 << 128) % P
    assert c == 45 * 2**40 - 1
    assert f"#define ZKB_C0 0x{c & 0xFFFFFFFF:08X}u" in src and f"#define ZKB_C1 0x{c >> 32:08X}u" in src
    k = (1 << 256) % P  # weight of the accumulator's ninth limb
    assert k == c * c and k < 2**92
    m = re.search(r"k0 = (0x[0-9A-Fa-f]+)u, k1 = (0x[0-9A-Fa-f]+)u, k2 = (0x[0-9A-Fa-f]+)u", src)
    assert m and [int(x, 16) for x in m.groups()] == [(k >> (32 * i)) & 0xFFFFFFFF for i in range(3)]
    # fe_inv: e_k = a^(2^k - 1); the chain in the source is (shift, multiply-by) pairs after e64
    steps = re.findall(r"r = fe_mul\(fe_sqr_n\((\w+), (\d+)\), (\w+)\);|return fe_mul\(fe_sqr_n\(r, (\d+)\), (\w+)\);", src)
    e = {"a": 1, "e2": 3, "e4": 15, "e8": 255, "e16": 2**16 - 1, "e32": 2**32 - 1, "e64": 2**64 - 1}
    exp = None
    for base, sh, mul, sh_last, mul_last in steps:
        if sh_last:
            exp = (exp << int(sh_last)) + e[mul_last]
        else:
            exp = ((e[base] if base != "r" else exp) << int(sh)) + e[mul]
    assert exp == P - 2


def test_chacha20_block_known_answer():
    """The tests' restatement of the device-side mask generator against the published ChaCha20 keystream for the all-zero key
    and nonce (block 0), so that the GPU comparison in test_device_side_training_trace pins the device code to real ChaCha20."""
    from tests import common as T
    ks = T.chacha20_block(bytes(32), 0)
    assert ks.hex() == ("76b8e0ada0f13d90405d6ae55386bd28bdd219b8a08ded1aa836efcc8b770dc7"
                        "da41597c5157488d7724e03fb8d84a376a43b8f41518a11cc387b669b2ee6586")
    assert T.chacha20_block(bytes(32), 1).hex().startswith("9f07e7be5551387a98ba977c732d080d")


def test_bench_counter_trace_is_seekable_and_canonical():
    """bench.py's counter-based synthetic trace: a rank that builds only its columns gets exactly the slice of the full trace
    (the sharded arm relies on it), every cell is a canonical field element, and the AIR description built from the two boundary
    rows equals the one built from the whole trace."""
    import numpy as np
    import bench
    import zk_stark_project_b200 as Z
    from zk_stark_project_b200 import synthetic as S
    w, n = 12, 64
    full = bench.counter_felts(w, n, 0x5EED2000)
    assert full.shape == (w, n, 2) and np.all(full[:, :, 1] < np.uint64(1 << 63))
    for r, world in ((0, 4), (3, 4), (1, 2)):
        wl = w // world
        assert np.array_equal(bench.counter_felts(w, n, 0x5EED2000, r * wl, wl), full[r * wl:(r + 1) * wl])
    assert not np.array_equal(bench.counter_felts(w, n, 1), full)
    opts = Z.ProofOptions(40, 16, 21, Z.FieldExtension.NONE, 16, 7)
    get = lambda c, r: int(full[c, r, 0]) | (int(full[c, r, 1]) << 64)
    a = bench.training_air_from_rows(n, w, opts, [get(j, 0) for j in range(w)], [get(j, n - 1) for j in range(w)])
    b = S.synthetic_training_air(n, opts, full)
    assert a == b


def test_bench_dump_outputs(oracle, tmp_path):
    """bench.py --dump-outputs (CPU arm, so no GPU is needed): float arrays that decode back to the proof of the last timed
    step, which the verifier accepts, and the transcript that came with it; --steps is the number of timed steps."""
    import json
    import subprocess
    import sys
    import bench
    cmd = [sys.executable, bench.__file__, "--impl", "reference", "--workload", "aggregation_16", "--warmup", "0", "--dump-outputs", str(tmp_path)]
    r = subprocess.run(cmd + ["--steps", "2"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout)["steps"] == 2
    arrays = {p.stem: np.load(p) for p in tmp_path.glob("*.npy")}
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values()) and sum(a.nbytes for a in arrays.values()) <= 64 << 20
    proof = arrays["proof"][0].astype(np.uint8).tobytes()
    air, _, _ = bench.build_workload("aggregation_16", 0x5EED0000)
    ts = oracle.verify(air, proof)
    assert arrays["transcript_z"][0].astype(np.uint8).tobytes() == bytes(ts.z)
    assert subprocess.run(cmd + ["--steps", "0"], capture_output=True).returncode == 2


def test_bench_algorithmic_bytes_match_survey():
    """SURVEY §8(d) totals: 9.47 GiB at configs[1], 33.5 GiB / 151.6 GiB at the two 2^20-row headline shapes."""
    import bench
    gib = 1 << 30
    assert abs(bench.algorithmic_bytes(1 << 16, 240, 16, 2, 1)["total"] / gib - 9.47) < 0.02
    assert abs(bench.algorithmic_bytes(1 << 20, 64, 8, 8, 6)["total"] / gib - 33.5) < 0.1
    assert abs(bench.algorithmic_bytes(1 << 20, 240, 16, 2, 1)["total"] / gib - 151.6) < 0.2


def test_library_rebuilds_when_any_source_changes(tmp_path, monkeypatch):
    """build.needs_build() watches every file in csrc/, not a list of names: a newer coin.cuh (the device Fiat-Shamir channel,
    included by kernels.cuh) makes the library stale."""
    import os
    import shutil
    from zk_stark_project_b200 import build
    csrc = tmp_path / "zk_stark_project_b200" / "csrc"
    shutil.copytree(build.CSRC, csrc)
    (tmp_path / "include").mkdir()
    shutil.copy(os.path.join(build.CSRC, "..", "..", "include", "zkb200.h"), tmp_path / "include")
    lib = tmp_path / "zk_stark_project_b200" / "libzkb200.so"
    lib.write_bytes(b"")
    monkeypatch.setattr(build, "CSRC", str(csrc))
    monkeypatch.setattr(build, "LIB", str(lib))
    t = os.path.getmtime(lib)
    for f in list(csrc.iterdir()) + [tmp_path / "include" / "zkb200.h"]:
        os.utime(f, (t - 60, t - 60))
    assert not build.needs_build()
    os.utime(csrc / "coin.cuh", (t + 60, t + 60))
    assert build.needs_build()
