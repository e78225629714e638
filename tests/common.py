"""Shared seeded inputs and checks for the parity tests (SURVEY §8d: none of the reference's thread_rng sites are used)."""
import ctypes as C
import json
import os
import random
import subprocess
import sys

import numpy as np

import zk_stark_project_b200 as Z
from zk_stark_project_b200 import field as F
from zk_stark_project_b200 import lib as L
from zk_stark_project_b200.training import AC, FE

P = Z.P
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def splitmix(seed):
    state = seed & 0xFFFFFFFFFFFFFFFF

    def nxt():
        nonlocal state
        state = (state + 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
        z = state
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF
        return z ^ (z >> 31)
    return nxt


from zk_stark_project_b200.synthetic import random_felts, synthetic_training_air  # noqa: E402,F401


def options(blowup=16, queries=40, grinding=8, folding=16, rem=7):
    return Z.ProofOptions(queries, blowup, grinding, Z.FieldExtension.NONE, folding, rem)


def model(rng, sigma):
    w = [[F.f64_to_signed_felt(rng.gauss(0, sigma), 1e6) for _ in range(FE)] for _ in range(AC)]
    b = [F.f64_to_signed_felt(rng.gauss(0, sigma), 1e6) for _ in range(AC)]
    return ([[v for v, _ in r] for r in w], [[s for _, s in r] for r in w], [v for v, _ in b], [s for _, s in b])


def training_prover(bs, opts, seed=0x5EED0002):
    """tests/integration_tests.rs:14-58 shaped inputs, but seeded."""
    rng = random.Random(seed)
    w, ws, b, bs_ = model(rng, 1.0)
    x = [[Z.f64_to_felt((i + j) * 0.1) for j in range(FE)] for i in range(bs)]
    xs = [[0] * FE for _ in range(bs)]
    y = [[Z.f64_to_felt(1.0) if a == i % AC else 0 for a in range(AC)] for i in range(bs)]
    return Z.TrainingUpdateProver(opts, w, b, ws, bs_, x, xs, y, Z.f64_to_felt(0.01), Z.f64_to_felt(1e6), bs, seed=seed)


def aggregation_prover(num_updates, opts, seed=0x5EED0003):
    """src/main.rs:440-459 shaped inputs, but seeded."""
    rng = random.Random(seed)
    gw, _, gb, _ = model(rng, 10000.0)
    reps = [rng.randrange(2**64) for _ in range(num_updates)]
    lw = [[[Z.f64_to_felt(r / 1e6)] * FE for _ in range(AC)] for r in reps]
    lb = [[Z.f64_to_felt(r / 1e6)] * AC for r in reps]
    return Z.GlobalUpdateProver(opts, gw, gb, lw, lb, Z.f64_to_felt(float(num_updates)), seed=seed)


def mimc_prover(width, steps, opts):
    return Z.MimcProver(opts, [j + 1 for j in range(width)], steps)


# ---- cases: (AIR description, contiguous [w][n][2] uint64 trace) -------------------------------------------------------------

def training_case(w, n, opts, seed):
    """Training AIR over a random training-shaped trace (the training prover is data-oblivious, see synthetic.py)."""
    data = random_felts(w * n, seed).reshape(w, n, 2)
    return synthetic_training_air(n, opts, data), data


def mimc_case(oracle, w, n, opts):
    """MiMC chains seeded 1..w; traces longer than 1024 rows come from the oracle, which builds them much faster."""
    p = mimc_prover(w, n, opts)
    if n <= 1024:
        return prover_case(p)
    data = np.frombuffer(oracle.mimc_trace(p.seeds, n, p.rc), dtype=np.uint64).reshape(w, n, 2)
    return p.describe(Z.TraceTable(data)), data


def prover_case(prover):
    trace = prover.build_trace()
    return prover.describe(trace), np.ascontiguousarray(trace.data)


def prove_both(ctx, oracle, air, data):
    """Proves `data` on the GPU and with the oracle: the transcripts and then the proof bytes must be equal, and the oracle's
    verifier and the product's Python verifier must accept the proof.  Returns the proof."""
    data = np.ascontiguousarray(data)
    ref, ts_o, _ = oracle.prove(air, data.tobytes())
    proof, ts = ctx.prove_host(air, data.ctypes.data)
    diff = transcript_diff(ts_o, ts)
    assert diff is None, f"transcripts diverge at `{diff}`"
    assert proof == ref, "proof bytes differ although the transcript matches"
    oracle.verify(air, proof)
    assert Z.verify(proof, air)
    return proof


# ---- the layout of Proof::to_bytes() -----------------------------------------------------------------------------------------

def proof_sections(proof):
    """Proof::to_bytes() cut into its data sections, in order: {name: slice}, length prefixes and constant bytes excluded.
    The tests' only reader of the proof layout, kept apart from the verifiers it checks."""
    pos = 0
    out = {}

    def take(name, k):
        nonlocal pos
        out[name] = slice(pos, pos + k)
        pos += k

    def vint():  # winter-utils vint64
        nonlocal pos
        first = proof[pos]
        length = 9 if first == 0 else (first & -first).bit_length()
        if length == 9:
            v = int.from_bytes(proof[pos + 1:pos + 9], "little")
        else:
            v = int.from_bytes(proof[pos:pos + length], "little") >> length
        pos += length
        return v

    def uint(k):
        nonlocal pos
        v = int.from_bytes(proof[pos:pos + k], "little")
        pos += k
        return v

    take("context", 4 + 2 + 1 + 16 + 8 + 2 + 1)
    take("commitments", uint(2))
    for name in ("trace rows", "trace paths", "constraint rows", "constraint paths"):
        take(name, vint())
    tl = uint(2)
    pos += 1
    take("ood trace", tl - 1)
    pos += 2
    take("ood constraints", uint(2))
    for layer in range(uint(1)):
        take(f"fri values {layer}", uint(4))
        take(f"fri paths {layer}", uint(4))
    take("remainder", uint(2))
    pos += 1
    take("nonce", 8)
    assert pos == len(proof)
    return out


def commitments(proof):
    """Trace root, constraint root, one root per FRI layer, remainder commitment."""
    blob = proof[proof_sections(proof)["commitments"]]
    return [blob[i:i + 32] for i in range(0, len(blob), 32)]


def fri_layers(proof):
    """(queried values, BatchMerkleProof bytes) of every FRI layer."""
    s = proof_sections(proof)
    return [(proof[s[f"fri values {l}"]], proof[s[f"fri paths {l}"]]) for l in range(sum(k.startswith("fri values") for k in s))]


# ---- the staged C ABI --------------------------------------------------------------------------------------------------------

class Staged:
    """One proof driven call by call through the staged surface of a Context (zkb_begin ... zkb_fri_remainder, zkb_query).
    Each method marshals its call's arguments, raises ZkbError when the call fails and returns what the call writes."""

    def __init__(self, ctx, air):
        self.lib, self.h, self.check = ctx.lib, ctx.handle, ctx.check
        self.w, self.n = air["trace_width"], air["trace_len"]
        self.desc = L.make_desc(air)
        self.check(self.lib.zkb_begin(self.h, C.byref(self.desc)))

    def trace_commit(self, data):
        """`data`: contiguous [w][n][2] trace.  Returns the trace root."""
        cols = (C.c_void_p * self.w)(*[data.ctypes.data + j * self.n * 16 for j in range(self.w)])
        root = C.create_string_buffer(32)
        self.check(self.lib.zkb_trace_commit(self.h, cols, root))
        return root.raw

    def read_frame(self, step):
        cur, nxt = C.create_string_buffer(16 * self.w), C.create_string_buffer(16 * self.w)
        self.check(self.lib.zkb_trace_read_frame(self.h, C.c_uint64(step), cur, nxt))
        return cur.raw, nxt.raw

    def read_frames(self, steps):
        k = len(steps)
        cur, nxt = C.create_string_buffer(16 * self.w * k), C.create_string_buffer(16 * self.w * k)
        self.check(self.lib.zkb_trace_read_frames(self.h, (C.c_uint64 * k)(*steps), C.c_uint32(k), cur, nxt))
        return cur.raw, nxt.raw

    def trace_polys(self):
        out = C.create_string_buffer(16 * self.n * self.w)
        self.check(self.lib.zkb_trace_polys_read(self.h, out))
        return out.raw

    def constraints_eval(self, alpha, ce=0):
        """Returns the ce * n constraint evaluations when the constraint blowup `ce` is given, else None."""
        ev = C.create_string_buffer(16 * self.n * ce) if ce else None
        self.check(self.lib.zkb_constraints_eval(self.h, alpha, ev))
        return ev.raw if ce else None

    def constraints_commit(self):
        root = C.create_string_buffer(32)
        self.check(self.lib.zkb_constraints_commit(self.h, root))
        return root.raw

    def ood_eval(self, z):
        self.check(self.lib.zkb_ood_eval(self.h, z, None, None, None))

    def deep_compose(self, alpha):
        self.check(self.lib.zkb_deep_compose(self.h, alpha))

    def fri_num_layers(self):
        nl = C.c_uint32()
        self.check(self.lib.zkb_fri_num_layers(self.h, C.byref(nl)))
        return nl.value

    def fri_commit_layer(self):
        root = C.create_string_buffer(32)
        self.check(self.lib.zkb_fri_commit_layer(self.h, root))
        return root.raw

    def fri_fold(self, alpha):
        self.check(self.lib.zkb_fri_fold(self.h, alpha))

    def fri_remainder(self):
        """Returns the remainder commitment."""
        coeffs, count, root = C.create_string_buffer(16 * 256), C.c_uint64(), C.create_string_buffer(32)
        self.check(self.lib.zkb_fri_remainder(self.h, coeffs, C.byref(count), root))
        return root.raw

    def query(self, which, positions, row_elems):
        """Rows of `row_elems` elements and the BatchMerkleProof bytes of commitment `which` (0 trace, 1 constraints, 2 + l FRI
        layer l) at `positions`."""
        k = len(positions)
        rows, po, ln = C.create_string_buffer(16 * row_elems * k), C.c_void_p(), C.c_uint64()
        self.check(self.lib.zkb_query(self.h, C.c_uint32(which), (C.c_uint32 * k)(*positions), C.c_uint32(k), rows, C.byref(po), C.byref(ln)))
        paths = C.string_at(po, ln.value)
        self.lib.zkb_free(po)
        return rows.raw, paths


# ---- column-sharded proofs ---------------------------------------------------------------------------------------------------

def run_sharded(ranks, port, cases, one_gpu):
    """tests/mg_worker.py on `ranks` ranks under torchrun: each case's column-sharded proof must equal its single-GPU proof.
    one_gpu: all ranks on the first visible GPU, talking over NCCL's socket transport on the loopback interface."""
    env = dict(os.environ)
    if one_gpu:
        env.update(CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0], NCCL_SOCKET_IFNAME="lo",
                   GLOO_SOCKET_IFNAME="lo", NCCL_IB_DISABLE="1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(ranks), "--master-addr", "127.0.0.1",
                        "--master-port", str(port), "tests/mg_worker.py", json.dumps(cases)], cwd=ROOT, env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0 and "mg ok" in r.stdout, f"{ranks} ranks: " + r.stdout[-2000:] + r.stderr[-2000:]


TS_FIELDS = ["trace_root", "constraint_alpha", "constraint_root", "z", "deep_alpha", "n_fri_layers", "fri_roots", "fri_alphas",
             "remainder_commitment", "pow_nonce", "n_positions", "positions"]


def transcript_diff(a, b):
    """First field where two transcripts (oracle / product ctypes structs with identical layout) differ."""
    for f in TS_FIELDS:
        x, y = getattr(a, f), getattr(b, f)
        xb = bytes(x) if hasattr(x, "__len__") else x
        yb = bytes(y) if hasattr(y, "__len__") else y
        if xb != yb:
            return f
    return None


def chacha20_block(key, counter):
    """ChaCha20 block function (20 rounds, 64-bit block counter in words 12-13, zero nonce): the device-side mask generator of
    zkb_training_trace_device restated for the tests.  Returns 64 keystream bytes."""
    import struct
    m = 0xFFFFFFFF
    rotl = lambda v, c: ((v << c) & m) | (v >> (32 - c))
    x = [0x61707865, 0x3320646E, 0x79622D32, 0x6B206574] + list(struct.unpack("<8I", key)) + [counter & m, (counter >> 32) & m, 0, 0]
    s = list(x)

    def qr(a, b, c, d):
        x[a] = (x[a] + x[b]) & m; x[d] = rotl(x[d] ^ x[a], 16)
        x[c] = (x[c] + x[d]) & m; x[b] = rotl(x[b] ^ x[c], 12)
        x[a] = (x[a] + x[b]) & m; x[d] = rotl(x[d] ^ x[a], 8)
        x[c] = (x[c] + x[d]) & m; x[b] = rotl(x[b] ^ x[c], 7)
    for _ in range(10):
        qr(0, 4, 8, 12); qr(1, 5, 9, 13); qr(2, 6, 10, 14); qr(3, 7, 11, 15)
        qr(0, 5, 10, 15); qr(1, 6, 11, 12); qr(2, 7, 8, 13); qr(3, 4, 9, 14)
    return struct.pack("<16I", *[(a + b) & m for a, b in zip(x, s)])


def training_mask(key, row, col, half):
    """Mask of trace cell (row, col) as zkb_training_trace_device generates it (include/zkb200.h)."""
    blocks = (half + 7) // 8
    ks = chacha20_block(key, row * blocks + col // 8)
    return int.from_bytes(ks[8 * (col % 8):8 * (col % 8) + 8], "little")
