"""ctypes binding of include/zkb200.h (libzkb200.so).  Fails loudly when the library or the GPU is missing."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ZKB_LIB", os.path.join(HERE, "libzkb200.so"))
_lib = None


class ZkbError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"zkb200 error {status}: {message}")
        self.status = status


class AirDesc(C.Structure):
    _fields_ = [
        ("air_id", C.c_uint32), ("trace_width", C.c_uint32), ("trace_len", C.c_uint64),
        ("num_queries", C.c_uint32), ("blowup", C.c_uint32), ("grinding_bits", C.c_uint32),
        ("field_extension", C.c_uint32), ("folding", C.c_uint32), ("rem_max_degree", C.c_uint32),
        ("batching_constraints", C.c_uint32), ("batching_deep", C.c_uint32),
        ("pub_elems", C.c_char_p), ("n_pub_elems", C.c_uint64),
        ("assert_cols", C.POINTER(C.c_uint32)), ("assert_steps", C.POINTER(C.c_uint64)),
        ("assert_values", C.c_char_p), ("n_assertions", C.c_uint64),
        ("params", C.c_char_p), ("n_params", C.c_uint64),
    ]


class Transcript(C.Structure):
    _fields_ = [
        ("trace_root", C.c_uint8 * 32), ("constraint_root", C.c_uint8 * 32), ("remainder_commitment", C.c_uint8 * 32),
        ("constraint_alpha", C.c_uint8 * 16), ("z", C.c_uint8 * 16), ("deep_alpha", C.c_uint8 * 16),
        ("n_fri_layers", C.c_uint32), ("n_positions", C.c_uint32),
        ("fri_roots", (C.c_uint8 * 32) * 16), ("fri_alphas", (C.c_uint8 * 16) * 16),
        ("pow_nonce", C.c_uint64), ("positions", C.c_uint32 * 256),
        ("comp_degree_ok", C.c_int32), ("_pad", C.c_int32),
    ]


class StageTimes(C.Structure):
    _fields_ = [(k, C.c_float) for k in ("h2d", "interpolate", "lde", "leaf_hash", "merkle", "constraints", "composition",
                                          "ood", "deep", "fri", "grind", "queries", "total")]

    def as_dict(self):
        return {k: float(getattr(self, k)) for k, _ in self._fields_}


def load():
    """Load libzkb200.so; there is deliberately no fallback of any kind."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(nvcc, sm_100a). zk_stark_project_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    lib.zkb_last_error.restype = C.c_char_p
    lib.zkb_last_error.argtypes = [C.c_void_p]
    lib.zkb_kernel_launches.restype = C.c_uint64
    lib.zkb_kernel_launches.argtypes = [C.c_void_p]
    lib.zkb_h2d_bytes.restype = C.c_uint64
    lib.zkb_h2d_bytes.argtypes = [C.c_void_p]
    lib.zkb_host_alloc.restype = C.c_void_p
    lib.zkb_host_alloc.argtypes = [C.c_size_t]
    lib.zkb_host_free.argtypes = [C.c_void_p]
    lib.zkb_free.argtypes = [C.c_void_p]
    lib.zkb_ctx_destroy.argtypes = [C.c_void_p]
    for name in EXPORTS:
        fn = getattr(lib, name)
        if name not in ("zkb_last_error", "zkb_kernel_launches", "zkb_h2d_bytes", "zkb_host_alloc", "zkb_host_free", "zkb_free", "zkb_ctx_destroy"):
            fn.restype = C.c_int32
    _lib = lib
    return lib


# every symbol include/zkb200.h declares
EXPORTS = [
    "zkb_ctx_create", "zkb_ctx_create_lane", "zkb_ctx_destroy", "zkb_last_error", "zkb_kernel_launches", "zkb_h2d_bytes", "zkb_last_stage_times", "zkb_host_alloc",
    "zkb_host_free", "zkb_prove", "zkb_prove_device", "zkb_free", "zkb_begin", "zkb_trace_commit", "zkb_trace_commit_device",
    "zkb_trace_read_frame", "zkb_trace_read_frames", "zkb_trace_polys_read", "zkb_constraints_eval", "zkb_constraints_commit", "zkb_ood_eval",
    "zkb_deep_compose", "zkb_fri_num_layers", "zkb_fri_commit_layer", "zkb_fri_fold", "zkb_fri_remainder", "zkb_grind",
    "zkb_query", "zkb_mg_unique_id", "zkb_mg_init", "zkb_mg_prove", "zkb_mg_prove_device", "zkb_prove_batch", "zkb_mimc_trace", "zkb_mimc_trace_device", "zkb_training_trace_device", "zkb_download", "zkb_blake3_host", "zkb_mimc_cipher_batch", "zkb_mimc_hash_matrix_batch", "zkb_upload_trace", "zkb_test_field", "zkb_test_hash_elements",
    "zkb_test_merkle_root", "zkb_test_lde", "zkb_verify_batch",
]


def mg_unique_id():
    """ncclGetUniqueId (call on rank 0 and broadcast the 128 bytes)."""
    buf = C.create_string_buffer(128)
    rc = load().zkb_mg_unique_id(buf)
    if rc != 0:
        raise ZkbError(rc, load().zkb_last_error(None).decode())
    return buf.raw


def fe_bytes(x):
    from .field import P
    return (int(x) % P).to_bytes(16, "little")


def fe_int(b):
    return int.from_bytes(bytes(b), "little")


def make_desc(air):
    """air: plain description dict from an Air's describe()."""
    d = AirDesc()
    o = air["options"]
    d.air_id, d.trace_width, d.trace_len = air["air_id"], air["trace_width"], air["trace_len"]
    d.num_queries, d.blowup, d.grinding_bits = o["num_queries"], o["blowup"], o["grinding"]
    d.field_extension, d.folding, d.rem_max_degree = o.get("field_extension", 1), o["folding"], o["rem_max_degree"]
    d.batching_constraints, d.batching_deep = o.get("batching_constraints", 1), o.get("batching_deep", 1)
    pub = b"".join(fe_bytes(x) for x in air["pub_elems"])
    d.pub_elems, d.n_pub_elems = pub, len(air["pub_elems"])
    na = len(air["assertions"])
    cols = (C.c_uint32 * max(na, 1))(*[a[0] for a in air["assertions"]])
    steps = (C.c_uint64 * max(na, 1))(*[a[1] for a in air["assertions"]])
    vals = b"".join(fe_bytes(a[2]) for a in air["assertions"])
    d.assert_cols, d.assert_steps, d.assert_values, d.n_assertions = cols, steps, vals, na
    par = b"".join(fe_bytes(x) for x in air.get("params", []))
    d.params, d.n_params = par, len(air.get("params", []))
    d._keep = [pub, cols, steps, vals, par]
    return d


class Context:
    """One zkb_ctx: a device + stream binding that owns all device memory of the proofs run through it."""

    def __init__(self, device=0, stream=None, own_stream=False):
        """stream: a cudaStream_t value (None = default stream); own_stream=True: a private stream (zkb_ctx_create_lane)."""
        self.lib = load()
        self.handle = C.c_void_p()
        if own_stream:
            rc = self.lib.zkb_ctx_create_lane(C.c_int32(device), C.byref(self.handle))
        else:
            rc = self.lib.zkb_ctx_create(C.c_int32(device), C.c_void_p(stream or 0), C.byref(self.handle))
        if rc != 0:
            raise ZkbError(rc, self.lib.zkb_last_error(None).decode())
        self.device = device

    def close(self):
        if self.handle:
            self.lib.zkb_ctx_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc):
        if rc != 0:
            raise ZkbError(rc, self.lib.zkb_last_error(self.handle).decode())

    def launches(self):
        return int(self.lib.zkb_kernel_launches(self.handle))

    def h2d_bytes(self):
        return int(self.lib.zkb_h2d_bytes(self.handle))

    def stage_times(self):
        t = StageTimes()
        self.check(self.lib.zkb_last_stage_times(self.handle, C.byref(t)))
        return t.as_dict()

    # ---- Prover::prove ----
    def _col_ptrs(self, trace_ptr, w, n):
        return (C.c_void_p * w)(*[trace_ptr + j * n * 16 for j in range(w)])

    @staticmethod
    def prepare(air):
        """Marshal an AIR description once (the Rust glue would hold this struct ready-made)."""
        return air if isinstance(air, AirDesc) else make_desc(air)

    def prove_host(self, air, trace_ptr, force_nonce=0):
        """trace_ptr: host address of a column-major [w][n] trace."""
        d = self.prepare(air)
        out, ln, ts = C.c_void_p(), C.c_uint64(), Transcript()
        cols = self._col_ptrs(trace_ptr, d.trace_width, d.trace_len)
        self.check(self.lib.zkb_prove(self.handle, C.byref(d), cols, C.c_uint64(force_nonce), C.byref(out), C.byref(ln), C.byref(ts)))
        proof = C.string_at(out, ln.value)
        self.lib.zkb_free(out)
        return proof, ts

    def prove_device(self, air, d_trace, force_nonce=0):
        d = self.prepare(air)
        out, ln, ts = C.c_void_p(), C.c_uint64(), Transcript()
        self.check(self.lib.zkb_prove_device(self.handle, C.byref(d), C.c_void_p(d_trace), C.c_uint64(force_nonce), C.byref(out),
                                             C.byref(ln), C.byref(ts)))
        proof = C.string_at(out, ln.value)
        self.lib.zkb_free(out)
        return proof, ts

    # ---- column-sharded single proof ----
    def mg_init(self, rank, world, unique_id):
        self.check(self.lib.zkb_mg_init(self.handle, C.c_int32(rank), C.c_int32(world), unique_id))

    def mg_prove_host(self, air, local_trace_ptr, world, force_nonce=0):
        """air: description of the WHOLE trace; local_trace_ptr: this rank's w/world columns, column-major."""
        d = self.prepare(air)
        out, ln, ts = C.c_void_p(), C.c_uint64(), Transcript()
        cols = self._col_ptrs(local_trace_ptr, d.trace_width // world, d.trace_len)
        self.check(self.lib.zkb_mg_prove(self.handle, C.byref(d), cols, C.c_uint64(force_nonce), C.byref(out), C.byref(ln), C.byref(ts)))
        proof = C.string_at(out, ln.value)
        self.lib.zkb_free(out)
        return proof, ts

    def mg_prove_device(self, air, d_local_trace, force_nonce=0):
        d = self.prepare(air)
        out, ln, ts = C.c_void_p(), C.c_uint64(), Transcript()
        self.check(self.lib.zkb_mg_prove_device(self.handle, C.byref(d), C.c_void_p(d_local_trace), C.c_uint64(force_nonce), C.byref(out),
                                                C.byref(ln), C.byref(ts)))
        proof = C.string_at(out, ln.value)
        self.lib.zkb_free(out)
        return proof, ts

    # ---- winterfell::verify for a batch ----
    def verify_batch(self, airs, proofs):
        """zkb_verify_batch: one zkb_verdict per proof (0 = accepted) and the transcripts the verifier re-derived.
        airs: AIR descriptions (dicts or AirDesc), proofs: bytes, one per AIR."""
        count = len(proofs)
        descs = [self.prepare(a) for a in airs]
        bufs = [bytes(p) for p in proofs]
        air_arr = (C.POINTER(AirDesc) * max(count, 1))(*[C.pointer(d) for d in descs])
        proof_arr = (C.c_char_p * max(count, 1))(*bufs)
        lens = (C.c_uint64 * max(count, 1))(*[len(b) for b in bufs])
        verdicts = (C.c_int32 * max(count, 1))()
        ts = (Transcript * max(count, 1))()
        self.check(self.lib.zkb_verify_batch(self.handle, air_arr, proof_arr, lens, C.c_uint32(count), verdicts, ts))
        return [int(verdicts[i]) for i in range(count)], [ts[i] for i in range(count)]

    def upload_trace(self, trace_ptr, w, n):
        cols = self._col_ptrs(trace_ptr, w, n)
        d = C.c_void_p()
        self.check(self.lib.zkb_upload_trace(self.handle, cols, C.c_uint32(w), C.c_uint64(n), C.byref(d)))
        return d.value

    def training_trace_device(self, raw_rows, n, key=None):
        """raw_rows: list of rows of `half` field elements (the distinct raw states); key: 32 bytes for the ChaCha20 mask stream
        (tests) or None = OS entropy, like the reference's thread_rng.  Returns (device ptr, first row, last row)."""
        if key is not None and len(key) != 32:
            raise ValueError("mask key must be 32 bytes")
        half = len(raw_rows[0])
        rb = b"".join(fe_bytes(x) for row in raw_rows for x in row)
        d = C.c_void_p()
        first, last = C.create_string_buffer(32 * half), C.create_string_buffer(32 * half)
        self.check(self.lib.zkb_training_trace_device(self.handle, rb, C.c_uint32(len(raw_rows)), C.c_uint32(half), C.c_uint64(n),
                                                      key, C.byref(d), first, last))
        dec = lambda buf: [fe_int(buf.raw[16 * i:16 * i + 16]) for i in range(2 * half)]
        return d.value, dec(first), dec(last)

    def download(self, d_ptr, nbytes):
        out = C.create_string_buffer(nbytes)
        self.check(self.lib.zkb_download(self.handle, C.c_void_p(d_ptr), C.c_uint64(nbytes), out))
        return out.raw

    def mimc_trace(self, seeds, n, rc, device=False):
        w = len(seeds)
        sb = b"".join(fe_bytes(s) for s in seeds)
        rb = b"".join(fe_bytes(x) for x in rc)
        if device:
            d = C.c_void_p()
            self.check(self.lib.zkb_mimc_trace_device(self.handle, sb, C.c_uint32(w), C.c_uint64(n), rb, C.c_uint32(len(rc)), C.byref(d)))
            return d.value
        out = C.create_string_buffer(16 * n * w)
        self.check(self.lib.zkb_mimc_trace(self.handle, sb, C.c_uint32(w), C.c_uint64(n), rb, C.c_uint32(len(rc)), out))
        return out.raw


def blake3_host(data):
    """BLAKE3-256 on the host through the library (no device needed)."""
    out = C.create_string_buffer(32)
    rc = load().zkb_blake3_host(bytes(data), C.c_uint64(len(data)), out)
    if rc != 0:
        raise ZkbError(rc, "zkb_blake3_host failed")
    return out.raw


def prove_batch(lanes, airs, trace_ptrs):
    """zkb_prove_batch: proof i (AIR description airs[i], column-major host trace at trace_ptrs[i]) runs on lanes[i % len(lanes)];
    the host threads live inside the library.  Returns the proofs in order."""
    count = len(airs)
    descs = [Context.prepare(a) for a in airs]
    lane_arr = (C.c_void_p * len(lanes))(*[l.handle for l in lanes])
    air_arr = (C.POINTER(AirDesc) * max(count, 1))(*[C.pointer(d) for d in descs])
    col_arrays = [lanes[0]._col_ptrs(p, d.trace_width, d.trace_len) for p, d in zip(trace_ptrs, descs)]
    cols_arr = (C.c_void_p * max(count, 1))(*[C.cast(c, C.c_void_p) for c in col_arrays])
    outs = (C.c_void_p * max(count, 1))()
    lens = (C.c_uint64 * max(count, 1))()
    lib = lanes[0].lib
    rc = lib.zkb_prove_batch(lane_arr, C.c_uint32(len(lanes)), air_arr, cols_arr, C.c_uint32(count), outs, lens)
    proofs = []
    for i in range(count):
        proofs.append(C.string_at(outs[i], lens[i]) if outs[i] else None)
        if outs[i]:
            lib.zkb_free(C.c_void_p(outs[i]))
    if rc != 0:
        msgs = [lib.zkb_last_error(l.handle).decode() for l in lanes]
        raise ZkbError(rc, "; ".join(m for m in msgs if m))
    return proofs


def mimc_cipher_batch(ctx, xs, rcs, zs):
    """GPU `mimc_cipher` over a batch (src/helper.rs:213-220)."""
    n = len(xs)
    out = C.create_string_buffer(16 * max(n, 1))
    pack = lambda v: b"".join(fe_bytes(x) for x in v)
    ctx.check(ctx.lib.zkb_mimc_cipher_batch(ctx.handle, pack(xs), pack(rcs), pack(zs), C.c_uint64(n), out))
    return [fe_int(out.raw[16 * i:16 * i + 16]) for i in range(n)]


def mimc_hash_matrix_batch(ctx, ws, bs, round_constants):
    """GPU `mimc_hash_matrix` over a batch of (w[ac][fe], b[ac]) pairs (src/helper.rs:222-233)."""
    n = len(ws)
    ac, fe_n = len(bs[0]), len(ws[0][0])
    wb = b"".join(fe_bytes(x) for w in ws for row in w for x in row)
    bb = b"".join(fe_bytes(x) for b in bs for x in b)
    rb = b"".join(fe_bytes(x) for x in round_constants)
    out = C.create_string_buffer(16 * n)
    ctx.check(ctx.lib.zkb_mimc_hash_matrix_batch(ctx.handle, wb, bb, C.c_uint32(ac), C.c_uint32(fe_n), rb, C.c_uint32(len(round_constants)),
                                                 C.c_uint64(n), out))
    return [fe_int(out.raw[16 * i:16 * i + 16]) for i in range(n)]


class PinnedBuffer:
    """Page-locked host memory for trace columns (zkb_host_alloc)."""

    def __init__(self, nbytes):
        self.lib = load()
        self.ptr = self.lib.zkb_host_alloc(C.c_size_t(nbytes))
        if not self.ptr:
            raise MemoryError("zkb_host_alloc failed")
        self.nbytes = nbytes

    def view(self):
        import numpy as np
        return np.ctypeslib.as_array((C.c_uint8 * self.nbytes).from_address(self.ptr))

    def free(self):
        if self.ptr:
            self.lib.zkb_host_free(C.c_void_p(self.ptr))
            self.ptr = None
