"""`winterfell::verify` for the three AIRs (src/main.rs:251-257, 430-436, 478-484), CPU, pure Python.

Verification is the caller's side of the reference and stays on the CPU there too.  This module is written independently
of the C++ prover driver (csrc/zkb200.cu) and of the test oracle: it parses `Proof::to_bytes()`, replays the Fiat-Shamir
transcript and checks the OOD consistency, the Merkle openings, the DEEP composition and FRI.  The conventions are the
recalled Winterfell 0.12 ones of SURVEY.md Appendix A (unverified against upstream, see DESIGN.md §6)."""
from . import lib as _lib
from .field import P, inv

OFFSET = 3  # StarkField::GENERATOR = domain offset


class VerifierError(Exception):
    """`winterfell::VerifierError` counterpart."""


def _h(data):
    return _lib.blake3_host(data)


def _hash_elements(elems):
    return _h(b"".join(int(e).to_bytes(16, "little") for e in elems))


def root_of_unity(log_n):
    return pow(23953097886125630542083529559205016746, 1 << (40 - log_n), P)


class _Reader:
    def __init__(self, data):
        self.d, self.p = bytes(data), 0

    def take(self, n):
        if self.p + n > len(self.d):
            raise VerifierError("proof deserialization failed: unexpected end of data")
        b = self.d[self.p:self.p + n]
        self.p += n
        return b

    def u8(self):
        return self.take(1)[0]

    def uint(self, n):
        return int.from_bytes(self.take(n), "little")

    def usize(self):  # winter-utils vint64
        first = self.u8()
        if first == 0:
            return self.uint(8)
        length = (first & -first).bit_length()
        v = first | (self.uint(length - 1) << 8 if length > 1 else 0)
        return v >> length

    def felt(self):
        v = self.uint(16)
        if v >= P:
            raise VerifierError("proof deserialization failed: non-canonical field element")
        return v

    def done(self):
        return self.p == len(self.d)


class _Coin:
    """DefaultRandomCoin<Blake3_256>."""

    def __init__(self, elems):
        self.seed, self.counter = _hash_elements(elems), 0

    def reseed(self, digest):
        self.seed, self.counter = _h(self.seed + digest), 0

    def _next(self):
        self.counter += 1
        return _h(self.seed + self.counter.to_bytes(8, "little"))

    def draw(self):
        for _ in range(1000):
            v = int.from_bytes(self._next()[:16], "little")
            if v < P:
                return v
        raise VerifierError("random coin failed to draw")

    def leading_zeros(self, nonce):
        head = int.from_bytes(_h(self.seed + nonce.to_bytes(8, "little"))[:8], "little")
        return 64 if head == 0 else (head & -head).bit_length() - 1

    def draw_integers(self, num, domain, nonce):
        self.seed, self.counter = _h(self.seed + nonce.to_bytes(8, "little")), 0
        return [int.from_bytes(self._next()[:8], "little") & (domain - 1) for _ in range(num)]


def _parse_batch_proof(data):
    r = _Reader(data)
    depth = r.u8()
    nodes = []
    for _ in range(r.usize()):
        nodes.append([r.take(32) for _ in range(r.usize())])
    if not r.done():
        raise VerifierError("trailing bytes in Merkle proof")
    return depth, nodes


def _batch_root(depth, nodes, indexes, leaves):
    """BatchMerkleProof::get_root."""
    n = 1 << depth
    index_map = {}
    for i, idx in enumerate(indexes):
        if idx >= n or idx in index_map:
            raise VerifierError("invalid Merkle proof indexes")
        index_map[idx] = i
    norm = sorted({i & ~1 for i in indexes})
    if len(norm) != len(nodes):
        raise VerifierError("invalid Merkle proof")
    v, nxt, ptr = {}, [], []
    for i, idx in enumerate(norm):
        a, b = index_map.get(idx), index_map.get(idx + 1)
        if a is not None:
            left = leaves[a]
            if b is not None:
                right = leaves[b]
                ptr.append(0)
            else:
                if not nodes[i]:
                    raise VerifierError("invalid Merkle proof")
                right = nodes[i][0]
                ptr.append(1)
        else:
            if not nodes[i] or b is None:
                raise VerifierError("invalid Merkle proof")
            left, right = nodes[i][0], leaves[b]
            ptr.append(1)
        parent = (n + idx) >> 1
        v[parent] = _h(left + right)
        nxt.append(parent)
    for _ in range(1, depth):
        cur, nxt, k = nxt, [], 0
        while k < len(cur):
            node, sib = cur[k], cur[k] ^ 1
            if k + 1 < len(cur) and cur[k + 1] == sib:
                sd = v[sib]
                k += 1
            else:
                # upstream indexes proof vectors with the per-level position k (SURVEY A.6)
                if ptr[k] >= len(nodes[k]):
                    raise VerifierError("invalid Merkle proof")
                sd = nodes[k][ptr[k]]
                ptr[k] += 1
            if node not in v:
                raise VerifierError("invalid Merkle proof")
            v[node >> 1] = _h(sd + v[node]) if node & 1 else _h(v[node] + sd)
            nxt.append(node >> 1)
            k += 1
    if 1 not in v:
        raise VerifierError("invalid Merkle proof")
    return v[1]


def _fold_positions(positions, domain, folding):
    target, out = domain // folding, []
    for p in positions:
        q = p % target
        if q not in out:
            out.append(q)
    return out


def _fold_row(row, x, alpha):
    """p(alpha) for the degree < F polynomial through (x * w_F^j, row[j]), F = len(row) (the folding factor)."""
    f = len(row)
    w_inv = inv(root_of_unity(f.bit_length() - 1))
    finv, t = inv(f), alpha * inv(x) % P
    acc, tk = 0, 1
    for k in range(f):
        ck = sum(row[j] * pow(w_inv, j * k, P) for j in range(f)) % P * finv % P
        acc = (acc + ck * tk) % P
        tk = tk * t % P
    return acc


def _evaluate_transition(air, cur, nxt, periodic):
    aid = air["air_id"]
    if aid == 1:  # training: current_step() == 0, every constraint evaluates to zero (src/training/air.rs:274-278)
        return [0] * air["trace_width"]
    if aid == 2:  # src/aggregation/air.rs:110-115
        d, k = air["trace_width"] // 2, air["params"][0]
        return [(k * nxt[i] - k * cur[i] - nxt[i + d]) % P for i in range(d)]
    return [(nxt[i] - pow((cur[i] + periodic) % P, 7, P)) % P for i in range(air["trace_width"])]


def verify(proof, air):
    """Raises VerifierError unless `proof` (bytes or Proof) is a valid proof for the AIR description `air`
    (an `Air.describe()` dict: it carries the public inputs, the assertions and the acceptable options)."""
    data = proof.to_bytes() if hasattr(proof, "to_bytes") else bytes(proof)
    o = air["options"]
    n, w, beta = air["trace_len"], air["trace_width"], o["blowup"]
    N = n * beta
    deg = 7 if air["air_id"] == 3 else 1
    c = max(1, (deg * (n - 1) - (n - 1) + n - 1) // n)
    folding = o["folding"]
    g = root_of_unity(n.bit_length() - 1)

    # ---- Proof::from_bytes ----
    r = _Reader(data)
    if (r.u8(), r.u8(), r.u8()) != (w, 0, 0) or (1 << r.u8()) != n or r.uint(2) != 0:
        raise VerifierError("trace info in the proof does not match the AIR")
    if r.u8() != 16 or r.uint(16) != P:
        raise VerifierError("inconsistent base field")
    got = [r.u8() for _ in range(8)]
    want = [o["num_queries"], beta, o["grinding"], o.get("field_extension", 1), folding, o["rem_max_degree"],
            o.get("batching_constraints", 1), o.get("batching_deep", 1)]
    if got != want or (r.u8(), r.u8()) != (1, 1):
        raise VerifierError("unacceptable proof options")  # AcceptableOptions::OptionSet
    n_unique = r.u8()
    clen = r.uint(2)
    commitments = [r.take(32) for _ in range(clen // 32)]
    trace_rows_b, trace_paths = r.take(r.usize()), r.take(r.usize())
    comp_rows_b, comp_paths = r.take(r.usize()), r.take(r.usize())
    tl = r.uint(2)
    if r.u8() != 2 or (tl - 1) != 2 * w * 16:
        raise VerifierError("malformed OOD trace frame")
    ood_states = [r.felt() for _ in range(2 * w)]
    if r.uint(2) != 0:
        raise VerifierError("unexpected Lagrange kernel frame")
    if r.uint(2) != c * 16:
        raise VerifierError("malformed OOD constraint evaluations")
    ood_h = [r.felt() for _ in range(c)]
    fri_layers = []
    for _ in range(r.u8()):
        vals = r.take(r.uint(4))
        paths = r.take(r.uint(4))
        fri_layers.append((vals, paths))
    remainder = [r.felt() for _ in range(r.uint(2) // 16)]
    if r.u8() != 1:
        raise VerifierError("unexpected FRI partition count")
    nonce = r.uint(8)
    if not r.done():
        raise VerifierError("trailing bytes in proof")

    # number of FRI layers for this domain
    nl, dom = 0, N
    while dom > (o["rem_max_degree"] + 1) * beta:
        dom //= folding
        nl += 1
    if len(commitments) != nl + 3 or len(fri_layers) != nl:
        raise VerifierError("wrong number of commitments / FRI layers")

    # ---- transcript ----
    asserts = sorted(air["assertions"], key=lambda a: (a[1], a[0]))
    nt = w // 2 if air["air_id"] == 2 else w
    ctx_elems = [w << 8, n, P & (2**64 - 1), P >> 64, len(asserts) + nt,
                 (o.get("field_extension", 1) << 24) | (folding << 16) | (o["rem_max_degree"] << 8) | beta, o["grinding"], o["num_queries"]]
    coin = _Coin(ctx_elems + [int(x) % P for x in air["pub_elems"]])
    coin.reseed(commitments[0])
    alpha = coin.draw()
    coin.reseed(commitments[1])
    z = coin.draw()

    # ---- OOD consistency ----
    cur, nxt = ood_states[0::2], ood_states[1::2]
    periodic = 0
    if air["air_id"] == 3:
        rc = air["params"]
        L = len(rc)
        wl = root_of_unity(L.bit_length() - 1)
        coeffs = [sum(rc[i] * pow(wl, -i * k % L, P) for i in range(L)) * inv(L) % P for k in range(L)]
        x = pow(z, n // L, P)
        periodic = sum(ck * pow(x, k, P) for k, ck in enumerate(coeffs)) % P
    tev = _evaluate_transition(air, cur, nxt, periodic)
    coef, t = 1, 0
    for e in tev:
        t = (t + coef * e) % P
        coef = coef * alpha % P
    lhs = t * ((z - pow(g, n - 1, P)) % P) % P * inv((pow(z, n, P) - 1) % P) % P
    groups = {}
    for col, step, value in asserts:
        groups.setdefault(step, 0)
        groups[step] = (groups[step] + coef * (cur[col] - value)) % P
        coef = coef * alpha % P
    for step, s in groups.items():
        lhs = (lhs + s * inv((z - pow(g, step, P)) % P)) % P
    coin.reseed(_hash_elements(ood_states))
    rhs = sum(pow(z, i * n, P) * h for i, h in enumerate(ood_h)) % P
    coin.reseed(_hash_elements(ood_h))
    if lhs != rhs:
        raise VerifierError("inconsistent OOD constraint evaluations")

    # ---- DEEP coefficients, FRI commitments, proof of work, query positions ----
    dalpha = coin.draw()
    alphas = []
    for cm in commitments[2:]:
        coin.reseed(cm)
        alphas.append(coin.draw())
    if coin.leading_zeros(nonce) < o["grinding"]:
        raise VerifierError("query seed proof-of-work verification failed")
    positions = sorted(set(coin.draw_integers(o["num_queries"], N, nonce)))
    if n_unique != len(positions):
        raise VerifierError("number of unique queries does not match the proof")
    nq = len(positions)
    if len(trace_rows_b) != nq * w * 16 or len(comp_rows_b) != nq * c * 16:
        raise VerifierError("malformed query values")
    trow = [[int.from_bytes(trace_rows_b[(q * w + j) * 16:(q * w + j + 1) * 16], "little") for j in range(w)] for q in range(nq)]
    crow = [[int.from_bytes(comp_rows_b[(q * c + j) * 16:(q * c + j + 1) * 16], "little") for j in range(c)] for q in range(nq)]
    d, nodes = _parse_batch_proof(trace_paths)
    if _batch_root(d, nodes, positions, [_h(trace_rows_b[q * w * 16:(q + 1) * w * 16]) for q in range(nq)]) != commitments[0]:
        raise VerifierError("trace query did not match the commitment")
    d, nodes = _parse_batch_proof(comp_paths)
    if _batch_root(d, nodes, positions, [_h(comp_rows_b[q * c * 16:(q + 1) * c * 16]) for q in range(nq)]) != commitments[1]:
        raise VerifierError("constraint query did not match the commitment")

    # ---- DEEP composition at the queried positions ----
    gN, zg = root_of_unity(N.bit_length() - 1), z * g % P
    gam = [pow(dalpha, i, P) for i in range(w + c)]
    evals = []
    for q, pos in enumerate(positions):
        x = OFFSET * pow(gN, pos, P) % P
        t1 = sum((trow[q][j] - cur[j]) * gam[j] for j in range(w)) % P
        t2 = sum((trow[q][j] - nxt[j]) * gam[j] for j in range(w)) % P
        hh = sum((crow[q][i] - ood_h[i]) * gam[w + i] for i in range(c)) % P
        d1, d2 = inv((x - z) % P), inv((x - zg) % P)
        evals.append(((t1 + hh) * d1 + t2 * d2) % P)

    # ---- FRI ----
    pos, dom, gen, max_deg_plus_1 = positions, N, gN, n
    for l in range(nl):
        folded = _fold_positions(pos, dom, folding)
        rows = dom // folding
        vals_b, paths_b = fri_layers[l]
        if len(vals_b) != len(folded) * folding * 16:
            raise VerifierError("malformed FRI layer")
        vals = [[int.from_bytes(vals_b[(i * folding + j) * 16:(i * folding + j + 1) * 16], "little") for j in range(folding)] for i in range(len(folded))]
        d, nodes = _parse_batch_proof(paths_b)
        if _batch_root(d, nodes, folded, [_h(vals_b[i * folding * 16:(i + 1) * folding * 16]) for i in range(len(folded))]) != commitments[2 + l]:
            raise VerifierError("FRI layer query did not match the commitment")
        for i, p in enumerate(pos):
            if vals[folded.index(p % rows)][p // rows] != evals[i]:
                raise VerifierError("invalid FRI layer folding")
        evals = [_fold_row(vals[i], pow(gen, fp, P) * OFFSET % P, alphas[l]) for i, fp in enumerate(folded)]
        if max_deg_plus_1 % folding:
            raise VerifierError("FRI degree truncation")
        gen, max_deg_plus_1, dom, pos = pow(gen, folding, P), max_deg_plus_1 // folding, rows, folded
    if len(remainder) > max_deg_plus_1 or _hash_elements(remainder) != commitments[2 + nl]:
        raise VerifierError("FRI remainder mismatch")
    for p, e in zip(pos, evals):
        x, acc = OFFSET * pow(gen, p, P) % P, 0
        for cf in remainder:  # eval_horner_rev: coefficients are stored highest degree first
            acc = (acc * x + cf) % P
        if acc != e:
            raise VerifierError("invalid FRI remainder folding")
    return True
