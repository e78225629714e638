// Batch verification on the device: winter-verifier 0.12 `verify` (the check run after every proof at /root/reference
// src/main.rs:251-257, 430-436, 478-484) for many proofs at once.  The host parses every proof, packs the parsed sections into
// one staging buffer (16-byte aligned, offsets in bytes from its base) and plans all index work; these kernels only hash,
// merge, evaluate and compare, at offsets and digest ids the host computed from checked lengths.
//
// A failed check is an ordinal (VO_*, in the order the sequential verifier runs its checks: stage, then FRI layer, then check
// within the layer) and a proof's verdict is the atomicMin of the ordinals of its failed checks, so it is the first failure a
// sequential verifier reports.
#pragma once
#include "kernels.cuh"

namespace zkb {

enum : uint32_t {
    VO_MALFORMED = 0, VO_TRACE_INFO, VO_OPTIONS, VO_COMMITMENTS, VO_OOD_SHAPE, VO_OOD, VO_POW, VO_UNIQUE,
    VO_TRACE_VALUES, VO_CONSTRAINT_VALUES, VO_TRACE_ROWS_PARSE, VO_CONSTRAINT_ROWS_PARSE,
    VO_TRACE_PATHS_PARSE, VO_TRACE_MERKLE, VO_CONSTRAINT_PATHS_PARSE, VO_CONSTRAINT_MERKLE,
    VO_FRI0 = 16,   // + VO_FRI_STEP * layer + VO_FRI_*
    VO_FRI_STEP = 6,
    VO_FRI_VALUES = 0, VO_FRI_ROWS_PARSE = 1, VO_FRI_PATHS_PARSE = 2, VO_FRI_MERKLE = 3, VO_FRI_FOLDING = 4, VO_FRI_TRUNCATION = 5,
    VO_REM = VO_FRI0 + VO_FRI_STEP * ZKB_MAX_FRI_LAYERS,   // + 0 degree, + 1 commitment, + 2 folding
    VO_ACCEPT = VO_REM + 3
};

// Per proof: where its sections sit in the staging buffer and what the channel and the OOD check need from the AIR
struct VProof {
    uint32_t seed[8];                  // coin seed: hash of Context ++ public inputs
    uint64_t o_comm, o_ood, o_h, o_rem;        // commitments (2 + layers + 1 digests), OOD frame (2w, interleaved), h_i(z) (c), remainder
    uint64_t o_aval, o_params, o_gpts, o_acol, o_goff;   // sorted assertion values, AIR params, g^step per group, columns, group offsets
    uint64_t nonce;
    uint32_t w, c, nt, na, ng, np, n_layers, rem_len, q, log_n, log_N, grinding, air_id, active, ood;
};

struct VLeafJob { uint64_t off; uint32_t count, out, proof, ord; };   // hash `count` elements at `off` into digest `out`
struct VMergeJob { uint32_t a, b, out; };                              // digest out = merge(a, b)
struct VRootJob { uint64_t commit_off; uint32_t id, proof, ord, pad; };   // digest id must equal the commitment at commit_off
// One evaluation to check: DEEP at a queried position (layer = ~0u) or the fold of one FRI row (layer l).  The result must equal
// the element at target_off, or (target_off = ~0) the remainder at 3 w_{2^rem_log}^rem_pos.
struct VEvalJob {
    uint64_t row_off, crow_off, target_off;   // DEEP: trace row, constraint row; FRI: the F row elements
    uint32_t proof, layer, pos, log_dom, rem_pos, rem_log, ord, folding;
};

struct VArgs {
    const uint8_t* base;               // staging buffer on the device
    const VProof* proofs;
    DevTs* ts;                         // per proof: the channel's draws (alpha, z, deep_alpha, fri_alpha) and raw positions
    uint32_t* verdict;                 // per proof: smallest failed ordinal
    const fe* roots;                   // roots[k] = primitive 2^k-th root of unity, k <= 40
    const uint32_t* nodes;             // digests supplied by the proofs (Merkle nodes), ids [0, n_nodes)
    uint32_t* dig;                     // digests computed here, ids [n_nodes, ...)
    uint32_t n_nodes;
    fe fold_wf_inv[4][8];              // [log F - 1][k] = w_F^{-k}, k < F/2
    fe fold_inv_f[4];                  // [log F - 1] = 1/F
};

__device__ __forceinline__ const fe* v_fe(const VArgs& a, uint64_t off) { return reinterpret_cast<const fe*>(a.base + off); }
__device__ __forceinline__ const uint32_t* v_digest(const VArgs& a, uint32_t id) {
    return id < a.n_nodes ? a.nodes + (size_t)id * 8 : a.dig + (size_t)(id - a.n_nodes) * 8;
}
__device__ __forceinline__ void v_fail(const VArgs& a, uint32_t proof, uint32_t ord) { atomicMin(a.verdict + proof, ord); }
__device__ __forceinline__ bool fe_noncanonical(const fe& v) {
    return v.x[3] == 0xFFFFFFFFu && v.x[2] == 0xFFFFFFFFu && (v.x[1] > 0xFFFFD300u || (v.x[1] == 0xFFFFD300u && v.x[0] >= 1u));
}
__device__ __forceinline__ fe fe_mul3(const fe& x) { const fe x2 = fe_add(x, x); return fe_add(x2, x); }

// Channel, one block per proof: the draws of the verifier's coin, the proof-of-work check and draw_integers.  Every step is
// the prover's (coin.cuh), fed from the proof instead of from the commitments the prover computed.
__global__ void __launch_bounds__(ZKB_FS_THREADS) k_v_channel(const VArgs a) {
    const VProof& p = a.proofs[blockIdx.x];
    if (!p.active) return;
    DevTs* ts = a.ts + blockIdx.x;
    __shared__ uint32_t cvs[16][8];
    __shared__ uint32_t s_seed[8];
    const uint32_t* comm = reinterpret_cast<const uint32_t*>(a.base + p.o_comm);
    uint32_t seed[8];
    if (threadIdx.x == 0) {
#pragma unroll
        for (int i = 0; i < 8; i++) seed[i] = p.seed[i];
        fs_reseed(seed, comm);
        ts->alpha = fs_draw(seed, &ts->coin_failed);
        fs_reseed(seed, comm + 8);
        ts->z = fs_draw(seed, &ts->coin_failed);
    }
    uint32_t h1[8], h2[8];
    fs_hash_elems_block(v_fe(a, p.o_ood), 2 * p.w, cvs, h1);
    fs_hash_elems_block(v_fe(a, p.o_h), p.c, cvs, h2);
    if (threadIdx.x == 0) {
        fs_reseed(seed, h1);
        fs_reseed(seed, h2);
        ts->deep_alpha = fs_draw(seed, &ts->coin_failed);
        for (uint32_t l = 0; l <= p.n_layers; l++) {   // the draw after the remainder commitment is not used
            fs_reseed(seed, comm + 8 * (2 + l));
            const fe al = fs_draw(seed, &ts->coin_failed);
            if (l < p.n_layers) ts->fri_alpha[l] = al;
        }
        // check_leading_zeros(nonce) and draw_integers' reseed with the nonce hash the same 40 bytes
        uint32_t d[8];
        b3_with_int(seed, p.nonce, d);
        const uint64_t head = ((uint64_t)d[1] << 32) | d[0];
        if (head & (((uint64_t)1 << p.grinding) - 1ull)) v_fail(a, blockIdx.x, VO_POW);
#pragma unroll
        for (int i = 0; i < 8; i++) s_seed[i] = d[i];
        ts->nonce = p.nonce;
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 8; i++) seed[i] = s_seed[i];
    const uint32_t mask = (uint32_t)(((uint64_t)1 << p.log_N) - 1u);
    for (uint32_t q = threadIdx.x; q < p.q; q += blockDim.x) {
        uint32_t d[8];
        b3_with_int(seed, (uint64_t)q + 1, d);
        ts->positions[q] = d[0] & mask;
    }
}

// warp sum of a field element; valid on lane 0
__device__ __forceinline__ fe fe_warp_sum(fe s) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        fe o;
        o.x[0] = __shfl_down_sync(0xffffffffu, s.x[0], off); o.x[1] = __shfl_down_sync(0xffffffffu, s.x[1], off);
        o.x[2] = __shfl_down_sync(0xffffffffu, s.x[2], off); o.x[3] = __shfl_down_sync(0xffffffffu, s.x[3], off);
        s = fe_add(s, o);
    }
    return s;
}
__device__ __forceinline__ fe fe_shfl(const fe& v, int src) {
    fe r;
#pragma unroll
    for (int i = 0; i < 4; i++) r.x[i] = __shfl_sync(0xffffffffu, v.x[i], src);
    return r;
}

// MiMC's periodic column at z: the polynomial through (w_L^i, rc_i) at y = z^(n/L), by the barycentric formula
//   P(y) = (y^L - 1)/L * sum_i rc_i w^i / (y - w^i),
// each lane summing its terms as one fraction (one inversion per warp); y = w^i exactly gives rc_i.  Called by a whole warp.
__device__ __forceinline__ fe v_periodic(const fe* rc, uint32_t L, uint32_t log_L, const fe& y, const fe* roots) {
    const uint32_t lane = threadIdx.x & 31u;
    const fe wl = roots[log_L];
    fe yl = y;
    for (uint32_t k = 0; k < log_L; k++) yl = fe_sqr(yl);
    const fe yl1 = fe_sub(yl, fe_one());
    const fe step = fe_pow_u64(wl, 32);
    if (fe_is_zero(yl1)) {   // y is an L-th root of unity
        fe val = fe_zero();
        bool hit = false;
        fe x = fe_pow_u64(wl, lane);
        for (uint32_t i = lane; i < L; i += 32) {
            if (fe_eq(x, y)) { val = fe_load(rc + i); hit = true; }
            x = fe_mul(x, step);
        }
        const uint32_t who = __ballot_sync(0xffffffffu, hit);
        return fe_shfl(val, who ? __ffs(who) - 1 : 0);
    }
    fe num = fe_zero(), den = fe_one();
    fe x = fe_pow_u64(wl, lane);
    for (uint32_t i = lane; i < L; i += 32) {   // num/den += rc_i x / (y - x)
        const fe d = fe_sub(y, x);
        num = fe_add(fe_mul(num, d), fe_mul(fe_mul(fe_load(rc + i), x), den));
        den = fe_mul(den, d);
        x = fe_mul(x, step);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {   // a/b + c/d = (a d + c b) / (b d)
        const fe on = fe_shfl(num, (lane + off) & 31), od = fe_shfl(den, (lane + off) & 31);
        num = fe_add(fe_mul(num, od), fe_mul(on, den));
        den = fe_mul(den, od);
    }
    const fe s = fe_mul(num, fe_inv_inline(den));
    return fe_shfl(fe_mul(fe_mul(s, yl1), fe_inv_inline(fe_from_u64(L))), 0);
}

// OOD consistency, one warp per proof (evaluate_constraints at z against sum_i z^(i n) h_i(z)).  The transition evaluations
// are restated per point here: k_eval_constraints evaluates them inline over LDE panels with a fused accumulator, and a shared
// per-constraint function would change its code.  inv(0) = 0, as in winter-math.
__global__ void __launch_bounds__(128) k_v_ood(const VArgs a, uint32_t count) {
    const uint32_t pi = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31u;
    if (pi >= count) return;   // warp-uniform
    const VProof& p = a.proofs[pi];
    if (!p.ood) return;
    const DevTs* ts = a.ts + pi;
    const fe alpha = ts->alpha, z = ts->z;
    const fe* frame = v_fe(a, p.o_ood);   // [T_0(z), T_0(zg), T_1(z), ...]
    const uint64_t n = (uint64_t)1 << p.log_n;
    fe per = fe_zero();
    if (p.air_id == ZKB_AIR_MIMC) {
        const uint32_t log_L = 31u - __clz(p.np);
        per = v_periodic(v_fe(a, p.o_params), p.np, log_L, fe_pow_u64(z, n >> log_L), a.roots);
    }
    // transition: sum_k alpha^k ev_k
    fe t = fe_zero();
    if (p.air_id != ZKB_AIR_TRAINING) {   // training: every transition evaluation is zero
        const fe step = fs_pow(alpha, 32);
        fe ak = fs_pow(alpha, lane);
        for (uint32_t k = lane; k < p.nt; k += 32) {
            fe ev;
            if (p.air_id == ZKB_AIR_AGGREGATION) {
                const fe kf = fe_load(v_fe(a, p.o_params));
                ev = fe_sub(fe_sub(fe_mul(kf, frame[2 * k + 1]), fe_mul(kf, frame[2 * k])), frame[2 * (k + p.nt) + 1]);
            } else {
                const fe a1 = fe_add(frame[2 * k], per);
                const fe a2 = fe_sqr(a1), a4 = fe_sqr(a2), a6 = fe_mul(a4, a2), a7 = fe_mul(a6, a1);
                ev = fe_sub(frame[2 * k + 1], a7);
            }
            t = fe_add(t, fe_mul(ak, ev));
            ak = fe_mul(ak, step);
        }
    }
    // boundary groups: sum_{a in g} alpha^(nt + a) (T_col(z) - value) / (z - g^step)
    fe b = fe_zero();
    const uint32_t* goff = reinterpret_cast<const uint32_t*>(a.base + p.o_goff);
    const uint32_t* acol = reinterpret_cast<const uint32_t*>(a.base + p.o_acol);
    const fe* aval = v_fe(a, p.o_aval);
    const fe* gpts = v_fe(a, p.o_gpts);
    for (uint32_t g = lane; g < p.ng; g += 32) {
        fe s = fe_zero();
        fe cf = fs_pow(alpha, p.nt + goff[g]);
        for (uint32_t i = goff[g]; i < goff[g + 1]; i++) {
            s = fe_add(s, fe_mul(cf, fe_sub(frame[2 * acol[i]], aval[i])));
            cf = fe_mul(cf, alpha);
        }
        b = fe_add(b, fe_mul(s, fe_inv_inline(fe_sub(z, gpts[g]))));
    }
    t = fe_warp_sum(t);
    b = fe_warp_sum(b);
    if (lane != 0) return;
    const fe g = a.roots[p.log_n];
    const fe zn = fe_pow_u64(z, n);
    const fe eval1 = fe_add(fe_mul(fe_mul(t, fe_sub(z, fe_pow_u64(g, n - 1))), fe_inv_inline(fe_sub(zn, fe_one()))), b);
    fe eval2 = fe_zero(), zi = fe_one();
    const fe* h = v_fe(a, p.o_h);
    for (uint32_t i = 0; i < p.c; i++) { eval2 = fe_add(eval2, fe_mul(zi, h[i])); zi = fe_mul(zi, zn); }
    if (!fe_eq(eval1, eval2)) v_fail(a, pi, VO_OOD);
}

// Leaves: one thread per queried row (trace, constraint, FRI layer) and per remainder.  A non-canonical element is the
// row's parse failure (the sequential verifier reads the rows before it hashes them).
__global__ void __launch_bounds__(128) k_v_leaves(const VArgs a, const VLeafJob* __restrict__ jobs, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const VLeafJob j = jobs[i];
    const fe* e = v_fe(a, j.off);
    bool bad = false;
    for (uint32_t k = 0; k < j.count; k++) bad |= fe_noncanonical(fe_load(e + k));
    if (bad) v_fail(a, j.proof, j.ord);
    uint32_t d[8];
    b3_hash_elems(e, 1, j.count, d, 256, 256, 0);
    uint4* out = reinterpret_cast<uint4*>(a.dig + (size_t)(j.out - a.n_nodes) * 8);
    out[0] = make_uint4(d[0], d[1], d[2], d[3]);
    out[1] = make_uint4(d[4], d[5], d[6], d[7]);
}

// One level of BatchMerkleProof::get_root over every tree of the batch
__global__ void __launch_bounds__(128) k_v_merge(const VArgs a, const VMergeJob* __restrict__ jobs, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const VMergeJob j = jobs[i];
    uint32_t d[8];
    b3_merge(v_digest(a, j.a), v_digest(a, j.b), d);
    uint4* out = reinterpret_cast<uint4*>(a.dig + (size_t)(j.out - a.n_nodes) * 8);
    out[0] = make_uint4(d[0], d[1], d[2], d[3]);
    out[1] = make_uint4(d[4], d[5], d[6], d[7]);
}

__global__ void __launch_bounds__(128) k_v_roots(const VArgs a, const VRootJob* __restrict__ jobs, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const VRootJob j = jobs[i];
    const uint32_t* d = v_digest(a, j.id);
    const uint32_t* c = reinterpret_cast<const uint32_t*>(a.base + j.commit_off);
    bool same = true;
#pragma unroll
    for (int k = 0; k < 8; k++) same &= d[k] == c[k];
    if (!same) v_fail(a, j.proof, j.ord);
}

// The prover's row fold (fri_fold_row) of the F = 2^LF elements at `row`, at x = 3 w^pos: alpha / x needs the one inversion
template <int LF>
__device__ __forceinline__ fe v_fold(const VArgs& a, const fe* row, const fe& alpha, const fe& x) {
    fe v;
    fri_fold_row<LF>([&](int k) { return fe_load(row + k); }, [&](int k) { return a.fold_wf_inv[LF - 1][k]; },
                     [&] { return fe_mul(alpha, fe_inv_inline(x)); }, a.fold_inv_f[LF - 1], [&](const fe& r) { v = r; });
    return v;
}

// DEEP composition at a queried position and the fold of one FRI row, each compared with the element the next layer holds for
// it, or with the remainder (reversed coefficients, Horner) after the last layer
__global__ void __launch_bounds__(128) k_v_eval(const VArgs a, const VEvalJob* __restrict__ jobs, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const VEvalJob j = jobs[i];
    const VProof& p = a.proofs[j.proof];
    const DevTs* ts = a.ts + j.proof;
    const fe x = fe_mul3(fe_pow_u64(a.roots[j.log_dom], j.pos));
    fe v;
    if (j.layer == ~0u) {   // DEEP: sum_j g^j ((T_j(x) - T_j(z)) / (x - z) + (T_j(x) - T_j(zg)) / (x - zg)) + sum_k g^(w+k) (H_k(x) - H_k(z)) / (x - z)
        const fe* tr = v_fe(a, j.row_off);
        const fe* cr = v_fe(a, j.crow_off);
        const fe* frame = v_fe(a, p.o_ood);
        const fe* h = v_fe(a, p.o_h);
        const fe da = ts->deep_alpha, z = ts->z, zg = fe_mul(z, a.roots[p.log_n]);
        fe t1 = fe_zero(), t2 = fe_zero(), hs = fe_zero(), gm = fe_one();
        for (uint32_t k = 0; k < p.w; k++) {
            const fe tv = fe_load(tr + k);
            t1 = fe_add(t1, fe_mul(fe_sub(tv, frame[2 * k]), gm));
            t2 = fe_add(t2, fe_mul(fe_sub(tv, frame[2 * k + 1]), gm));
            gm = fe_mul(gm, da);
        }
        for (uint32_t k = 0; k < p.c; k++) { hs = fe_add(hs, fe_mul(fe_sub(fe_load(cr + k), h[k]), gm)); gm = fe_mul(gm, da); }
        const fe d1 = fe_inv_inline(fe_sub(x, z)), d2 = fe_inv_inline(fe_sub(x, zg));
        v = fe_add(fe_add(fe_mul(t1, d1), fe_mul(t2, d2)), fe_mul(hs, d1));
    } else {
        const fe* row = v_fe(a, j.row_off);
        const fe al = ts->fri_alpha[j.layer];
        switch (j.folding) {
            case 2: v = v_fold<1>(a, row, al, x); break;
            case 4: v = v_fold<2>(a, row, al, x); break;
            case 8: v = v_fold<3>(a, row, al, x); break;
            default: v = v_fold<4>(a, row, al, x); break;
        }
    }
    fe want;
    if (j.target_off != ~0ull) want = fe_load(v_fe(a, j.target_off));
    else {
        const fe xr = fe_mul3(fe_pow_u64(a.roots[j.rem_log], j.rem_pos));
        const fe* rem = v_fe(a, p.o_rem);
        want = fe_zero();
        for (uint32_t k = 0; k < p.rem_len; k++) want = fe_add(fe_mul(want, xr), fe_load(rem + k));
    }
    if (!fe_eq(v, want)) v_fail(a, j.proof, j.ord);
}

}  // namespace zkb
