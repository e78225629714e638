// Device-resident Fiat-Shamir channel (SURVEY §8f rank 3): winter-crypto `DefaultRandomCoin<Blake3_256>` and the
// ProverChannel steps of winter-prover's `generate_proof` (reached from /root/reference src/main.rs:228,424,468 with the coin
// type fixed at src/training/prover.rs:227, src/aggregation/prover.rs:200), run by single-block kernels between the bulk
// stages so that a proof needs no host round trip until its last byte is on the device.
//
// Every kernel here is launched <<<1, ZKB_FS_THREADS>>>: the hashes are a few compressions each (the OOD frame, up to 8 KiB,
// is hashed chunk-parallel), and the challenge-dependent scalars the next bulk kernel needs (coefficient powers, powers of z,
// DEEP constants) are derived in the same launch.
#pragma once
#include "blake3.cuh"
#include "f128.cuh"

namespace zkb {

#define ZKB_FS_THREADS 256
// FRI layers a proof may have: folding by 2 down to a remainder of at least the blowup (>= 2) from the largest LDE domain
// (2^30) takes 29
#define ZKB_MAX_FRI_LAYERS 32

// Transcript of the proof in flight, in device memory; the host receives it with the final download.
struct DevTs {
    uint32_t seed[8];                 // coin state (the counter restarts at every reseed, so it is not kept)
    uint32_t trace_root[8], constraint_root[8], rem_commit[8];
    uint32_t fri_roots[ZKB_MAX_FRI_LAYERS][8];
    fe alpha, z, zg, zR, zgR, deep_alpha, az, abz, azg;   // zR = z^64, zgR = (z g)^64
    fe fri_alpha[ZKB_MAX_FRI_LAYERS];
    unsigned long long nonce;
    uint32_t bad_degree, coin_failed;
    uint32_t positions[256];          // raw query draws: unsorted, duplicates kept (the host sorts and dedups)
};

// ---- BLAKE3 pieces -------------------------------------------------------------------------------------------------------
// RandomCoin::draw: first 16 bytes of next() as a little-endian u128, rejected while >= p.  One thread.
__device__ __forceinline__ fe fs_draw(const uint32_t seed[8], uint32_t* failed) {
    for (uint64_t counter = 1; counter <= 1000; counter++) {
        uint32_t d[8];
        b3_with_int(seed, counter, d);
        // v < p  <=>  not (limbs 3,2 all ones and (limb1, limb0) >= (0xFFFFD300, 1))
        const bool ge = d[3] == 0xFFFFFFFFu && d[2] == 0xFFFFFFFFu && (d[1] > 0xFFFFD300u || (d[1] == 0xFFFFD300u && d[0] >= 1u));
        if (!ge) { fe r; r.x[0] = d[0]; r.x[1] = d[1]; r.x[2] = d[2]; r.x[3] = d[3]; return r; }
    }
    *failed = 1;
    return fe_zero();
}
__device__ __forceinline__ void fs_reseed(uint32_t seed[8], const uint32_t digest[8]) {
    uint32_t t[8];
    b3_merge(seed, digest, t);
#pragma unroll
    for (int i = 0; i < 8; i++) seed[i] = t[i];
}

// Blake3_256::hash_elements of `count` contiguous elements (count <= 1024 -> up to 16 chunks) by a thread block: thread c
// hashes chunk c (64 elements), thread 0 folds the chunk chaining values with BLAKE3's stack rule.  `cvs` is shared memory
// for 16 chaining values.  All threads of the block must call it; the digest is valid in thread 0 only.
__device__ __forceinline__ void fs_hash_elems_block(const fe* __restrict__ e, uint32_t count, uint32_t (*cvs)[8], uint32_t out[8]) {
    const uint32_t nchunks = count <= 64 ? 1u : (count + 63u) / 64u;
    if (threadIdx.x < nchunks) {
        const uint32_t c = threadIdx.x;
        uint32_t cv[8];
        b3_iv(cv);
        const uint32_t e0 = c * 64u;
        const uint32_t ne = (count - e0) < 64u ? (count - e0) : 64u;
        const uint32_t nblk = ne == 0 ? 1u : (ne + 3u) / 4u;
        for (uint32_t b = 0; b < nblk; b++) {
            uint32_t m[16];
            const uint32_t eb = e0 + 4u * b;
            const uint32_t nb = (e0 + ne - eb) < 4u ? (e0 + ne - eb) : 4u;
#pragma unroll
            for (uint32_t q = 0; q < 4; q++) {
                uint4 v = make_uint4(0, 0, 0, 0);
                if (q < nb) v = *reinterpret_cast<const uint4*>(e + eb + q);
                m[4 * q] = v.x; m[4 * q + 1] = v.y; m[4 * q + 2] = v.z; m[4 * q + 3] = v.w;
            }
            uint32_t flags = (b == 0 ? B3_CHUNK_START : 0u);
            if (b + 1 == nblk) flags |= B3_CHUNK_END | (nchunks == 1 ? B3_ROOT : 0u);
            b3_compress(cv, m, c, nb * 16u, flags);
        }
#pragma unroll
        for (int i = 0; i < 8; i++) cvs[c][i] = cv[i];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (nchunks == 1) {
#pragma unroll
            for (int i = 0; i < 8; i++) out[i] = cvs[0][i];
        } else {
            // chaining-value stack: after chunk i (all but the last) merge once per trailing zero bit of i + 1; the last chunk's
            // value is then merged down the stack, the final merge carrying ROOT
            uint32_t stack[5][8];
            int sp = 0;
            for (uint32_t i = 0; i + 1 < nchunks; i++) {
#pragma unroll
                for (int q = 0; q < 8; q++) stack[sp][q] = cvs[i][q];
                sp++;
                for (uint32_t t = i + 1; (t & 1u) == 0; t >>= 1) {
                    uint32_t p[8];
                    b3_parent(stack[sp - 2], stack[sp - 1], false, p);
                    sp--;
#pragma unroll
                    for (int q = 0; q < 8; q++) stack[sp - 1][q] = p[q];
                }
            }
            uint32_t cur[8];
#pragma unroll
            for (int q = 0; q < 8; q++) cur[q] = cvs[nchunks - 1][q];
            while (sp > 0) {
                uint32_t p[8];
                b3_parent(stack[sp - 1], cur, sp == 1, p);
                sp--;
#pragma unroll
                for (int q = 0; q < 8; q++) cur[q] = p[q];
            }
#pragma unroll
            for (int q = 0; q < 8; q++) out[q] = cur[q];
        }
    }
    __syncthreads();
}

// base^e by square-and-multiply (e < 2^16 here: coefficient indices)
__device__ __forceinline__ fe fs_pow(fe b, uint32_t e) {
    fe r = fe_one();
    while (e) { if (e & 1u) r = fe_mul(r, b); b = fe_sqr(b); e >>= 1; }
    return r;
}

// ---- channel steps ---------------------------------------------------------------------------------------------------------
// ProverChannel::new: the coin seed (hash of Context ++ public inputs) is computed by the host, which knows the AIR, and
// uploaded into ts->seed before the first stage; nothing to do on the device.

// channel.commit_trace(root) + get_constraint_composition_coeffs() (one draw alpha; transition coefficients alpha^0.., boundary
// coefficients continuing over the assertions sorted by (step, column)).  digest == nullptr: alpha was provided by the host
// (staged API) and is already in ts->alpha.  coef[0 .. nt + na) = alpha^i.
__global__ void __launch_bounds__(ZKB_FS_THREADS) k_fs_trace_root(DevTs* ts, const uint32_t* __restrict__ digest, uint32_t n_coef, fe* __restrict__ coef,
                                                                 uint32_t* __restrict__ degree_flag) {
    __shared__ uint4 s_alpha;
    if (threadIdx.x == 0) {
        *degree_flag = 0;   // raised by k_scale_pow if the composition polynomial does not fit (constraints_commit)
        if (digest) {
            uint32_t seed[8], d[8];
#pragma unroll
            for (int i = 0; i < 8; i++) { seed[i] = ts->seed[i]; d[i] = digest[i]; ts->trace_root[i] = d[i]; }
            fs_reseed(seed, d);
#pragma unroll
            for (int i = 0; i < 8; i++) ts->seed[i] = seed[i];
            ts->alpha = fs_draw(seed, &ts->coin_failed);
        }
        const fe a = ts->alpha;
        s_alpha = make_uint4(a.x[0], a.x[1], a.x[2], a.x[3]);
    }
    __syncthreads();
    fe a; a.x[0] = s_alpha.x; a.x[1] = s_alpha.y; a.x[2] = s_alpha.z; a.x[3] = s_alpha.w;
    for (uint32_t i = threadIdx.x; i < n_coef; i += blockDim.x) fe_store(coef + i, fs_pow(a, i));
}

// channel.commit_constraints(root) + get_ood_point(); also the powers of z the OOD kernels consume.  g = trace-domain generator.
__global__ void k_fs_constraint_root(DevTs* ts, const uint32_t* __restrict__ digest, const uint32_t* __restrict__ bad_degree, fe g) {
    if (threadIdx.x != 0) return;
    if (digest) {
        uint32_t seed[8], d[8];
#pragma unroll
        for (int i = 0; i < 8; i++) { seed[i] = ts->seed[i]; d[i] = digest[i]; ts->constraint_root[i] = d[i]; }
        fs_reseed(seed, d);
#pragma unroll
        for (int i = 0; i < 8; i++) ts->seed[i] = seed[i];
        ts->z = fs_draw(seed, &ts->coin_failed);
        ts->bad_degree = *bad_degree;
    }
    const fe z = ts->z, zg = fe_mul(z, g);
    ts->zg = zg;
    fe a = z, b = zg;
#pragma unroll 1
    for (int i = 0; i < 6; i++) { a = fe_sqr(a); b = fe_sqr(b); }   // ^64: the row-chunk length of k_ood_partial / k_poly_eval_partial
    ts->zR = a; ts->zgR = b;
}

// send_ood_trace_states (hash of the frame interleaved [T_0(z), T_0(zg), T_1(z), ...]) + send_ood_constraint_evaluations +
// get_deep_composition_coeffs (one draw; gamma^0.. over the trace columns, continuing over the composition columns), and the
// DEEP constants A(z), (A+B)(z), A(zg).   ood = [T_j(z) w][T_j(zg) w][H_i(z) c];  scratch: 2w elements;  gamma: w + c.
// with_coin = 0: the staged API supplied deep_alpha in ts->deep_alpha.
__global__ void __launch_bounds__(ZKB_FS_THREADS) k_fs_ood(DevTs* ts, const fe* __restrict__ ood, uint32_t w, uint32_t c, fe* __restrict__ scratch,
                                                          fe* __restrict__ gamma, uint32_t with_coin) {
    __shared__ uint32_t cvs[16][8];
    __shared__ uint4 s_da;
    __shared__ uint4 red[3][ZKB_FS_THREADS];
    if (with_coin) {
        for (uint32_t j = threadIdx.x; j < w; j += blockDim.x) { fe_store(scratch + 2 * j, fe_load(ood + j)); fe_store(scratch + 2 * j + 1, fe_load(ood + w + j)); }
        __syncthreads();
        uint32_t h1[8], h2[8];
        fs_hash_elems_block(scratch, 2 * w, cvs, h1);
        fs_hash_elems_block(ood + 2 * (size_t)w, c, cvs, h2);
        if (threadIdx.x == 0) {
            uint32_t seed[8];
#pragma unroll
            for (int i = 0; i < 8; i++) seed[i] = ts->seed[i];
            fs_reseed(seed, h1);
            fs_reseed(seed, h2);
#pragma unroll
            for (int i = 0; i < 8; i++) ts->seed[i] = seed[i];
            ts->deep_alpha = fs_draw(seed, &ts->coin_failed);
        }
    }
    if (threadIdx.x == 0) { const fe a = ts->deep_alpha; s_da = make_uint4(a.x[0], a.x[1], a.x[2], a.x[3]); }
    __syncthreads();
    fe da; da.x[0] = s_da.x; da.x[1] = s_da.y; da.x[2] = s_da.z; da.x[3] = s_da.w;
    fe az = fe_zero(), azg = fe_zero(), bz = fe_zero();
    for (uint32_t i = threadIdx.x; i < w + c; i += blockDim.x) {
        const fe gm = fs_pow(da, i);
        fe_store(gamma + i, gm);
        if (i < w) { az = fe_add(az, fe_mul(gm, fe_load(ood + i))); azg = fe_add(azg, fe_mul(gm, fe_load(ood + w + i))); }
        else bz = fe_add(bz, fe_mul(gm, fe_load(ood + 2 * (size_t)w + (i - w))));
    }
    red[0][threadIdx.x] = make_uint4(az.x[0], az.x[1], az.x[2], az.x[3]);
    red[1][threadIdx.x] = make_uint4(azg.x[0], azg.x[1], azg.x[2], azg.x[3]);
    red[2][threadIdx.x] = make_uint4(bz.x[0], bz.x[1], bz.x[2], bz.x[3]);
    __syncthreads();
    for (uint32_t h = blockDim.x / 2; h > 0; h >>= 1) {
        if (threadIdx.x < h) {
#pragma unroll
            for (int q = 0; q < 3; q++) {
                const uint4 x = red[q][threadIdx.x], y = red[q][threadIdx.x + h];
                fe a, b; a.x[0] = x.x; a.x[1] = x.y; a.x[2] = x.z; a.x[3] = x.w; b.x[0] = y.x; b.x[1] = y.y; b.x[2] = y.z; b.x[3] = y.w;
                const fe s = fe_add(a, b);
                red[q][threadIdx.x] = make_uint4(s.x[0], s.x[1], s.x[2], s.x[3]);
            }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        fe a, g_, b;
        { const uint4 x = red[0][0]; a.x[0] = x.x; a.x[1] = x.y; a.x[2] = x.z; a.x[3] = x.w; }
        { const uint4 x = red[1][0]; g_.x[0] = x.x; g_.x[1] = x.y; g_.x[2] = x.z; g_.x[3] = x.w; }
        { const uint4 x = red[2][0]; b.x[0] = x.x; b.x[1] = x.y; b.x[2] = x.z; b.x[3] = x.w; }
        ts->az = a; ts->azg = g_; ts->abz = fe_add(a, b);
    }
}

// channel.commit_fri_layer(root) + draw the layer's folding challenge
__global__ void k_fs_fri_root(DevTs* ts, const uint32_t* __restrict__ digest, uint32_t layer) {
    if (threadIdx.x != 0) return;
    uint32_t seed[8], d[8];
#pragma unroll
    for (int i = 0; i < 8; i++) { seed[i] = ts->seed[i]; d[i] = digest[i]; ts->fri_roots[layer][i] = d[i]; }
    fs_reseed(seed, d);
#pragma unroll
    for (int i = 0; i < 8; i++) ts->seed[i] = seed[i];
    ts->fri_alpha[layer] = fs_draw(seed, &ts->coin_failed);
}

// FriProver::set_remainder: coef = the last layer after the inverse transform; the first rs coefficients are scaled here
// (interpolation over the coset 3*<w_M>: coefficient m times scale * 3^-m, scale = 1/M), stored REVERSED (SURVEY A.10),
// committed with hash_elements, and the coin is reseeded.  with_coin = 0: hash only (staged API).
__global__ void __launch_bounds__(ZKB_FS_THREADS) k_fs_remainder(DevTs* ts, const fe* __restrict__ coef, uint32_t rs, fe* __restrict__ rem, uint32_t with_coin,
                                                                const fe* __restrict__ inv3_lo, const fe* __restrict__ inv3_hi, uint32_t inv3_l1, fe scale) {
    __shared__ uint32_t cvs[16][8];
    for (uint32_t i = threadIdx.x; i < rs; i += blockDim.x) {
        const uint32_t m = rs - 1 - i;
        const fe f = fe_mul(fe_mul(fe_ldg(inv3_lo + (m & ((1u << inv3_l1) - 1u))), fe_ldg(inv3_hi + (m >> inv3_l1))), scale);
        fe_store(rem + i, fe_mul(fe_load(coef + m), f));
    }
    __syncthreads();
    uint32_t h[8];
    fs_hash_elems_block(rem, rs, cvs, h);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int i = 0; i < 8; i++) ts->rem_commit[i] = h[i];
        if (with_coin) {
            uint32_t seed[8];
#pragma unroll
            for (int i = 0; i < 8; i++) seed[i] = ts->seed[i];
            fs_reseed(seed, h);
#pragma unroll
            for (int i = 0; i < 8; i++) ts->seed[i] = seed[i];
        }
        ts->nonce = ~0ull;   // armed for the proof-of-work search
    }
}

// ProverChannel::grind_query_seed: the smallest nonce >= 1 whose merge_with_int(seed, nonce) has >= bits trailing zero bits in
// its first little-endian u64.  One persistent launch: thread t tests nonces 1 + t, 1 + t + T, ...; a thread is done as soon as its
// next candidate exceeds the best nonce found so far (ts->nonce only ever decreases), so the minimum survives without a
// grid-wide barrier.  `limit`: give up beyond this nonce (ts->nonce stays ~0).
// The loop is warp-uniform on purpose: every lane stays in it until the whole warp is done and the vote reconverges the warp
// each iteration.  With a per-lane `break`, the lane that found a nonce sits on a divergent path that is not scheduled while
// its 31 warp-mates keep spinning, its atomicMin is published only when they leave too, and the search degenerates to
// ~2^bits iterations per warp (measured: 3.7 s instead of 0.15 ms at 21 bits).
__global__ void __launch_bounds__(256) k_fs_grind(DevTs* ts, uint32_t bits, unsigned long long limit) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const uint64_t mask = bits >= 64 ? ~0ull : (((uint64_t)1 << bits) - 1ull);
    uint32_t seed[8];
#pragma unroll
    for (int i = 0; i < 8; i++) seed[i] = ts->seed[i];
    volatile unsigned long long* best = &ts->nonce;
    bool done = false;
    for (uint64_t x = 1 + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;; x += stride) {
        if (!done && (x > limit || x > *best)) done = true;
        if (!done) {
            uint32_t d[8];
            b3_with_int(seed, x, d);
            const uint64_t head = ((uint64_t)d[1] << 32) | d[0];
            if ((head & mask) == 0) { atomicMin(&ts->nonce, (unsigned long long)x); done = true; }
        }
        if (__all_sync(0xffffffffu, done)) break;
    }
}

// get_query_positions: draw_integers(num_queries, N, nonce) — reseed with the nonce, then position_i = low bits of the first
// u64 of merge_with_int(seed, i), i = 1..  (sorting / dedup is the host's job when it assembles the proof)
__global__ void __launch_bounds__(ZKB_FS_THREADS) k_fs_positions(DevTs* ts, uint32_t num_queries, uint32_t domain_mask) {
    __shared__ uint32_t s_seed[8];
    if (threadIdx.x == 0) {
        uint32_t seed[8], t[8];
#pragma unroll
        for (int i = 0; i < 8; i++) seed[i] = ts->seed[i];
        b3_with_int(seed, ts->nonce, t);
#pragma unroll
        for (int i = 0; i < 8; i++) { s_seed[i] = t[i]; ts->seed[i] = t[i]; }
    }
    __syncthreads();
    uint32_t seed[8];
#pragma unroll
    for (int i = 0; i < 8; i++) seed[i] = s_seed[i];
    for (uint32_t q = threadIdx.x; q < num_queries; q += blockDim.x) {
        uint32_t d[8];
        b3_with_int(seed, (uint64_t)q + 1, d);
        ts->positions[q] = d[0] & domain_mask;
    }
}

}  // namespace zkb
