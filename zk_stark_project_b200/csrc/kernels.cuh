// CUDA kernels of the proving hot path (sm_100a).  Stage numbering K1..K11 follows SURVEY.md §2.4;
// each kernel names the Winterfell stage it replaces and the reference line that selects that stage.
//
// Data layouts in HBM (all elements 16 B little-endian canonical f128):
//   trace      column-major [w][n]                    as handed over by the caller (TraceTable columns)
//   polys      row-major    [n][w]  (coefficient m major, column j minor)
//   LDE        "panel" layout: rows that the last NTT pass of one coset produces together form a panel
//              of P = 2^log_p rows, stored column-major inside the panel:
//                 row r = i*beta + k  (i = trace-domain index, k = coset),  T = n/P,
//                 panel = k*T + (i mod T),  slot = i div T,
//                 addr(r, j) = ((panel*w + j) << log_p) + slot
//              so that a kernel with one thread per row (hashing, constraint evaluation, DEEP) reads
//              column j of 32 consecutive slots as one coalesced 512-byte request.
#pragma once
#include "f128.cuh"
#include "blake3.cuh"
#include "coin.cuh"

namespace zkb {

// two-level power table: base^e = lo[e & (2^l1 - 1)] * hi[e >> l1]
struct PowTab {
    const fe* lo;
    const fe* hi;
    uint32_t l1;
};
__device__ __forceinline__ fe powtab(const PowTab& t, uint32_t e) {
    fe a = fe_ldg(t.lo + (e & ((1u << t.l1) - 1u)));
    fe b = fe_ldg(t.hi + (e >> t.l1));
    return fe_mul(a, b);
}

// LDE matrix descriptor.  Single GPU: log_shard = 0, bw = w and the layout is the panel layout above.
// Column-sharded multi-GPU proofs (G = 2^log_shard ranks) store the array as [G][panels][bw][P'] with P' = P/G = 2^log_p:
//   send view (view = 0) on rank r: its bw = w/G columns, all rows; chunk index = slot div P' (the destination rank)
//   recv view (view = 1) on rank q: all w columns, its rows (slots [q P', (q+1) P')); chunk index = column div bw (the source)
// The NVLink all-to-all exchanges chunk q of rank r with chunk r of rank q, so both views share one address formula.
struct LdeMat {
    fe* data;
    uint32_t log_n, log_beta, w, log_p;   // log_p: slots per stored chunk (P' = P >> log_shard)
    uint32_t log_shard, bw, bw_magic, view, q_self;   // bw_magic = ceil(2^16 / bw): j / bw == (j * bw_magic) >> 16 for j, bw <= 256
    uint64_t blk_stride;                  // elements between column blocks (recv view): panels * bw * P'
    uint32_t k0, log_kc;                  // cosets stored: k in [k0, k0 + 2^log_kc) (all of them: k0 = 0, log_kc = log_beta)
};
__device__ __forceinline__ uint32_t lde_full_log_p(const LdeMat& m) { return m.log_p + m.log_shard; }
// address of (row (k, i), column 0 of block 0)
__device__ __forceinline__ size_t lde_row_base(const LdeMat& m, uint32_t k, uint32_t i) {
    const uint32_t lt = m.log_n - lde_full_log_p(m);
    const uint32_t t_low = i & ((1u << lt) - 1u), slot = i >> lt;
    const size_t panel = ((size_t)(k - m.k0) << lt) + t_low;
    const size_t np = (size_t)1 << (m.log_kc + lt);
    const uint32_t chunk = m.view == 0 ? (slot >> m.log_p) : 0u;
    return (((size_t)chunk * np + panel) * m.bw << m.log_p) + (slot & ((1u << m.log_p) - 1u));
}
// The rows a rank stores, enumerated (panel, slot): consecutive row numbers are consecutive slots of one panel.  Row `gid` is
// (coset k, trace-domain index i); its Merkle leaf is r = i*beta + k - leaf0, or, compact (coset-sharded matrices),
// r = i * (stored cosets) + local coset.
struct LdeLeaf { uint32_t k, i; uint64_t r; };
__device__ __forceinline__ LdeLeaf lde_leaf(const LdeMat& m, uint64_t gid, uint64_t leaf0, uint32_t compact) {
    const uint32_t lpf = lde_full_log_p(m), lt = m.log_n - lpf;
    const uint32_t lslots = m.view == 0 ? lpf : m.log_p;
    const uint32_t s = (uint32_t)gid & ((1u << lslots) - 1u);
    const uint32_t panel = (uint32_t)(gid >> lslots);
    const uint32_t slot = m.view == 0 ? s : ((m.q_self << m.log_p) + s);
    const uint32_t k = m.k0 + (panel >> lt), t_low = panel & ((1u << lt) - 1u);
    const uint32_t i = t_low + (slot << lt);
    return {k, i, compact ? (((uint64_t)i << m.log_kc) + (k - m.k0)) : (((uint64_t)i << m.log_beta) + k - leaf0)};
}
__device__ __forceinline__ size_t lde_col_off(const LdeMat& m, uint32_t j) {
    const uint32_t blk = (j * m.bw_magic) >> 16;
    return (size_t)blk * m.blk_stride + ((size_t)(j - blk * m.bw) << m.log_p);
}
__device__ __forceinline__ size_t lde_addr(const LdeMat& m, uint32_t k, uint32_t i, uint32_t j) {
    return lde_row_base(m, k, i) + lde_col_off(m, j);
}

// ------------------------------------------------------------------------------------------------
// transpose: `wc` columns of a column-major matrix (column length n) -> columns [0, wc) of a row-major matrix
// with row stride `out_stride`   (first step of K1; called per column group).  This is where caller data enters the field
// arithmetic: a raw u128 in [p, 2^128) is reduced here, as winter-math's BaseElement::new does (one add-and-select per cell).
__global__ void k_transpose_cols(const fe* __restrict__ in, fe* __restrict__ out, uint32_t n, uint32_t wc, uint32_t out_stride) {
    __shared__ uint4 tile[32][33];
    const uint32_t i0 = blockIdx.x * 32, j0 = blockIdx.y * 32;
    for (uint32_t jj = threadIdx.y; jj < 32; jj += blockDim.y) {
        uint32_t j = j0 + jj, i = i0 + threadIdx.x;
        if (j < wc && i < n) {
            const fe v = fe_canon(fe_load(in + (size_t)j * n + i), 0);
            tile[jj][threadIdx.x] = make_uint4(v.x[0], v.x[1], v.x[2], v.x[3]);
        }
    }
    __syncthreads();
    for (uint32_t ii = threadIdx.y; ii < 32; ii += blockDim.y) {
        uint32_t i = i0 + ii, j = j0 + threadIdx.x;
        if (j < wc && i < n) reinterpret_cast<uint4*>(out)[(size_t)i * out_stride + j] = tile[threadIdx.x][ii];
    }
}

// ------------------------------------------------------------------------------------------------
// K1/K2/K6/K8: one pass of a column-batched radix-2 DIT NTT over layers (a, b].
//
// Mathematics (Winterfell fft::interpolate_poly / evaluate_poly_with_offset, reached through
// DefaultTraceLde::new at src/training/prover.rs:280 and DefaultConstraintCommitment::new at :299):
//   A_l[u][t] = sum_{m' < 2^l} c[u + (n/2^l) m'] * s_l^{m'} * w_{2^l}^{m' t},   s_l = s^{n/2^l}
//   A_l[u][t'], A_l[u][t' + 2^{l-1}] = A_{l-1}[u][t'] +- (s_l w_{2^l}^{t'}) * A_{l-1}[u + n/2^l][t']
// with s = 3*w_N^k for coset k of the LDE (the coset shift is folded into the twiddles, so the LDE costs
// exactly (n/2) log n multiplications per coset and column), s = 1 and inverse roots for interpolation.
// Between passes the array holds A_b as  index = u*2^b + t  (row-major [index][column]).
// A tile = S = 2^(b-a) rows (u = u0 + (n/2^b) v, fixed t_low) x cj columns staged in shared memory;
// its S-1 twiddles are generated once per tile and shared by all columns of the batch.
struct NttPass {
    const fe* in;
    fe* out;
    uint32_t log_n, a, b;          // transform size, layer range
    uint32_t w_in, w_out;          // row widths of the in / out matrices (elements)
    uint32_t col0_in, col0_out, ncols, cj;
    uint32_t n_cosets, coset0;     // cosets k = coset0 + kk; ignored when `coset` == 0
    uint64_t in_coset_stride, out_coset_stride;  // elements between consecutive cosets (0 = shared input)
    uint32_t coset;                // 1: s = 3*w_N^k (forward roots); 0: s = 1
    uint32_t inverse;              // 1: inverse roots (interpolation)
    uint32_t log_tab;              // root table covers <w_{2^log_tab}>
    uint32_t log_lde;              // log2(n * beta) for coset transforms
    uint32_t out_panel;            // final pass of an LDE: write the panel layout
    uint32_t log_shard;            // panel layout split into 2^log_shard slot chunks (multi-GPU send view)
    uint32_t panel_k0, log_kc;     // the output stores cosets [panel_k0, panel_k0 + 2^log_kc) only (coset-sharded LDEs)
    uint32_t do_scale;             // multiply outputs by `scale` (1/n for interpolation)
    fe scale;
    PowTab roots;                  // w_{2^log_tab}^e
    const fe* pow3;                // pow3[l] = 3^(n >> l), l = 0..log_n
    const fe* tw_tab;              // optional: precomputed tile twiddles [(k << a) + t_low][S - 1] (k_build_twiddles); null = generate
    uint32_t tw_four;              // tw_tab holds every twiddle as its four pre-shifted copies (fe4, four fe per entry)
    uint32_t tile0;                // (t_low, u0) index of blockIdx.z == 0: launches of more than 65535 of them are split
};

__device__ __forceinline__ uint32_t bitrev(uint32_t v, uint32_t bits) { return bits == 0 ? 0u : (__brev(v) >> (32 - bits)); }

// twiddle multiply of a butterfly: plain twiddles (fe) or four pre-shifted copies (fe4, f128.cuh)
__device__ __forceinline__ fe tw_mul(const fe& x, const fe& w) { return fe_mul(x, w); }
__device__ __forceinline__ fe tw_mul(const fe& x, const fe4& w) { return fe_mul_pre4(x, w); }

// RHO consecutive DIT layers (lam0, lam0 + RHO] of NC columns, done in registers: the 2^RHO elements of a unit sit at
// positions base + d * 2^lam0.  Layer lam uses tw[2^(lam-1) - 1 + (p0 mod 2^(lam-1))] for the pair (p0, p0 + 2^(lam-1)).
// With four-copy twiddles (TW = fe4) one 64-byte load serves NC * 2^(RHO-1-s) butterflies of layer s; narrow tiles (1-2
// columns) reuse a twiddle too rarely for the three shift-folds of fe4_from to pay and take plain ones (TW = fe, NC = 1).
// The NC columns of a thread are `cstride` apart so that the threads of a quarter-warp touch one contiguous 128-byte run.
template <int RHO, int NC, class TW>
__device__ __forceinline__ void ntt_unit(fe* __restrict__ col, const uint32_t rs, const uint32_t cstride, const TW* __restrict__ tw,
                                         const uint32_t base, const uint32_t lam0) {
    constexpr int R = 1 << RHO;
    fe x[NC][R];
    const uint32_t step = rs << lam0;
    fe* p = col + base * rs;
#pragma unroll
    for (int c = 0; c < NC; c++)
#pragma unroll
        for (int d = 0; d < R; d++) x[c][d] = p[d * step + c * cstride];
    const uint32_t base_low = base & ((1u << lam0) - 1u);
#pragma unroll
    for (int s = 0; s < RHO; s++) {
        const TW* twl = tw + ((1u << (lam0 + s)) - 1u) + base_low;
#pragma unroll
        for (int t = 0; t < (1 << s); t++) {
            const TW w = twl[(uint32_t)t << lam0];
#pragma unroll
            for (int g = 0; g < (R >> (s + 1)); g++) {
                const int d0 = g * (2 << s) + t, d1 = d0 + (1 << s);
#pragma unroll
                for (int c = 0; c < NC; c++) {
                    const fe u = x[c][d0];
                    const fe v = tw_mul(x[c][d1], w);
                    x[c][d0] = fe_add(u, v);
                    x[c][d1] = fe_sub(u, v);
                }
            }
        }
    }
#pragma unroll
    for (int c = 0; c < NC; c++)
#pragma unroll
        for (int d = 0; d < R; d++) p[d * step + c * cstride] = x[c][d];
}

// twiddle q of the tile (coset k, t_low) of a pass: layer lam = floor(log2(q + 1)) + 1, position th = q + 1 - 2^(lam-1)
__device__ __forceinline__ fe ntt_twiddle(const NttPass& p, uint32_t k, uint32_t t_low, uint32_t q) {
    const uint32_t logS = p.b - p.a;
    const uint32_t tab_mask = (1u << p.log_tab) - 1u;
    const uint32_t lam = 32 - __clz(q + 1);      // 1..logS
    const uint32_t th = q + 1 - (1u << (lam - 1));
    const uint32_t l = p.a + lam;
    (void)logS;
    // exponent in units of w_{2^log_tab}
    uint32_t e = (t_low << (p.log_tab - l)) + (th << (p.log_tab - lam));
    if (p.coset) e += (k << (p.log_n - l)) << (p.log_tab - p.log_lde);
    e &= tab_mask;
    if (p.inverse) e = (0u - e) & tab_mask;
    fe t = powtab(p.roots, e);
    if (p.coset) t = fe_mul(t, fe_ldg(p.pow3 + l));
    return t;
}
// all tile twiddles of a pass, for cosets [0, n_cosets): table[((k << a) + t_low) * (S - 1) + q], as four pre-shifted copies
// (fe4) when p.tw_four, so that the tiles of k_ntt_pass<true> only copy them
__global__ void k_build_twiddles(const NttPass p, fe* __restrict__ table) {
    const uint32_t S = 1u << (p.b - p.a);
    const uint64_t total = ((uint64_t)p.n_cosets << p.a) * (S - 1u);
    const uint64_t id = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= total) return;
    const uint32_t q = (uint32_t)(id % (S - 1u));
    const uint32_t tile = (uint32_t)(id / (S - 1u));
    const fe w = ntt_twiddle(p, tile >> p.a, tile & ((1u << p.a) - 1u), q);
    if (p.tw_four) {
        const fe4 t = fe4_from(w);
#pragma unroll
        for (int i = 0; i < 4; i++) fe_store(table + 4 * id + i, t.w[i]);
    } else fe_store(table + id, w);
}
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}

template <int RHO, int NC, class TW>
__device__ __forceinline__ void ntt_round(fe* sm, const TW* tw, uint32_t rs, uint32_t log_cj, uint32_t logS, uint32_t lam0) {
    // a thread owns columns jj and (NC == 2) jj + cj/2 of one unit
    const uint32_t log_cw = log_cj - (NC == 2 ? 1u : 0u);
    const uint32_t cw_mask = (1u << log_cw) - 1u;
    const uint32_t units = (1u << (logS - RHO)) << log_cw;
    for (uint32_t idx = threadIdx.x; idx < units; idx += blockDim.x) {
        const uint32_t jj = idx & cw_mask, u = idx >> log_cw;
        const uint32_t base = (u & ((1u << lam0) - 1u)) + ((u >> lam0) << (lam0 + RHO));
        ntt_unit<RHO, NC>(sm + jj, rs, 1u << log_cw, tw, base, lam0);
    }
}
template <int NC, class TW>
__device__ __forceinline__ void ntt_rounds(fe* sm, const TW* tw, uint32_t rs, uint32_t log_cj, uint32_t logS) {
    // rounds of up to three layers held in registers
    if (NC == 2 && log_cj == 4 && logS == 8) {
        // 256 x 16 tiles (every pass of the 2^16-row transforms of >= 9 columns): with the strides and layer offsets known at
        // compile time the 16 element addresses of a unit are immediate offsets from one register
        uint32_t lam0 = 0;
        asm("" : "+r"(lam0));   // kept opaque: constant twiddle addresses would be hoisted (112 registers) and spilled
        ntt_round<3, NC>(sm, tw, 17, 4, 8, lam0); __syncthreads();
        ntt_round<3, NC>(sm, tw, 17, 4, 8, 3); __syncthreads();
        ntt_round<2, NC>(sm, tw, 17, 4, 8, 6); __syncthreads();
        return;
    }
    for (uint32_t lam0 = 0; lam0 < logS;) {
        const uint32_t left = logS - lam0;
        if (left >= 3 && left != 4) { ntt_round<3, NC>(sm, tw, rs, log_cj, logS, lam0); lam0 += 3; }
        else if (left >= 2) { ntt_round<2, NC>(sm, tw, rs, log_cj, logS, lam0); lam0 += 2; }
        else { ntt_round<1, NC>(sm, tw, rs, log_cj, logS, lam0); lam0 += 1; }
        __syncthreads();
    }
}

// PRE = true (tiles of >= 4 columns): four-copy twiddles; two blocks of 256 threads per SM, a thread carries a two-column radix-8
// unit (16 elements + one fe4 twiddle in registers, ILP 8), and a 256-row x 16-column tile plus its 255 four-copy twiddles is
// 86 KB of shared memory.  PRE = false (1-2 columns): plain twiddles, one column per thread, three blocks per SM when they fit.
template <bool PRE>
__global__ void __launch_bounds__(256, PRE ? 2 : 3) k_ntt_pass(const NttPass p) {
    extern __shared__ uint4 smem_raw[];
    fe* sm = reinterpret_cast<fe*>(smem_raw);
    const uint32_t logS = p.b - p.a, S = 1u << logS, cj = p.cj;
    const uint32_t log_cj = 31 - __clz(cj);
    const uint32_t rs = cj + (cj > 1 ? 1u : 0u);  // padded row stride: conflict-free column reads
    fe4* tw = reinterpret_cast<fe4*>(sm + (size_t)S * rs);
    fe* tw1 = sm + (size_t)S * rs;

    // tile coordinates (x = column tile, y = coset, z = (t_low, u0)): blocks are dispatched x fastest, so the cosets of one input
    // tile run back to back and reuse it out of L2
    const uint32_t ct = blockIdx.x, kk = blockIdx.y, id = p.tile0 + blockIdx.z;
    const uint32_t t_low = id & ((1u << p.a) - 1u);
    const uint32_t u0 = id >> p.a;
    const uint32_t k = p.coset0 + kk;
    // twiddles: tw[2^(lam-1) - 1 + th] = s_l * w_{2^l}^{t_low} * w_{2^lam}^{th},  l = a + lam.  A four-copy table is copied as it
    // is (cp.async, overlapped with the tile load); otherwise the three shifted copies are derived here, once per tile
    if (PRE && p.tw_four) {
        const uint4* t = reinterpret_cast<const uint4*>(p.tw_tab) + ((size_t)(k << p.a) + t_low) * (4u * (S - 1u));
        uint4* d = reinterpret_cast<uint4*>(tw);
#pragma unroll 1
        for (uint32_t q = threadIdx.x; q < 4u * (S - 1u); q += blockDim.x) cp_async16(d + q, t + q);
        asm volatile("cp.async.commit_group;" ::: "memory");
    } else {
        const fe* t = p.tw_tab ? p.tw_tab + ((size_t)(k << p.a) + t_low) * (S - 1u) : nullptr;
        for (uint32_t q = threadIdx.x; q + 1 < S; q += blockDim.x) {
            const fe w = t ? fe_ldg(t + q) : ntt_twiddle(p, k, t_low, q);
            if (PRE) tw[q] = fe4_from(w); else tw1[q] = w;
        }
    }
    // load: row v of the tile is input row (u0 + (n/2^b) v) * 2^a + t_low; store bit-reversed.
    // blockDim (a power of two >= cj) is a multiple of cj, so a thread keeps its column and walks rows v_t, v_t + dv, .. with a
    // constant pointer stride; counting them with shifts keeps integer divisions out of the loops.
    const uint32_t c_base = ct << log_cj;
    const uint32_t log_bd = 31 - __clz(blockDim.x), log_dv = log_bd - log_cj;
    const uint32_t jj_t = threadIdx.x & (cj - 1u), v_t = threadIdx.x >> log_cj, dv = 1u << log_dv;
    const uint32_t nrow = v_t < S ? ((S - 1u - v_t) >> log_dv) + 1u : 0u;   // rows of this thread
    const bool col_ok = c_base + jj_t < p.ncols;
    {
        const size_t vstride = ((size_t)p.w_in << (p.log_n - p.b)) << p.a;
        const fe* src = p.in + (size_t)kk * p.in_coset_stride + (((size_t)u0 << p.a) + t_low) * p.w_in + p.col0_in + c_base + jj_t +
                        (size_t)v_t * vstride;
        const size_t dstride = (size_t)dv * vstride;
        char* smc = reinterpret_cast<char*>(sm + jj_t);
        const uint32_t brs = (32u - logS) & 31u;  // logS == 0: the only row is v = 0 and brev(0) == 0
        const uint32_t rs16 = rs * 16u;
        uint32_t vs = v_t << brs;                 // brev(vs) = brev(v) >> brs: row v's bit-reversed position
        const uint32_t dvs = dv << brs;
        if (col_ok) {
#pragma unroll 4
            for (uint32_t i = 0; i < nrow; i++, vs += dvs, src += dstride) *reinterpret_cast<fe*>(smc + __brev(vs) * rs16) = fe_load(src);
        } else {  // columns past the end of a ragged last tile are zero-filled
            for (uint32_t i = 0; i < nrow; i++, vs += dvs) *reinterpret_cast<fe*>(smc + __brev(vs) * rs16) = fe_zero();
        }
    }
    if (PRE) asm volatile("cp.async.wait_all;" ::: "memory");
    __syncthreads();
    // butterflies
    if (PRE) { if (cj >= 16) ntt_rounds<2>(sm, tw, rs, log_cj, logS); else ntt_rounds<1>(sm, tw, rs, log_cj, logS); }   // narrow tiles: one column per thread
    else ntt_rounds<1>(sm, tw1, rs, log_cj, logS);
    // store
    if (p.out_panel) {
        // panel = k*2^a + t_low, slot = t_high; consecutive threads write consecutive slots of one column.  A thread keeps its
        // slot(s) and walks columns: with S >= blockDim every thread covers slots tid, tid + blockDim, .. of each column; smaller
        // tiles put blockDim / S columns side by side
        const size_t panel = ((size_t)(k - p.panel_k0) << p.a) + t_low;
        const uint32_t lp = logS - p.log_shard;                       // slots per stored chunk
        const size_t np = (size_t)1 << (p.log_kc + p.a);              // panels = stored cosets * 2^a
        const size_t chunk_stride = (np * p.w_out) << lp;             // elements between slot chunks (multi-GPU send view)
        const bool wide = S >= blockDim.x;
        const uint32_t th0 = wide ? threadIdx.x : (threadIdx.x & (S - 1u)), dth = wide ? blockDim.x : S;
        const uint32_t jj0 = wide ? 0u : (threadIdx.x >> logS), log_djj = wide ? 0u : log_bd - logS, djj = 1u << log_djj;
        const uint32_t jend = min(cj, p.ncols - c_base);
        const uint32_t ncol = jj0 < jend ? ((jend - 1u - jj0) >> log_djj) + 1u : 0u;
        const size_t cstep = (size_t)djj << lp;                      // elements between the thread's columns
        fe* colp = p.out + ((panel * p.w_out + p.col0_out + c_base + jj0) << lp);
#pragma unroll 1
        for (uint32_t th = th0; th < S; th += dth) {
            fe* d = colp + (size_t)(th >> lp) * chunk_stride + (th & ((1u << lp) - 1u));
            const fe* s = sm + th * rs + jj0;
#pragma unroll 4
            for (uint32_t j = 0; j < ncol; j++, d += cstep, s += djj) fe_store(d, *s);
        }
    } else {
        const size_t tstride = (size_t)p.w_out << p.a;
        fe* dst = p.out + (size_t)kk * p.out_coset_stride + (((size_t)u0 << p.b) + t_low) * p.w_out + p.col0_out + c_base + jj_t +
                  (size_t)v_t * tstride;
        const size_t dstride = (size_t)dv * tstride;
        const fe* s = sm + v_t * rs + jj_t;
        const uint32_t sstep = dv * rs;
        if (col_ok) {
            if (p.do_scale) {
                for (uint32_t i = 0; i < nrow; i++, dst += dstride, s += sstep) fe_store(dst, fe_mul(*s, p.scale));
            } else {
#pragma unroll 4
                for (uint32_t i = 0; i < nrow; i++, dst += dstride, s += sstep) fe_store(dst, *s);
            }
        }
    }
}

// x[m] *= scale * base^m   (interpolate_poly_with_offset: base = 1/offset).  Coefficients at m >= keep are dropped by the caller
// (CompositionPoly::new keeps c*n of the ce*n); a non-zero one means the trace violates the AIR: *bad_degree is raised.
__global__ void k_scale_pow(fe* x, uint64_t n, PowTab base, fe scale, uint64_t keep, uint32_t* __restrict__ bad_degree) {
    uint64_t m = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n) return;
    const fe v = fe_load(x + m);
    if (m >= keep) { if (!fe_is_zero(v)) atomicOr(bad_degree, 1u); return; }
    fe f = fe_mul(powtab(base, (uint32_t)m), scale);
    fe_store(x + m, fe_mul(v, f));
}

// ------------------------------------------------------------------------------------------------
// K3: leaf = Blake3_256::hash_elements(LDE row)  (RowMatrix::commit_to_rows; src/training/prover.rs:225,280)
// one thread per stored LDE row, enumerated (panel, slot) so that a warp reads 32 consecutive slots per column.
// leaves: digest array indexed by (global leaf index - leaf0); in the multi-GPU recv view a rank stores and hashes only
// the rows of its slot chunk, which are the contiguous leaves [q N/G, (q+1) N/G).
__global__ void __launch_bounds__(128) k_hash_lde_rows(const LdeMat m, uint32_t* __restrict__ leaves, uint64_t leaf0, uint32_t compact) {
    const uint64_t gid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t lpf = lde_full_log_p(m), lt = m.log_n - lpf;
    const uint32_t log_rows = m.log_kc + lt + (m.view == 0 ? lpf : m.log_p);   // rows stored on this rank
    if (gid >> log_rows) return;
    const LdeLeaf L = lde_leaf(m, gid, leaf0, compact);
    uint32_t d[8];
    b3_hash_elems(m.data + lde_row_base(m, L.k, L.i), (size_t)1 << m.log_p, m.w, d, m.bw, m.bw_magic, m.blk_stride);
    uint4* o = reinterpret_cast<uint4*>(leaves + L.r * 8);
    o[0] = make_uint4(d[0], d[1], d[2], d[3]);
    o[1] = make_uint4(d[4], d[5], d[6], d[7]);
}
// The same leaves for a matrix of a few thousand rows (the aggregation proof: 512 rows x 120 columns): one thread per
// (row, 1 KiB chunk) — a row's chunks are independent until their chaining values meet in the BLAKE3 tree, so a 1920-byte
// row costs 16 + 1 dependent compressions instead of 31.  Four lanes per row; lanes past the row's chunk count idle.
__global__ void __launch_bounds__(128) k_hash_lde_rows_split(const LdeMat m, uint32_t* __restrict__ leaves, uint64_t leaf0, uint32_t compact) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t c = (uint32_t)t & 3u;
    const uint32_t lpf = lde_full_log_p(m), lt = m.log_n - lpf;
    const uint32_t log_rows = m.log_kc + lt + (m.view == 0 ? lpf : m.log_p);
    const bool live = ((t >> 2) >> log_rows) == 0;      // whole warps take part in the shuffles; dead rows hash row 0 and drop it
    const LdeLeaf L = lde_leaf(m, live ? (t >> 2) : 0, leaf0, compact);
    const uint32_t nchunks = (m.w + 63u) / 64u;         // 2..4 (the caller sends single-chunk rows to k_hash_lde_rows)
    uint32_t cv[8], nb[8];
    if (c < nchunks) b3_chunk_cv_elems(m.data + lde_row_base(m, L.k, L.i), (size_t)1 << m.log_p, m.w, c, cv, m.bw, m.bw_magic, m.blk_stride);
    else {
#pragma unroll
        for (int q = 0; q < 8; q++) cv[q] = 0;
    }
    // tree: 2 chunks parent(0,1); 3 chunks parent(parent(0,1), 2); 4 chunks parent(parent(0,1), parent(2,3))
#pragma unroll
    for (int q = 0; q < 8; q++) nb[q] = __shfl_down_sync(0xffffffffu, cv[q], 1);
    if (c == 0 || (c == 2 && nchunks == 4)) {
        uint32_t o[8];
        b3_parent(cv, nb, nchunks == 2, o);
#pragma unroll
        for (int q = 0; q < 8; q++) cv[q] = o[q];
    }
    if (nchunks > 2) {
#pragma unroll
        for (int q = 0; q < 8; q++) nb[q] = __shfl_down_sync(0xffffffffu, cv[q], 2);
        if (c == 0) {
            uint32_t o[8];
            b3_parent(cv, nb, true, o);
#pragma unroll
            for (int q = 0; q < 8; q++) cv[q] = o[q];
        }
    }
    if (live && c == 0) {
        uint4* o = reinterpret_cast<uint4*>(leaves + L.r * 8);
        o[0] = make_uint4(cv[0], cv[1], cv[2], cv[3]);
        o[1] = make_uint4(cv[4], cv[5], cv[6], cv[7]);
    }
}
// multi-GPU: after an all-gather of per-rank compact arrays [src][i * kc + kl] (kc = stored cosets per rank), put item
// (i, k = src*kc + kl) at natural LDE position i*beta + k.  `words` 32-bit words per item (8: digests, 4: field elements).
__global__ void k_permute_coset_items(const uint32_t* __restrict__ gathered, uint32_t* __restrict__ out, uint32_t log_n, uint32_t log_beta,
                                      uint32_t log_kc, uint32_t words) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;   // one thread per (item, 16-byte quarter)
    const uint32_t q4 = words >> 2;
    const uint64_t item = t / q4;
    if (item >> (log_n + log_beta)) return;
    const uint32_t part = (uint32_t)(t - item * q4);
    const uint32_t k = (uint32_t)item & ((1u << log_beta) - 1u);
    const uint64_t i = item >> log_beta;
    const uint32_t src = k >> log_kc, kl = k & ((1u << log_kc) - 1u);
    const uint64_t from = ((uint64_t)src << (log_n + log_kc)) + (i << log_kc) + kl;
    reinterpret_cast<uint4*>(out)[item * q4 + part] = reinterpret_cast<const uint4*>(gathered)[from * q4 + part];
}

// FRI layer rows: leaf_i = hash_elements([e[i + j*rows]]_{j<F})   (winter-fri build_layer / transpose_slice)
__global__ void __launch_bounds__(128) k_hash_strided_rows(const fe* __restrict__ e, uint64_t rows, uint32_t count, uint32_t* __restrict__ leaves) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows) return;
    uint32_t d[8];
    b3_hash_elems(e + i, rows, count, d, 256, 256, 0);
    uint4* o = reinterpret_cast<uint4*>(leaves + i * 8);
    o[0] = make_uint4(d[0], d[1], d[2], d[3]);
    o[1] = make_uint4(d[4], d[5], d[6], d[7]);
}

// K4: one level of MerkleTree::new (build_merkle_nodes): dst[i] = merge(src[2i], src[2i+1])
__global__ void __launch_bounds__(256) k_merkle_level(const uint32_t* __restrict__ src, uint32_t* __restrict__ dst, uint64_t count) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const uint4* s = reinterpret_cast<const uint4*>(src + i * 16);
    const uint4 a = s[0], b = s[1], c = s[2], d = s[3];
    const uint32_t l[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w}, r[8] = {c.x, c.y, c.z, c.w, d.x, d.y, d.z, d.w};
    uint32_t cv[8];
    b3_merge(l, r, cv);
    uint4* o = reinterpret_cast<uint4*>(dst + i * 8);
    o[0] = make_uint4(cv[0], cv[1], cv[2], cv[3]);
    o[1] = make_uint4(cv[4], cv[5], cv[6], cv[7]);
}

// top of a Merkle heap in one launch: levels top, top/2, ..., 1 (top <= 512 nodes) by a single block; every level is
// read back from global memory after a block barrier (the data is a few KB and stays in L1/L2)
__global__ void __launch_bounds__(512) k_merkle_top(uint32_t* __restrict__ heap, uint32_t top) {
    for (uint32_t lvl = top; lvl >= 1; lvl >>= 1) {
        const uint32_t i = threadIdx.x;
        if (i < lvl) {
            const uint4* s = reinterpret_cast<const uint4*>(heap + (size_t)(2 * (lvl + i)) * 8);
            const uint4 a = s[0], b = s[1], c = s[2], d = s[3];
            const uint32_t l[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w}, r[8] = {c.x, c.y, c.z, c.w, d.x, d.y, d.z, d.w};
            uint32_t cv[8];
            b3_merge(l, r, cv);
            uint4* o = reinterpret_cast<uint4*>(heap + (size_t)(lvl + i) * 8);
            o[0] = make_uint4(cv[0], cv[1], cv[2], cv[3]);
            o[1] = make_uint4(cv[4], cv[5], cv[6], cv[7]);
        }
        __threadfence_block();
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------
// K5: DefaultConstraintEvaluator::evaluate (src/training/prover.rs:283-290) fused with
// ConstraintEvaluationTable::combine: one thread per constraint-evaluation-domain point.
enum { ZKB_AIR_TRAINING = 1, ZKB_AIR_AGGREGATION = 2, ZKB_AIR_MIMC = 3 };
#define ZKB_MAX_GROUPS 4
struct EvalParams {
    LdeMat lde;
    uint32_t air_id, log_ce;      // ce blowup = 2^log_ce
    uint32_t n_trans;             // number of transition constraints
    const fe* tcoef;              // transition coefficients (alpha^0 ..)
    uint32_t n_groups;
    uint32_t g_off[ZKB_MAX_GROUPS + 1];  // assertion ranges per boundary group
    const uint32_t* a_col;        // per assertion of this column window: column, index into the global (sorted) assertion list
    const uint32_t* a_sel;
    const fe* a_val;              // global assertion values / coefficients (device-resident: written per proof, read by index)
    const fe* a_coef;
    const fe* div;                // divisor table of the shape, [(n_groups + 1)][ce n] (k_build_divisors)
    const fe* params;             // aggregation: params[0] = scaling factor k (src/aggregation/air.rs:108)
    const fe* periodic;           // MiMC: round-constant column over the ce domain, length per_len
    uint32_t per_mask;
    fe* out;                      // composition trace, natural ce-domain order
    // boundary numerators as polynomials: bnd column g holds B_g(x) = sum_a coef_a (T_col_a(x) - value_a) over the ce domain
    // (combined in coefficient space by k_boundary_combine, extended once); used when that is cheaper than per-point sums
    uint32_t bnd_poly;
    LdeMat bnd;
};

// Row-wise combinations of the trace polynomials (k_boundary_combine, k_deep_combine): ZKB_ROW_LANES lanes share a coefficient row
#define ZKB_ROW_LANES 8
__device__ __forceinline__ fe fe_group_sum(fe s) {   // sum over the ZKB_ROW_LANES lanes of a row group; valid on its first lane
#pragma unroll
    for (int off = ZKB_ROW_LANES / 2; off > 0; off >>= 1) {
        fe o;
        o.x[0] = __shfl_down_sync(0xffffffffu, s.x[0], off, ZKB_ROW_LANES); o.x[1] = __shfl_down_sync(0xffffffffu, s.x[1], off, ZKB_ROW_LANES);
        o.x[2] = __shfl_down_sync(0xffffffffu, s.x[2], off, ZKB_ROW_LANES); o.x[3] = __shfl_down_sync(0xffffffffu, s.x[3], off, ZKB_ROW_LANES);
        s = fe_add(s, o);
    }
    return s;
}
// B_g coefficients: bc[m][g] = sum_{a in group g} coef_a * polys[m][col_a]  (minus sum_a coef_a * value_a at m = 0);
// a lane group per coefficient row, its lanes stride over the assertions of each boundary group
struct BoundaryGroups { uint32_t n_groups; uint32_t g_off[ZKB_MAX_GROUPS + 1]; };
__global__ void __launch_bounds__(256) k_boundary_combine(const fe* __restrict__ polys, uint32_t n, uint32_t w, const uint32_t* __restrict__ a_col,
                                                          const uint32_t* __restrict__ a_sel, const fe* __restrict__ a_coef, const fe* __restrict__ a_val,
                                                          const BoundaryGroups bg, fe* __restrict__ bc) {
    const uint32_t row = (blockIdx.x * blockDim.x + threadIdx.x) / ZKB_ROW_LANES, sub = threadIdx.x & (ZKB_ROW_LANES - 1);
    if (row >= n) return;
    const fe* pr = polys + (size_t)row * w;
    for (uint32_t g = 0; g < bg.n_groups; g++) {
        acc288 acc; acc288_zero(acc);
        acc288 cst; acc288_zero(cst);   // row 0 only: sum_a coef_a * value_a
        for (uint32_t a = bg.g_off[g] + sub; a < bg.g_off[g + 1]; a += ZKB_ROW_LANES) {
            const uint32_t ai = __ldg(a_sel + a);
            const fe cf = fe_ldg(a_coef + ai);
            acc288_mad(acc, fe_load(pr + __ldg(a_col + a)), cf);
            if (row == 0) acc288_mad(cst, fe_ldg(a_val + ai), cf);
        }
        fe s = acc288_reduce(acc);
        if (row == 0) s = fe_sub(s, acc288_reduce(cst));
        s = fe_group_sum(s);
        if (sub == 0) fe_store(bc + (size_t)row * bg.n_groups + g, s);
    }
}

// Divisor table of a shape: everything in the combination that depends only on the evaluation point x = 3 * w_{ce n}^ci —
//   div[g][ci]  = 1 / (x - g^step_g)                    boundary divisors (Air::get_assertions groups)
//   div[ng][ci] = (x - g^(n-1)) / (x^n - 1)             inverse of the transition divisor (x^n - 1)/(x - g^(n-1))
// It does not depend on the trace or on any challenge, so it is built once per (n, ce, assertion steps) and cached by the
// context: the ~45 multiplications per point that the batch inversions cost are paid by the first proof of a shape only.
struct DivParams {
    uint32_t log_cen, log_ce, n_groups;
    fe g_point[ZKB_MAX_GROUPS];
    fe g_last;
    const fe* zinv;               // 1/(x^n - 1) for the 2^log_ce cosets of the ce domain
    PowTab roots; uint32_t log_tab;
    fe* out;                      // [(n_groups + 1)][2^log_cen]
};
#define ZKB_DIV_RPT 8
__global__ void __launch_bounds__(128) k_build_divisors(const DivParams p) {
    const uint64_t total = (uint64_t)1 << p.log_cen;
    const uint64_t nthreads = total / ZKB_DIV_RPT;    // ce * n >= 16: a multiple of 8
    const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (tid >= nthreads) return;
    const uint32_t ng = p.n_groups;
    fe den[ZKB_DIV_RPT * ZKB_MAX_GROUPS], pre[ZKB_DIV_RPT * ZKB_MAX_GROUPS];
    fe acc = fe_one();
    for (int s = 0; s < ZKB_DIV_RPT; s++) {
        const uint32_t ci = (uint32_t)(tid + (uint64_t)s * nthreads);
        fe x = powtab(p.roots, ci << (p.log_tab - p.log_cen));
        { fe x2 = fe_add(x, x); x = fe_add(x2, x); }     // x = 3 * w^ci
        fe_store(p.out + ((size_t)ng << p.log_cen) + ci, fe_mul(fe_sub(x, p.g_last), fe_ldg(p.zinv + (ci & ((1u << p.log_ce) - 1u)))));
        for (uint32_t g = 0; g < ng; g++) {
            const uint32_t q = s * ZKB_MAX_GROUPS + g;
            den[q] = fe_sub(x, p.g_point[g]);
            pre[q] = acc;
            acc = fe_mul(acc, den[q]);
        }
    }
    fe ia = ng ? fe_inv(acc) : fe_one();     // one inversion shared by 8 points (Montgomery's trick)
    for (int s = ZKB_DIV_RPT - 1; s >= 0; s--) {
        const uint32_t ci = (uint32_t)(tid + (uint64_t)s * nthreads);
        for (int g = (int)ng - 1; g >= 0; g--) {
            const uint32_t q = s * ZKB_MAX_GROUPS + g;
            fe_store(p.out + ((size_t)g << p.log_cen) + ci, fe_mul(ia, pre[q]));
            ia = fe_mul(ia, den[q]);
        }
    }
}

// One point of the constraint evaluation domain:  sum_c coef_c * transition_c(frame) * div[ng]  +  sum_g numerator_g * div[g].
// LANES = 1: one thread per point (large domains: every SM is full of points).  LANES = 32: one warp per point, lanes stride
// over the constraints and assertions and their partial results are added by shuffles — for domains of a few hundred points
// (the aggregation proof: 64 points x 60 constraints + 120 assertions) the per-point chain of dependent loads is what the
// proof waits for, not throughput.  Field addition is exact, so both variants store the same canonical element.
template <int LANES>
__global__ void __launch_bounds__(128) k_eval_constraints(const EvalParams p) {
    const LdeMat& m = p.lde;
    const uint64_t total = (uint64_t)1 << (m.log_n + p.log_ce);
    const uint64_t gthread = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t gid = LANES == 1 ? gthread : gthread / LANES;
    const uint32_t lane = LANES == 1 ? 0u : (uint32_t)(threadIdx.x & (LANES - 1));
    if (gid >= total) return;   // LANES = 32: warp-uniform
    const uint32_t lpf = lde_full_log_p(m), lt = m.log_n - lpf;
    const size_t cs = (size_t)1 << m.log_p;  // column stride
    const uint32_t ng = p.n_groups;
    // enumerate points (coset, panel, slot) so that a warp reads 32 consecutive slots of every column
    const uint32_t slot = (uint32_t)gid & ((1u << lpf) - 1u);
    const uint32_t t_low = (uint32_t)(gid >> lpf) & ((1u << lt) - 1u);
    const uint32_t kc = (uint32_t)(gid >> m.log_n);
    const uint32_t k = kc << (m.log_beta - p.log_ce);
    const uint32_t i = t_low + (slot << lt);
    const uint32_t i1 = (i + 1u) & ((1u << m.log_n) - 1u);  // frame.next = row + blowup (mod N)
    const uint32_t ci = (i << p.log_ce) + kc;
    const uint32_t log_cen = m.log_n + p.log_ce;
    const fe* cur = m.data + lde_row_base(m, k, i);   // send view / single GPU: columns are local, stride 2^log_p
    const fe* nxt = m.data + lde_row_base(m, k, i1);

    // transition constraints, merged with their coefficients.  sum_c coef_c * ev_c is accumulated as an exact 288-bit
    // integer and reduced once per point (acc288): same field element, one reduction instead of one per column
    acc288 tacc; acc288_zero(tacc);
    if (p.air_id == ZKB_AIR_AGGREGATION) {
        const uint32_t d = p.n_trans;
        const fe kf = fe_ldg(p.params);
        for (uint32_t c = lane; c < d; c += LANES) {
            fe dn = fe_sub(fe_load(nxt + c * cs), fe_load(cur + c * cs));
            fe ev = fe_sub(fe_mul(kf, dn), fe_load(nxt + (size_t)(c + d) * cs));
            acc288_mad(tacc, fe_ldg(p.tcoef + c), ev);
        }
    } else if (p.air_id == ZKB_AIR_MIMC) {
        const fe rc = fe_ldg(p.periodic + (ci & p.per_mask));
        for (uint32_t c = lane; c < p.n_trans; c += LANES) {
            fe a1 = fe_add(fe_load(cur + c * cs), rc);
            fe a2 = fe_sqr(a1), a4 = fe_sqr(a2), a6 = fe_mul(a4, a2), a7 = fe_mul(a6, a1);
            fe ev = fe_sub(fe_load(nxt + c * cs), a7);
            acc288_mad(tacc, fe_ldg(p.tcoef + c), ev);
        }
    }  // TRAINING: every transition evaluation is zero (src/training/air.rs:274-278, src/helper.rs:141-146)
    fe res = fe_zero();
    if (p.air_id != ZKB_AIR_TRAINING) res = fe_mul(acc288_reduce(tacc), fe_ldg(p.div + ((size_t)ng << log_cen) + ci));

    // boundary groups: sum coef * (cur[col] - value) / (x - g^step)
    const fe* bp = p.bnd_poly ? p.bnd.data + lde_row_base(p.bnd, kc, i) : nullptr;
    for (uint32_t g = 0; g < ng; g++) {
        fe sum;
        if (p.bnd_poly) {
            sum = lane == 0 ? fe_load(bp + ((size_t)g << p.bnd.log_p)) : fe_zero();
        } else {
            acc288 bacc; acc288_zero(bacc);
            for (uint32_t a = p.g_off[g] + lane; a < p.g_off[g + 1]; a += LANES) {
                const uint32_t ai = __ldg(p.a_sel + a);
                fe v = fe_sub(fe_load(cur + (size_t)__ldg(p.a_col + a) * cs), fe_ldg(p.a_val + ai));
                acc288_mad(bacc, fe_ldg(p.a_coef + ai), v);
            }
            sum = acc288_reduce(bacc);
        }
        res = fe_add(res, fe_mul(sum, fe_ldg(p.div + ((size_t)g << log_cen) + ci)));
    }
    if (LANES > 1) {   // every lane holds the terms of its constraints and assertions, each already times its divisor
#pragma unroll
        for (int off = LANES / 2; off > 0; off >>= 1) {
            fe o;
            o.x[0] = __shfl_down_sync(0xffffffffu, res.x[0], off); o.x[1] = __shfl_down_sync(0xffffffffu, res.x[1], off);
            o.x[2] = __shfl_down_sync(0xffffffffu, res.x[2], off); o.x[3] = __shfl_down_sync(0xffffffffu, res.x[3], off);
            res = fe_add(res, o);
        }
        if (lane != 0) return;
    }
    fe_store(p.out + ci, res);
}

// ------------------------------------------------------------------------------------------------
// K7: TracePolyTable::get_ood_frame — T_j(z), T_j(z*g) for all columns (inside Prover::prove, SURVEY §3.2 step 4)
// polys row-major [n][w]; block c handles rows [c*R, (c+1)*R), thread j handles column j.
// A block of 256 threads = nsub row-chunks x wq columns (wq = power of two >= w); chunk q covers rows [q*R, (q+1)*R).
__global__ void __launch_bounds__(256) k_ood_partial(const fe* __restrict__ polys, uint32_t n, uint32_t w, uint32_t R, uint32_t log_wq,
                                                      const DevTs* __restrict__ ts, fe* __restrict__ part_z, fe* __restrict__ part_zg) {
    const fe z = ts->z, zg = ts->zg, zR = ts->zR, zgR = ts->zgR;   // R must be 64 (k_fs_constraint_root)
    // z^(R c), (zg)^(R c) of each row chunk in the block: one thread per chunk raises z^R to the chunk index (<= 2 log2(n/R)
    // multiplications, against 2 R wq for the chunk itself) instead of the host tabulating n/R powers per proof
    // The chunk itself is a dot product with z^0..z^(R-1) (tabulated once per block, R <= 64) accumulated as exact 288-bit
    // integers and reduced once: no dependent Horner chain, one reduction per chunk instead of one per coefficient.
    __shared__ uint4 zs[2][256];
    __shared__ uint4 zp[2][64];
    const uint32_t j = threadIdx.x & ((1u << log_wq) - 1u), sub = threadIdx.x >> log_wq;
    const uint32_t c = blockIdx.x * (256u >> log_wq) + sub;
    const uint32_t m0 = c * R;
    if (threadIdx.x < R) {
        const fe a = fe_pow_u64(z, threadIdx.x), b = fe_pow_u64(zg, threadIdx.x);
        zp[0][threadIdx.x] = make_uint4(a.x[0], a.x[1], a.x[2], a.x[3]);
        zp[1][threadIdx.x] = make_uint4(b.x[0], b.x[1], b.x[2], b.x[3]);
    }
    if (j == 0 && m0 < n) {
        const fe a = fe_pow_u64(zR, c), b = fe_pow_u64(zgR, c);
        zs[0][sub] = make_uint4(a.x[0], a.x[1], a.x[2], a.x[3]);
        zs[1][sub] = make_uint4(b.x[0], b.x[1], b.x[2], b.x[3]);
    }
    __syncthreads();
    if (j >= w || m0 >= n) return;
    const uint32_t m1 = min(n, m0 + R);
    acc288 az, ag; acc288_zero(az); acc288_zero(ag);
    for (uint32_t m = m0; m < m1; m++) {
        const fe v = fe_load(polys + (size_t)m * w + j);
        fe pz, pg;
        { const uint4 t = zp[0][m - m0]; pz.x[0] = t.x; pz.x[1] = t.y; pz.x[2] = t.z; pz.x[3] = t.w; }
        { const uint4 t = zp[1][m - m0]; pg.x[0] = t.x; pg.x[1] = t.y; pg.x[2] = t.z; pg.x[3] = t.w; }
        acc288_mad(az, v, pz);
        acc288_mad(ag, v, pg);
    }
    fe pa, pb;
    { const uint4 t = zs[0][sub]; pa.x[0] = t.x; pa.x[1] = t.y; pa.x[2] = t.z; pa.x[3] = t.w; }
    { const uint4 t = zs[1][sub]; pb.x[0] = t.x; pb.x[1] = t.y; pb.x[2] = t.z; pb.x[3] = t.w; }
    fe_store(part_z + (size_t)c * w + j, fe_mul(acc288_reduce(az), pa));
    fe_store(part_zg + (size_t)c * w + j, fe_mul(acc288_reduce(ag), pb));
}
// out[j] = sum_c part[c][j]; block = 32 columns x 32 chunk lanes, tree-reduced in shared memory
__global__ void __launch_bounds__(1024) k_col_sum(const fe* __restrict__ part, uint32_t nchunks, uint32_t w, fe* __restrict__ out) {
    __shared__ uint4 red[32][33];
    const uint32_t jx = threadIdx.x, gy = threadIdx.y;
    const uint32_t j = blockIdx.x * 32 + jx;
    fe s = fe_zero();
    if (j < w) for (uint32_t c = gy; c < nchunks; c += 32) s = fe_add(s, fe_load(part + (size_t)c * w + j));
    red[gy][jx] = make_uint4(s.x[0], s.x[1], s.x[2], s.x[3]);
    __syncthreads();
    for (uint32_t h = 16; h > 0; h >>= 1) {
        if (gy < h) {
            uint4 o = red[gy + h][jx];
            fe t; t.x[0] = o.x; t.x[1] = o.y; t.x[2] = o.z; t.x[3] = o.w;
            s = fe_add(s, t);
            red[gy][jx] = make_uint4(s.x[0], s.x[1], s.x[2], s.x[3]);
        }
        __syncthreads();
    }
    if (gy == 0 && j < w) fe_store(out + j, s);
}
// CompositionPoly::evaluate_at: H_i(z) for contiguous coefficient columns [c][n]; one block per column chunk
__global__ void __launch_bounds__(256) k_poly_eval_partial(const fe* __restrict__ coef, uint32_t n, uint32_t Q, const DevTs* __restrict__ ts,
                                                           fe* __restrict__ part) {
    const fe z = ts->z, zQ = ts->zR;   // Q must be 64
    // block handles column blockIdx.y; thread t handles coefficients [t*Q, (t+1)*Q); partial = Horner * z^(t*Q)
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t nt = (n + Q - 1) / Q;
    if (t >= nt) return;
    const fe* c = coef + (size_t)blockIdx.y * n;
    const uint32_t m0 = t * Q, m1 = min(n, m0 + Q);
    fe a = fe_zero();
    for (uint32_t m = m1; m-- > m0;) a = fe_add(fe_mul(a, z), fe_load(c + m));
    fe_store(part + (size_t)t * gridDim.y + blockIdx.y, fe_mul(a, fe_pow_u64(zQ, t)));  // [chunk][column], summed by k_col_sum
}

// ------------------------------------------------------------------------------------------------
// K8: DEEP composition (winter-prover composer; SURVEY A.9), evaluation form:
//   A(x) = sum_j gamma_j T_j(x),  B(x) = sum_i gamma'_i H_i(x)
//   DEEP(x) = (A(x)+B(x) - A(z)-B(z))/(x - z) + (A(x) - A(zg))/(x - zg)
// which equals Winterfell's coefficient-form quotient at every LDE point.
// k_deep_combine: AB[m][0] = A coefficients, AB[m][1] = (A+B) coefficients.  ZKB_ROW_LANES lanes share a coefficient row (its
// elements are consecutive in memory, so the group reads whole 128-byte lines); with a full warp per row the shuffle reduction
// and the H tail on one lane cost more issue slots than the w products they serve (ncu, MiMC 2^20: 1.37 ms for a 1 GiB read).
__global__ void __launch_bounds__(256) k_deep_combine(const fe* __restrict__ polys, uint32_t n, uint32_t w,
                                                      const fe* __restrict__ gamma, const fe* __restrict__ hcoef, uint32_t c,
                                                      const fe* __restrict__ gamma_h, fe* __restrict__ ab) {
    const uint32_t row = (blockIdx.x * blockDim.x + threadIdx.x) / ZKB_ROW_LANES, sub = threadIdx.x & (ZKB_ROW_LANES - 1);
    if (row >= n) return;   // n >= 8: whole warps leave together
    acc288 acc; acc288_zero(acc);
    const fe* pr = polys + (size_t)row * w;
    // four loads in flight per lane: the loop is bound by load latency, not by the products (ncu: long-scoreboard stalls)
    uint32_t j = sub;
    for (; j + 3 * ZKB_ROW_LANES < w; j += 4 * ZKB_ROW_LANES) {
        const fe v0 = fe_load(pr + j), v1 = fe_load(pr + j + ZKB_ROW_LANES), v2 = fe_load(pr + j + 2 * ZKB_ROW_LANES), v3 = fe_load(pr + j + 3 * ZKB_ROW_LANES);
        acc288_mad(acc, v0, fe_ldg(gamma + j));
        acc288_mad(acc, v1, fe_ldg(gamma + j + ZKB_ROW_LANES));
        acc288_mad(acc, v2, fe_ldg(gamma + j + 2 * ZKB_ROW_LANES));
        acc288_mad(acc, v3, fe_ldg(gamma + j + 3 * ZKB_ROW_LANES));
    }
    for (; j < w; j += ZKB_ROW_LANES) acc288_mad(acc, fe_load(pr + j), fe_ldg(gamma + j));
    acc288 hacc; acc288_zero(hacc);
    for (uint32_t i = sub; i < c; i += ZKB_ROW_LANES) acc288_mad(hacc, fe_load(hcoef + (size_t)i * n + row), fe_ldg(gamma_h + i));
    const fe s = fe_group_sum(acc288_reduce(acc));
    const fe b = c ? fe_group_sum(acc288_reduce(hacc)) : fe_zero();
    if (sub == 0) {
        fe_store(ab + (size_t)row * 2, s);
        fe_store(ab + (size_t)row * 2 + 1, fe_add(s, b));
    }
}
// k_deep_eval: each thread handles ZKB_DEEP_RPT rows (one Montgomery batch inversion per thread); RPT = 1 for domains of a
// few thousand rows, where the proof waits for one thread's chain (inversion + 6 multiplications per extra row), not for throughput
#define ZKB_DEEP_RPT 8
// compact = 1 (coset-sharded AB matrix): out index = i * (stored cosets) + local coset, else the natural position i*beta + k
template <int RPT>
__global__ void __launch_bounds__(128) k_deep_eval(const LdeMat m, const DevTs* __restrict__ ts, PowTab roots, uint32_t log_tab,
                                                   fe* __restrict__ out, uint32_t compact) {
    const fe z = ts->z, zg = ts->zg, abz = ts->abz, azg = ts->azg;
    const uint32_t log_N = m.log_n + m.log_beta;
    const uint64_t N = (uint64_t)1 << (m.log_n + m.log_kc);   // rows stored
    const uint64_t nthreads = N / RPT;
    const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (tid >= nthreads) return;
    const uint32_t lt = m.log_n - m.log_p;
    fe d[2 * RPT], pre[2 * RPT], n1[RPT], n2[RPT];
    uint32_t rr[RPT];
    fe acc = fe_one();
#pragma unroll
    for (int s = 0; s < RPT; s++) {
        const uint64_t gid = tid + (uint64_t)s * nthreads;
        const uint32_t slot = (uint32_t)gid & ((1u << m.log_p) - 1u);
        const uint32_t panel = (uint32_t)(gid >> m.log_p);
        const uint32_t k = m.k0 + (panel >> lt), t_low = panel & ((1u << lt) - 1u);
        const uint32_t i = t_low + (slot << lt);
        const uint32_t r = (i << m.log_beta) + k;
        rr[s] = compact ? ((i << m.log_kc) + (k - m.k0)) : r;
        const fe* row = m.data + (((size_t)panel * 2) << m.log_p) + slot;
        fe a = fe_load(row), ab = fe_load(row + ((size_t)1 << m.log_p));
        fe x = powtab(roots, r << (log_tab - log_N));
        { fe x2 = fe_add(x, x); x = fe_add(x2, x); }
        n1[s] = fe_sub(ab, abz);
        n2[s] = fe_sub(a, azg);
        d[2 * s] = fe_sub(x, z);
        d[2 * s + 1] = fe_sub(x, zg);
        pre[2 * s] = acc; acc = fe_mul(acc, d[2 * s]);
        pre[2 * s + 1] = acc; acc = fe_mul(acc, d[2 * s + 1]);
    }
    fe ia = fe_inv(acc);
#pragma unroll
    for (int s = RPT - 1; s >= 0; s--) {
        fe i2 = fe_mul(ia, pre[2 * s + 1]); ia = fe_mul(ia, d[2 * s + 1]);
        fe i1 = fe_mul(ia, pre[2 * s]); ia = fe_mul(ia, d[2 * s]);
        fe_store(out + rr[s], fe_add(fe_mul(n1[s], i1), fe_mul(n2[s], i2)));
    }
}

// ------------------------------------------------------------------------------------------------
// K9: FRI degree-respecting projection with folding factor F = 2^LOG_F in {2, 4, 8, 16} (winter-fri folding::apply_drp;
// ProofOptions accepts these four).  next[i] = p_i(alpha), p_i interpolating (x_i w_F^j, e[i + j*rows]), rows = M / F,
// x_i = 3 * w_M^i  — the offset 3 is NOT raised to the F-th power between layers (SURVEY A.10).
struct FriFoldParams {
    const fe* in; fe* out;
    uint32_t log_m;            // current domain size M = 2^log_m
    const fe* alpha;           // the layer's folding challenge (device transcript)
    fe inv3, inv_f;            // 1/3, 1/F
    fe wf_inv[8];              // w_F^{-k}, k = 0..F/2-1
    PowTab roots; uint32_t log_tab;
};
// One row of the projection, shared by the prover (k_fri_fold) and the verifier (k_v_eval): load(j) = the row's element at
// x_i w_F^j, wf_inv(k) = w_F^{-k} (k < F/2), alpha_over_x() = alpha / x_i, inv_f = 1/F; store(v) receives p(alpha).  The loads,
// the twiddles, alpha / x_i and the store are callables so that each kernel keeps its own addressing and the prover's
// instructions are what they were before the split.
template <int LOG_F, class Load, class WfInv, class AlphaOverX, class Store>
__device__ __forceinline__ void fri_fold_row(Load load, WfInv wf_inv, AlphaOverX alpha_over_x, const fe& inv_f, Store store) {
    constexpr int F = 1 << LOG_F;
    fe v[F];
    // bit-reversed load for an in-register DIT inverse DFT (__brev folds to a constant per unrolled j; a shift-and-or loop
    // for the reversal changes the register allocation of the F = 16 instance: 100 registers and 30 more instructions)
#pragma unroll
    for (int j = 0; j < F; j++) {
        const int br = (int)(__brev((unsigned)j) >> (32 - LOG_F));
        v[br] = load(j);
    }
#pragma unroll
    for (int lam = 1; lam <= LOG_F; lam++) {
        const int half = 1 << (lam - 1);
#pragma unroll
        for (int q = 0; q < F / 2; q++) {
            const int th = q & (half - 1);
            const int p0 = ((q >> (lam - 1)) << lam) + th;
            fe u = v[p0];
            fe t = th == 0 ? v[p0 + half] : fe_mul(v[p0 + half], wf_inv(th * ((F / 2) >> (lam - 1))));
            v[p0] = fe_add(u, t);
            v[p0 + half] = fe_sub(u, t);
        }
    }
    // p(alpha) = (1/F) sum_k c_k (alpha / x_i)^k
    const fe t = alpha_over_x();
    fe acc = v[F - 1];
#pragma unroll
    for (int kq = F - 2; kq >= 0; kq--) acc = fe_add(fe_mul(acc, t), v[kq]);
    store(fe_mul(acc, inv_f));
}
template <int LOG_F>
__global__ void __launch_bounds__(128) k_fri_fold(const FriFoldParams p) {
    constexpr int F = 1 << LOG_F;
    static_assert(LOG_F >= 1 && F / 2 <= (int)(sizeof(p.wf_inv) / sizeof(fe)), "folding factor out of range");
    const uint64_t rows = ((uint64_t)1 << p.log_m) >> LOG_F;
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows) return;
    fe* const out = p.out + i;   // formed before the row fold: this keeps the address arithmetic where the unfactored kernel had it
    fri_fold_row<LOG_F>([&](int j) { return fe_load(p.in + i + (uint64_t)j * rows); }, [&](int k) { return p.wf_inv[k]; }, [&] {
        // 1/x_i = (1/3) w_M^{-i}
        const uint32_t tab_mask = (1u << p.log_tab) - 1u;
        const uint32_t e = (0u - ((uint32_t)i << (p.log_tab - p.log_m))) & tab_mask;
        return fe_mul(fe_mul(fe_ldg(p.alpha), p.inv3), powtab(p.roots, e));
    }, p.inv_f, [&](const fe& r) { fe_store(out, r); });
}

// ------------------------------------------------------------------------------------------------
// K11: TraceLde::query / ConstraintCommitment::query — gather LDE rows at the query positions (row-major out)
__global__ void k_gather_lde_rows(const LdeMat m, const uint32_t* __restrict__ pos, uint32_t npos, fe* __restrict__ out) {
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= npos * m.w) return;
    const uint32_t q = idx / m.w, j = idx - q * m.w;
    const uint32_t r = __ldg(pos + q);
    const uint32_t k = r & ((1u << m.log_beta) - 1u), i = r >> m.log_beta;
    if (k - m.k0 >= (1u << m.log_kc)) { fe_store(out + idx, fe_zero()); return; }   // coset held by another rank
    fe_store(out + idx, fe_load(m.data + lde_addr(m, k, i, j)));
}
// Openings in ONE launch (blockIdx.y + first = commitment): rows at the raw query positions plus the full authentication path
// of each, because for small proofs every launch is a measurable part of the latency.  Commitments 0, 1: LDE matrices (trace,
// constraint composition); 2 + l: FRI layer l, rows [e[p + j*rows]]_{j<F} (folding a position is p mod rows).
// Sharded proofs: an entry this rank does not hold is written as zeros, every other entry is the same on all ranks, so a
// byte-wise max over the ranks assembles the openings.  Trace rows and the path levels below lsub belong to the rank that owns
// the queried row (r >> lsub); the levels at or above lsub are read from the replicated cap heap.  A composition row is held
// by the rank that stores its coset.
#define ZKB_MAX_OPEN (2 + ZKB_MAX_FRI_LAYERS)
struct OpenJobs {
    uint32_t first, q;
    const uint32_t* pos;                 // raw positions (device transcript)
    LdeMat mat[2];
    const fe* fri_evals[ZKB_MAX_OPEN - 2];
    uint64_t fri_rows[ZKB_MAX_OPEN - 2];
    const uint32_t* heap[ZKB_MAX_OPEN];
    uint32_t depth[ZKB_MAX_OPEN], width[ZKB_MAX_OPEN];
    fe* rows_out[ZKB_MAX_OPEN];
    uint32_t* paths_out[ZKB_MAX_OPEN];
    const uint32_t* cap;                 // trace commitment: heap of the top depth - lsub levels (one GPU: lsub = depth)
    uint32_t lsub, rank;                 // trace commitment: log2 rows per rank, this rank
};
static_assert(sizeof(OpenJobs) <= 4096, "k_open_all takes OpenJobs by value: it must fit the 4 KiB of kernel parameters");
__global__ void __launch_bounds__(128) k_open_all(const OpenJobs J) {
    const uint32_t t = blockIdx.y + J.first;
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t w = J.width[t], depth = J.depth[t];
    const uint32_t nrow = J.q * w, npath = J.q * depth * 2;
    if (idx < nrow) {
        const uint32_t q = idx / w, j = idx - q * w;
        const uint32_t r = __ldg(J.pos + q);
        if (t < 2) {
            const LdeMat& m = J.mat[t];
            const uint32_t k = r & ((1u << m.log_beta) - 1u), i = r >> m.log_beta;
            const bool held = k - m.k0 < (1u << m.log_kc) && (t != 0 || (r >> J.lsub) == J.rank);
            fe_store(J.rows_out[t] + idx, held ? fe_load(m.data + lde_addr(m, k, i, j)) : fe_zero());
        } else {
            const uint64_t rows = J.fri_rows[t - 2];
            fe_store(J.rows_out[t] + idx, fe_load(J.fri_evals[t - 2] + (r & (uint32_t)(rows - 1)) + (uint64_t)j * rows));
        }
    } else if (idx - nrow < npath) {
        const uint32_t tt = idx - nrow;
        const uint32_t half = tt & 1u, ql = tt >> 1, q = ql / depth, level = ql - q * depth;
        const uint32_t r = __ldg(J.pos + q) & ((1u << depth) - 1u);
        const uint32_t lsub = t == 0 ? J.lsub : depth;
        uint4 v = make_uint4(0, 0, 0, 0);
        if (level >= lsub) {   // the top levels of a heap coincide with the heap of its cap
            const uint64_t node = ((((uint64_t)1 << depth) + r) >> level) ^ 1ull;
            v = reinterpret_cast<const uint4*>(J.cap)[node * 2 + half];
        } else if (t != 0 || (r >> lsub) == J.rank) {
            const uint64_t node = ((((uint64_t)1 << lsub) + (r & ((1u << lsub) - 1u))) >> level) ^ 1ull;
            v = reinterpret_cast<const uint4*>(J.heap[t])[node * 2 + half];
        }
        reinterpret_cast<uint4*>(J.paths_out[t])[tt] = v;
    }
}

// ------------------------------------------------------------------------------------------------
// multi-GPU: out[i] = sum_g parts[g * stride + i]  (field sum of per-rank partial vectors after an all-gather;
// NCCL has no mod-p reduction for 128-bit elements)
__global__ void k_sum_partials(const fe* __restrict__ parts, uint32_t g, uint64_t stride, uint64_t n, fe* __restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fe s = fe_load(parts + i);
    for (uint32_t q = 1; q < g; q++) s = fe_add(s, fe_load(parts + (uint64_t)q * stride + i));
    fe_store(out + i, s);
}
// multi-GPU DEEP: ab[m][1] += sum_i gamma'_i H_i[m]   (ab[m][0] = ab[m][1] = A[m] on entry)
__global__ void k_deep_add_h(fe* __restrict__ ab, uint32_t n, const fe* __restrict__ hcoef, uint32_t c, const fe* __restrict__ gamma_h) {
    const uint32_t m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n) return;
    fe b = fe_zero();
    for (uint32_t i = 0; i < c; i++) b = fe_add(b, fe_mul(fe_load(hcoef + (size_t)i * n + m), fe_ldg(gamma_h + i)));
    fe_store(ab + (size_t)m * 2 + 1, fe_add(fe_load(ab + (size_t)m * 2 + 1), b));
}

// device-side MiMC chain trace (SURVEY §8f rank 2): col_j[0] = seed_j, col_j[i+1] = (col_j[i] + rc[i mod L])^7
// round function from src/helper.rs:213-220, constants from :404-406; output column-major [w][n]
__global__ void k_mimc_trace(const fe* __restrict__ seeds, uint32_t w, uint64_t n, const fe* __restrict__ rc, uint32_t L, fe* __restrict__ out) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= w) return;
    fe x = fe_canon(fe_load(seeds + j), 0);
    for (uint64_t i = 0; i < n; i++) {
        fe_store(out + (size_t)j * n + i, x);
        fe a1 = fe_add(x, fe_canon(fe_ldg(rc + (i & (L - 1))), 0));
        fe a2 = fe_sqr(a1), a4 = fe_sqr(a2), a6 = fe_mul(a4, a2);
        x = fe_mul(a6, a1);
    }
}

// device-side training trace (SURVEY §8f rank 2; src/training/prover.rs:117-130,188-199): row i = [raw_i + mask_i || mask_i] with
// a fresh 64-bit mask per cell.  The raw state only changes during the first `n_raw - 1` steps (the batch), afterwards it is
// constant (src/training/prover.rs:185), so the caller uploads n_raw rows of `half` raw values and the masks are generated
// here.  The masks are the only thing hiding the raw model state (masked rows 0 and n-1 are public inputs), and the
// reference draws them from rand::thread_rng(), an OS-seeded ChaCha CSPRNG: so do we — ChaCha20 keystream under a 256-bit
// key (drawn from OS entropy by the host unless the caller passes one), block counter = row * blocks_per_row + column block,
// eight 64-bit masks per 64-byte block.  Output: column-major [2*half][n].
__device__ __forceinline__ void chacha20_block(const uint32_t key[8], uint64_t counter, uint32_t out[16]) {
    uint32_t x[16] = {0x61707865u, 0x3320646eu, 0x79622d32u, 0x6b206574u, key[0], key[1], key[2], key[3], key[4], key[5], key[6], key[7],
                      (uint32_t)counter, (uint32_t)(counter >> 32), 0u, 0u};
    uint32_t s[16];
#pragma unroll
    for (int i = 0; i < 16; i++) s[i] = x[i];
#define ZKB_QR(a, b, c, d)                                                                     \
    x[a] += x[b]; x[d] = __funnelshift_l(x[d] ^ x[a], x[d] ^ x[a], 16); x[c] += x[d]; x[b] = __funnelshift_l(x[b] ^ x[c], x[b] ^ x[c], 12); \
    x[a] += x[b]; x[d] = __funnelshift_l(x[d] ^ x[a], x[d] ^ x[a], 8);  x[c] += x[d]; x[b] = __funnelshift_l(x[b] ^ x[c], x[b] ^ x[c], 7);
#pragma unroll
    for (int r = 0; r < 10; r++) {
        ZKB_QR(0, 4, 8, 12) ZKB_QR(1, 5, 9, 13) ZKB_QR(2, 6, 10, 14) ZKB_QR(3, 7, 11, 15)
        ZKB_QR(0, 5, 10, 15) ZKB_QR(1, 6, 11, 12) ZKB_QR(2, 7, 8, 13) ZKB_QR(3, 4, 9, 14)
    }
#undef ZKB_QR
#pragma unroll
    for (int i = 0; i < 16; i++) out[i] = x[i] + s[i];
}
struct ChaChaKey { uint32_t k[8]; };
__global__ void k_training_trace(const fe* __restrict__ raw, uint32_t n_raw, uint32_t half, uint64_t n, const ChaChaKey key, fe* __restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t jb = blockIdx.y, nb = gridDim.y;   // column block: masks of columns [8 jb, 8 jb + 8)
    if (i >= n) return;
    uint32_t ks[16];
    chacha20_block(key.k, i * nb + jb, ks);
    const uint64_t r = i < n_raw ? i : (uint64_t)n_raw - 1;
#pragma unroll
    for (int q = 0; q < 8; q++) {
        const uint32_t j = jb * 8 + q;
        if (j >= half) break;
        fe mask; mask.x[0] = ks[2 * q]; mask.x[1] = ks[2 * q + 1]; mask.x[2] = mask.x[3] = 0;
        fe_store(out + (size_t)j * n + i, fe_add(fe_canon(fe_load(raw + r * half + j), 0), mask));
        fe_store(out + (size_t)(half + j) * n + i, mask);
    }
}
// read two rows of a column-major device trace (boundary rows for get_pub_inputs)
__global__ void k_read_rows(const fe* __restrict__ trace, uint32_t w, uint64_t n, uint64_t r0, uint64_t r1, fe* __restrict__ out) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= w) return;
    fe_store(out + j, fe_load(trace + (size_t)j * n + r0));
    fe_store(out + w + j, fe_load(trace + (size_t)j * n + r1));
}

// batched MiMC helpers of the reference: mimc_cipher (src/helper.rs:213-220) and mimc_hash_matrix (:222-233), one thread
// per instance — the GPU counterpart of benches/bench_mimc.rs:17-57
__device__ __forceinline__ fe mimc_cipher_dev(fe inp, const fe rc, const fe z) {
    const fe k = fe_add(rc, z);
    for (int r = 0; r < 64; r++) {
        fe a1 = fe_add(inp, k);
        fe a2 = fe_sqr(a1), a4 = fe_sqr(a2), a6 = fe_mul(a4, a2);
        inp = fe_mul(a6, a1);
    }
    return fe_add(inp, z);
}
__global__ void k_mimc_cipher_batch(const fe* __restrict__ x, const fe* __restrict__ rc, const fe* __restrict__ z, uint64_t n, fe* __restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fe_store(out + i, mimc_cipher_dev(fe_canon(fe_load(x + i), 0), fe_canon(fe_load(rc + i), 0), fe_canon(fe_load(z + i), 0)));
}
// w: [count][ac][fe], b: [count][ac]
__global__ void k_mimc_hash_matrix_batch(const fe* __restrict__ w, const fe* __restrict__ b, uint32_t ac, uint32_t fe_n, const fe* __restrict__ rc,
                                         uint32_t n_rc, uint64_t count, fe* __restrict__ out) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    fe z = fe_zero();
    for (uint32_t i = 0; i < ac; i++) {
        for (uint32_t j = 0; j < fe_n; j++) z = mimc_cipher_dev(fe_canon(fe_load(w + (t * ac + i) * fe_n + j), 0), fe_canon(fe_ldg(rc + j % n_rc), 0), z);
        z = mimc_cipher_dev(fe_canon(fe_load(b + t * ac + i), 0), fe_canon(fe_ldg(rc + i % n_rc), 0), z);
    }
    fe_store(out + t, z);
}

// elementwise kernels used by tests (KATs of the device field / hash against the oracle)
__global__ void k_test_field(const fe* a, const fe* b, fe* mul, fe* add, fe* sub, fe* inv, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fe x = fe_load(a + i), y = fe_load(b + i);
    fe m = fe_mul(x, y);
    {   // the lazy 288-bit accumulator and the dedicated squaring must agree with reduce-every-product arithmetic;
        // a disagreement poisons the product the host checks
        acc288 acc; acc288_zero(acc);
        acc288_mad(acc, x, y); acc288_mad(acc, y, x); acc288_mad(acc, x, x); acc288_mad(acc, y, y); acc288_mad(acc, x, y);
        const fe want = fe_add(fe_add(fe_add(m, m), m), fe_add(fe_mul(x, x), fe_mul(y, y)));
        const fe sq = fe_add(fe_sqr(x), fe_sqr(y));
        if (!fe_eq(acc288_reduce(acc), want) || !fe_eq(sq, fe_add(fe_mul(x, x), fe_mul(y, y)))) m.x[0] ^= 0xDEADBEEFu;
    }
    fe_store(mul + i, m); fe_store(add + i, fe_add(x, y)); fe_store(sub + i, fe_sub(x, y));
    fe_store(inv + i, fe_inv(x));
}
__global__ void k_test_hash(const fe* data, uint32_t count, uint32_t nrows, uint32_t* out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nrows) return;
    uint32_t d[8];
    b3_hash_elems(data + (size_t)i * count, 1, count, d, 256, 256, 0);
    for (int q = 0; q < 8; q++) out[i * 8 + q] = d[q];
}

}  // namespace zkb
