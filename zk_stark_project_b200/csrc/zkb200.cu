// libzkb200.so — B200-native STARK proving backend behind the C ABI of include/zkb200.h.
//
// This file is the host-side driver: it owns device memory, plans the NTT passes, issues the kernels of
// kernels.cuh on the context's stream and runs the Fiat-Shamir channel between stages (a 32-byte root
// up, a 16-byte challenge down).  It re-composes Winterfell 0.12's `Prover::prove` / `generate_proof`
// (driven by the reference at /root/reference src/main.rs:228,424,468 through the Prover impls at
// src/training/prover.rs:221-301 and src/aggregation/prover.rs:194-249) with every stage on the GPU.
// There is no CPU fallback: without a CUDA device every entry point fails.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <sys/random.h>
#include <nccl.h>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <functional>
#include <map>
#include <mutex>
#include <thread>
#include <tuple>
#include <memory>
#include "kernels.cuh"
#include "verify.cuh"
#include "host.hpp"

namespace zkb {

struct CudaError : std::runtime_error { using std::runtime_error::runtime_error; };
struct StateError : std::runtime_error { using std::runtime_error::runtime_error; };

#define CK(call)                                                                                              \
    do {                                                                                                      \
        cudaError_t e_ = (call);                                                                              \
        if (e_ != cudaSuccess)                                                                                \
            throw CudaError(std::string(#call) + " failed: " + cudaGetErrorString(e_) + " (" + __FILE__ + ":" + \
                            std::to_string(__LINE__) + ")");                                                  \
    } while (0)

static thread_local std::string g_last_error;

}  // namespace zkb
#include "nccl_loader.hpp"
namespace zkb {

// bumped whenever any device buffer is (re)allocated or released: a captured CUDA graph holds raw device addresses and is only
// replayed while the epoch it was captured in is still current
static std::atomic<uint64_t> g_alloc_epoch{1};

#define ZKB_CAP_BYTES 4096   // 2 G digests of the replicated Merkle cap of a sharded trace commitment (G <= 64)
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    void ensure(size_t bytes) {
        if (bytes <= cap) return;
        g_alloc_epoch++;
        if (p) { cudaFree(p); p = nullptr; cap = 0; }
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) { p = nullptr; throw CudaError(std::string("cudaMalloc of ") + std::to_string(bytes) + " bytes failed: " + cudaGetErrorString(e)); }
        cap = bytes;
    }
    void release() { if (p) { cudaFree(p); g_alloc_epoch++; } p = nullptr; cap = 0; }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

// Device tables kept per shape (twiddles, evaluator inputs, divisors), so that captured graphs of several shapes stay valid
// side by side.  A long-lived context that has seen many shapes would hold them all: an entry that does not fit the budget
// next to the others releases every entry first (after the stream is done with them) and the cache starts over.
template <class Key>
struct ShapeCache {
    std::map<Key, DevBuf> map;
    size_t bytes = 0;
    const size_t budget;
    explicit ShapeCache(size_t budget_bytes) : budget(budget_bytes) {}
    DevBuf* find(const Key& k) {
        auto it = map.find(k);
        return it == map.end() ? nullptr : &it->second;
    }
    bool full(size_t size) const { return bytes + size > budget && !map.empty(); }
    DevBuf& insert(const Key& k, size_t size, cudaStream_t stream) {
        if (full(size)) {
            CK(cudaStreamSynchronize(stream));
            release();
        }
        DevBuf& b = map[k];
        try { b.ensure(size); } catch (...) { map.erase(k); throw; }   // no entry without memory behind it
        bytes += size;
        return b;
    }
    void release() {
        for (auto& kv : map) kv.second.release();
        map.clear();
        bytes = 0;
    }
};

static inline fe to_fe(const HF& h) {
    fe r;
    r.x[0] = (uint32_t)h.v; r.x[1] = (uint32_t)(h.v >> 32); r.x[2] = (uint32_t)(h.v >> 64); r.x[3] = (uint32_t)(h.v >> 96);
    return r;
}

enum Stage { ST_IDLE = 0, ST_BEGUN, ST_TRACE, ST_EVAL, ST_COMP, ST_OOD, ST_DEEP, ST_FRI_DONE, ST_QUERY };

}  // namespace zkb

using namespace zkb;

struct zkb_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    std::string err;
    uint64_t launches = 0;
    uint64_t h2d_bytes = 0;   // host-to-device bytes copied by this context's calls (zkb_h2d_bytes)
    int sm_count = 148;

    // ---- per-proof state -------------------------------------------------------------------------------------
    AirSpec air;
    Stage stage = ST_IDLE;
    uint32_t log_n = 0, log_beta = 0, log_N = 0, log_ce = 0, c = 0;
    uint32_t log_tab = 0;  // root table domain (= LDE domain)
    HostCoin coin;
    ProofParts parts;
    zkb_transcript ts;
    zkb_stage_times times;
    HF z, zg, deep_alpha;
    std::vector<HF> ood_cur, ood_next, ood_h;
    uint32_t fri_layer = 0, fri_layers = 0;
    bool fri_committed = false;
    std::vector<uint32_t> positions;

    // ---- device memory (grown on demand, reused between proofs) ----------------------------------------------
    DevBuf d_trace, d_bufA, d_bufB, d_tmp1, d_tmp2, d_lde, d_tree, d_small, d_comp_evals, d_comp_lde, d_comp_tree, d_ab, d_ab_lde,
        d_deep, d_roots_lo, d_roots_hi, d_inv3_lo, d_inv3_hi, d_pow3, d_aux, d_gather, d_user_trace, d_flags;
    std::vector<DevBuf> d_fri_evals, d_fri_tree;
    fe* d_polys = nullptr;  // points into bufA or bufB
    uint32_t lde_log_p = 0, comp_log_p = 0, ab_log_p = 0;
    uint32_t tab_log_built = 0, pow3_for_log_n = 0, pow3_for_beta = 0;
    PowTab roots{}, inv3tab{};
    uint32_t inv3_l1 = 0;
    // per-stage CUDA events; elapsed times are collected lazily (no host synchronisation inside a proof just for timing)
    enum { TS_LDE, TS_XCHG, TS_LEAF, TS_MERKLE, TS_CONSTR, TS_COMP, TS_OOD, TS_DEEP, TS_FRI, TS_GRIND, TS_QUERY, TS_TOTAL, TS_COUNT };
    cudaEvent_t tev[TS_COUNT][2];
    bool trec[TS_COUNT] = {};
    bool times_valid = true;
    // pinned host staging for the small per-stage uploads (coefficients, challenges, positions): truly asynchronous H2D
    uint8_t* h_stage = nullptr;
    size_t h_stage_cap = 0, h_stage_used = 0;
    // MiMC periodic-column table over the ce domain, cached across proofs of the same shape
    std::vector<HF> per_cache, per_cache_params;
    uint64_t per_cache_n = 0, per_cache_ce = 0;
    cudaEvent_t ev_group[17];          // per column group: "H2D of this group has landed"
    cudaStream_t copy_stream = nullptr;  // trace ingest overlaps the NTTs of earlier column groups
    bool owns_stream = false;            // zkb_ctx_create_lane: `stream` was created by the context
    cudaStream_t xchg_stream = nullptr;  // sharded proofs: the NVLink all-to-all of finished coset batches overlaps the LDE of the next
    bool ev_ok = false;

    // ---- multi-GPU (column-sharded single proof) -----------------------------------------------------------------
    ncclComm_t comm = nullptr;
    int mg_rank = 0, mg_world = 1;
    uint32_t log_g = 0;
    bool mg_active = false;             // the proof in flight is sharded
    DevBuf d_bnd_coef, d_bnd_lde;       // boundary numerators as polynomials (constraints_eval_window)

    // ---- device-resident Fiat-Shamir transcript (csrc/coin.cuh) and the openings gathered for the final download -------
    // d_fs = [DevTs][OOD frame 2w+c][remainder][per commitment: queried rows, full authentication paths] | device-only:
    // [coefficient powers nt+na][DEEP gammas w+c][scratch 2w].  The first `host_bytes` travel to the host in ONE copy at the
    // end of a proof; nothing else crosses PCIe after the trace went up.
    struct FsTree { size_t o_rows, o_paths; uint32_t width, depth; };
    struct FsLayout { size_t o_ood = 0, o_rem = 0, host_bytes = 0, o_coef = 0, o_gamma = 0, o_scr = 0, total = 0; uint32_t rem_cap = 0; std::vector<FsTree> trees; } fs;
    DevBuf d_fs, d_in, d_rem_coef;      // d_in: per-proof inputs [assertion values na][AIR params]
    // shape-only evaluator inputs (periodic column, assertion columns / indices) and divisor tables (k_build_divisors)
    ShapeCache<std::string> pack_cache{(size_t)64 << 20};
    ShapeCache<std::vector<uint64_t>> div_cache{(size_t)2 << 30};
    // ---- CUDA graphs for small proofs: the whole enqueue sequence of a shape, replayed with one launch ---------------------
    struct GraphEntry { cudaGraphExec_t exec = nullptr; uint64_t epoch = 0; uint32_t seen = 0; uint64_t launches = 0; };
    std::map<std::string, GraphEntry> graphs;
    bool capturing = false;
    uint8_t* h_out = nullptr;           // pinned landing area of the final download
    size_t h_out_cap = 0;
    cudaEvent_t ev_done = nullptr;      // blocking-sync event: the host thread sleeps instead of spinning while the device works
    DevTs* dts() const { return d_fs.as<DevTs>(); }
    fe* fs_fe(size_t off) const { return reinterpret_cast<fe*>(d_fs.as<uint8_t>() + off); }
    const fe* d_aval() const { return d_in.as<fe>(); }
    const fe* d_params() const { return d_in.as<fe>() + air.assertions.size(); }
    DevBuf d_lde_rows, d_mg_a, d_mg_b;  // recv view of the LDE; all-gather staging
    DevBuf d_cap;                       // sharded trace commitment: heap of the replicated top log G levels, cap[1] = root
    // ---- batch verification (csrc/verify.cuh): staging of the parsed proofs, the plan, the channel's draws, computed digests ----
    DevBuf d_vstage, d_vplan, d_vts, d_vdig;
    uint8_t* h_vstage = nullptr;        // pinned, grown on demand
    size_t h_vstage_cap = 0;
    uint8_t* h_vplan = nullptr;
    size_t h_vplan_cap = 0;

    // ==========================================================================================================
    void count() { launches++; }
    static uint32_t magic16(uint32_t d) { return (65536u + d - 1) / d; }
    LdeMat std_mat(fe* data, uint32_t w, uint32_t log_p) const { return LdeMat{data, log_n, log_beta, w, log_p, 0, w, magic16(w), 0, 0, 0, 0, log_beta}; }
    // coset-sharded matrices of a multi-GPU proof (composition columns, DEEP pair): rank r stores cosets [r*kc, (r+1)*kc)
    bool mg_coset() const { return mg_active && (uint32_t)mg_world <= air.blowup; }
    uint32_t mg_log_kc() const { return log_beta - log_g; }
    LdeMat coset_mat(fe* data, uint32_t w, uint32_t log_p) const {
        LdeMat m = std_mat(data, w, log_p);
        if (mg_coset()) { m.log_kc = mg_log_kc(); m.k0 = (uint32_t)mg_rank << m.log_kc; }
        return m;
    }
    // single GPU: the whole trace LDE; multi-GPU: the send view (this rank's columns, all rows)
    LdeMat lde_mat() const {
        if (!mg_active) return std_mat(d_lde.as<fe>(), air.w, lde_log_p);
        const uint32_t wl = air.w / (uint32_t)mg_world;
        return LdeMat{d_lde.as<fe>(), log_n, log_beta, wl, lde_log_p - log_g, log_g, wl, magic16(wl), 0, (uint32_t)mg_rank, 0, 0, log_beta};
    }
    // multi-GPU recv view: all columns, this rank's rows
    LdeMat lde_rows_mat() const {
        const uint32_t wl = air.w / (uint32_t)mg_world, lp = lde_log_p - log_g;
        const uint64_t np = (uint64_t)1 << (log_beta + log_n - lde_log_p);
        return LdeMat{d_lde_rows.as<fe>(), log_n, log_beta, air.w, lp, log_g, wl, magic16(wl), 1, (uint32_t)mg_rank, (np * wl) << lp, 0, log_beta};
    }
    LdeMat comp_mat() const { return coset_mat(d_comp_lde.as<fe>(), c, comp_log_p); }
    LdeMat ab_mat() const { return coset_mat(d_ab_lde.as<fe>(), 2, ab_log_p); }

    void init(int dev, void* strm) {
        int ndev = 0;
        cudaError_t e = cudaGetDeviceCount(&ndev);
        if (e != cudaSuccess || ndev == 0) throw CudaError(std::string("no CUDA device available: ") + cudaGetErrorString(e));
        if (dev < 0 || dev >= ndev) throw InvalidArg("device index out of range");
        device = dev;
        CK(cudaSetDevice(device));
        stream = (cudaStream_t)strm;
        cudaDeviceProp prop;
        CK(cudaGetDeviceProperties(&prop, device));
        sm_count = prop.multiProcessorCount;
        CK(cudaFuncSetAttribute(k_ntt_pass<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        CK(cudaFuncSetAttribute(k_ntt_pass<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        for (auto& pr : tev) for (auto& x : pr) CK(cudaEventCreate(&x));
        h_stage_cap = (size_t)8 << 20;
        CK(cudaHostAlloc((void**)&h_stage, h_stage_cap, cudaHostAllocDefault));
        for (auto& x : ev_group) CK(cudaEventCreateWithFlags(&x, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ev_done, cudaEventBlockingSync | cudaEventDisableTiming));
        CK(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking));
        {   // highest priority: the exchange's few blocks must get SM slots as soon as LDE blocks retire
            int lo = 0, hi = 0;
            CK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
            CK(cudaStreamCreateWithPriority(&xchg_stream, cudaStreamNonBlocking, hi));
        }
        ev_ok = true;
        memset(&times, 0, sizeof(times));
    }
    void destroy() {
        cudaSetDevice(device);
        cudaStreamSynchronize(stream);
        for (DevBuf* b : {&d_trace, &d_bufA, &d_bufB, &d_tmp1, &d_tmp2, &d_lde, &d_tree, &d_small, &d_comp_evals, &d_comp_lde, &d_comp_tree,
                          &d_ab, &d_ab_lde, &d_deep, &d_roots_lo, &d_roots_hi, &d_inv3_lo, &d_inv3_hi, &d_pow3, &d_aux, &d_gather, &d_user_trace, &d_flags,
                          &d_lde_rows, &d_mg_a, &d_mg_b, &d_cap, &d_bnd_coef, &d_bnd_lde, &d_fs, &d_in, &d_rem_coef, &d_vstage, &d_vplan,
                          &d_vts, &d_vdig})
            b->release();
        if (comm) { g_nccl.CommDestroy(comm); comm = nullptr; }
        for (auto& b : d_fri_evals) b.release();
        for (auto& b : d_fri_tree) b.release();
        tw_cache.release();
        pack_cache.release();
        div_cache.release();
        for (auto& kv : graphs) if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
        if (ev_ok) { for (auto& pr : tev) for (auto& x : pr) cudaEventDestroy(x); for (auto& x : ev_group) cudaEventDestroy(x); cudaStreamDestroy(copy_stream); cudaStreamDestroy(xchg_stream); }
        if (h_stage) cudaFreeHost(h_stage);
        if (h_out) cudaFreeHost(h_out);
        if (h_vstage) cudaFreeHost(h_vstage);
        if (h_vplan) cudaFreeHost(h_vplan);
        if (ev_done) cudaEventDestroy(ev_done);
        if (owns_stream && stream) { cudaStreamDestroy(stream); stream = nullptr; }
    }

    void h2d(void* dst, const void* src, size_t bytes) { CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream)); h2d_bytes += bytes; }
    // small upload through the pinned staging area: returns immediately, `src` may be released right away.  The area is
    // rewound at the start of every proof (every proof ends with a stream synchronisation).
    void h2d_small(void* dst, const void* src, size_t bytes) {
        if (bytes == 0) return;
        h2d_bytes += bytes;
        const size_t need = (bytes + 255) & ~(size_t)255;
        if (h_stage_used + need > h_stage_cap) {  // does not fit: plain (staged by the driver) copy, then wait so `src` can go away
            CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream));
            CK(cudaStreamSynchronize(stream));
            return;
        }
        memcpy(h_stage + h_stage_used, src, bytes);
        CK(cudaMemcpyAsync(dst, h_stage + h_stage_used, bytes, cudaMemcpyHostToDevice, stream));
        h_stage_used += need;
    }
    void t_begin(int st) { if (!capturing) CK(cudaEventRecord(tev[st][0], stream)); }
    void t_end(int st) { if (!capturing) { CK(cudaEventRecord(tev[st][1], stream)); trec[st] = true; times_valid = false; } }
    void collect_times() {
        if (times_valid) return;
        CK(cudaSetDevice(device));
        CK(cudaStreamSynchronize(stream));
        float* slot[TS_COUNT] = {&times.lde, &times.interpolate, &times.leaf_hash, &times.merkle, &times.constraints, &times.composition,
                                 &times.ood, &times.deep, &times.fri, &times.grind, &times.queries, &times.total};
        for (int st = 0; st < TS_COUNT; st++) if (trec[st]) CK(cudaEventElapsedTime(slot[st], tev[st][0], tev[st][1]));
        times_valid = true;
    }
    void d2h(void* dst, const void* src, size_t bytes) {
        CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
    }
    void check_launch() { CK(cudaGetLastError()); count(); }

    // ---- tables ---------------------------------------------------------------------------------------------
    static void build_powtab(HF base, uint32_t log_size, std::vector<HF>& lo, std::vector<HF>& hi, uint32_t& l1) {
        l1 = (log_size + 1) / 2;
        uint32_t l2 = log_size - l1;
        lo.resize((size_t)1 << l1); hi.resize((size_t)1 << l2);
        HF x = HF::raw(1);
        for (auto& v : lo) { v = x; x = x * base; }
        HF step = x;  // base^(2^l1)
        x = HF::raw(1);
        for (auto& v : hi) { v = x; x = x * step; }
    }
    void ensure_tables() {
        if (tab_log_built != log_N) {
            std::vector<HF> lo, hi; uint32_t l1;
            build_powtab(HF::root_of_unity(log_N), log_N, lo, hi, l1);
            d_roots_lo.ensure(lo.size() * 16); d_roots_hi.ensure(hi.size() * 16);
            h2d(d_roots_lo.p, lo.data(), lo.size() * 16); h2d(d_roots_hi.p, hi.data(), hi.size() * 16);
            roots = PowTab{d_roots_lo.as<fe>(), d_roots_hi.as<fe>(), l1};
            build_powtab(HF::from_u64(3).inv(), log_N, lo, hi, l1);
            d_inv3_lo.ensure(lo.size() * 16); d_inv3_hi.ensure(hi.size() * 16);
            h2d(d_inv3_lo.p, lo.data(), lo.size() * 16); h2d(d_inv3_hi.p, hi.data(), hi.size() * 16);
            inv3tab = PowTab{d_inv3_lo.as<fe>(), d_inv3_hi.as<fe>(), l1};
            CK(cudaStreamSynchronize(stream));  // host vectors go out of scope
            tab_log_built = log_N;
            pow3_for_log_n = 0;
        }
        log_tab = log_N;
        if (pow3_for_log_n != log_n) {
            std::vector<HF> p3(log_n + 1);
            for (uint32_t l = 0; l <= log_n; l++) p3[l] = HF::from_u64(3).pow((u128)(air.n >> l));
            d_pow3.ensure(64 * 16);
            h2d(d_pow3.p, p3.data(), p3.size() * 16);
            CK(cudaStreamSynchronize(stream));
            pow3_for_log_n = log_n;
        }
    }

    // ---- NTT planning ---------------------------------------------------------------------------------------
    // 16-column tiles (256 rows, 3 blocks/SM) were measured against 8-column tiles at 4 blocks/SM (64 registers): no gain,
    // the pass kernel is bound by integer issue, not occupancy (DESIGN.md §3)
    static uint32_t pick_cj(uint32_t ncols) { return ncols >= 9 ? 16 : ncols >= 5 ? 8 : ncols >= 3 ? 4 : ncols == 2 ? 2 : 1; }
    // tiles of >= 4 columns keep four pre-shifted copies of every twiddle (k_ntt_pass<true>)
    static bool pre_twiddles(uint32_t cj) { return cj >= 4; }
    static std::vector<uint32_t> plan_layers(uint32_t log_len, uint32_t cj) {
        // plain twiddles: S * cj <= 4096 elements in shared memory; four-copy twiddles: tile + 4 S twiddles <= ~107 KB so that two
        // blocks share an SM (256 x 16, 512 x 8, 512 x 4)
        uint32_t maxlog = pre_twiddles(cj) ? (cj >= 16 ? 8 : 9) : 12 - log2u(cj);
        uint32_t passes = (log_len + maxlog - 1) / maxlog;
        if (passes == 0) passes = 1;
        std::vector<uint32_t> b;  // cumulative layer boundaries
        uint32_t done = 0;
        for (uint32_t q = 0; q < passes; q++) { uint32_t take = (log_len - done + (passes - q) - 1) / (passes - q); done += take; b.push_back(done); }
        return b;
    }
    // Tile twiddles depend only on (transform size, layer range, coset, t_low): tables are built once per shape (k_build_twiddles)
    // and re-read from L2 by every column tile, column group and proof instead of being regenerated (two multiplications per
    // twiddle) by each of the thousands of tiles that share them.  Wide tiles (k_ntt_pass<true>) take a table of four pre-shifted
    // copies (64 B per twiddle) when it fits in 64 MiB — the tiles then only copy it — else a plain one (16 B per twiddle, shifted
    // by every tile) within the same cap; narrow tiles (1-2 columns) have as many twiddles as elements, so their plain tables may
    // take 192 MiB.  Sets p.tw_tab (null: the tiles generate their twiddles) and p.tw_four.
    ShapeCache<std::tuple<uint32_t, uint32_t, uint32_t, uint32_t, uint32_t, uint32_t, uint32_t>> tw_cache{(size_t)768 << 20};
    void twiddle_table(NttPass& p, uint32_t all_cosets) {
        const uint32_t S = 1u << (p.b - p.a);
        const uint64_t entries = ((uint64_t)all_cosets << p.a) * (S - 1u);
        const bool pre = pre_twiddles(p.cj);
        const uint64_t cap = (uint64_t)(pre ? 64 : 192) << 20;
        p.tw_tab = nullptr; p.tw_four = 0;
        static const bool log_tables = getenv("ZKB_HOST_PROFILE") != nullptr;   // diagnostics: which passes get which table
        if (S < 2 || entries * 16 > cap) {
            if (log_tables && S >= 2)
                fprintf(stderr, "[zkb twiddles] log_n %u layers [%u, %u) coset %u inverse %u cj %u: no table (%.2f MiB plain), generated\n", p.log_n,
                        p.a, p.b, p.coset, p.inverse, p.cj, entries * 16 / 1048576.0);
            return;
        }
        const uint32_t four = pre && entries * 64 <= cap ? 1u : 0u;
        const uint64_t bytes = entries * (four ? 64 : 16);
        const auto key = std::make_tuple(p.log_n, p.a, p.b, p.coset, p.inverse, p.coset ? p.log_lde : 0u, four);
        DevBuf* tab = tw_cache.find(key);
        if (!tab) {
            if (log_tables && tw_cache.full(bytes)) fprintf(stderr, "[zkb twiddles] cache of %.2f MiB over budget: cleared\n", tw_cache.bytes / 1048576.0);
            tab = &tw_cache.insert(key, bytes, stream);
            if (log_tables)
                fprintf(stderr, "[zkb twiddles] log_n %u layers [%u, %u) coset %u inverse %u cj %u: %s table %.2f MiB, cache %.2f MiB\n", p.log_n, p.a,
                        p.b, p.coset, p.inverse, p.cj, four ? "four-copy" : "plain", bytes / 1048576.0, tw_cache.bytes / 1048576.0);
            NttPass q = p;
            q.n_cosets = all_cosets; q.coset0 = 0; q.tw_four = four;
            k_build_twiddles<<<(unsigned)((entries + 255) / 256), 256, 0, stream>>>(q, tab->as<fe>());
            check_launch();
        }
        p.tw_tab = tab->as<fe>(); p.tw_four = four;
    }
    void launch_pass(NttPass p) {
        const uint32_t S = 1u << (p.b - p.a);
        const uint32_t rs = p.cj + (p.cj > 1 ? 1 : 0);
        const bool pre = pre_twiddles(p.cj);
        const size_t smem = ((size_t)S * rs + (pre ? 4 : 1) * (size_t)S) * 16;   // tile + twiddles (four copies each for wide tiles)
        // grid: x = column tile, y = coset, z = (t_low, u0) tile; z is limited to 65535 per launch
        const uint32_t n_ct = (p.ncols + p.cj - 1) / p.cj;
        const uint64_t tiles = (uint64_t)1 << (p.log_n - (p.b - p.a));
        if (p.n_cosets > 65535) throw InvalidArg("transform too large for one launch");
        uint32_t threads = 256;
        if (pre) {
            // one two-column radix-8 unit per thread and round: S * cj / 16 threads keep every thread busy (128-row tiles of the
            // three-pass transforms get 128-thread blocks, four per SM); never fewer than the panel store needs (min(S, 256))
            const uint32_t units = p.cj >= 16 ? S * p.cj / 16 : S * p.cj / 8;   // radix-8 units per round (two columns each for 16-wide tiles)
            threads = std::max<uint32_t>(units, std::min<uint32_t>(S, 256));
            threads = std::min<uint32_t>(256, std::max<uint32_t>(32, threads));
        }
        for (uint64_t z0 = 0; z0 < tiles; z0 += 65535) {
            p.tile0 = (uint32_t)z0;
            const dim3 grid(n_ct, p.n_cosets, (unsigned)std::min<uint64_t>(65535, tiles - z0));
            if (pre) k_ntt_pass<true><<<grid, threads, smem, stream>>>(p);
            else k_ntt_pass<false><<<grid, threads, smem, stream>>>(p);
            check_launch();
        }
    }
    // generic multi-pass transform of `ncols` columns of length 2^log_len.
    //  in : row-major [len][w_in] (column window col0_in..)         bufs: scratch buffers for intermediate passes
    //  out: row-major natural [len][w_out] (inverse / plain) or the panel layout (coset LDE, one launch per coset batch)
    struct Xform {
        const fe* in; uint32_t w_in, col0_in;
        fe* out; uint32_t w_out, col0_out;
        uint32_t ncols, log_len;
        bool inverse, coset_lde;
        uint32_t log_lde;  // coset LDE only
        bool scale; HF scale_by;
        uint32_t log_shard = 0;  // coset LDE only: split every panel into 2^log_shard slot chunks (multi-GPU send view)
        uint32_t coset_lo = 0, coset_cnt = 0;  // coset LDE only: evaluate cosets [lo, lo + cnt) (0 = all) into a buffer holding just those
        uint32_t batch_cosets = 0;  // coset LDE only: cosets per launch batch (0 = as many as the scratch budget allows)
        std::function<void(uint32_t, uint32_t)> after_batch;  // called with (first coset, count) once a batch's last pass is enqueued
        uint32_t cj = 0;  // column-tile width; 0 = from ncols.  Column groups of one matrix must share it: it fixes the pass plan
                          // and with it the panel size of the LDE layout
    };
    // returns log_p of the panel layout for LDEs (size of the last pass)
    uint32_t run_xform(const Xform& x, DevBuf& s1, DevBuf& s2) {
        const uint32_t cj = x.cj ? x.cj : pick_cj(x.ncols);
        std::vector<uint32_t> bnd = plan_layers(x.log_len, cj);
        const uint32_t passes = (uint32_t)bnd.size();
        const uint64_t len = (uint64_t)1 << x.log_len;
        const uint32_t all_cosets = x.coset_lde ? (1u << (x.log_lde - x.log_len)) : 1;
        const uint32_t n_cosets = (x.coset_lde && x.coset_cnt) ? x.coset_cnt : all_cosets;
        // coset batches bound the scratch size
        uint32_t batch = x.batch_cosets ? std::min(x.batch_cosets, n_cosets) : n_cosets;
        if (passes > 1) {
            const uint64_t per = len * x.ncols * 16;
            uint64_t budget = (uint64_t)6 << 30;
            batch = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(batch, budget / std::max<uint64_t>(per, 1)));
            s1.ensure(per * batch);
            if (passes > 2) s2.ensure(per * batch);
        }
        for (uint32_t k0 = 0; k0 < n_cosets; k0 += batch) {
            const uint32_t nk = std::min(batch, n_cosets - k0);
            uint32_t a = 0;
            const fe* src = x.in; uint32_t w_src = x.w_in, c0_src = x.col0_in; uint64_t src_stride = 0;
            for (uint32_t q = 0; q < passes; q++) {
                NttPass p{};
                const bool last = (q + 1 == passes);
                p.in = src; p.w_in = w_src; p.col0_in = c0_src; p.in_coset_stride = src_stride;
                p.log_n = x.log_len; p.a = a; p.b = bnd[q];
                p.ncols = x.ncols; p.cj = cj; p.n_cosets = nk; p.coset0 = x.coset_lo + k0;
                p.panel_k0 = x.coset_lo; p.log_kc = log2u(n_cosets);
                p.coset = x.coset_lde ? 1 : 0; p.inverse = x.inverse ? 1 : 0;
                p.log_tab = log_tab; p.log_lde = x.coset_lde ? x.log_lde : 0;
                p.roots = roots; p.pow3 = d_pow3.as<fe>();
                twiddle_table(p, all_cosets);
                if (last) {
                    p.out = x.out; p.w_out = x.w_out; p.col0_out = x.col0_out;
                    p.out_panel = x.coset_lde ? 1 : 0;
                    p.log_shard = x.coset_lde ? x.log_shard : 0;
                    if (p.log_shard > p.b - p.a) throw InvalidArg("trace too short to shard its LDE panels across this many GPUs");
                    p.out_coset_stride = 0;
                    p.do_scale = x.scale ? 1 : 0; p.scale = to_fe(x.scale_by);
                } else {
                    fe* dst = (q % 2 == 0) ? s1.as<fe>() : s2.as<fe>();
                    p.out = dst; p.w_out = x.ncols; p.col0_out = 0; p.out_coset_stride = len * x.ncols;
                    src = dst; w_src = x.ncols; c0_src = 0; src_stride = len * x.ncols;
                }
                launch_pass(p);
                a = bnd[q];
            }
            if (x.after_batch) x.after_batch(x.coset_lo + k0, nk);
        }
        return bnd.back() - (passes > 1 ? bnd[passes - 2] : 0);
    }

    // ---- Merkle heap: heap[1] root, heap[N + l] leaves -----------------------------------------------------------
    void build_merkle(uint32_t* heap, uint64_t n_leaves) {
        uint64_t lvl = n_leaves / 2;
        for (; lvl > 512; lvl >>= 1) {   // wide levels: one launch each
            k_merkle_level<<<(unsigned)((lvl + 255) / 256), 256, 0, stream>>>(heap + 2 * lvl * 8, heap + lvl * 8, lvl);
            check_launch();
        }
        k_merkle_top<<<1, 512, 0, stream>>>(heap, (uint32_t)lvl);   // the last <= 10 levels in one launch
        check_launch();
    }

    // ==========================================================================================================
    // stages
    void begin(const zkb_air_desc* desc) {
        CK(cudaSetDevice(device));
        air = AirSpec::from_desc(desc);
        log_n = log2u(air.n); log_beta = log2u(air.blowup); log_N = log_n + log_beta;
        log_ce = log2u(air.ce_blowup()); c = air.num_comp_cols();
        if ((1u << log_ce) > air.blowup) throw InvalidArg("constraint evaluation blowup exceeds the LDE blowup");
        {   // distinct assertion steps = boundary groups
            std::set<uint64_t> steps;
            for (auto& a : air.assertions) steps.insert(a.step);
            if (steps.size() > ZKB_MAX_GROUPS) throw InvalidArg("too many distinct assertion steps (boundary groups)");
        }
        ensure_tables();
        parts = ProofParts();
        memset(&ts, 0, sizeof(ts));
        ts.comp_degree_ok = 1;
        memset(&times, 0, sizeof(times));
        for (auto& r : trec) r = false;
        times_valid = true;
        h_stage_used = 0;
        coin.init(air.coin_seed());
        fri_layers = air.num_fri_layers();
        if (fri_layers > ZKB_MAX_FRI_LAYERS) throw InvalidArg("too many FRI layers");
        fri_layer = 0; fri_committed = false;
        positions.clear();
        mg_active = false;
        {   // device transcript + openings layout (everything is determined by the shape)
            auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
            const uint32_t w = air.w, q = air.num_queries;
            const uint64_t m_last = fri_domain(fri_layers);
            fs = FsLayout();
            fs.o_ood = al(sizeof(DevTs));
            fs.o_rem = fs.o_ood + (2 * (size_t)w + c) * 16;
            fs.rem_cap = (uint32_t)std::max<uint64_t>(1, m_last / air.blowup);
            size_t off = al(fs.o_rem + (size_t)fs.rem_cap * 16);
            auto add_tree = [&](uint32_t width, uint32_t depth) {
                FsTree t{off, off + (size_t)q * width * 16, width, depth};
                off = al(t.o_paths + (size_t)q * depth * 32);
                fs.trees.push_back(t);
            };
            add_tree(w, log_N);
            add_tree(c, log_N);
            for (uint32_t l = 0; l < fri_layers; l++) add_tree(air.folding, log2u(fri_rows(l)));
            fs.host_bytes = off;
            fs.o_coef = off; off += ((size_t)air.num_transition() + air.assertions.size()) * 16;
            fs.o_gamma = off; off += ((size_t)w + c) * 16;
            fs.o_scr = off; off += 2 * (size_t)w * 16;
            fs.total = off;
            d_fs.ensure(fs.total);
            d_flags.ensure(256);
            if (h_out_cap < fs.host_bytes) {
                if (h_out) { cudaFreeHost(h_out); h_out = nullptr; h_out_cap = 0; }
                g_alloc_epoch++;
                CK(cudaHostAlloc((void**)&h_out, fs.host_bytes, cudaHostAllocDefault));
                h_out_cap = fs.host_bytes;
            }
            // transcript: coin seed = hash(Context ++ public inputs), computed here because the host holds the AIR; all else zero
            DevTs h0;
            memset(&h0, 0, sizeof(h0));
            memcpy(h0.seed, coin.seed, 32);
            h0.nonce = ~0ull;
            h2d_small(d_fs.p, &h0, sizeof(h0));
            // per-proof inputs: assertion values (sorted order) and AIR parameters
            const size_t na = air.assertions.size(), np = air.params.size();
            std::vector<HF> in(na + np);
            for (size_t i = 0; i < na; i++) in[i] = air.assertions[i].value;
            for (size_t i = 0; i < np; i++) in[na + i] = air.params[i];
            d_in.ensure((na + np + 1) * 16);
            h2d_small(d_in.p, in.data(), in.size() * 16);
        }
        stage = ST_BEGUN;
    }

    // staged API: a commitment's root, downloaded from `d_root`, joins the proof and the transcript slot `ts_root`
    void take_root(const uint32_t* d_root, uint8_t ts_root[32], uint8_t* root_out) {
        Digest32 root;
        d2h(root.b, d_root, 32);
        parts.commitments.push_back(root);
        memcpy(ts_root, root.b, 32);
        if (root_out) memcpy(root_out, root.b, 32);
    }

    // K1-K4.  The trace is committed column group by column group (16 columns): [H2D] -> transpose -> inverse NTT ->
    // coset LDE.  Column groups are independent until the rows are hashed, so the host-to-device copy of group g+1
    // (copy stream) overlaps the transforms of group g, and a group's polynomials (n*16 elements) stay L2-resident
    // while all beta cosets are evaluated from them.
    // Group widths: a trace that is already in HBM is one group (no launch tails).  A host trace is cut into groups of
    // 16, 32, 48, 48, ... columns: the first copy, which nothing can hide, is short (16 columns), later groups are wide enough
    // that every launch still fills > 25 waves of resident blocks.
    void trace_commit(const uint8_t* const* host_cols, const fe* d_src, uint8_t root_out[32]) {
        trace_commit_dev(host_cols, d_src);
        take_root(d_tree.as<uint32_t>() + 8, ts.trace_root, root_out);
    }
    // leaves the root at d_tree + 8 words
    void trace_commit_dev(const uint8_t* const* host_cols, const fe* d_src) {
        if (stage != ST_BEGUN) throw StateError("zkb_trace_commit: call zkb_begin first");
        const uint64_t n = air.n, N = air.lde_size();
        const uint32_t w = air.w;
        std::vector<std::pair<uint32_t, uint32_t>> groups;  // (first column, width)
        if (!host_cols) groups.push_back({0, w});
        else for (uint32_t c0 = 0, step = 16; c0 < w; c0 += groups.back().second, step = std::min(step + 16, 48u)) groups.push_back({c0, std::min(step, w - c0)});
        const uint32_t ngroups = (uint32_t)groups.size();
        d_bufA.ensure(n * w * 16); d_bufB.ensure(n * w * 16);
        d_lde.ensure(N * w * 16);
        d_tree.ensure(2 * N * 32);
        t_begin(TS_LDE);
        if (host_cols) {
            d_trace.ensure((size_t)w * n * 16);
            for (uint32_t j = 0; j < w; j++) if (!host_cols[j]) throw InvalidArg("null trace column");
            // the copy stream must not start before earlier work on the compute stream (previous proof) is done
            CK(cudaEventRecord(ev_group[16], stream));
            CK(cudaStreamWaitEvent(copy_stream, ev_group[16], 0));
            if (ngroups > 16) throw InvalidArg("too many column groups");
            for (uint32_t g = 0; g < ngroups; g++) {
                const uint32_t c0 = groups[g].first;
                copy_cols(host_cols + c0, groups[g].second, n, d_trace.as<uint8_t>() + (size_t)c0 * n * 16, copy_stream);
                h2d_bytes += (size_t)groups[g].second * n * 16;
                CK(cudaEventRecord(ev_group[g], copy_stream));
            }
            d_src = d_trace.as<fe>();
        }
        d_polys = d_bufB.as<fe>();
        const HF n_inv = HF::from_u64(n).inv();
        for (uint32_t g = 0; g < ngroups; g++) {
            const uint32_t c0 = groups[g].first, wc = groups[g].second;
            if (host_cols) CK(cudaStreamWaitEvent(stream, ev_group[g], 0));
            {
                dim3 grid((unsigned)((n + 31) / 32), (wc + 31) / 32), block(32, 8);
                k_transpose_cols<<<grid, block, 0, stream>>>(d_src + (size_t)c0 * n, d_bufA.as<fe>() + c0, (uint32_t)n, wc, w);
                check_launch();
            }
            // K1: interpolate (inverse NTT, scaled by 1/n) -> polys row-major [n][w]
            Xform xi{d_bufA.as<fe>(), w, c0, d_bufB.as<fe>(), w, c0, wc, log_n, true, false, 0, true, n_inv};
            xi.cj = pick_cj(w);
            run_xform(xi, d_tmp1, d_tmp2);
            // K2: coset LDE into the panel layout
            Xform xl{d_polys, w, c0, d_lde.as<fe>(), w, c0, wc, log_n, false, true, log_N, false, HF()};
            xl.cj = pick_cj(w);
            lde_log_p = run_xform(xl, d_tmp1, d_tmp2);
        }
        t_end(TS_LDE);
        // K3: leaves
        t_begin(TS_LEAF);
        // few, wide rows: hash a row's 1 KiB chunks on separate lanes (a shorter chain of compressions, same digests)
        if (N <= 8192 && w > 64) k_hash_lde_rows_split<<<(unsigned)((N * 4 + 127) / 128), 128, 0, stream>>>(lde_mat(), d_tree.as<uint32_t>() + N * 8, 0, 0);
        else k_hash_lde_rows<<<(unsigned)((N + 127) / 128), 128, 0, stream>>>(lde_mat(), d_tree.as<uint32_t>() + N * 8, 0, 0);
        check_launch();
        t_end(TS_LEAF);
        // K4: tree
        t_begin(TS_MERKLE);
        build_merkle(d_tree.as<uint32_t>(), N);
        t_end(TS_MERKLE);
        // interpolation and LDE are interleaved per group: they are reported together under `lde`
        stage = ST_TRACE;
    }
    void trace_commit_device(const fe* d_src, uint8_t root_out[32]) { trace_commit(nullptr, d_src, root_out); }
    void trace_commit_host(const uint8_t* const* cols, uint8_t root_out[32]) {
        if (!cols) throw InvalidArg("null trace columns");
        trace_commit(cols, nullptr, root_out);
    }
    // host columns cols[0 .. w) of n elements into the column-major `dst`: one copy when they are contiguous in host memory
    static void copy_cols(const uint8_t* const* cols, uint32_t w, uint64_t n, uint8_t* dst, cudaStream_t st) {
        const size_t cb = (size_t)n * 16;
        bool contiguous = true;
        for (uint32_t j = 1; j < w; j++) if (cols[j] != cols[0] + j * cb) contiguous = false;
        if (contiguous) CK(cudaMemcpyAsync(dst, cols[0], w * cb, cudaMemcpyHostToDevice, st));
        else for (uint32_t j = 0; j < w; j++) CK(cudaMemcpyAsync(dst + j * cb, cols[j], cb, cudaMemcpyHostToDevice, st));
    }
    const fe* upload_cols(const uint8_t* const* cols, uint32_t w, uint64_t n, DevBuf& dst) {
        if (!cols) throw InvalidArg("null trace columns");
        for (uint32_t j = 0; j < w; j++) if (!cols[j]) throw InvalidArg("null trace column");
        dst.ensure((size_t)w * n * 16);
        copy_cols(cols, w, n, dst.as<uint8_t>(), stream);
        h2d_bytes += (size_t)w * n * 16;
        return dst.as<fe>();
    }

    // ---- column-sharded single proof (SURVEY §8e, BASELINE.json configs[4]) ---------------------------------------
    // Rank r owns columns [r w/G, (r+1) w/G): ingest, interpolation and the coset LDE are column-local.  The LDE's last
    // pass writes the sharded panel layout [G][panels][w/G][P/G]; one NCCL all-to-all over NVLink (chunk q of rank r <->
    // chunk r of rank q) turns it into the recv view "all columns x my rows", rows [q N/G, (q+1) N/G) being contiguous
    // Merkle leaves.  Every rank hashes its rows and builds its subtree; an all-gather of the G subtree roots lets every
    // rank finish the top log G levels redundantly.
    void mg_init(int rank, int world, const uint8_t* id_bytes) {
        if (world < 1 || !is_pow2((uint64_t)world) || rank < 0 || rank >= world) throw InvalidArg("multi-GPU world size must be a power of two");
        g_nccl.load();
        CK(cudaSetDevice(device));
        if (comm) { g_nccl.CommDestroy(comm); comm = nullptr; }
        ncclUniqueId id;
        static_assert(sizeof(ncclUniqueId) == 128, "unexpected ncclUniqueId size");
        memcpy(&id, id_bytes, sizeof(id));
        NK(g_nccl.CommInitRank(&comm, world, id, rank));
        mg_rank = rank; mg_world = world; log_g = log2u((uint64_t)world);
    }
    // leaves the root at d_cap + 8 words
    void trace_commit_mg(const uint8_t* const* host_cols_local, const fe* d_src) {
        if (stage != ST_BEGUN) throw StateError("zkb_mg_prove: call zkb_begin first");
        if (!comm) throw StateError("zkb_mg_init has not been called on this context");
        const uint64_t n = air.n, N = air.lde_size();
        const uint32_t w = air.w, G = (uint32_t)mg_world;
        if (w % G) throw InvalidArg("trace width must be divisible by the number of GPUs");
        const uint32_t wl = w / G;
        if (air.id == ZKB_AIR_ID_AGGREGATION) throw InvalidArg("the aggregation AIR cannot be column-sharded (replicas only)");
        if (N / G < 2) throw InvalidArg("LDE domain too small to shard");
        mg_active = true;
        t_begin(TS_LDE);
        if (host_cols_local) d_src = upload_cols(host_cols_local, wl, n, d_trace);
        d_bufA.ensure(n * wl * 16); d_bufB.ensure(n * wl * 16);
        {
            dim3 grid((unsigned)((n + 31) / 32), (wl + 31) / 32), block(32, 8);
            k_transpose_cols<<<grid, block, 0, stream>>>(d_src, d_bufA.as<fe>(), (uint32_t)n, wl, wl);
            check_launch();
        }
        Xform xi{d_bufA.as<fe>(), wl, 0, d_bufB.as<fe>(), wl, 0, wl, log_n, true, false, 0, true, HF::from_u64(n).inv()};
        run_xform(xi, d_tmp1, d_tmp2);
        d_polys = d_bufB.as<fe>();
        d_lde.ensure(N * wl * 16);
        Xform xl{d_polys, wl, 0, d_lde.as<fe>(), wl, 0, wl, log_n, false, true, log_N, false, HF()};
        xl.log_shard = log_g;
        // NVLink transpose, column shards -> row shards, pipelined behind the LDE.  In the send view [dest][coset][...] the
        // data of one coset batch bound for one destination is contiguous, so a finished batch is shipped on xchg_stream
        // while the next batch is still being evaluated; only the last batch's transfer is exposed.
        d_lde_rows.ensure(N * wl * 16);
        const size_t chunk = (size_t)(N / G) * wl * 16;  // bytes per (source, destination) pair
        const size_t per_coset = chunk >> log_beta;
        uint32_t n_batches = std::min<uint32_t>(air.blowup, 8);   // only the last batch's transfer is exposed
        while (n_batches > 1 && (uint64_t)n * wl * (air.blowup / n_batches) < ((uint64_t)1 << 20)) n_batches >>= 1;  // keep launches wide
        xl.batch_cosets = (uint32_t)air.blowup / n_batches;
        uint32_t shipped = 0;
        xl.after_batch = [&](uint32_t k0, uint32_t nk) {
            cudaEvent_t ev = ev_group[shipped++ & 15];
            CK(cudaEventRecord(ev, stream));
            CK(cudaStreamWaitEvent(xchg_stream, ev, 0));
            NK(g_nccl.GroupStart());
            for (uint32_t q = 0; q < G; q++) {
                const size_t off = q * chunk + (size_t)k0 * per_coset;
                NK(g_nccl.Send(d_lde.as<uint8_t>() + off, (size_t)nk * per_coset, ncclUint8, (int)q, comm, xchg_stream));
                NK(g_nccl.Recv(d_lde_rows.as<uint8_t>() + off, (size_t)nk * per_coset, ncclUint8, (int)q, comm, xchg_stream));
            }
            NK(g_nccl.GroupEnd());
        };
        lde_log_p = run_xform(xl, d_tmp1, d_tmp2);
        t_end(TS_LDE);
        t_begin(TS_XCHG);
        CK(cudaEventRecord(ev_group[16], xchg_stream));
        CK(cudaStreamWaitEvent(stream, ev_group[16], 0));
        t_end(TS_XCHG);
        t_begin(TS_LEAF);
        // K3/K4 on this rank's rows
        const uint64_t Nl = N / G;
        d_tree.ensure(2 * Nl * 32);
        k_hash_lde_rows<<<(unsigned)((Nl + 127) / 128), 128, 0, stream>>>(lde_rows_mat(), d_tree.as<uint32_t>() + Nl * 8, (uint64_t)mg_rank * Nl, 0);
        check_launch();
        t_end(TS_LEAF);
        t_begin(TS_MERKLE);
        build_merkle(d_tree.as<uint32_t>(), Nl);
        // all-gather of the subtree roots into the leaves of the cap heap, which every rank finishes: cap[1] = root
        if (2 * (size_t)G * 32 > ZKB_CAP_BYTES) throw InvalidArg("too many GPUs for one sharded commitment");
        d_cap.ensure(ZKB_CAP_BYTES);
        NK(g_nccl.AllGather(d_tree.as<uint8_t>() + 32, d_cap.as<uint8_t>() + (size_t)G * 32, 32, ncclUint8, comm, stream));
        k_merkle_top<<<1, 512, 0, stream>>>(d_cap.as<uint32_t>(), G / 2);
        check_launch();
        t_end(TS_MERKLE);
        // (the `interpolate` slot of zkb_stage_times carries the NVLink all-to-all time of a sharded proof)
        stage = ST_TRACE;
    }

    // ---- Fiat-Shamir steps.  `digest` = device address of the commitment the coin is reseeded with (one-shot proofs: the whole
    // channel runs on the device, csrc/coin.cuh); nullptr = the staged API handed us the challenge, which is uploaded instead.
    void fs_upload(fe* dst, const HF& v) { h2d_small(dst, &v, 16); }
    void fs_after_trace_root(const uint32_t* digest, const HF* alpha) {
        if (!digest) fs_upload(&dts()->alpha, *alpha);
        k_fs_trace_root<<<1, ZKB_FS_THREADS, 0, stream>>>(dts(), digest, air.num_transition() + (uint32_t)air.assertions.size(), fs_fe(fs.o_coef), d_flags.as<uint32_t>());
        check_launch();
    }
    void fs_after_constraint_root(const uint32_t* digest, const HF* zz) {
        if (!digest) fs_upload(&dts()->z, *zz);
        k_fs_constraint_root<<<1, 32, 0, stream>>>(dts(), digest, d_flags.as<uint32_t>(), to_fe(HF::root_of_unity(log_n)));
        check_launch();
    }
    void fs_after_ood(bool with_coin, const HF* deep_alpha) {
        if (!with_coin) fs_upload(&dts()->deep_alpha, *deep_alpha);
        k_fs_ood<<<1, ZKB_FS_THREADS, 0, stream>>>(dts(), fs_fe(fs.o_ood), air.w, c, fs_fe(fs.o_scr), fs_fe(fs.o_gamma), with_coin ? 1u : 0u);
        check_launch();
    }

    // K5.  The evaluator works on a window of `ncols` trace columns starting at global column `col0` (the whole trace on
    // one GPU; this rank's columns in a column-sharded proof).  Every term of the combined evaluation is linear in
    // per-column sums, so per-rank partial results add up to the full composition trace.
    // The coefficient powers alpha^0.. (transition constraints, then the assertions sorted by (step, column): draw_algebraic,
    // [A.5]) are in device memory already (k_fs_trace_root); assertion values and AIR parameters are the per-proof inputs d_in.
    void constraints_eval_window(const LdeMat& mat, uint32_t col0, uint32_t ncols, fe* out) {
        const uint32_t nt = air.num_transition(), na = (uint32_t)air.assertions.size();
        const uint64_t n = air.n, ce = (uint64_t)1 << log_ce;
        const bool windowed = !(col0 == 0 && ncols == air.w);
        if (windowed && air.id == ZKB_AIR_ID_AGGREGATION) throw InvalidArg("the aggregation AIR couples columns i and i+d and cannot be column-sharded");
        EvalParams p{};
        p.lde = mat; p.air_id = air.id; p.log_ce = log_ce;
        p.n_trans = windowed ? ncols : nt;
        const HF g = HF::root_of_unity(log_n);
        std::vector<uint32_t> acol, asel;
        std::vector<uint64_t> gsteps;
        uint32_t ng = 0;
        for (uint32_t i = 0; i < na; i++) {
            if (i == 0 || air.assertions[i].step != air.assertions[i - 1].step) {
                p.g_off[ng] = (uint32_t)acol.size(); gsteps.push_back(air.assertions[i].step); ng++;
            }
            const uint32_t col = air.assertions[i].col;
            if (col >= col0 && col < col0 + ncols) { acol.push_back(col - col0); asel.push_back(i); }
        }
        const uint32_t nl = (uint32_t)acol.size();
        p.g_off[ng] = nl; p.n_groups = ng;
        // divisor table of the shape (k_build_divisors): cached until the trace length, the ce blowup or the assertion steps change
        std::vector<uint64_t> dkey{n, ce};
        dkey.insert(dkey.end(), gsteps.begin(), gsteps.end());
        DevBuf* divbuf = div_cache.find(dkey);
        const bool build_div = !divbuf;
        // 1/(x^n - 1) on the cosets used by the ce domain: x^n = 3^n * w_beta^k, k = kc * beta/ce   (input of the table build only)
        std::vector<HF> zinv(ce);
        if (build_div) {
            HF on = HF::from_u64(3).pow((u128)n), wb = HF::root_of_unity(log_beta);
            for (uint64_t kc = 0; kc < ce; kc++) zinv[kc] = (on * wb.pow((u128)(kc << (log_beta - log_ce))) - HF::raw(1)).inv();
        }
        // periodic column over the ce domain (PeriodicValueTable): P_L(x^(n/L)) tabulated on 3^(n/L) * <w_{L*ce}>
        if (air.id == ZKB_AIR_ID_MIMC && !(per_cache_n == n && per_cache_ce == ce && per_cache_params.size() == air.params.size() &&
                                           std::equal(per_cache_params.begin(), per_cache_params.end(), air.params.begin()))) {
            const size_t L = air.params.size();
            std::vector<HF> poly = host_interpolate(air.params, HF::raw(1));
            const HF off = HF::from_u64(3).pow((u128)(n / L)), wl = HF::root_of_unity(log2u(L * ce));
            per_cache.resize(L * ce);
            HF x = off;
            for (size_t t = 0; t < L * ce; t++) { HF acc; for (size_t q = L; q-- > 0;) acc = acc * x + poly[q]; per_cache[t] = acc; x = x * wl; }
            per_cache_params = air.params; per_cache_n = n; per_cache_ce = ce;
        }
        static const std::vector<HF> no_per;
        const std::vector<HF>& per = air.id == ZKB_AIR_ID_MIMC ? per_cache : no_per;
        // pack the shape-dependent small arrays into one device buffer
        size_t off_p = 0, off_col = off_p + per.size() * 16, off_sel = off_col + (size_t)nl * 4, total = off_sel + (size_t)nl * 4 + 16;
        std::vector<uint8_t> pack(total);
        if (!per.empty()) memcpy(&pack[off_p], per.data(), per.size() * 16);
        if (nl) { memcpy(&pack[off_col], acol.data(), (size_t)nl * 4); memcpy(&pack[off_sel], asel.data(), (size_t)nl * 4); }
        // shape-only data: uploaded once per distinct content and kept (a captured graph of that shape keeps reading it), never
        // per proof and never inside a graph capture
        const std::string pk((const char*)pack.data(), pack.size());
        DevBuf* packbuf = pack_cache.find(pk);
        if (!packbuf) {
            if (capturing) throw StateError("evaluator tables changed during a graph capture");
            packbuf = &pack_cache.insert(pk, total, stream);
            h2d_small(packbuf->p, pack.data(), total);
        }
        uint8_t* base = packbuf->as<uint8_t>();
        const fe* coef = fs_fe(fs.o_coef);
        p.tcoef = coef + (windowed ? col0 : 0); p.a_coef = coef + nt; p.a_val = d_aval(); p.params = d_params();
        p.periodic = (const fe*)(base + off_p);
        p.a_col = (const uint32_t*)(base + off_col); p.a_sel = (const uint32_t*)(base + off_sel);
        p.per_mask = per.empty() ? 0 : (uint32_t)per.size() - 1;
        p.out = out;
        if (build_div) {
            if (capturing) throw StateError("divisor table changed during a graph capture");
            divbuf = &div_cache.insert(dkey, (size_t)(ng + 1) * n * ce * 16, stream);
            d_aux.ensure(ce * 16);
            h2d_small(d_aux.p, zinv.data(), ce * 16);
            DivParams dp{};
            dp.log_cen = log_n + log_ce; dp.log_ce = log_ce; dp.n_groups = ng;
            for (uint32_t gi = 0; gi < ng; gi++) dp.g_point[gi] = to_fe(g.pow((u128)gsteps[gi]));
            dp.g_last = to_fe(g.pow((u128)(n - 1)));
            dp.zinv = d_aux.as<fe>();
            dp.roots = roots; dp.log_tab = log_tab;
            dp.out = divbuf->as<fe>();
            const uint64_t threads = (n * ce) / ZKB_DIV_RPT;
            k_build_divisors<<<(unsigned)((threads + 127) / 128), 128, 0, stream>>>(dp);
            check_launch();
        }
        p.div = divbuf->as<fe>();
        // Boundary numerators.  Per-point sums cost nl multiplications at each of the ce*n points; combining the asserted
        // columns in coefficient space (nl per coefficient row) and extending the ng combined polynomials once costs
        // nl*n + ng * ce*n * (log2(n)/2 + ~6).  MiMC on one GPU (128 assertions, ce = 8) is 2.7x cheaper that way; the training
        // AIR (ce = 2) and narrow column shards are not, and tiny domains would only pay the extra launches.
        p.bnd_poly = 0;
        {
            const uint64_t direct = (uint64_t)nl * ce * n, poly = (uint64_t)nl * n + (uint64_t)ng * ce * n * (log_n / 2 + 6);
            static const char* force = getenv("ZKB_BOUNDARY_POLY");  // "0" / "1": A/B measurements and tests of both paths
            const bool want = force ? (force[0] == '1') : (n * ce >= ((uint64_t)1 << 16) && direct > 2 * poly);
            if (nl && want) {
                BoundaryGroups bg{};
                bg.n_groups = ng;
                for (uint32_t gi = 0; gi <= ng; gi++) bg.g_off[gi] = p.g_off[gi];
                d_bnd_coef.ensure(n * ng * 16);
                d_bnd_lde.ensure(n * ce * ng * 16);
                k_boundary_combine<<<(unsigned)((n * ZKB_ROW_LANES + 255) / 256), 256, 0, stream>>>(d_polys, (uint32_t)n, ncols, p.a_col, p.a_sel, p.a_coef, p.a_val, bg,
                                                                                        d_bnd_coef.as<fe>());
                check_launch();
                Xform xb{d_bnd_coef.as<fe>(), ng, 0, d_bnd_lde.as<fe>(), ng, 0, ng, log_n, false, true, log_n + log_ce, false, HF()};
                const uint32_t lp = run_xform(xb, d_tmp1, d_tmp2);
                p.bnd_poly = 1;
                p.bnd = LdeMat{d_bnd_lde.as<fe>(), log_n, log_ce, ng, lp, 0, ng, magic16(ng), 0, 0, 0, 0, log_ce};
            }
        }
        const uint64_t points = n * ce;
        // a few hundred points cannot fill the GPU with one thread each: give every point a warp (same values, shorter chain)
        if (points <= 4096 && !p.bnd_poly) k_eval_constraints<32><<<(unsigned)((points * 32 + 127) / 128), 128, 0, stream>>>(p);
        else k_eval_constraints<1><<<(unsigned)((points + 127) / 128), 128, 0, stream>>>(p);
        check_launch();
    }
    // out[i] = sum over ranks of partial[i] (mod p), on every rank.  NCCL cannot add 128-bit field elements, so the reduction is
    // a hand-written reduce-scatter — slice q of every rank's vector goes to rank q (grouped send/recv), which sums the G slices
    // (k_sum_partials) — followed by an all-gather of the summed slices: no rank ever receives G full vectors.
    void mg_field_allreduce(const fe* partial, uint64_t count, fe* out) {
        const uint32_t G = (uint32_t)mg_world;
        if (count % G) throw InvalidArg("vector length must be divisible by the number of GPUs");
        const uint64_t sl = count / G;
        d_mg_b.ensure(count * 16 + sl * 16);
        NK(g_nccl.GroupStart());
        for (uint32_t q = 0; q < G; q++) {
            NK(g_nccl.Send(partial + q * sl, sl * 16, ncclUint8, (int)q, comm, stream));
            NK(g_nccl.Recv(d_mg_b.as<fe>() + q * sl, sl * 16, ncclUint8, (int)q, comm, stream));
        }
        NK(g_nccl.GroupEnd());
        fe* mine = d_mg_b.as<fe>() + count;
        k_sum_partials<<<(unsigned)((sl + 255) / 256), 256, 0, stream>>>(d_mg_b.as<fe>(), G, sl, sl, mine);
        check_launch();
        NK(g_nccl.AllGather(mine, out, sl * 16, ncclUint8, comm, stream));
    }
    // the coefficient powers must be in place (fs_after_trace_root)
    void constraints_eval_dev() {
        if (stage != ST_TRACE) throw StateError("zkb_constraints_eval: trace is not committed");
        t_begin(TS_CONSTR);
        const uint64_t n = air.n, ce = (uint64_t)1 << log_ce;
        d_comp_evals.ensure(n * ce * 16);
        if (!mg_active) {
            constraints_eval_window(lde_mat(), 0, air.w, d_comp_evals.as<fe>());
        } else {
            // column-sharded: partial evaluation over this rank's columns, then a field all-reduce
            const uint32_t wl = air.w / (uint32_t)mg_world;
            d_mg_a.ensure(n * ce * 16);
            constraints_eval_window(lde_mat(), mg_rank * wl, wl, d_mg_a.as<fe>());
            mg_field_allreduce(d_mg_a.as<fe>(), n * ce, d_comp_evals.as<fe>());
        }
        t_end(TS_CONSTR);
        stage = ST_EVAL;
    }
    void constraints_eval(const HF& alpha, uint8_t* evals_out) {
        if (stage != ST_TRACE) throw StateError("zkb_constraints_eval: trace is not committed");
        fs_after_trace_root(nullptr, &alpha);
        constraints_eval_dev();
        if (evals_out) d2h(evals_out, d_comp_evals.p, (air.n << log_ce) * 16);
    }

    // K6.  Leaves the root at d_comp_tree + 8 words and the degree flag in d_flags.
    void constraints_commit_dev() {
        if (stage != ST_EVAL) throw StateError("zkb_constraints_commit: constraints are not evaluated");
        t_begin(TS_COMP);
        const uint64_t n = air.n, N = air.lde_size(), cen = n << log_ce;
        // CompositionPoly::new: interpolate over 3*<w_{ce n}>, then split into c columns of n coefficients
        d_bufA.ensure(cen * 16);
        fe* coef = d_bufA.as<fe>();  // the trace-sized transposed input is dead by now
        {
            Xform x{d_comp_evals.as<fe>(), 1, 0, coef, 1, 0, 1, log_n + log_ce, true, false, 0, false, HF()};
            run_xform(x, d_tmp1, d_tmp2);
            // inv3tab covers exponents < 2^log_N >= ce*n
            // the c*n kept coefficients are scaled; the dropped tail must be zero, else the trace violates the AIR (flag in d_flags)
            // (the flag was cleared by k_fs_trace_root)
            k_scale_pow<<<(unsigned)((cen + 255) / 256), 256, 0, stream>>>(coef, cen, inv3tab, to_fe(HF::from_u64(cen).inv()), (uint64_t)c * n,
                                                                            d_flags.as<uint32_t>());
            check_launch();
        }
        // evaluate the c column polynomials over the LDE domain (panel layout, width c)
        d_comp_lde.ensure(N * c * 16);
        // multi-GPU: every rank extends the columns over its own beta/G cosets only, hashes those rows, and the leaf digests
        // are all-gathered and put in leaf order; the (small) tree is then built by every rank
        const bool cs = mg_coset();
        const uint32_t kc = cs ? (1u << mg_log_kc()) : (uint32_t)air.blowup;
        const uint64_t Nloc = n * kc;
        // (measured twice, rounds 1 and 2: c single-column transforms with 4096-point tiles — two passes at n = 2^20 — beat one
        // 8-wide tile, which shares twiddles and takes the four-copy multiplier but needs a third pass: 5.45 vs 6.64 ms at MiMC 2^20)
        for (uint32_t i = 0; i < c; i++) {
            Xform x{coef + (size_t)i * n, 1, 0, d_comp_lde.as<fe>(), c, i, 1, log_n, false, true, log_N, false, HF()};
            if (cs) { x.coset_lo = (uint32_t)mg_rank * kc; x.coset_cnt = kc; }
            comp_log_p = run_xform(x, d_tmp1, d_tmp2);
        }
        d_comp_tree.ensure(2 * N * 32);
        if (!cs) {
            k_hash_lde_rows<<<(unsigned)((N + 127) / 128), 128, 0, stream>>>(comp_mat(), d_comp_tree.as<uint32_t>() + N * 8, 0, 0);
            check_launch();
        } else {
            d_mg_a.ensure(Nloc * 32); d_mg_b.ensure(N * 32);
            k_hash_lde_rows<<<(unsigned)((Nloc + 127) / 128), 128, 0, stream>>>(comp_mat(), d_mg_a.as<uint32_t>(), 0, 1);
            check_launch();
            NK(g_nccl.AllGather(d_mg_a.p, d_mg_b.p, Nloc * 32, ncclUint8, comm, stream));
            k_permute_coset_items<<<(unsigned)((N * 2 + 255) / 256), 256, 0, stream>>>(d_mg_b.as<uint32_t>(), d_comp_tree.as<uint32_t>() + N * 8, log_n,
                                                                                   log_beta, mg_log_kc(), 8);
            check_launch();
        }
        build_merkle(d_comp_tree.as<uint32_t>(), N);
        t_end(TS_COMP);
        stage = ST_COMP;
    }
    void constraints_commit(uint8_t root_out[32]) {
        constraints_commit_dev();
        uint32_t bad_degree = 0;
        CK(cudaMemcpyAsync(&bad_degree, d_flags.p, 4, cudaMemcpyDeviceToHost, stream));
        take_root(d_comp_tree.as<uint32_t>() + 8, ts.constraint_root, root_out);
        // as the oracle (and a release build of Winterfell) the proof is still produced; it will not verify
        if (bad_degree) ts.comp_degree_ok = 0;
    }

    // K7.  Trace polynomials are held per rank for its own columns (all of them on one GPU); a column-sharded proof
    // all-gathers the 2*w_local evaluations.  z and its powers are read from the device transcript (k_fs_constraint_root);
    // the frame lands in d_fs: [T_j(z) w][T_j(zg) w][H_i(z) c].
    void ood_eval_dev() {
        if (stage != ST_COMP) throw StateError("zkb_ood_eval: constraint commitment is missing");
        t_begin(TS_OOD);
        const uint64_t n = air.n; const uint32_t w = air.w;
        const uint32_t wl = mg_active ? (w / (uint32_t)mg_world) : w;   // columns of d_polys
        const uint32_t R = 64;                                          // k_fs_constraint_root tabulates z^64
        const uint32_t nch = (uint32_t)((n + R - 1) / R);
        uint32_t log_wq = 0; while ((1u << log_wq) < wl) log_wq++;
        const uint32_t nsub = 256u >> log_wq;
        // layout of d_small: [part_z nch*wl][part_zg nch*wl][hpart nt*c][local frame 2wl][gathered 2w][scratch]
        const uint32_t Q = 64;
        const uint32_t nt = (uint32_t)((n + Q - 1) / Q);
        size_t o_pz = 0, o_pzg = o_pz + (size_t)nch * wl, o_hp = o_pzg + (size_t)nch * wl, o_loc = o_hp + (size_t)c * nt,
               o_ga = o_loc + 2 * (size_t)wl, o_sc = o_ga + 2 * (size_t)w, total = o_sc + 64 * 256;
        d_small.ensure(total * 16);
        fe* sm = d_small.as<fe>();
        fe* frame = fs_fe(fs.o_ood);
        fe* cur_out = mg_active ? sm + o_loc : frame;
        fe* nxt_out = mg_active ? sm + o_loc + wl : frame + w;
        // column sums of a [chunks][cols] matrix; many chunks are first folded 64-fold by treating the matrix as
        // [chunks/64][64*cols], so the reduction is spread over 2*cols blocks instead of cols/32
        auto col_sum = [&](const fe* part, uint32_t chunks, uint32_t cols, fe* out) {
            if (chunks >= 4096 && chunks % 64 == 0) {
                k_col_sum<<<(64 * cols + 31) / 32, dim3(32, 32), 0, stream>>>(part, chunks / 64, 64 * cols, sm + o_sc);
                check_launch();
                part = sm + o_sc; chunks = 64;
            }
            k_col_sum<<<(cols + 31) / 32, dim3(32, 32), 0, stream>>>(part, chunks, cols, out);
            check_launch();
        };
        // (a single chunk — traces of <= 64 rows — needs no column sums: the partials are the frame)
        k_ood_partial<<<(nch + nsub - 1) / nsub, 256, 0, stream>>>(d_polys, (uint32_t)n, wl, R, log_wq, dts(), nch == 1 ? cur_out : sm + o_pz,
                                                                   nch == 1 ? nxt_out : sm + o_pzg);
        check_launch();
        if (nch > 1) { col_sum(sm + o_pz, nch, wl, cur_out); col_sum(sm + o_pzg, nch, wl, nxt_out); }
        // H_i(z) from the composition column coefficients (still in d_bufA; replicated on every rank)
        {
            dim3 grid((nt + 255) / 256, c);
            k_poly_eval_partial<<<grid, 256, 0, stream>>>(d_bufA.as<fe>(), (uint32_t)n, Q, dts(), nt == 1 ? frame + 2 * (size_t)w : sm + o_hp);
            check_launch();
            if (nt > 1) col_sum(sm + o_hp, nt, c, frame + 2 * (size_t)w);
        }
        if (mg_active) {
            // per-rank [cur wl][next wl] blocks -> the global frame [cur w][next w]: two strided copies on the device
            NK(g_nccl.AllGather(sm + o_loc, sm + o_ga, 2 * (size_t)wl * 16, ncclUint8, comm, stream));
            for (uint32_t h = 0; h < 2; h++)
                CK(cudaMemcpy2DAsync(frame + (size_t)h * w, (size_t)wl * 16, sm + o_ga + (size_t)h * wl, 2 * (size_t)wl * 16, (size_t)wl * 16, (size_t)mg_world,
                                     cudaMemcpyDeviceToDevice, stream));
        }
        t_end(TS_OOD);
        stage = ST_OOD;
    }
    void ood_fetch() {   // host copy of the frame (staged API)
        const uint32_t w = air.w;
        std::vector<HF> host(2 * (size_t)w + c);
        d2h(host.data(), fs_fe(fs.o_ood), host.size() * 16);
        ood_cur.assign(host.begin(), host.begin() + w);
        ood_next.assign(host.begin() + w, host.begin() + 2 * (size_t)w);
        ood_h.assign(host.begin() + 2 * (size_t)w, host.end());
    }
    void ood_eval(const HF& z_) {
        if (stage != ST_COMP) throw StateError("zkb_ood_eval: constraint commitment is missing");
        z = z_; zg = z * HF::root_of_unity(log_n);
        fs_after_constraint_root(nullptr, &z_);
        ood_eval_dev();
        ood_fetch();
    }

    // K8.  The DEEP coefficients gamma^0.. (trace columns, then composition columns: draw_algebraic [A.5]) and the constants
    // A(z), (A+B)(z), A(zg) are in device memory (k_fs_ood).
    void deep_compose_dev() {
        if (stage != ST_OOD) throw StateError("zkb_deep_compose: OOD frame is missing");
        t_begin(TS_DEEP);
        const uint64_t n = air.n, N = air.lde_size(); const uint32_t w = air.w;
        const fe* gamma = fs_fe(fs.o_gamma);
        d_ab.ensure(n * 2 * 16);
        if (!mg_active) {
            k_deep_combine<<<(unsigned)((n * ZKB_ROW_LANES + 255) / 256), 256, 0, stream>>>(d_polys, (uint32_t)n, w, gamma, d_bufA.as<fe>(), c, gamma + w, d_ab.as<fe>());
            check_launch();
        } else {
            // partial A over this rank's columns -> field all-reduce -> add the (replicated) H part
            const uint32_t wl = w / (uint32_t)mg_world;
            d_mg_a.ensure(n * 2 * 16);
            k_deep_combine<<<(unsigned)((n * ZKB_ROW_LANES + 255) / 256), 256, 0, stream>>>(d_polys, (uint32_t)n, wl, gamma + (size_t)mg_rank * wl, d_bufA.as<fe>(), 0,
                                                                              gamma + w, d_mg_a.as<fe>());
            check_launch();
            mg_field_allreduce(d_mg_a.as<fe>(), 2 * n, d_ab.as<fe>());
            k_deep_add_h<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(d_ab.as<fe>(), (uint32_t)n, d_bufA.as<fe>(), c, gamma + w);
            check_launch();
        }
        d_ab_lde.ensure(N * 2 * 16);
        d_deep.ensure(N * 16);
        if (!mg_coset()) {
            Xform x{d_ab.as<fe>(), 2, 0, d_ab_lde.as<fe>(), 2, 0, 2, log_n, false, true, log_N, false, HF()};
            ab_log_p = run_xform(x, d_tmp1, d_tmp2);
            if (N <= 8192) k_deep_eval<1><<<(unsigned)((N + 127) / 128), 128, 0, stream>>>(ab_mat(), dts(), roots, log_tab, d_deep.as<fe>(), 0);
            else k_deep_eval<ZKB_DEEP_RPT><<<(unsigned)((N / ZKB_DEEP_RPT + 127) / 128), 128, 0, stream>>>(ab_mat(), dts(), roots, log_tab, d_deep.as<fe>(), 0);
            check_launch();
        } else {
            // multi-GPU: extend and evaluate on this rank's cosets, all-gather the evaluations, restore natural order
            const uint32_t kc = 1u << mg_log_kc();
            const uint64_t Nloc = n * kc;
            Xform x{d_ab.as<fe>(), 2, 0, d_ab_lde.as<fe>(), 2, 0, 2, log_n, false, true, log_N, false, HF()};
            x.coset_lo = (uint32_t)mg_rank * kc; x.coset_cnt = kc;
            ab_log_p = run_xform(x, d_tmp1, d_tmp2);
            d_mg_a.ensure(Nloc * 16); d_mg_b.ensure(N * 16);
            const uint64_t threads = Nloc / ZKB_DEEP_RPT;
            k_deep_eval<ZKB_DEEP_RPT><<<(unsigned)((threads + 127) / 128), 128, 0, stream>>>(ab_mat(), dts(), roots, log_tab, d_mg_a.as<fe>(), 1);
            check_launch();
            NK(g_nccl.AllGather(d_mg_a.p, d_mg_b.p, Nloc * 16, ncclUint8, comm, stream));
            k_permute_coset_items<<<(unsigned)((N + 255) / 256), 256, 0, stream>>>(d_mg_b.as<uint32_t>(), d_deep.as<uint32_t>(), log_n, log_beta,
                                                                               mg_log_kc(), 4);
            check_launch();
        }
        t_end(TS_DEEP);
        if (d_fri_evals.size() < fri_layers + 1) { d_fri_evals.resize(fri_layers + 1); d_fri_tree.resize(fri_layers + 1); }
        fri_layer = 0; fri_committed = false;
        stage = ST_DEEP;
    }
    void deep_compose(const HF& alpha) {
        if (stage != ST_OOD) throw StateError("zkb_deep_compose: OOD frame is missing");
        deep_alpha = alpha;
        fs_after_ood(false, &alpha);
        deep_compose_dev();
    }

    // K9
    const fe* fri_cur_evals() const { return fri_layer == 0 ? d_deep.as<fe>() : d_fri_evals[fri_layer].as<fe>(); }
    uint64_t fri_domain(uint32_t layer) const { return air.lde_size() >> (air.log_folding() * layer); }
    uint64_t fri_rows(uint32_t layer) const { return fri_domain(layer) >> air.log_folding(); }   // leaves of layer `layer`
    // leaves the layer's root at d_fri_tree[layer] + 8 words
    void fri_commit_layer_dev() {
        if (stage != ST_DEEP || fri_layer >= fri_layers || fri_committed) throw StateError("zkb_fri_commit_layer: out of order");
        const uint64_t rows = fri_rows(fri_layer);
        DevBuf& tree = d_fri_tree[fri_layer];
        tree.ensure(2 * rows * 32);
        k_hash_strided_rows<<<(unsigned)((rows + 127) / 128), 128, 0, stream>>>(fri_cur_evals(), rows, air.folding, tree.as<uint32_t>() + rows * 8);
        check_launch();
        build_merkle(tree.as<uint32_t>(), rows);
        fri_committed = true;
    }
    // the public transcript keeps the first 16 layers' roots and challenges; the proof carries every layer
    static constexpr uint32_t TS_FRI_SLOTS = sizeof(zkb_transcript::fri_roots) / sizeof(zkb_transcript::fri_roots[0]);
    void fri_commit_layer(uint8_t root_out[32]) {
        fri_commit_layer_dev();
        uint8_t spare[32];
        take_root(d_fri_tree[fri_layer].as<uint32_t>() + 8, fri_layer < TS_FRI_SLOTS ? ts.fri_roots[fri_layer] : spare, root_out);
    }
    // the folding challenge is dts()->fri_alpha[fri_layer]
    void fri_fold_dev() {
        if (stage != ST_DEEP || !fri_committed) throw StateError("zkb_fri_fold: commit the layer first");
        const uint64_t rows = fri_rows(fri_layer);
        DevBuf& nxt = d_fri_evals[fri_layer + 1];
        nxt.ensure(rows * sizeof(fe));
        FriFoldParams p{};
        p.in = fri_cur_evals(); p.out = nxt.as<fe>(); p.log_m = log2u(fri_domain(fri_layer));
        p.alpha = &dts()->fri_alpha[fri_layer]; p.inv3 = to_fe(HF::from_u64(3).inv()); p.inv_f = to_fe(HF::from_u64(air.folding).inv());
        HF wi = HF::root_of_unity(air.log_folding()).inv(), x = HF::raw(1);
        for (uint32_t q = 0; q < air.folding / 2; q++) { p.wf_inv[q] = to_fe(x); x = x * wi; }
        p.roots = roots; p.log_tab = log_tab;
        const dim3 grid((unsigned)((rows + 127) / 128)), block(128);
        switch (air.log_folding()) {
            case 1: k_fri_fold<1><<<grid, block, 0, stream>>>(p); break;
            case 2: k_fri_fold<2><<<grid, block, 0, stream>>>(p); break;
            case 3: k_fri_fold<3><<<grid, block, 0, stream>>>(p); break;
            case 4: k_fri_fold<4><<<grid, block, 0, stream>>>(p); break;
            default: throw InvalidArg("FRI folding factor must be one of 2, 4, 8, 16");
        }
        check_launch();
        fri_layer++;
        fri_committed = false;
        ts.n_fri_layers = fri_layer;
    }
    void fri_fold(const HF& alpha) {
        if (stage != ST_DEEP || !fri_committed) throw StateError("zkb_fri_fold: commit the layer first");
        if (fri_layer < TS_FRI_SLOTS) alpha.to_bytes(ts.fri_alphas[fri_layer]);
        fs_upload(&dts()->fri_alpha[fri_layer], alpha);
        fri_fold_dev();
    }
    // FriProver::set_remainder  [A.10]: interpolate the last layer over 3*<w_M> on the device (the ordinary inverse transform
    // + the offset scaling of CompositionPoly::new), keep M/beta coefficients reversed, commit them (k_fs_remainder)
    void fri_remainder_dev(bool with_coin) {
        if (stage != ST_DEEP || fri_layer != fri_layers || fri_committed) throw StateError("zkb_fri_remainder: fold all layers first");
        const uint64_t M = fri_domain(fri_layer);
        const uint32_t rs = (uint32_t)(M / air.blowup);
        // (rs == 0 — the last layer is shorter than the blowup — yields an empty remainder, which the verifier rejects as it
        // does Winterfell's: the options do not fit the trace length)
        if (rs > fs.rem_cap || rs > 1024) throw InvalidArg("unsupported FRI remainder size");
        d_rem_coef.ensure(M * 16);
        Xform x{fri_cur_evals(), 1, 0, d_rem_coef.as<fe>(), 1, 0, 1, log2u(M), true, false, 0, false, HF()};
        run_xform(x, d_tmp1, d_tmp2);
        k_fs_remainder<<<1, ZKB_FS_THREADS, 0, stream>>>(dts(), d_rem_coef.as<fe>(), rs, fs_fe(fs.o_rem), with_coin ? 1u : 0u, inv3tab.lo, inv3tab.hi, inv3tab.l1,
                                                         to_fe(HF::from_u64(M).inv()));
        check_launch();
        stage = ST_FRI_DONE;
    }
    void fri_remainder(uint8_t commitment_out[32]) {
        fri_remainder_dev(false);
        const uint32_t rs = (uint32_t)(fri_domain(fri_layer) / air.blowup);
        parts.remainder.assign(rs, HF());
        CK(cudaMemcpyAsync(parts.remainder.data(), fs_fe(fs.o_rem), (size_t)rs * 16, cudaMemcpyDeviceToHost, stream));
        take_root(dts()->rem_commit, ts.remainder_commitment, commitment_out);
    }

    // K10: the smallest nonce >= 1 for `t->seed` into t->nonce, which must hold ~0; it stays ~0 when there is none up to 2^44
    void enqueue_grind(DevTs* t, uint32_t bits) {
        k_fs_grind<<<(unsigned)sm_count * 8, 256, 0, stream>>>(t, bits, 1ull << 44);
        check_launch();
    }
    // staged zkb_grind: a scratch transcript, so that the proof's own (d_fs) stays untouched
    uint64_t grind(const uint8_t seed[32], uint32_t bits) {
        if (bits > 32) throw InvalidArg("grinding factor must be <= 32");
        d_gather.ensure(sizeof(DevTs));
        DevTs* t = d_gather.as<DevTs>();
        const unsigned long long none = ~0ull;
        h2d_small(t->seed, seed, 32);
        h2d_small(&t->nonce, &none, 8);
        enqueue_grind(t, bits);
        unsigned long long nonce;
        d2h(&nonce, &t->nonce, 8);
        if (nonce == ~0ull) throw std::runtime_error("proof-of-work nonce not found");
        return nonce;
    }

    // K11 (TraceLde::query, ConstraintCommitment::query, FriProver::build_proof): rows and full authentication paths of
    // commitments [first, first + n) at the J.q positions J.pos, into J.rows_out / J.paths_out, in one launch
    void open_commitments(OpenJobs& J, uint32_t first, uint32_t n) {
        J.first = first;
        J.mat[0] = mg_active ? lde_rows_mat() : lde_mat(); J.mat[1] = comp_mat();
        J.cap = d_cap.as<uint32_t>(); J.lsub = log_N - (mg_active ? log_g : 0); J.rank = mg_active ? (uint32_t)mg_rank : 0;
        uint32_t items = 0;
        for (uint32_t t = first; t < first + n; t++) {
            const FsTree& tr = fs.trees[t];
            J.depth[t] = tr.depth; J.width[t] = tr.width;
            if (t == 0) J.heap[t] = d_tree.as<uint32_t>();
            else if (t == 1) J.heap[t] = d_comp_tree.as<uint32_t>();
            else {
                const uint32_t l = t - 2;
                J.fri_evals[l] = l == 0 ? d_deep.as<fe>() : d_fri_evals[l].as<fe>();
                J.fri_rows[l] = fri_rows(l);
                J.heap[t] = d_fri_tree[l].as<uint32_t>();
            }
            items = std::max(items, J.q * tr.width + J.q * tr.depth * 2);
        }
        k_open_all<<<dim3((items + 127) / 128, n), 128, 0, stream>>>(J);
        check_launch();
    }
    // staged zkb_query: one commitment at the caller's positions
    void query(uint32_t which, const std::vector<uint32_t>& pos, std::vector<uint8_t>& rows, std::vector<uint8_t>& paths) {
        if (mg_active) throw StateError("zkb_query: not available for a column-sharded proof");
        const uint32_t np = (uint32_t)pos.size();
        if (np == 0 || np > 255) throw InvalidArg("bad number of query positions");
        if (which >= fs.trees.size()) throw InvalidArg("no such FRI layer");
        const FsTree& tr = fs.trees[which];
        const uint64_t domain = which < 2 ? air.lde_size() : fri_rows(which - 2);
        for (uint32_t p : pos) if (p >= domain) throw InvalidArg("query position out of range");
        // device scratch: [positions np u32][rows np*width fe][full paths np*depth digests]
        const size_t o_rows = 1024, rb = (size_t)np * tr.width * 16, pb = (size_t)np * tr.depth * 32;
        d_gather.ensure(o_rows + rb + pb);
        uint8_t* base = d_gather.as<uint8_t>();
        h2d_small(base, pos.data(), np * 4);
        OpenJobs J{};
        J.q = np; J.pos = (const uint32_t*)base;
        J.rows_out[which] = (fe*)(base + o_rows); J.paths_out[which] = (uint32_t*)(base + o_rows + rb);
        open_commitments(J, which, 1);
        std::vector<uint8_t> host(rb + pb);
        d2h(host.data(), base + o_rows, host.size());
        pick_openings(host.data(), host.data() + rb, tr.width, tr.depth, pos, pos, (uint32_t)(domain - 1), rows, paths);
    }

    // ==========================================================================================================
    // Prover::prove  (SURVEY §3.2).  One GPU: the Fiat-Shamir channel runs on the device (csrc/coin.cuh) — the host enqueues
    // every stage back to back, waits ONCE on a blocking event, and assembles Proof::to_bytes() from a single download
    // (transcript, OOD frame, remainder, and for every commitment the rows and full authentication paths at the raw query
    // positions, from which the host picks what BatchMerkleProof needs after sorting / deduplicating the positions).
    // sharded = true: `cols` / `d_trace_in` hold only this rank's w/G columns and the proof is produced cooperatively by all
    // ranks of the NCCL communicator, the channel replicated on every rank's device (every rank returns the same bytes); the
    // openings are completed by one all-reduce before the download, so a sharded proof also waits on the device once.
    std::vector<uint8_t> prove(const zkb_air_desc* desc, const uint8_t* const* cols, const fe* d_trace_in, uint64_t force_nonce,
                               bool sharded = false) {
        static const bool host_prof = getenv("ZKB_HOST_PROFILE") != nullptr;   // diagnostics: host phases of a proof on stderr
        static const bool graphs_on = !(getenv("ZKB_GRAPH") && getenv("ZKB_GRAPH")[0] == '0');
        const auto hp0 = std::chrono::steady_clock::now();
        begin(desc);
        const auto hp1 = std::chrono::steady_clock::now();
        t_begin(TS_TOTAL);
        if (!d_trace_in && !cols) throw InvalidArg("null trace columns");
        // Small proofs are launch-bound (tens of 3-8 us kernels): from the second proof of a shape on, the whole enqueue sequence
        // is captured into a CUDA graph and replayed with one launch.  What varies between proofs of a shape — coin seed,
        // assertion values, AIR parameters (uploaded by begin()) and the trace — sits at fixed device addresses.
        const bool small = graphs_on && !sharded && !force_nonce && ((air.lde_size() * air.w) >> 22) == 0;
        if (!small) enqueue_proof(cols, d_trace_in, force_nonce, sharded);
        else {
            const fe* src = d_trace_in ? d_trace_in : upload_cols(cols, air.w, air.n, d_trace);
            std::string key((const char*)desc, offsetof(zkb_air_desc, pub_elems));
            key.append((const char*)desc->assert_cols, desc->n_assertions * 4).append((const char*)desc->assert_steps, desc->n_assertions * 8);
            // AIR parameters are part of the key: the MiMC round constants are baked into the evaluator's periodic-column table,
            // which a replay does not rebuild (the aggregation factor k is read from the per-proof inputs either way)
            key.append((const char*)&desc->n_params, 8).append((const char*)desc->params, desc->n_params * 16).append((const char*)&src, sizeof(src));
            GraphEntry& g = graphs[key];
            if (g.exec && g.epoch != g_alloc_epoch.load()) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; }
            if (g.exec) {
                CK(cudaGraphLaunch(g.exec, stream));
                launches += g.launches;
            } else if (g.seen == 0) {
                g.seen = 1;                              // first proof of a shape: eager (buffers, tables and caches get built)
                enqueue_proof(nullptr, src, 0);
            } else {
                const uint64_t e0 = g_alloc_epoch.load(), l0 = launches;
                cudaGraph_t graph = nullptr;
                bool ok = false;
                // captured on the context's side stream (the caller's stream may be the legacy default stream, which cannot be
                // captured); nothing executes during a capture, and the instantiated graph is launched into the caller's stream
                cudaStream_t user_stream = stream;
                stream = copy_stream;
                cudaError_t ce = cudaStreamBeginCapture(stream, cudaStreamCaptureModeRelaxed);
                if (ce == cudaSuccess) {
                    capturing = true;
                    try { enqueue_proof(nullptr, src, 0); ok = true; } catch (const std::exception&) {}
                    capturing = false;
                    ce = cudaStreamEndCapture(stream, &graph);
                }
                stream = user_stream;
                if (ok && ce == cudaSuccess && graph && g_alloc_epoch.load() == e0) {
                    cudaGraphExec_t ex = nullptr;
                    if (cudaGraphInstantiate(&ex, graph, 0) == cudaSuccess) { g.exec = ex; g.epoch = e0; g.launches = launches - l0; }
                }
                if (graph) cudaGraphDestroy(graph);
                cudaGetLastError();                      // a failed capture leaves a sticky-looking (but cleared here) error
                launches = l0;
                begin_stage_reset();
                if (g.exec) { CK(cudaGraphLaunch(g.exec, stream)); launches += g.launches; }
                else { g.seen = 0; enqueue_proof(nullptr, src, 0); }   // could not capture (e.g. a buffer grew): run it eagerly
            }
        }
        t_end(TS_TOTAL);
        const auto hp2 = std::chrono::steady_clock::now();
        // small proofs: spin on the stream (a blocking wait costs a wake-up, tens of microseconds, which is a large part of a
        // sub-millisecond proof); large proofs: sleep on the event so that a lane does not burn a host core while the GPU works
        if ((air.lde_size() * air.w) >> 22) { CK(cudaEventRecord(ev_done, stream)); CK(cudaEventSynchronize(ev_done)); }
        else CK(cudaStreamSynchronize(stream));
        const auto hp3 = std::chrono::steady_clock::now();
        stage = ST_QUERY;
        std::vector<uint8_t> out = assemble_proof();
        if (host_prof) {
            const auto hp4 = std::chrono::steady_clock::now();
            auto us = [](auto a, auto b) { return std::chrono::duration<double, std::micro>(b - a).count(); };
            fprintf(stderr, "[zkb host] begin %.1f us, enqueue %.1f us, wait %.1f us, assemble %.1f us, launches so far %llu\n", us(hp0, hp1), us(hp1, hp2),
                    us(hp2, hp3), us(hp3, hp4), (unsigned long long)launches);
        }
        return out;
    }
    // host-side stage bookkeeping back to "begun" (after a capture walked it through all stages without executing anything)
    void begin_stage_reset() { stage = ST_BEGUN; fri_layer = 0; fri_committed = false; }

    // Everything between "the trace is available" and "the last byte of the proof is on its way to the host": no host
    // synchronisation and no per-proof upload — the sequence depends on the shape only, which is what makes it capturable.
    void enqueue_proof(const uint8_t* const* cols, const fe* d_trace_in, uint64_t force_nonce, bool sharded = false) {
        if (sharded) trace_commit_mg(cols, d_trace_in);
        else if (d_trace_in) trace_commit_dev(nullptr, d_trace_in);
        else trace_commit_dev(cols, nullptr);
        fs_after_trace_root((sharded ? d_cap : d_tree).as<uint32_t>() + 8, nullptr);   // channel.commit_trace; get_constraint_composition_coeffs
        constraints_eval_dev();
        constraints_commit_dev();
        fs_after_constraint_root(d_comp_tree.as<uint32_t>() + 8, nullptr);   // channel.commit_constraints; get_ood_point
        ood_eval_dev();
        fs_after_ood(true, nullptr);                                   // send_ood_*; get_deep_composition_coeffs
        deep_compose_dev();
        enqueue_fri_to_positions(force_nonce);
        {   // every commitment at the raw positions
            OpenJobs J{};
            uint8_t* base = d_fs.as<uint8_t>();
            J.q = air.num_queries; J.pos = dts()->positions;
            for (size_t t = 0; t < fs.trees.size(); t++) { J.rows_out[t] = (fe*)(base + fs.trees[t].o_rows); J.paths_out[t] = (uint32_t*)(base + fs.trees[t].o_paths); }
            open_commitments(J, 0, (uint32_t)fs.trees.size());
            // sharded: trace rows and paths, and coset-sharded composition rows, are the owner's value or zero on each rank
            if (mg_active) {
                const size_t o = fs.trees[0].o_rows;
                NK(g_nccl.AllReduce(base + o, base + o, fs.trees[1].o_paths - o, ncclUint8, ncclMax, comm, stream));
            }
        }
        t_end(TS_QUERY);
        CK(cudaMemcpyAsync(h_out, d_fs.p, fs.host_bytes, cudaMemcpyDeviceToHost, stream));
    }

    // FRI layers, remainder, proof of work and query positions: replicated on every rank of a sharded proof
    void enqueue_fri_to_positions(uint64_t force_nonce) {
        t_begin(TS_FRI);
        for (uint32_t l = 0; l < fri_layers; l++) {                    // FriProver::build_layers
            fri_commit_layer_dev();
            k_fs_fri_root<<<1, 32, 0, stream>>>(dts(), d_fri_tree[l].as<uint32_t>() + 8, l);
            check_launch();
            fri_fold_dev();
        }
        fri_remainder_dev(true);
        t_end(TS_FRI);
        t_begin(TS_GRIND);
        if (force_nonce) { const unsigned long long v = force_nonce; h2d_small(&dts()->nonce, &v, 8); }
        else enqueue_grind(dts(), air.grinding);                       // grind_query_seed
        t_end(TS_GRIND);
        t_begin(TS_QUERY);
        k_fs_positions<<<1, ZKB_FS_THREADS, 0, stream>>>(dts(), air.num_queries, (uint32_t)(air.lde_size() - 1));   // get_query_positions
        check_launch();
    }

    // Proof assembly from the single download: sort / dedup the positions (get_query_positions), fold them per FRI layer
    // (fold_positions), select rows, and build every BatchMerkleProof from the full paths gathered on the device — each node of
    // a batch proof is the sibling of an ancestor of some queried leaf, so it is in one of those paths.
    // transcript, commitments, OOD frame, remainder, nonce and the sorted / deduplicated positions from the single download;
    // returns the raw positions
    std::vector<uint32_t> assemble_transcript() {
        const DevTs* h = reinterpret_cast<const DevTs*>(h_out);
        if (h->coin_failed) throw std::runtime_error("random coin failed to draw a field element");
        if (h->nonce == ~0ull) throw std::runtime_error("proof-of-work nonce not found");
        const uint32_t w = air.w, q = air.num_queries;
        memcpy(ts.trace_root, h->trace_root, 32); memcpy(ts.constraint_root, h->constraint_root, 32);
        memcpy(ts.remainder_commitment, h->rem_commit, 32);
        memcpy(ts.constraint_alpha, &h->alpha, 16); memcpy(ts.z, &h->z, 16); memcpy(ts.deep_alpha, &h->deep_alpha, 16);
        ts.n_fri_layers = fri_layers;
        if (h->bad_degree) ts.comp_degree_ok = 0;
        auto dg = [](const uint32_t* p) { Digest32 d; memcpy(d.b, p, 32); return d; };
        parts.commitments.push_back(dg(h->trace_root));
        parts.commitments.push_back(dg(h->constraint_root));
        for (uint32_t l = 0; l < fri_layers; l++) {
            parts.commitments.push_back(dg(h->fri_roots[l]));
            if (l < TS_FRI_SLOTS) { memcpy(ts.fri_roots[l], h->fri_roots[l], 32); memcpy(ts.fri_alphas[l], &h->fri_alpha[l], 16); }
        }
        parts.commitments.push_back(dg(h->rem_commit));
        const HF* frame = reinterpret_cast<const HF*>(h_out + fs.o_ood);
        parts.ood_trace_interleaved.resize(2 * (size_t)w);   // [T_0(z), T_0(zg), T_1(z), ...]  [A.5]
        for (uint32_t j = 0; j < w; j++) { parts.ood_trace_interleaved[2 * j] = frame[j]; parts.ood_trace_interleaved[2 * j + 1] = frame[w + j]; }
        parts.ood_h.assign(frame + 2 * (size_t)w, frame + 2 * (size_t)w + c);
        const uint32_t rs = (uint32_t)(fri_domain(fri_layers) / air.blowup);
        const HF* rem = reinterpret_cast<const HF*>(h_out + fs.o_rem);
        parts.remainder.assign(rem, rem + rs);
        parts.nonce = h->nonce; ts.pow_nonce = h->nonce;
        std::vector<uint32_t> raw(h->positions, h->positions + q);
        positions = raw;
        std::sort(positions.begin(), positions.end());
        positions.erase(std::unique(positions.begin(), positions.end()), positions.end());
        parts.n_unique = (uint32_t)positions.size();
        ts.n_positions = parts.n_unique;
        for (size_t i = 0; i < positions.size() && i < 256; i++) ts.positions[i] = positions[i];
        return raw;
    }
    // One commitment from the rows `hrows` and full paths `hpaths` gathered at the positions `raw`: the rows of `pos` (each found
    // among the raw positions reduced by `mask`) and the batch proof of `pos`
    static void pick_openings(const uint8_t* hrows, const uint8_t* hpaths, uint32_t width, uint32_t depth, const std::vector<uint32_t>& raw,
                              const std::vector<uint32_t>& pos, uint32_t mask, std::vector<uint8_t>& rows, std::vector<uint8_t>& paths) {
        const size_t rb = (size_t)width * 16;
        std::vector<std::pair<uint32_t, uint32_t>> first(raw.size());   // (reduced position, a raw index that carries it), sorted
        for (uint32_t i = 0; i < raw.size(); i++) first[i] = {raw[i] & mask, i};
        std::sort(first.begin(), first.end());
        auto raw_index_in = [&](uint64_t lo, uint64_t hi_excl) -> uint32_t {   // a raw index whose reduced position is in [lo, hi)
            auto it = std::lower_bound(first.begin(), first.end(), std::make_pair((uint32_t)lo, 0u));
            if (it == first.end() || it->first >= hi_excl) throw std::runtime_error("internal error: opening not gathered");
            return it->second;
        };
        rows.resize(pos.size() * rb);
        for (size_t i = 0; i < pos.size(); i++) memcpy(&rows[i * rb], hrows + (size_t)raw_index_in(pos[i], (uint64_t)pos[i] + 1) * rb, rb);
        // node `hi` of the heap sits `lv` levels above the leaves and is the sibling of an ancestor of some queried leaf: that
        // leaf lies under hi ^ 1, and its gathered path holds `hi` at position lv
        std::vector<std::vector<uint64_t>> plan = plan_batch_proof(depth, pos);
        std::vector<uint8_t> gathered;
        for (auto& v : plan)
            for (uint64_t hi : v) {
                const uint32_t lv = depth - (63u - (uint32_t)__builtin_clzll(hi));
                const uint64_t anc = hi ^ 1ull, lo = (anc << lv) - ((uint64_t)1 << depth);
                const uint8_t* d = hpaths + ((size_t)raw_index_in(lo, lo + ((uint64_t)1 << lv)) * depth + lv) * 32;
                gathered.insert(gathered.end(), d, d + 32);
            }
        paths = batch_proof_bytes(depth, plan, gathered.data());
    }
    std::vector<uint8_t> assemble_proof() {
        const std::vector<uint32_t> raw = assemble_transcript();
        auto open = [&](const FsTree& tr, const std::vector<uint32_t>& pos, uint32_t mask, std::vector<uint8_t>& rows, std::vector<uint8_t>& paths) {
            pick_openings(h_out + tr.o_rows, h_out + tr.o_paths, tr.width, tr.depth, raw, pos, mask, rows, paths);
        };
        open(fs.trees[0], positions, (uint32_t)(air.lde_size() - 1), parts.trace_rows, parts.trace_paths);
        open(fs.trees[1], positions, (uint32_t)(air.lde_size() - 1), parts.comp_rows, parts.comp_paths);
        parts.fri_rows.resize(fri_layers); parts.fri_paths.resize(fri_layers);
        std::vector<uint32_t> fpos = positions;
        uint64_t dom = air.lde_size();
        for (uint32_t l = 0; l < fri_layers; l++) {
            fpos = fold_positions(fpos, dom, air.folding);
            dom /= air.folding;
            open(fs.trees[2 + l], fpos, (uint32_t)(dom - 1), parts.fri_rows[l], parts.fri_paths[l]);
        }
        return serialize_proof(air, parts);
    }

    // ==========================================================================================================
    // winter-verifier `verify` for a batch (csrc/verify.cuh).  Host: parse every proof and check every length, count and depth
    // against the AIR before anything that depends on it is uploaded; pack the parsed sections into one pinned staging buffer
    // (one copy up).  Device: the channel and the OOD check.  Host, after the first synchronisation: positions, position folding
    // and the Merkle merge plans.  Device: leaves, merges level by level, roots, DEEP and FRI checks.  Second synchronisation:
    // the verdicts.  Host-found failures and device-found failures are ordinals of the same order; the smaller one wins.
    struct VItem {
        AirSpec air;
        ProofLayout L;
        uint32_t fail = VO_ACCEPT, nl = 0, c = 0;
        std::vector<BatchProofLayout> bp;                         // 0 trace, 1 constraint, 2 + l FRI layer l
        std::vector<std::vector<std::vector<uint32_t>>> node_ids; // digest ids of bp[k].nodes
        uint64_t o_comm = 0, o_ood = 0, o_h = 0, o_rem = 0, o_trows = 0, o_crows = 0;
        std::vector<uint64_t> o_fri;
        std::vector<uint32_t> positions;                          // sorted, unique
    };
    static void grow_pinned(uint8_t*& p, size_t& cap, size_t need) {
        if (need <= cap) return;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        CK(cudaHostAlloc((void**)&p, need, cudaHostAllocDefault));
        cap = need;
    }
    static int32_t verdict_of(uint32_t ord) {
        static const int32_t head[VO_FRI0] = {ZKB_VERIFY_MALFORMED, ZKB_VERIFY_TRACE_INFO, ZKB_VERIFY_OPTIONS, ZKB_VERIFY_COMMITMENTS,
                                              ZKB_VERIFY_OOD_FRAME, ZKB_VERIFY_OOD_CONSISTENCY, ZKB_VERIFY_POW, ZKB_VERIFY_UNIQUE_QUERIES,
                                              ZKB_VERIFY_TRACE_VALUES, ZKB_VERIFY_CONSTRAINT_VALUES, ZKB_VERIFY_MALFORMED, ZKB_VERIFY_MALFORMED,
                                              ZKB_VERIFY_MALFORMED, ZKB_VERIFY_TRACE_MERKLE, ZKB_VERIFY_MALFORMED, ZKB_VERIFY_CONSTRAINT_MERKLE};
        static const int32_t layer[VO_FRI_STEP] = {ZKB_VERIFY_FRI_VALUES, ZKB_VERIFY_MALFORMED, ZKB_VERIFY_MALFORMED, ZKB_VERIFY_FRI_MERKLE,
                                                   ZKB_VERIFY_FRI_FOLDING, ZKB_VERIFY_FRI_TRUNCATION};
        static const int32_t rem[3] = {ZKB_VERIFY_REMAINDER_DEGREE, ZKB_VERIFY_REMAINDER_COMMITMENT, ZKB_VERIFY_REMAINDER_FOLDING};
        if (ord < VO_FRI0) return head[ord];
        if (ord < VO_REM) return layer[(ord - VO_FRI0) % VO_FRI_STEP];
        if (ord < VO_ACCEPT) return rem[ord - VO_REM];
        return ZKB_VERIFY_OK;
    }

    // fn(i) for every i < n, on up to one host thread per core when n is large enough to pay for starting them; the first
    // exception thrown is rethrown once every thread has finished
    template <class F>
    static void host_parallel(uint32_t n, F&& fn) {
        const uint32_t T = n < 16 ? 1u : std::min<uint32_t>(n / 8, std::max(1u, std::thread::hardware_concurrency()));
        if (T <= 1) { for (uint32_t i = 0; i < n; i++) fn(i); return; }
        std::vector<std::thread> th;
        std::exception_ptr err;
        std::mutex m;
        for (uint32_t t = 0; t < T; t++)
            th.emplace_back([&, t] {
                try { for (uint32_t i = t; i < n; i += T) fn(i); }
                catch (...) { std::lock_guard<std::mutex> g(m); if (!err) err = std::current_exception(); }
            });
        for (auto& x : th) x.join();
        if (err) std::rethrow_exception(err);
    }
    // digest ids a proof's plan gives its own leaves and merges, relocated after every proof is planned
    static constexpr uint32_t LOCAL_ID = 0x80000000u;
    struct VPlan {
        std::vector<VLeafJob> leaves;
        std::vector<std::vector<MergeJob>> merges;
        std::vector<VRootJob> roots;
        std::vector<VEvalJob> evals;
        uint32_t ids = 0;
    };

    void verify_batch(const zkb_air_desc* const* airs, const uint8_t* const* proofs, const uint64_t* lens, uint32_t count, int32_t* verdicts,
                      zkb_transcript* tss) {
        if (count == 0) return;
        if (!airs || !proofs || !lens || !verdicts) throw InvalidArg("null argument");
        CK(cudaSetDevice(device));
        static const bool host_prof = getenv("ZKB_HOST_PROFILE") != nullptr;   // diagnostics: host phases of a call on stderr
        const auto hp0 = std::chrono::steady_clock::now();
        std::vector<VItem> it(count);
        for (uint32_t i = 0; i < count; i++) if (!proofs[i]) throw InvalidArg("null proof");
        auto al = [](size_t x) { return (x + 15) & ~(size_t)15; };
        size_t off = al((size_t)count * 4);               // [verdicts][VProof x count][roots of unity][per proof sections][nodes]
        const size_t o_proofs = off;
        off = al(off + (size_t)count * sizeof(VProof));
        const size_t o_roots = off;
        off += 41 * 16;
        // ---- parse: everything the sequential verifier checks before its first draw, and every position-independent check ----
        host_parallel(count, [&](uint32_t i) {
            VItem& x = it[i];
            x.air = AirSpec::from_desc(airs[i]);
            const AirSpec& a = x.air;
            const uint8_t* b = proofs[i];
            auto fail = [&](uint32_t ord) { x.fail = std::min(x.fail, ord); };
            if (!parse_proof(b, (size_t)lens[i], x.L)) { fail(VO_MALFORMED); return; }
            ProofLayout& L = x.L;
            const uint8_t want[8] = {(uint8_t)a.num_queries, (uint8_t)a.blowup, (uint8_t)a.grinding, (uint8_t)a.field_ext, (uint8_t)a.folding,
                                     (uint8_t)a.rem_max_degree, (uint8_t)a.batch_c, (uint8_t)a.batch_d};
            x.nl = a.num_fri_layers(); x.c = a.num_comp_cols();
            if (L.w != a.w || L.log_n != log2u(a.n)) { fail(VO_TRACE_INFO); return; }
            if (memcmp(L.opt, want, 8)) { fail(VO_OPTIONS); return; }
            if (L.n_commitments() != 2 + x.nl + 1 || L.fri_rows.size() != x.nl) { fail(VO_COMMITMENTS); return; }
            if (L.ood_trace.len != 2 * (size_t)a.w * 16 || L.ood_h.len != (size_t)x.c * 16) { fail(VO_OOD_SHAPE); return; }
            // batch Merkle proofs: read where the verifier reads them
            x.bp.resize(2 + x.nl);
            for (uint32_t k = 0; k < 2 + x.nl; k++) {
                const Span& sp = k == 0 ? L.trace_paths : k == 1 ? L.comp_paths : L.fri_paths[k - 2];
                const uint32_t ord = k == 0 ? VO_TRACE_PATHS_PARSE : k == 1 ? VO_CONSTRAINT_PATHS_PARSE : VO_FRI0 + VO_FRI_STEP * (k - 2) + VO_FRI_PATHS_PARSE;
                if (!parse_batch_proof(b + sp.off, sp.len, x.bp[k])) { fail(ord); x.bp[k] = BatchProofLayout(); }
            }
            {   // degree bookkeeping of FriVerifier::verify
                uint64_t md = a.n;
                for (uint32_t l = 0; l < x.nl; l++) {
                    if (md % a.folding) fail(VO_FRI0 + VO_FRI_STEP * l + VO_FRI_TRUNCATION);
                    md /= a.folding;
                }
                if (L.remainder.len / 16 > md) fail(VO_REM);
            }
        });
        // staging offsets and the digest ids of the proofs' Merkle nodes, in proof order
        uint32_t n_nodes = 0;
        for (uint32_t i = 0; i < count; i++) {
            VItem& x = it[i];
            if (x.fail <= VO_OOD_SHAPE) continue;
            const ProofLayout& L = x.L;
            x.node_ids.resize(x.bp.size());
            for (size_t k = 0; k < x.bp.size(); k++)
                for (auto& v : x.bp[k].nodes) {
                    std::vector<uint32_t> ids(v.size());
                    for (auto& d : ids) d = n_nodes++;
                    x.node_ids[k].push_back(std::move(ids));
                }
            auto place = [&](size_t len) { const size_t o = off; off = al(off + len); return (uint64_t)o; };
            x.o_comm = place(L.commitments.len); x.o_ood = place(L.ood_trace.len); x.o_h = place(L.ood_h.len); x.o_rem = place(L.remainder.len);
            x.o_trows = place(L.trace_rows.len); x.o_crows = place(L.comp_rows.len);
            for (uint32_t l = 0; l < x.nl; l++) x.o_fri.push_back(place(L.fri_rows[l].len));
        }
        // AIR data of the OOD check, then the nodes
        std::vector<uint64_t> o_air(count, 0);
        for (uint32_t i = 0; i < count; i++) {
            if (it[i].fail <= VO_OOD_SHAPE) continue;
            const AirSpec& a = it[i].air;
            o_air[i] = off;
            off = al(off + a.assertions.size() * 16) ; off = al(off + a.params.size() * 16); off = al(off + a.assertions.size() * 16);
            off = al(off + a.assertions.size() * 4); off = al(off + (a.assertions.size() + 1) * 4);
        }
        const size_t o_nodes = off;
        const size_t total = off + (size_t)n_nodes * 32;
        grow_pinned(h_vstage, h_vstage_cap, total);
        uint8_t* H = h_vstage;
        VProof* hp = reinterpret_cast<VProof*>(H + o_proofs);
        {
            HF* r = reinterpret_cast<HF*>(H + o_roots);
            for (int k = 0; k <= 40; k++) r[k] = HF::root_of_unity(k);
        }
        if (n_nodes >= LOCAL_ID) throw InvalidArg("too many Merkle nodes in one batch");
        host_parallel(count, [&](uint32_t i) {   // every proof writes its own parts of the staging buffer
            VItem& x = it[i];
            reinterpret_cast<uint32_t*>(H)[i] = x.fail;
            VProof& p = hp[i];
            memset(&p, 0, sizeof(p));
            if (x.fail <= VO_OOD_SHAPE) return;   // not a proof of this AIR: no device work
            const AirSpec& a = x.air;
            const ProofLayout& L = x.L;
            const uint8_t* b = proofs[i];
            auto put = [&](uint64_t o, const Span& s) { memcpy(H + o, b + s.off, s.len); };
            put(x.o_comm, L.commitments); put(x.o_ood, L.ood_trace); put(x.o_h, L.ood_h); put(x.o_rem, L.remainder);
            put(x.o_trows, L.trace_rows); put(x.o_crows, L.comp_rows);
            for (uint32_t l = 0; l < x.nl; l++) put(x.o_fri[l], L.fri_rows[l]);
            for (uint32_t k = 0; k < x.bp.size(); k++) {
                const Span& sp = k == 0 ? L.trace_paths : k == 1 ? L.comp_paths : L.fri_paths[k - 2];
                for (size_t v = 0; v < x.bp[k].nodes.size(); v++)
                    for (size_t q = 0; q < x.bp[k].nodes[v].size(); q++)
                        memcpy(H + o_nodes + (size_t)x.node_ids[k][v][q] * 32, b + sp.off + x.bp[k].nodes[v][q], 32);
            }
            HostCoin coin;
            coin.init(a.coin_seed());
            memcpy(p.seed, coin.seed, 32);
            p.o_comm = x.o_comm; p.o_ood = x.o_ood; p.o_h = x.o_h; p.o_rem = x.o_rem;
            p.nonce = L.nonce;
            p.w = a.w; p.c = x.c; p.nt = a.num_transition(); p.na = (uint32_t)a.assertions.size(); p.np = (uint32_t)a.params.size();
            p.n_layers = x.nl; p.rem_len = (uint32_t)(L.remainder.len / 16); p.q = a.num_queries;
            p.log_n = log2u(a.n); p.log_N = log2u(a.lde_size()); p.grinding = a.grinding; p.air_id = a.id;
            p.active = 1; p.ood = x.fail > VO_OOD ? 1 : 0;
            // sorted assertions, parameters, boundary groups (g^step), columns, group offsets
            const size_t na = a.assertions.size();
            std::vector<uint32_t> goff;
            std::vector<HF> gpts;
            const HF g = HF::root_of_unity((int)p.log_n);
            for (size_t k = 0; k < na; k++)
                if (k == 0 || a.assertions[k].step != a.assertions[k - 1].step) { goff.push_back((uint32_t)k); gpts.push_back(g.pow((u128)a.assertions[k].step)); }
            goff.push_back((uint32_t)na);
            p.ng = (uint32_t)gpts.size();
            uint64_t o = o_air[i];
            p.o_aval = o; for (size_t k = 0; k < na; k++) memcpy(H + o + 16 * k, &a.assertions[k].value, 16); o = al(o + na * 16);
            p.o_params = o; memcpy(H + o, a.params.data(), a.params.size() * 16); o = al(o + a.params.size() * 16);
            p.o_gpts = o; memcpy(H + o, gpts.data(), gpts.size() * 16); o = al(o + na * 16);
            p.o_acol = o; for (size_t k = 0; k < na; k++) memcpy(H + o + 4 * k, &a.assertions[k].col, 4); o = al(o + na * 4);
            p.o_goff = o; memcpy(H + o, goff.data(), goff.size() * 4);
        });
        const auto hp1 = std::chrono::steady_clock::now();
        d_vstage.ensure(total);
        d_vts.ensure((size_t)count * sizeof(DevTs));
        h2d(d_vstage.p, H, total);
        VArgs A{};
        A.base = d_vstage.as<uint8_t>();
        A.proofs = reinterpret_cast<const VProof*>(A.base + o_proofs);
        A.ts = d_vts.as<DevTs>();
        A.verdict = d_vstage.as<uint32_t>();
        A.roots = reinterpret_cast<const fe*>(A.base + o_roots);
        A.nodes = reinterpret_cast<const uint32_t*>(A.base + o_nodes);
        A.n_nodes = n_nodes;
        for (uint32_t lf = 1; lf <= 4; lf++) {   // folding constants of every factor (the prover's FriFoldParams has them per layer)
            const HF wi = HF::root_of_unity((int)lf).inv();
            HF x = HF::raw(1);
            for (uint32_t k = 0; k < (1u << lf) / 2; k++) { A.fold_wf_inv[lf - 1][k] = to_fe(x); x = x * wi; }
            A.fold_inv_f[lf - 1] = to_fe(HF::from_u64(1u << lf).inv());
        }
        k_v_channel<<<count, ZKB_FS_THREADS, 0, stream>>>(A);
        check_launch();
        k_v_ood<<<(unsigned)(((uint64_t)count * 32 + 127) / 128), 128, 0, stream>>>(A, count);
        check_launch();
        std::vector<DevTs> hts(count);
        std::vector<uint32_t> dv(count);
        CK(cudaMemcpyAsync(hts.data(), d_vts.p, (size_t)count * sizeof(DevTs), cudaMemcpyDeviceToHost, stream));
        CK(cudaMemcpyAsync(dv.data(), d_vstage.p, (size_t)count * 4, cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));   // synchronisation 1: positions and the channel's verdicts
        const auto hp2 = std::chrono::steady_clock::now();

        // ---- plan: positions, position folding, Merkle merges, DEEP / FRI evaluations ----
        std::vector<VPlan> plans(count);
        host_parallel(count, [&](uint32_t i) {
            VItem& x = it[i];
            if (x.fail <= VO_OOD_SHAPE) return;
            std::vector<VLeafJob>& leaves = plans[i].leaves;
            std::vector<std::vector<MergeJob>>& merges = plans[i].merges;
            std::vector<VRootJob>& roots_chk = plans[i].roots;
            std::vector<VEvalJob>& evals = plans[i].evals;
            uint32_t next_id = LOCAL_ID;
            const AirSpec& a = x.air;
            const ProofLayout& L = x.L;
            uint32_t f = std::min(x.fail, dv[i]);
            const uint32_t F = a.folding, w = a.w, c = x.c;
            const uint32_t log_N = log2u(a.lde_size()), log_F = a.log_folding();
            x.positions.assign(hts[i].positions, hts[i].positions + a.num_queries);
            std::sort(x.positions.begin(), x.positions.end());
            x.positions.erase(std::unique(x.positions.begin(), x.positions.end()), x.positions.end());
            const std::vector<uint32_t>& pos = x.positions;
            const size_t nq = pos.size();
            auto leaf = [&](uint64_t o, uint32_t cnt, uint32_t ord) { leaves.push_back({o, cnt, next_id, i, ord}); return next_id++; };
            auto tree = [&](uint32_t k, const std::vector<uint32_t>& idx, const std::vector<uint32_t>& ids, uint32_t ord) {
                uint32_t root = 0;
                if (!plan_batch_root(x.bp[k].depth, idx, ids, x.node_ids[k], merges, next_id, &root)) f = std::min(f, ord);
                else roots_chk.push_back({x.o_comm + 32 * (uint64_t)k, root, i, ord, 0});
            };
            do {
                if (f <= VO_UNIQUE) break;
                if (L.n_unique != nq) { f = VO_UNIQUE; break; }
                if (L.trace_rows.len != nq * w * 16) { f = VO_TRACE_VALUES; break; }
                if (L.comp_rows.len != nq * c * 16) { f = VO_CONSTRAINT_VALUES; break; }
                std::vector<uint32_t> tid, cid;
                if (f > VO_TRACE_ROWS_PARSE) for (size_t q = 0; q < nq; q++) tid.push_back(leaf(x.o_trows + q * w * 16, w, VO_TRACE_ROWS_PARSE));
                if (f > VO_CONSTRAINT_ROWS_PARSE) for (size_t q = 0; q < nq; q++) cid.push_back(leaf(x.o_crows + q * c * 16, c, VO_CONSTRAINT_ROWS_PARSE));
                if (f > VO_TRACE_MERKLE) tree(0, pos, tid, VO_TRACE_MERKLE);
                if (f > VO_CONSTRAINT_MERKLE) tree(1, pos, cid, VO_CONSTRAINT_MERKLE);
                auto deep_job = [&](size_t q, uint64_t target, uint32_t ord) {
                    evals.push_back({x.o_trows + q * w * 16, x.o_crows + q * c * 16, target, i, ~0u, pos[q], log_N, pos[q], log_N, ord, F});
                };
                std::vector<uint32_t> cur = pos, prev;
                uint64_t dom = a.lde_size();
                for (uint32_t l = 0; l < x.nl; l++) {
                    const uint32_t base = VO_FRI0 + VO_FRI_STEP * l;
                    if (f <= base) break;
                    const std::vector<uint32_t> folded = fold_positions(cur, dom, F);
                    const uint64_t rows = dom / F;
                    if (L.fri_rows[l].len != folded.size() * F * 16) { f = base + VO_FRI_VALUES; break; }
                    std::vector<uint32_t> ids;
                    if (f > base + VO_FRI_ROWS_PARSE) for (size_t r = 0; r < folded.size(); r++) ids.push_back(leaf(x.o_fri[l] + r * F * 16, F, base + VO_FRI_ROWS_PARSE));
                    if (f > base + VO_FRI_MERKLE) tree(2 + l, folded, ids, base + VO_FRI_MERKLE);
                    if (f > base + VO_FRI_FOLDING) {   // get_query_values: position q sits in row (q mod rows), slot (q div rows)
                        std::vector<std::pair<uint32_t, uint32_t>> row_of(folded.size());   // (folded position, row), ascending
                        for (size_t r = 0; r < folded.size(); r++) row_of[r] = {folded[r], (uint32_t)r};
                        std::sort(row_of.begin(), row_of.end());
                        auto target = [&](uint32_t q) {
                            const uint32_t fq = (uint32_t)(q % rows);
                            const uint32_t r = std::lower_bound(row_of.begin(), row_of.end(), std::make_pair(fq, 0u))->second;
                            return x.o_fri[l] + ((uint64_t)r * F + q / rows) * 16;
                        };
                        const uint32_t ord = base + VO_FRI_FOLDING;
                        if (l == 0) for (size_t q = 0; q < nq; q++) deep_job(q, target(pos[q]), ord);
                        else for (size_t r = 0; r < prev.size(); r++)
                            evals.push_back({x.o_fri[l - 1] + r * F * 16, 0, target(prev[r]), i, l - 1, prev[r], log2u(dom * F), 0, 0, ord, F});
                    }
                    prev = folded; cur = folded; dom = rows;
                }
                if (f > VO_REM + 1) roots_chk.push_back({x.o_comm + 32 * (uint64_t)(2 + x.nl), leaf(x.o_rem, (uint32_t)(L.remainder.len / 16), VO_REM + 1), i, VO_REM + 1, 0});
                if (f > VO_REM + 2) {   // the last evaluations against the remainder polynomial
                    if (x.nl == 0) for (size_t q = 0; q < nq; q++) deep_job(q, ~0ull, VO_REM + 2);
                    else for (size_t r = 0; r < prev.size(); r++)
                        evals.push_back({x.o_fri[x.nl - 1] + r * F * 16, 0, ~0ull, i, x.nl - 1, prev[r], log2u(dom) + log_F, prev[r], log2u(dom), VO_REM + 2, F});
                }
            } while (false);
            x.fail = f;
            plans[i].ids = next_id - LOCAL_ID;
        });
        // one id space for the batch: each proof's ids follow the nodes and the ids of the proofs before it
        std::vector<VLeafJob> leaves;
        std::vector<std::vector<MergeJob>> merges;
        std::vector<VRootJob> roots_chk;
        std::vector<VEvalJob> evals;
        uint32_t next_id = n_nodes;
        for (uint32_t i = 0; i < count; i++) {
            VPlan& pl = plans[i];
            if ((uint64_t)next_id + pl.ids >= LOCAL_ID) throw InvalidArg("too many digests in one batch");
            const uint32_t base = next_id;
            auto reloc = [base](uint32_t id) { return id >= LOCAL_ID ? base + (id - LOCAL_ID) : id; };
            for (VLeafJob j : pl.leaves) { j.out = reloc(j.out); leaves.push_back(j); }
            if (merges.size() < pl.merges.size()) merges.resize(pl.merges.size());
            for (size_t d = 0; d < pl.merges.size(); d++)
                for (const MergeJob& j : pl.merges[d]) merges[d].push_back({reloc(j.a), reloc(j.b), reloc(j.out)});
            for (VRootJob j : pl.roots) { j.id = reloc(j.id); roots_chk.push_back(j); }
            evals.insert(evals.end(), pl.evals.begin(), pl.evals.end());
            next_id += pl.ids;
        }
        const auto hp3 = std::chrono::steady_clock::now();
        // ---- plan upload: [leaves][merges, level by level][roots][evaluations] ----
        std::vector<size_t> lvl_off(merges.size() + 1, 0);
        size_t po = al(leaves.size() * sizeof(VLeafJob));
        for (size_t d = 0; d < merges.size(); d++) { lvl_off[d] = po; po = al(po + merges[d].size() * sizeof(VMergeJob)); }
        const size_t o_rchk = po; po = al(po + roots_chk.size() * sizeof(VRootJob));
        const size_t o_eval = po; po = al(po + evals.size() * sizeof(VEvalJob));
        const size_t plan_bytes = std::max<size_t>(po, 16);
        grow_pinned(h_vplan, h_vplan_cap, plan_bytes);
        memcpy(h_vplan, leaves.data(), leaves.size() * sizeof(VLeafJob));
        for (size_t d = 0; d < merges.size(); d++) {
            static_assert(sizeof(MergeJob) == sizeof(VMergeJob), "merge job layouts differ");
            memcpy(h_vplan + lvl_off[d], merges[d].data(), merges[d].size() * sizeof(VMergeJob));
        }
        memcpy(h_vplan + o_rchk, roots_chk.data(), roots_chk.size() * sizeof(VRootJob));
        memcpy(h_vplan + o_eval, evals.data(), evals.size() * sizeof(VEvalJob));
        d_vplan.ensure(plan_bytes);
        d_vdig.ensure(std::max<size_t>(32, (size_t)(next_id - n_nodes) * 32));
        h2d(d_vplan.p, h_vplan, plan_bytes);
        A.dig = d_vdig.as<uint32_t>();
        const uint8_t* P = d_vplan.as<uint8_t>();
        auto grid = [](size_t n) { return (unsigned)((n + 127) / 128); };
        if (!leaves.empty()) { k_v_leaves<<<grid(leaves.size()), 128, 0, stream>>>(A, (const VLeafJob*)P, (uint32_t)leaves.size()); check_launch(); }
        for (size_t d = 0; d < merges.size(); d++) {
            if (merges[d].empty()) continue;
            k_v_merge<<<grid(merges[d].size()), 128, 0, stream>>>(A, (const VMergeJob*)(P + lvl_off[d]), (uint32_t)merges[d].size());
            check_launch();
        }
        if (!roots_chk.empty()) { k_v_roots<<<grid(roots_chk.size()), 128, 0, stream>>>(A, (const VRootJob*)(P + o_rchk), (uint32_t)roots_chk.size()); check_launch(); }
        if (!evals.empty()) { k_v_eval<<<grid(evals.size()), 128, 0, stream>>>(A, (const VEvalJob*)(P + o_eval), (uint32_t)evals.size()); check_launch(); }
        CK(cudaMemcpyAsync(dv.data(), d_vstage.p, (size_t)count * 4, cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));   // synchronisation 2: the verdicts
        if (host_prof) {
            const auto hp4 = std::chrono::steady_clock::now();
            auto us = [](auto a, auto b) { return std::chrono::duration<double, std::micro>(b - a).count(); };
            fprintf(stderr, "[zkb verify] %u proofs: parse + pack %.1f us, upload + channel + OOD %.1f us, plan %.1f us (%zu leaves, %zu levels, "
                    "%zu evaluations), upload + checks %.1f us\n", count, us(hp0, hp1), us(hp1, hp2), us(hp2, hp3), leaves.size(), merges.size(),
                    evals.size(), us(hp3, hp4));
        }
        for (uint32_t i = 0; i < count; i++) {
            VItem& x = it[i];
            verdicts[i] = verdict_of(std::min(x.fail, dv[i]));
            if (!tss) continue;
            zkb_transcript& t = tss[i];
            memset(&t, 0, sizeof(t));
            t.comp_degree_ok = 1;
            if (x.bp.empty()) continue;   // the channel did not run
            const uint8_t* cm = proofs[i] + x.L.commitments.off;
            const DevTs& h = hts[i];
            memcpy(t.trace_root, cm, 32); memcpy(t.constraint_root, cm + 32, 32); memcpy(t.remainder_commitment, cm + 32 * (2 + x.nl), 32);
            memcpy(t.constraint_alpha, &h.alpha, 16); memcpy(t.z, &h.z, 16); memcpy(t.deep_alpha, &h.deep_alpha, 16);
            t.n_fri_layers = x.nl;
            for (uint32_t l = 0; l < x.nl && l < TS_FRI_SLOTS; l++) { memcpy(t.fri_roots[l], cm + 32 * (2 + l), 32); memcpy(t.fri_alphas[l], &h.fri_alpha[l], 16); }
            t.pow_nonce = x.L.nonce;
            t.n_positions = (uint32_t)x.positions.size();
            for (size_t q = 0; q < x.positions.size() && q < 256; q++) t.positions[q] = x.positions[q];
        }
    }
};

// ================================================================================================================
// C ABI
template <class F>
static int32_t guarded(zkb_ctx* ctx, F&& f) {
    try {
        if (!ctx) throw InvalidArg("null context");
        f();
        return ZKB_OK;
    } catch (const InvalidArg& e) { (ctx ? ctx->err : g_last_error) = e.what(); return ZKB_ERR_INVALID; }
    catch (const StateError& e) { (ctx ? ctx->err : g_last_error) = e.what(); return ZKB_ERR_STATE; }
    catch (const CudaError& e) {
        (ctx ? ctx->err : g_last_error) = e.what();
        return std::string(e.what()).find("out of memory") != std::string::npos ? ZKB_ERR_OOM : ZKB_ERR_CUDA;
    } catch (const std::exception& e) { (ctx ? ctx->err : g_last_error) = e.what(); return ZKB_ERR_INVALID; }
}
static uint8_t* dup_bytes(const std::vector<uint8_t>& v) {
    uint8_t* p = (uint8_t*)malloc(v.size() ? v.size() : 1);
    if (v.size()) memcpy(p, v.data(), v.size());
    return p;
}

// the proving entry points: Prover::prove, then the proof bytes (malloc'ed, released with zkb_free) and the transcript out
static void prove_out(zkb_ctx* ctx, const zkb_air_desc* air, const uint8_t* const* cols, const void* d_trace, uint64_t force_nonce, bool sharded,
                      uint8_t** proof_out, uint64_t* proof_len, zkb_transcript* transcript) {
    std::vector<uint8_t> b = ctx->prove(air, cols, (const fe*)d_trace, force_nonce, sharded);
    if (transcript) *transcript = ctx->ts;
    if (proof_len) *proof_len = b.size();
    if (proof_out) *proof_out = dup_bytes(b);
}

extern "C" {

int32_t zkb_ctx_create(int32_t device, void* stream, zkb_ctx** out) {
    if (!out) { g_last_error = "null output pointer"; return ZKB_ERR_INVALID; }
    *out = nullptr;
    zkb_ctx* c = new zkb_ctx();
    try {
        c->init(device, stream);
    } catch (const InvalidArg& e) { g_last_error = e.what(); delete c; return ZKB_ERR_INVALID; }
    catch (const std::exception& e) { g_last_error = e.what(); delete c; return ZKB_ERR_CUDA; }
    *out = c;
    return ZKB_OK;
}
int32_t zkb_ctx_create_lane(int32_t device, zkb_ctx** out) {
    if (!out) { g_last_error = "null output pointer"; return ZKB_ERR_INVALID; }
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { g_last_error = "no CUDA device available"; return ZKB_ERR_CUDA; }
    if (device < 0 || device >= ndev) { g_last_error = "device index out of range"; return ZKB_ERR_INVALID; }
    cudaStream_t st = nullptr;
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess) {
        g_last_error = "cannot create a stream for the lane"; return ZKB_ERR_CUDA;
    }
    const int32_t rc = zkb_ctx_create(device, st, out);
    if (rc != ZKB_OK) { cudaStreamDestroy(st); return rc; }
    (*out)->owns_stream = true;
    return ZKB_OK;
}
void zkb_ctx_destroy(zkb_ctx* ctx) { if (ctx) { ctx->destroy(); delete ctx; } }
const char* zkb_last_error(const zkb_ctx* ctx) { return ctx ? ctx->err.c_str() : g_last_error.c_str(); }
uint64_t zkb_kernel_launches(const zkb_ctx* ctx) { return ctx ? ctx->launches : 0; }
uint64_t zkb_h2d_bytes(const zkb_ctx* ctx) { return ctx ? ctx->h2d_bytes : 0; }
int32_t zkb_last_stage_times(const zkb_ctx* ctx, zkb_stage_times* out) {
    if (!ctx || !out) return ZKB_ERR_INVALID;
    zkb_ctx* c = const_cast<zkb_ctx*>(ctx);  // elapsed times are read from the recorded events on first request
    int32_t rc = guarded(c, [&] { c->collect_times(); });
    *out = ctx->times;
    return rc;
}
void* zkb_host_alloc(size_t bytes) { void* p = nullptr; if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) return nullptr; return p; }
void zkb_host_free(void* p) { if (p) cudaFreeHost(p); }
void zkb_free(void* p) { free(p); }

int32_t zkb_prove(zkb_ctx* ctx, const zkb_air_desc* air, const uint8_t* const* cols, uint64_t force_nonce, uint8_t** proof_out,
                  uint64_t* proof_len, zkb_transcript* transcript) {
    return guarded(ctx, [&] {
        if (!cols) throw InvalidArg("null trace columns");
        prove_out(ctx, air, cols, nullptr, force_nonce, false, proof_out, proof_len, transcript);
    });
}
int32_t zkb_prove_device(zkb_ctx* ctx, const zkb_air_desc* air, const void* d_trace, uint64_t force_nonce, uint8_t** proof_out,
                         uint64_t* proof_len, zkb_transcript* transcript) {
    return guarded(ctx, [&] {
        if (!d_trace) throw InvalidArg("null device trace");
        prove_out(ctx, air, nullptr, d_trace, force_nonce, false, proof_out, proof_len, transcript);
    });
}

int32_t zkb_prove_batch(zkb_ctx* const* lanes, uint32_t n_lanes, const zkb_air_desc* const* airs, const uint8_t* const* const* cols,
                        uint32_t count, uint8_t** proofs_out, uint64_t* lens_out) {
    if (!lanes || n_lanes == 0 || !proofs_out || !lens_out || (count && (!airs || !cols))) { g_last_error = "zkb_prove_batch: null argument"; return ZKB_ERR_INVALID; }
    for (uint32_t l = 0; l < n_lanes; l++) if (!lanes[l]) { g_last_error = "zkb_prove_batch: null lane"; return ZKB_ERR_INVALID; }
    for (uint32_t i = 0; i < count; i++) { proofs_out[i] = nullptr; lens_out[i] = 0; }
    std::vector<int32_t> rc(n_lanes, ZKB_OK);
    std::vector<uint32_t> failed(n_lanes, UINT32_MAX);
    auto work = [&](uint32_t l) {
        for (uint32_t i = l; i < count; i += n_lanes) {
            const int32_t r = zkb_prove(lanes[l], airs[i], cols[i], 0, &proofs_out[i], &lens_out[i], nullptr);
            if (r != ZKB_OK) { rc[l] = r; failed[l] = i; return; }   // the lane stops at its first failure
        }
    };
    std::vector<std::thread> threads;
    for (uint32_t l = 1; l < n_lanes && l < count; l++) threads.emplace_back(work, l);
    work(0);
    for (auto& t : threads) t.join();
    uint32_t first = UINT32_MAX; int32_t out = ZKB_OK;
    for (uint32_t l = 0; l < n_lanes; l++) if (rc[l] != ZKB_OK && failed[l] < first) { first = failed[l]; out = rc[l]; }
    return out;
}

int32_t zkb_verify_batch(zkb_ctx* ctx, const zkb_air_desc* const* airs, const uint8_t* const* proofs, const uint64_t* lens, uint32_t count,
                         int32_t* verdicts_out, zkb_transcript* transcripts_out) {
    return guarded(ctx, [&] { ctx->verify_batch(airs, proofs, lens, count, verdicts_out, transcripts_out); });
}

int32_t zkb_begin(zkb_ctx* ctx, const zkb_air_desc* air) { return guarded(ctx, [&] { ctx->begin(air); }); }
int32_t zkb_trace_commit(zkb_ctx* ctx, const uint8_t* const* cols, uint8_t root_out[32]) { return guarded(ctx, [&] { ctx->trace_commit_host(cols, root_out); }); }
int32_t zkb_trace_commit_device(zkb_ctx* ctx, const void* d, uint8_t root_out[32]) {
    return guarded(ctx, [&] { if (!d) throw InvalidArg("null device trace"); ctx->trace_commit_device((const fe*)d, root_out); });
}
// TraceLde::read_main_trace_frame_into for `count` LDE steps at once: one upload of the row indices, one gather launch, one
// download (the single-step call is the count = 1 case).  An evaluator that walks the whole domain should ask for thousands
// of steps per call — or, better, not read frames at all and use zkb_constraints_eval.
int32_t zkb_trace_read_frames(zkb_ctx* ctx, const uint64_t* lde_steps, uint32_t count, uint8_t* cur, uint8_t* nxt) {
    return guarded(ctx, [&] {
        if (ctx->stage < ST_TRACE) throw StateError("zkb_trace_read_frames: trace is not committed");
        if (ctx->mg_active) throw StateError("zkb_trace_read_frames: not available for a column-sharded trace");
        const uint64_t N = ctx->air.lde_size();
        if (!lde_steps || !cur || !nxt) throw InvalidArg("bad frame request");
        if (count == 0) return;
        if (count > (1u << 20)) throw InvalidArg("at most 2^20 frames per call");
        std::vector<uint32_t> pos(2 * (size_t)count);
        for (uint32_t q = 0; q < count; q++) {
            if (lde_steps[q] >= N) throw InvalidArg("LDE step out of range");
            pos[q] = (uint32_t)lde_steps[q];
            pos[count + q] = (uint32_t)((lde_steps[q] + ctx->air.blowup) % N);   // frame.next wraps around the LDE domain
        }
        CK(cudaSetDevice(ctx->device));
        const uint32_t w = ctx->air.w;
        const size_t o_rows = ((pos.size() * 4 + 255) / 256) * 256, row_bytes = (size_t)count * w * 16;
        ctx->d_gather.ensure(o_rows + 2 * row_bytes);
        uint8_t* base = ctx->d_gather.as<uint8_t>();
        ctx->h2d(base, pos.data(), pos.size() * 4);
        const uint64_t th = 2 * (uint64_t)count * w;
        k_gather_lde_rows<<<(unsigned)((th + 127) / 128), 128, 0, ctx->stream>>>(ctx->lde_mat(), (const uint32_t*)base, 2 * count, (fe*)(base + o_rows));
        ctx->check_launch();
        CK(cudaMemcpyAsync(cur, base + o_rows, row_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        ctx->d2h(nxt, base + o_rows + row_bytes, row_bytes);
    });
}
int32_t zkb_trace_read_frame(zkb_ctx* ctx, uint64_t lde_step, uint8_t* cur, uint8_t* nxt) {
    return zkb_trace_read_frames(ctx, &lde_step, 1, cur, nxt);
}
int32_t zkb_trace_polys_read(zkb_ctx* ctx, uint8_t* out) {
    return guarded(ctx, [&] {
        if (ctx->stage < ST_TRACE || ctx->stage >= ST_DEEP) throw StateError("zkb_trace_polys_read: trace polynomials are not available");
        if (!out) throw InvalidArg("null output");
        ctx->d2h(out, ctx->d_polys, (size_t)ctx->air.n * ctx->air.w * 16);
    });
}
int32_t zkb_constraints_eval(zkb_ctx* ctx, const uint8_t alpha[16], uint8_t* evals_out) {
    return guarded(ctx, [&] { if (!alpha) throw InvalidArg("null alpha"); ctx->constraints_eval(HF::reduce(HF::from_bytes(alpha).v), evals_out); });
}
int32_t zkb_constraints_commit(zkb_ctx* ctx, uint8_t root_out[32]) { return guarded(ctx, [&] { ctx->constraints_commit(root_out); }); }
int32_t zkb_ood_eval(zkb_ctx* ctx, const uint8_t z[16], uint8_t* cur, uint8_t* nxt, uint8_t* h) {
    return guarded(ctx, [&] {
        if (!z) throw InvalidArg("null z");
        ctx->ood_eval(HF::reduce(HF::from_bytes(z).v));
        if (cur) memcpy(cur, ctx->ood_cur.data(), ctx->ood_cur.size() * 16);
        if (nxt) memcpy(nxt, ctx->ood_next.data(), ctx->ood_next.size() * 16);
        if (h) memcpy(h, ctx->ood_h.data(), ctx->ood_h.size() * 16);
    });
}
int32_t zkb_deep_compose(zkb_ctx* ctx, const uint8_t a[16]) {
    return guarded(ctx, [&] { if (!a) throw InvalidArg("null alpha"); ctx->deep_compose(HF::reduce(HF::from_bytes(a).v)); });
}
int32_t zkb_fri_num_layers(zkb_ctx* ctx, uint32_t* out) { return guarded(ctx, [&] { if (!out) throw InvalidArg("null output"); *out = ctx->fri_layers; }); }
int32_t zkb_fri_commit_layer(zkb_ctx* ctx, uint8_t root_out[32]) { return guarded(ctx, [&] { ctx->fri_commit_layer(root_out); }); }
int32_t zkb_fri_fold(zkb_ctx* ctx, const uint8_t a[16]) {
    return guarded(ctx, [&] { if (!a) throw InvalidArg("null alpha"); ctx->fri_fold(HF::reduce(HF::from_bytes(a).v)); });
}
int32_t zkb_fri_remainder(zkb_ctx* ctx, uint8_t* coeffs_out, uint64_t* n_out, uint8_t commitment_out[32]) {
    return guarded(ctx, [&] {
        ctx->fri_remainder(commitment_out);
        if (coeffs_out) memcpy(coeffs_out, ctx->parts.remainder.data(), ctx->parts.remainder.size() * 16);
        if (n_out) *n_out = ctx->parts.remainder.size();
    });
}
int32_t zkb_grind(zkb_ctx* ctx, const uint8_t seed[32], uint32_t bits, uint64_t* nonce_out) {
    return guarded(ctx, [&] { if (!seed || !nonce_out) throw InvalidArg("null argument"); CK(cudaSetDevice(ctx->device)); *nonce_out = ctx->grind(seed, bits); });
}
int32_t zkb_query(zkb_ctx* ctx, uint32_t which, const uint32_t* positions, uint32_t n_pos, uint8_t* rows_out, uint8_t** proof_out,
                  uint64_t* proof_len) {
    return guarded(ctx, [&] {
        // a commitment can be opened as soon as it exists: Winterfell's own generate_proof (associated-type integration) runs
        // DEEP and FRI on the host and then calls TraceLde::query / ConstraintCommitment::query
        if (which == 0 && ctx->stage < ST_TRACE) throw StateError("zkb_query: the trace is not committed");
        if (which == 1 && ctx->stage < ST_COMP) throw StateError("zkb_query: the constraint composition is not committed");
        if (which >= 2 && ctx->stage < ST_FRI_DONE) throw StateError("zkb_query: the FRI commit phase is not finished");
        if (!positions) throw InvalidArg("null positions");
        std::vector<uint32_t> pos(positions, positions + n_pos);
        std::vector<uint8_t> rows, paths;
        ctx->query(which, pos, rows, paths);
        if (rows_out) memcpy(rows_out, rows.data(), rows.size());
        if (proof_len) *proof_len = paths.size();
        if (proof_out) *proof_out = dup_bytes(paths);
    });
}

int32_t zkb_mg_unique_id(uint8_t out[128]) {
    try {
        if (!out) throw InvalidArg("null output");
        g_nccl.load();
        ncclUniqueId id;
        NK(g_nccl.GetUniqueId(&id));
        memcpy(out, &id, 128);
        return ZKB_OK;
    } catch (const InvalidArg& e) { g_last_error = e.what(); return ZKB_ERR_INVALID; }
    catch (const std::exception& e) { g_last_error = e.what(); return ZKB_ERR_CUDA; }
}
int32_t zkb_mg_init(zkb_ctx* ctx, int32_t rank, int32_t world, const uint8_t id[128]) {
    return guarded(ctx, [&] { if (!id) throw InvalidArg("null NCCL id"); ctx->mg_init(rank, world, id); });
}
int32_t zkb_mg_prove(zkb_ctx* ctx, const zkb_air_desc* air, const uint8_t* const* local_cols, uint64_t force_nonce, uint8_t** proof_out,
                     uint64_t* proof_len, zkb_transcript* transcript) {
    return guarded(ctx, [&] {
        if (!local_cols) throw InvalidArg("null trace columns");
        prove_out(ctx, air, local_cols, nullptr, force_nonce, true, proof_out, proof_len, transcript);
    });
}
int32_t zkb_mg_prove_device(zkb_ctx* ctx, const zkb_air_desc* air, const void* d_local_trace, uint64_t force_nonce, uint8_t** proof_out,
                            uint64_t* proof_len, zkb_transcript* transcript) {
    return guarded(ctx, [&] {
        if (!d_local_trace) throw InvalidArg("null device trace");
        prove_out(ctx, air, nullptr, d_local_trace, force_nonce, true, proof_out, proof_len, transcript);
    });
}

int32_t zkb_mimc_trace_device(zkb_ctx* ctx, const uint8_t* seeds, uint32_t w, uint64_t n, const uint8_t* rc, uint32_t n_rc, void** d_out) {
    return guarded(ctx, [&] {
        if (!seeds || !rc || !d_out || w == 0 || n == 0 || !is_pow2(n_rc)) throw InvalidArg("bad mimc trace request");
        CK(cudaSetDevice(ctx->device));
        ctx->d_user_trace.ensure((size_t)w * n * 16);
        ctx->d_aux.ensure(((size_t)w + n_rc) * 16);
        ctx->h2d(ctx->d_aux.p, seeds, (size_t)w * 16);
        ctx->h2d(ctx->d_aux.as<fe>() + w, rc, (size_t)n_rc * 16);
        k_mimc_trace<<<(w + 31) / 32, 32, 0, ctx->stream>>>(ctx->d_aux.as<fe>(), w, n, ctx->d_aux.as<fe>() + w, n_rc, ctx->d_user_trace.as<fe>());
        ctx->check_launch();
        CK(cudaStreamSynchronize(ctx->stream));
        *d_out = ctx->d_user_trace.p;
    });
}
int32_t zkb_mimc_trace(zkb_ctx* ctx, const uint8_t* seeds, uint32_t w, uint64_t n, const uint8_t* rc, uint32_t n_rc, uint8_t* out) {
    void* d = nullptr;
    int32_t r = zkb_mimc_trace_device(ctx, seeds, w, n, rc, n_rc, &d);
    if (r != ZKB_OK) return r;
    return guarded(ctx, [&] { if (!out) throw InvalidArg("null output"); ctx->d2h(out, d, (size_t)w * n * 16); });
}
// host-side BLAKE3 (the channel's hash) for callers that verify proofs on the CPU; needs no device
int32_t zkb_blake3_host(const uint8_t* data, uint64_t len, uint8_t out[32]) {
    if ((!data && len) || !out) { g_last_error = "null argument"; return ZKB_ERR_INVALID; }
    b3_hash_host(data, len, out);
    return ZKB_OK;
}
int32_t zkb_mimc_cipher_batch(zkb_ctx* ctx, const uint8_t* inputs, const uint8_t* round_constants, const uint8_t* zs, uint64_t count, uint8_t* out) {
    return guarded(ctx, [&] {
        if (!inputs || !round_constants || !zs || !out) throw InvalidArg("null argument");
        if (count == 0) return;
        CK(cudaSetDevice(ctx->device));
        ctx->d_aux.ensure(count * 16 * 4);
        fe* b = ctx->d_aux.as<fe>();
        ctx->h2d(b, inputs, count * 16); ctx->h2d(b + count, round_constants, count * 16); ctx->h2d(b + 2 * count, zs, count * 16);
        k_mimc_cipher_batch<<<(unsigned)((count + 127) / 128), 128, 0, ctx->stream>>>(b, b + count, b + 2 * count, count, b + 3 * count);
        ctx->check_launch();
        ctx->d2h(out, b + 3 * count, count * 16);
    });
}
int32_t zkb_mimc_hash_matrix_batch(zkb_ctx* ctx, const uint8_t* w, const uint8_t* b, uint32_t ac, uint32_t fe_, const uint8_t* round_constants,
                                   uint32_t n_rc, uint64_t count, uint8_t* out) {
    return guarded(ctx, [&] {
        if (!w || !b || !round_constants || !out || ac == 0 || fe_ == 0 || n_rc == 0) throw InvalidArg("bad mimc_hash_matrix request");
        if (count == 0) return;
        CK(cudaSetDevice(ctx->device));
        const size_t per = (size_t)ac * fe_ + ac;
        ctx->d_aux.ensure((count * per + n_rc + count) * 16);
        fe* base = ctx->d_aux.as<fe>();
        ctx->h2d(base, w, count * ac * fe_ * 16); ctx->h2d(base + count * ac * fe_, b, count * ac * 16);
        ctx->h2d(base + count * per, round_constants, (size_t)n_rc * 16);
        k_mimc_hash_matrix_batch<<<(unsigned)((count + 127) / 128), 128, 0, ctx->stream>>>(base, base + count * ac * fe_, ac, fe_, base + count * per, n_rc,
                                                                                          count, base + count * per + n_rc);
        ctx->check_launch();
        ctx->d2h(out, base + count * per + n_rc, count * 16);
    });
}
int32_t zkb_training_trace_device(zkb_ctx* ctx, const uint8_t* raw_rows, uint32_t n_raw, uint32_t half, uint64_t n, const uint8_t* key32,
                                  void** d_out, uint8_t* first_row_out, uint8_t* last_row_out) {
    return guarded(ctx, [&] {
        if (!raw_rows || !d_out || n_raw == 0 || half == 0 || half > 127 || n < n_raw) throw InvalidArg("bad training trace request");
        CK(cudaSetDevice(ctx->device));
        const uint32_t w = 2 * half;
        ctx->d_user_trace.ensure((size_t)w * n * 16);
        ctx->d_aux.ensure(((size_t)n_raw * half + 2 * w) * 16);
        fe* d_raw = ctx->d_aux.as<fe>();
        ctx->h2d(d_raw, raw_rows, (size_t)n_raw * half * 16);
        // mask key: the caller's (tests, reproducible runs) or 256 bits of OS entropy, as rand::thread_rng() is seeded
        ChaChaKey key;
        if (key32) memcpy(key.k, key32, 32);
        else {
            size_t got = 0;
            while (got < 32) {
                const ssize_t r = getrandom((uint8_t*)key.k + got, 32 - got, 0);
                if (r <= 0) throw std::runtime_error("getrandom failed: no entropy for the blinding masks");
                got += (size_t)r;
            }
        }
        dim3 grid((unsigned)((n + 255) / 256), (half + 7) / 8);
        k_training_trace<<<grid, 256, 0, ctx->stream>>>(d_raw, n_raw, half, n, key, ctx->d_user_trace.as<fe>());
        ctx->check_launch();
        fe* d_rows = d_raw + (size_t)n_raw * half;
        k_read_rows<<<(w + 127) / 128, 128, 0, ctx->stream>>>(ctx->d_user_trace.as<fe>(), w, n, 0, n - 1, d_rows);
        ctx->check_launch();
        std::vector<uint8_t> rows(2 * (size_t)w * 16);
        ctx->d2h(rows.data(), d_rows, rows.size());
        if (first_row_out) memcpy(first_row_out, rows.data(), (size_t)w * 16);
        if (last_row_out) memcpy(last_row_out, rows.data() + (size_t)w * 16, (size_t)w * 16);
        *d_out = ctx->d_user_trace.p;
    });
}
int32_t zkb_download(zkb_ctx* ctx, const void* d_src, uint64_t bytes, uint8_t* out) {
    return guarded(ctx, [&] { if (!d_src || !out) throw InvalidArg("null argument"); CK(cudaSetDevice(ctx->device)); ctx->d2h(out, d_src, bytes); });
}
int32_t zkb_upload_trace(zkb_ctx* ctx, const uint8_t* const* cols, uint32_t w, uint64_t n, void** d_out) {
    return guarded(ctx, [&] {
        if (!d_out) throw InvalidArg("null output");
        CK(cudaSetDevice(ctx->device));
        *d_out = (void*)ctx->upload_cols(cols, w, n, ctx->d_user_trace);
        CK(cudaStreamSynchronize(ctx->stream));
    });
}

int32_t zkb_test_field(zkb_ctx* ctx, const uint8_t* a, const uint8_t* b, uint32_t n, uint8_t* mul, uint8_t* add, uint8_t* sub, uint8_t* inv) {
    return guarded(ctx, [&] {
        CK(cudaSetDevice(ctx->device));
        ctx->d_aux.ensure((size_t)n * 16 * 6);
        fe* base = ctx->d_aux.as<fe>();
        ctx->h2d(base, a, (size_t)n * 16); ctx->h2d(base + n, b, (size_t)n * 16);
        k_test_field<<<(n + 127) / 128, 128, 0, ctx->stream>>>(base, base + n, base + 2 * (size_t)n, base + 3 * (size_t)n, base + 4 * (size_t)n, base + 5 * (size_t)n, n);
        ctx->check_launch();
        ctx->d2h(mul, base + 2 * (size_t)n, (size_t)n * 16); ctx->d2h(add, base + 3 * (size_t)n, (size_t)n * 16);
        ctx->d2h(sub, base + 4 * (size_t)n, (size_t)n * 16); ctx->d2h(inv, base + 5 * (size_t)n, (size_t)n * 16);
    });
}
int32_t zkb_test_hash_elements(zkb_ctx* ctx, const uint8_t* rows, uint32_t count, uint32_t n_rows, uint8_t* out) {
    return guarded(ctx, [&] {
        CK(cudaSetDevice(ctx->device));
        size_t in_bytes = (size_t)count * n_rows * 16;
        ctx->d_aux.ensure(in_bytes + 16 + (size_t)n_rows * 32);
        uint8_t* base = ctx->d_aux.as<uint8_t>();
        size_t o = ((in_bytes + 15) / 16) * 16;
        if (in_bytes) ctx->h2d(base, rows, in_bytes);
        k_test_hash<<<(n_rows + 127) / 128, 128, 0, ctx->stream>>>((const fe*)base, count, n_rows, (uint32_t*)(base + o));
        ctx->check_launch();
        ctx->d2h(out, base + o, (size_t)n_rows * 32);
    });
}
int32_t zkb_test_merkle_root(zkb_ctx* ctx, const uint8_t* leaves, uint64_t n, uint8_t root_out[32]) {
    return guarded(ctx, [&] {
        if (n < 2 || !is_pow2(n)) throw InvalidArg("leaf count must be a power of two >= 2");
        CK(cudaSetDevice(ctx->device));
        ctx->d_aux.ensure(2 * n * 32);
        ctx->h2d(ctx->d_aux.as<uint8_t>() + n * 32, leaves, n * 32);
        ctx->build_merkle(ctx->d_aux.as<uint32_t>(), n);
        ctx->d2h(root_out, ctx->d_aux.as<uint8_t>() + 32, 32);
    });
}
int32_t zkb_test_lde(zkb_ctx* ctx, const uint8_t* const* cols, uint32_t w, uint64_t n, uint32_t blowup, uint8_t* polys_out, uint8_t* lde_out) {
    return guarded(ctx, [&] {
        // drive K1+K2 through a throw-away training-shaped description
        std::vector<uint8_t> zero(16, 0);
        uint32_t col = 0; uint64_t step = 0;
        zkb_air_desc d{};
        d.air_id = ZKB_AIR_ID_TRAINING; d.trace_width = w; d.trace_len = n; d.num_queries = 1; d.blowup = blowup; d.grinding_bits = 0;
        d.field_extension = 1; d.folding = 16; d.rem_max_degree = 7; d.batching_constraints = 1; d.batching_deep = 1;
        d.assert_cols = &col; d.assert_steps = &step; d.assert_values = zero.data(); d.n_assertions = 1;
        ctx->begin(&d);
        uint8_t root[32];
        ctx->trace_commit_host(cols, root);
        if (polys_out) ctx->d2h(polys_out, ctx->d_polys, (size_t)n * w * 16);
        if (lde_out) {
            const uint64_t N = n * blowup;
            std::vector<uint32_t> pos;
            // gather in slices of 128 rows to reuse the query gather kernel
            ctx->d_gather.ensure(1024 + (size_t)128 * w * 16);
            uint8_t* base = ctx->d_gather.as<uint8_t>();
            for (uint64_t r0 = 0; r0 < N; r0 += 128) {
                uint32_t cnt = (uint32_t)std::min<uint64_t>(128, N - r0);
                pos.resize(cnt);
                for (uint32_t q = 0; q < cnt; q++) pos[q] = (uint32_t)(r0 + q);
                ctx->h2d(base, pos.data(), cnt * 4);
                k_gather_lde_rows<<<(cnt * w + 127) / 128, 128, 0, ctx->stream>>>(ctx->lde_mat(), (const uint32_t*)base, cnt, (fe*)(base + 1024));
                ctx->check_launch();
                ctx->d2h(lde_out + r0 * w * 16, base + 1024, (size_t)cnt * w * 16);
            }
        }
        ctx->stage = ST_IDLE;
    });
}

}  // extern "C"
