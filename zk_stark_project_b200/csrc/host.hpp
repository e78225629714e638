// Host-side pieces of the prover that are not bulk arithmetic: AIR description, Fiat-Shamir coin,
// batch-Merkle-proof planning and the Proof wire format.  These mirror (independently of oracle/) the
// Winterfell 0.12 behaviour recalled in SURVEY.md Appendix A; every convention that could not be read
// from upstream source is tagged [A.x] with the appendix item it depends on.
#pragma once
#include <algorithm>
#include <map>
#include <set>
#include <stdexcept>
#include <string>
#include <vector>
#include "hostfield.hpp"
#include "blake3.cuh"
#include "../../include/zkb200.h"

namespace zkb {

struct InvalidArg : std::runtime_error { using std::runtime_error::runtime_error; };

static inline uint32_t log2u(uint64_t n) { uint32_t l = 0; while (((uint64_t)1 << l) < n) l++; return l; }
static inline bool is_pow2(uint64_t n) { return n && !(n & (n - 1)); }

struct Digest32 { uint8_t b[32]; };

// ---- AIR + options (winter-air AirContext / ProofOptions; src/main.rs:98-107) --------------------------------
struct HostAssertion { uint32_t col; uint64_t step; HF value; };
struct AirSpec {
    uint32_t id = 0, w = 0;
    uint64_t n = 0;
    uint32_t num_queries = 0, blowup = 0, grinding = 0, field_ext = 1, folding = 0, rem_max_degree = 0, batch_c = 1, batch_d = 1;
    std::vector<HF> pub_elems, params;
    std::vector<HostAssertion> assertions;  // sorted by (step, column): winter-air prepare_assertions

    uint32_t num_transition() const { return id == ZKB_AIR_ID_AGGREGATION ? w / 2 : w; }
    uint32_t degree() const { return id == ZKB_AIR_ID_MIMC ? 7 : 1; }
    uint32_t ce_blowup() const { uint32_t b = 2; while (b < degree()) b <<= 1; return b; }   // [A.3]
    uint32_t num_comp_cols() const {                                                           // [A.3]
        uint64_t eval_deg = (uint64_t)degree() * (n - 1), div_deg = n - 1;
        uint64_t c = (eval_deg - div_deg + n - 1) / n;
        return c < 1 ? 1 : (uint32_t)c;
    }
    uint64_t lde_size() const { return n * blowup; }
    // every FRI size (layer domain, rows per layer, leaf width, position folding) derives from this
    uint32_t log_folding() const { return log2u(folding); }
    uint32_t num_fri_layers() const {                                                          // [A.10]
        uint64_t d = lde_size(), max_rem = (uint64_t)(rem_max_degree + 1) * blowup;
        uint32_t r = 0;
        while (d > max_rem) { d /= folding; r++; }
        return r;
    }

    static AirSpec from_desc(const zkb_air_desc* d) {
        if (!d) throw InvalidArg("null air description");
        AirSpec a;
        a.id = d->air_id; a.w = d->trace_width; a.n = d->trace_len;
        a.num_queries = d->num_queries; a.blowup = d->blowup; a.grinding = d->grinding_bits; a.field_ext = d->field_extension;
        a.folding = d->folding; a.rem_max_degree = d->rem_max_degree; a.batch_c = d->batching_constraints; a.batch_d = d->batching_deep;
        if (a.id < 1 || a.id > 3) throw InvalidArg("unknown air id");
        if (a.n < 8 || !is_pow2(a.n)) throw InvalidArg("trace length must be a power of two >= 8");
        if (a.w < 1 || a.w > 255) throw InvalidArg("trace width must be in 1..=255");
        if (!is_pow2(a.blowup) || a.blowup < 2 || a.blowup > 128) throw InvalidArg("blowup factor must be a power of two in 2..=128");
        if (a.blowup < a.ce_blowup()) throw InvalidArg("blowup factor too small for the constraint degree");
        if (a.folding != 2 && a.folding != 4 && a.folding != 8 && a.folding != 16)
            throw InvalidArg("FRI folding factor must be one of 2, 4, 8, 16");
        if (a.num_queries < 1 || a.num_queries > 255) throw InvalidArg("number of queries must be in 1..=255");
        if (a.grinding > 32) throw InvalidArg("grinding factor must be <= 32");
        if (a.rem_max_degree > 255 || ((a.rem_max_degree + 1) & a.rem_max_degree)) throw InvalidArg("bad FRI remainder max degree");
        if (a.field_ext != 1) throw InvalidArg("only FieldExtension::None is supported (src/main.rs:102)");
        if (a.batch_c != 1 || a.batch_d != 1) throw InvalidArg("only BatchingMethod::Algebraic is supported (src/main.rs:105-106)");
        if (a.lde_size() > ((uint64_t)1 << 30)) throw InvalidArg("LDE domain too large");
        if (d->n_assertions == 0) throw InvalidArg("at least one assertion is required");
        if ((d->n_pub_elems && !d->pub_elems) || !d->assert_cols || !d->assert_steps || !d->assert_values) throw InvalidArg("null pointer in air description");
        for (uint64_t i = 0; i < d->n_pub_elems; i++) a.pub_elems.push_back(HF::reduce(HF::from_bytes(d->pub_elems + 16 * i).v));
        for (uint64_t i = 0; i < d->n_params; i++) a.params.push_back(HF::reduce(HF::from_bytes(d->params + 16 * i).v));
        for (uint64_t i = 0; i < d->n_assertions; i++) {
            HostAssertion h{d->assert_cols[i], d->assert_steps[i], HF::reduce(HF::from_bytes(d->assert_values + 16 * i).v)};
            if (h.col >= a.w || h.step >= a.n) throw InvalidArg("assertion out of range");
            a.assertions.push_back(h);
        }
        std::stable_sort(a.assertions.begin(), a.assertions.end(), [](const HostAssertion& x, const HostAssertion& y) {
            return x.step != y.step ? x.step < y.step : x.col < y.col; });
        for (size_t i = 0; i + 1 < a.assertions.size(); i++)
            if (a.assertions[i].step == a.assertions[i + 1].step && a.assertions[i].col == a.assertions[i + 1].col)
                throw InvalidArg("overlapping assertions");
        if (a.id == ZKB_AIR_ID_AGGREGATION && ((a.w & 1) || a.params.size() != 1)) throw InvalidArg("aggregation air needs an even width and the factor k");
        if (a.id == ZKB_AIR_ID_MIMC && (a.params.size() < 2 || !is_pow2(a.params.size()) || a.params.size() > a.n))
            throw InvalidArg("mimc air needs a power-of-two round-constant cycle");
        return a;
    }

    // Context::to_elements() ++ PublicInputs::to_elements()   [A.5, Appendix D items 1-2]
    std::vector<HF> coin_seed() const {
        std::vector<HF> e;
        e.push_back(HF::raw(((u128)w << 8)));            // (main width << 8) | num aux segments
        e.push_back(HF::raw((u128)n));                   // trace length
        e.push_back(HF::raw((u128)(uint64_t)HF::modulus()));
        e.push_back(HF::raw((u128)(uint64_t)(HF::modulus() >> 64)));
        e.push_back(HF::raw((u128)(assertions.size() + num_transition())));  // number of constraints
        uint32_t buf = field_ext;
        buf = (buf << 8) | folding; buf = (buf << 8) | rem_max_degree; buf = (buf << 8) | blowup;
        e.push_back(HF::raw(buf));
        e.push_back(HF::raw(grinding));
        e.push_back(HF::raw(num_queries));
        e.insert(e.end(), pub_elems.begin(), pub_elems.end());
        return e;
    }
};

// ---- DefaultRandomCoin<Blake3_256> (src/training/prover.rs:227)  [A.5]: the seed; the channel itself runs on the device
// (csrc/coin.cuh) -----------------------------------------------------------------------------------------------------------
struct HostCoin {
    uint8_t seed[32];
    void init(const std::vector<HF>& e) { b3_hash_host((const uint8_t*)e.data(), e.size() * 16, seed); }
};

// ---- MerkleTree::prove_batch as an index plan  [A.6] ---------------------------------------------------------
// The tree lives on the device as a heap of 2N digests: heap[1] = root, heap[N + l] = leaf l.
// The plan lists, per output vector of BatchMerkleProof.nodes, the heap indices to gather.
static inline std::vector<std::vector<uint64_t>> plan_batch_proof(uint32_t depth, const std::vector<uint32_t>& positions) {
    const uint64_t N = (uint64_t)1 << depth;
    std::set<uint64_t> have(positions.begin(), positions.end());
    if (have.size() != positions.size()) throw std::runtime_error("duplicate query position");
    std::set<uint64_t> norm;
    for (uint32_t p : positions) norm.insert((uint64_t)p & ~(uint64_t)1);
    std::vector<std::vector<uint64_t>> plan;
    std::vector<uint64_t> next;
    for (uint64_t idx : norm) {
        std::vector<uint64_t> v;
        for (uint64_t i = idx; i < idx + 2; i++) if (!have.count(i)) v.push_back(N + i);
        plan.push_back(v);
        next.push_back((idx + N) >> 1);
    }
    for (uint32_t d = 1; d < depth; d++) {
        std::vector<uint64_t> cur = next;
        next.clear();
        size_t i = 0;
        while (i < cur.size()) {
            uint64_t sib = cur[i] ^ 1;
            if (i + 1 < cur.size() && cur[i + 1] == sib) i++;
            else plan[i].push_back(sib);  // upstream pushes into nodes[i] with the per-level index i
            next.push_back(sib >> 1);
            i++;
        }
    }
    return plan;
}

// ---- winter-utils ByteWriter  ----------------------------------------------------------------------------------
struct ByteWriter {
    std::vector<uint8_t> buf;
    void u8(uint8_t v) { buf.push_back(v); }
    void raw(const void* p, size_t n) { const uint8_t* q = (const uint8_t*)p; buf.insert(buf.end(), q, q + n); }
    void u16(uint16_t v) { raw(&v, 2); }
    void u32(uint32_t v) { raw(&v, 4); }
    void u64(uint64_t v) { raw(&v, 8); }
    void usize(uint64_t value) {  // vint64
        int zeros = value == 0 ? 64 : __builtin_clzll(value);
        int len = (zeros > 0 ? zeros - 1 : 0) / 7;
        int length = 9 - std::min(len, 8);
        if (length == 9) { u8(0); u64(value); }
        else { uint64_t enc = ((value << 1) | 1) << (length - 1); raw(&enc, length); }
    }
};

// BatchMerkleProof::write_into  [A.6, Appendix D]
static inline std::vector<uint8_t> batch_proof_bytes(uint32_t depth, const std::vector<std::vector<uint64_t>>& plan, const uint8_t* gathered) {
    ByteWriter w;
    w.u8((uint8_t)depth);
    w.usize(plan.size());
    size_t k = 0;
    for (auto& v : plan) {
        w.usize(v.size());
        for (size_t i = 0; i < v.size(); i++) { w.raw(gathered + 32 * k, 32); k++; }
    }
    return w.buf;
}

// Proof::to_bytes()  [A.5, Appendix D]: Context, num_unique_queries, Commitments, trace Queries, constraint Queries,
// OodFrame, FriProof, pow_nonce
struct ProofParts {
    std::vector<Digest32> commitments;
    std::vector<uint8_t> trace_rows, trace_paths, comp_rows, comp_paths;
    std::vector<HF> ood_trace_interleaved, ood_h, remainder;
    std::vector<std::vector<uint8_t>> fri_rows, fri_paths;
    uint64_t nonce = 0;
    uint32_t n_unique = 0;
};
static inline std::vector<uint8_t> serialize_proof(const AirSpec& a, const ProofParts& p) {
    ByteWriter w;
    w.u8((uint8_t)a.w); w.u8(0); w.u8(0); w.u8((uint8_t)log2u(a.n)); w.u16(0);          // TraceInfo
    w.u8(16); { u128 m = HF::modulus(); w.raw(&m, 16); }                                 // field modulus bytes
    w.u8((uint8_t)a.num_queries); w.u8((uint8_t)a.blowup); w.u8((uint8_t)a.grinding); w.u8((uint8_t)a.field_ext);
    w.u8((uint8_t)a.folding); w.u8((uint8_t)a.rem_max_degree); w.u8((uint8_t)a.batch_c); w.u8((uint8_t)a.batch_d);
    w.u8(1); w.u8(1);                                                                      // PartitionOptions(1, 1)
    w.u8((uint8_t)p.n_unique);
    w.u16((uint16_t)(p.commitments.size() * 32));
    for (auto& d : p.commitments) w.raw(d.b, 32);
    w.usize(p.trace_rows.size()); w.raw(p.trace_rows.data(), p.trace_rows.size());
    w.usize(p.trace_paths.size()); w.raw(p.trace_paths.data(), p.trace_paths.size());
    w.usize(p.comp_rows.size()); w.raw(p.comp_rows.data(), p.comp_rows.size());
    w.usize(p.comp_paths.size()); w.raw(p.comp_paths.data(), p.comp_paths.size());
    w.u16((uint16_t)(1 + p.ood_trace_interleaved.size() * 16)); w.u8(2);
    w.raw(p.ood_trace_interleaved.data(), p.ood_trace_interleaved.size() * 16);
    w.u16(0);
    w.u16((uint16_t)(p.ood_h.size() * 16)); w.raw(p.ood_h.data(), p.ood_h.size() * 16);
    w.u8((uint8_t)p.fri_rows.size());
    for (size_t i = 0; i < p.fri_rows.size(); i++) {
        w.u32((uint32_t)p.fri_rows[i].size()); w.raw(p.fri_rows[i].data(), p.fri_rows[i].size());
        w.u32((uint32_t)p.fri_paths[i].size()); w.raw(p.fri_paths[i].data(), p.fri_paths[i].size());
    }
    w.u16((uint16_t)(p.remainder.size() * 16)); w.raw(p.remainder.data(), p.remainder.size() * 16);
    w.u8(1);
    w.u64(p.nonce);
    return w.buf;
}

// ---- readers: the inverse of serialize_proof / batch_proof_bytes over untrusted bytes ------------------------------------
// Every read is bounds-checked before it happens (lengths are compared with what is left, never added to a position first).
struct ByteReader {
    const uint8_t* p; size_t n, pos = 0;
    bool ok = true;
    ByteReader(const uint8_t* p_, size_t n_) : p(p_), n(n_) {}
    bool need(size_t k) { if (!ok || k > n - pos) ok = false; return ok; }
    uint64_t le(size_t k) { if (!need(k)) return 0; uint64_t v = 0; memcpy(&v, p + pos, k); pos += k; return v; }
    uint8_t u8() { return (uint8_t)le(1); }
    uint16_t u16() { return (uint16_t)le(2); }
    uint32_t u32() { return (uint32_t)le(4); }
    uint64_t u64() { return le(8); }
    size_t skip(uint64_t k) { const size_t at = pos; if (need(k)) pos += (size_t)k; return at; }   // offset of the skipped bytes
    uint64_t usize() {  // vint64
        const uint8_t first = u8();
        if (!ok) return 0;
        const int length = first == 0 ? 9 : __builtin_ctz(first) + 1;
        if (length == 9) return u64();
        uint64_t enc = first;
        for (int i = 1; i < length; i++) enc |= (uint64_t)u8() << (8 * i);
        return enc >> length;
    }
};
static inline bool canonical(const uint8_t* e) { u128 v; memcpy(&v, e, 16); return v < HF::modulus(); }

// Where each section of Proof::to_bytes() lies in the input (byte offsets, lengths in bytes), as serialize_proof writes them
struct Span { size_t off = 0, len = 0; };
struct ProofLayout {
    uint32_t w = 0, log_n = 0;
    uint8_t opt[8] = {};             // num_queries, blowup, grinding, field extension, folding, remainder degree, batching x2
    uint32_t n_unique = 0;
    Span commitments, trace_rows, trace_paths, comp_rows, comp_paths, ood_trace, ood_h, remainder;
    std::vector<Span> fri_rows, fri_paths;
    uint64_t nonce = 0;
    size_t n_commitments() const { return commitments.len / 32; }
};
// false: not a proof (the sequential verifier's deserialization error).  The OOD frame and the remainder must be canonical
// here; queried rows are checked where the verifier reads them.
static inline bool parse_proof(const uint8_t* b, size_t len, ProofLayout& L) {
    ByteReader r(b, len);
    L = ProofLayout();
    L.w = r.u8();
    if (r.u8() != 0 || r.u8() != 0) return false;
    L.log_n = r.u8();
    if (!r.ok || L.log_n < 3 || L.log_n > 32) return false;
    if (r.u16() != 0 || r.u8() != 16) return false;
    { const size_t m = r.skip(16); u128 P = HF::modulus(); if (!r.ok || memcmp(b + m, &P, 16)) return false; }
    for (auto& o : L.opt) o = r.u8();
    if (r.u8() != 1 || r.u8() != 1) return false;
    L.n_unique = r.u8();
    { const uint16_t cl = r.u16(); if (cl % 32) return false; L.commitments = {r.skip(cl), cl}; }
    auto vec = [&](Span& s) { const uint64_t k = r.usize(); s = {r.skip(k), (size_t)k}; };
    vec(L.trace_rows); vec(L.trace_paths); vec(L.comp_rows); vec(L.comp_paths);
    auto elems = [&](Span& s, size_t bytes) {
        s = {r.skip(bytes), bytes};
        if (r.ok) for (size_t i = 0; i < bytes; i += 16) if (!canonical(b + s.off + i)) r.ok = false;
    };
    { const uint16_t tl = r.u16(); if (!r.ok || tl < 1 || (tl - 1) % 16 || r.u8() != 2) return false; elems(L.ood_trace, tl - 1u); }
    if (r.u16() != 0) return false;
    { const uint16_t el = r.u16(); if (el % 16) return false; elems(L.ood_h, el); }
    const uint8_t nl = r.u8();
    L.fri_rows.resize(nl); L.fri_paths.resize(nl);
    for (uint32_t i = 0; i < nl; i++) {
        const uint32_t a = r.u32(); L.fri_rows[i] = {r.skip(a), a};
        const uint32_t c = r.u32(); L.fri_paths[i] = {r.skip(c), c};
    }
    { const uint16_t rl = r.u16(); if (rl % 16) return false; elems(L.remainder, rl); }
    if (r.u8() != 1) return false;
    L.nonce = r.u64();
    return r.ok && r.pos == len;
}

// BatchMerkleProof::read_from: depth and, per vector of `nodes`, the offsets of its digests.  false: not a batch proof.
struct BatchProofLayout { uint32_t depth = 0; std::vector<std::vector<size_t>> nodes; };
static inline bool parse_batch_proof(const uint8_t* b, size_t len, BatchProofLayout& L) {
    ByteReader r(b, len);
    L = BatchProofLayout();
    L.depth = r.u8();
    const uint64_t nv = r.usize();
    if (!r.ok || nv > len) return false;
    L.nodes.resize((size_t)nv);
    for (auto& v : L.nodes) {
        const uint64_t k = r.usize();
        if (!r.ok || k > 64) return false;
        for (uint64_t i = 0; i < k; i++) { const size_t at = r.skip(32); if (!r.ok) return false; v.push_back(at); }
    }
    return r.ok && r.pos == len;
}

// BatchMerkleProof::get_root as a plan of merges, for the device: `leaf_ids[i]` is the digest id of the leaf at indexes[i]
// (any order), node_ids[i] the ids of the digests of nodes[i].  Every merge gets a fresh id from `next_id` and is appended to
// jobs[level] (level 0 merges leaves).  Returns false, like get_root, when the proof's structure does not fit the indexes
// (an index out of range, a duplicate, a missing or surplus node vector, a node vector that runs out); *root_id is the id of
// the computed root otherwise.  get_root's node map is replaced by one array per level: the nodes a level computes are
// ascending and distinct, and a node's sibling, when it is computed too, is its neighbour in that array.
struct MergeJob { uint32_t a, b, out; };
static inline bool plan_batch_root(uint32_t depth, const std::vector<uint32_t>& indexes, const std::vector<uint32_t>& leaf_ids,
                                   const std::vector<std::vector<uint32_t>>& node_ids, std::vector<std::vector<MergeJob>>& all_jobs,
                                   uint32_t& all_next_id, uint32_t* root_id) {
    if (indexes.empty() || depth < 1 || depth > 32) return false;
    const uint64_t n = (uint64_t)1 << depth;
    std::vector<std::pair<uint64_t, uint32_t>> leaf(indexes.size());   // (leaf index, digest id), ascending
    for (size_t i = 0; i < indexes.size(); i++) {
        if (indexes[i] >= n) return false;
        leaf[i] = {indexes[i], leaf_ids[i]};
    }
    std::sort(leaf.begin(), leaf.end());
    size_t pairs = 0;   // distinct (index & ~1): one node vector each
    for (size_t i = 0; i < leaf.size(); i++) {
        if (i && leaf[i].first == leaf[i - 1].first) return false;
        if (!i || (leaf[i].first & ~1ull) != (leaf[i - 1].first & ~1ull)) pairs++;
    }
    if (pairs != node_ids.size()) return false;
    std::vector<std::vector<MergeJob>> jobs(depth);   // appended to all_jobs only if the structure fits
    uint32_t next_id = all_next_id;
    std::vector<uint64_t> cur, nxt;                   // heap indices of the nodes computed at a level, ascending
    std::vector<uint32_t> cur_id, nxt_id;
    std::vector<size_t> ptr;                          // next unread node of each vector
    for (size_t i = 0, k = 0; i < leaf.size(); k++) {
        const uint64_t idx = leaf[i].first & ~1ull;
        uint32_t l, r;
        if (leaf[i].first == idx) {
            l = leaf[i].second;
            if (i + 1 < leaf.size() && leaf[i + 1].first == idx + 1) { r = leaf[i + 1].second; ptr.push_back(0); i += 2; }
            else { if (node_ids[k].empty()) return false; r = node_ids[k][0]; ptr.push_back(1); i += 1; }
        } else {
            if (node_ids[k].empty()) return false;
            l = node_ids[k][0]; r = leaf[i].second; ptr.push_back(1); i += 1;
        }
        jobs[0].push_back({l, r, next_id});
        cur.push_back((n + idx) >> 1);
        cur_id.push_back(next_id++);
    }
    for (uint32_t d = 1; d < depth; d++) {
        nxt.clear(); nxt_id.clear();
        for (size_t k = 0; k < cur.size(); k++) {
            const uint64_t node = cur[k], sib = node ^ 1;
            const uint32_t nd = cur_id[k];
            uint32_t sd;
            if (k + 1 < cur.size() && cur[k + 1] == sib) { sd = cur_id[k + 1]; k++; }
            else { if (node_ids[k].size() <= ptr[k]) return false; sd = node_ids[k][ptr[k]++]; }
            jobs[d].push_back((node & 1) ? MergeJob{sd, nd, next_id} : MergeJob{nd, sd, next_id});
            nxt.push_back(node >> 1);
            nxt_id.push_back(next_id++);
        }
        cur.swap(nxt); cur_id.swap(nxt_id);
    }
    if (cur.empty() || cur[0] != 1) return false;
    *root_id = cur_id[0];
    if (all_jobs.size() < depth) all_jobs.resize(depth);
    for (uint32_t d = 0; d < depth; d++) all_jobs[d].insert(all_jobs[d].end(), jobs[d].begin(), jobs[d].end());
    all_next_id = next_id;
    return true;
}

// winter-fri fold_positions  [A.10]
static inline std::vector<uint32_t> fold_positions(const std::vector<uint32_t>& pos, uint64_t domain, uint32_t folding) {
    uint64_t target = domain / folding;
    std::vector<uint32_t> r;
    for (uint32_t p : pos) { uint32_t q = (uint32_t)(p % target); if (std::find(r.begin(), r.end(), q) == r.end()) r.push_back(q); }
    return r;
}

}  // namespace zkb
