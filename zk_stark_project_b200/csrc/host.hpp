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

// winter-fri fold_positions  [A.10]
static inline std::vector<uint32_t> fold_positions(const std::vector<uint32_t>& pos, uint64_t domain, uint32_t folding) {
    uint64_t target = domain / folding;
    std::vector<uint32_t> r;
    for (uint32_t p : pos) { uint32_t q = (uint32_t)(p % target); if (std::find(r.begin(), r.end(), q) == r.end()) r.push_back(q); }
    return r;
}

}  // namespace zkb
