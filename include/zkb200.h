/*
 * zkb200 — C ABI of the B200-native STARK proving backend (libzkb200.so).
 *
 * This is the drop-in boundary for the Winterfell 0.12 `Prover` plug-in points the reference uses.
 * The reference is Rust (no cargo/rustc in the build image), so the boundary is this C ABI; the Rust
 * glue that binds it is shown in INTEGRATION.md and rust/zkb200-winterfell/.  Citations are relative
 * to /root/reference.
 *
 * Conventions
 *   - every function returns 0 on success and a negative zkb_status on failure; the message is
 *     available through zkb_last_error(ctx) (or zkb_last_error(NULL) for context creation);
 *     nothing panics or throws across the boundary;
 *   - field elements are 16-byte little-endian canonical values of
 *     p = 2^128 - 45*2^40 + 1 (winter-math f128::BaseElement, src/training/prover.rs:9);
 *     digests are 32-byte BLAKE3 outputs (Blake3_256<Felt>, src/training/prover.rs:225);
 *   - the caller owns every host buffer; the library owns all device memory until zkb_ctx_destroy;
 *   - a context is bound to one device and one stream and must be used from one thread at a time;
 *     different contexts may be used concurrently;
 *   - there is no CPU fallback: without a CUDA device every call fails with ZKB_ERR_CUDA.
 */
#ifndef ZKB200_H
#define ZKB200_H
#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct zkb_ctx zkb_ctx;

typedef enum {
    ZKB_OK = 0,
    ZKB_ERR_INVALID = -1, /* bad argument / unsupported option (the reference panics: src/training/prover.rs:59-61) */
    ZKB_ERR_CUDA = -2,    /* CUDA runtime failure, including "no device" */
    ZKB_ERR_STATE = -3,   /* staged call out of order */
    ZKB_ERR_OOM = -4
} zkb_status;

/* AIRs on the hot path */
#define ZKB_AIR_ID_TRAINING 1u    /* src/training/air.rs:105-287   */
#define ZKB_AIR_ID_AGGREGATION 2u /* src/aggregation/air.rs:93-147 */
#define ZKB_AIR_ID_MIMC 3u        /* defined by this build from src/helper.rs:213-220,404-406 (SURVEY D1) */

/*
 * Everything `Prover::prove` derives from (Air, ProofOptions, PublicInputs):
 *   options       winterfell::ProofOptions::new argument order, src/main.rs:98-107; folding (the FRI folding factor) is one of
 *                 2, 4, 8, 16, as ProofOptions::new accepts; any other value is ZKB_ERR_INVALID
 *   pub_elems     PublicInputs::to_elements(): src/training/air.rs:70-94, src/aggregation/air.rs:57-81
 *   assertions    Air::get_assertions(): src/training/air.rs:130-151, src/aggregation/air.rs:121-147
 *   params        aggregation: the scaling factor k (src/aggregation/air.rs:108);
 *                 mimc: the periodic round-constant column (power-of-two length)
 */
typedef struct {
    uint32_t air_id, trace_width;
    uint64_t trace_len;
    uint32_t num_queries, blowup, grinding_bits, field_extension, folding, rem_max_degree, batching_constraints,
        batching_deep;
    const uint8_t* pub_elems;
    uint64_t n_pub_elems;
    const uint32_t* assert_cols;
    const uint64_t* assert_steps;
    const uint8_t* assert_values;
    uint64_t n_assertions;
    const uint8_t* params;
    uint64_t n_params;
} zkb_air_desc;

/* Fiat-Shamir transcript of one proof, exported for stage-by-stage parity checks.
 * n_fri_layers is the proof's true number of FRI layers; fri_roots / fri_alphas hold the first min(n_fri_layers, 16) of them
 * (a small folding factor can need more than 16 layers, up to 29 at folding 2).  The proof bytes carry every layer. */
typedef struct {
    uint8_t trace_root[32], constraint_root[32], remainder_commitment[32];
    uint8_t constraint_alpha[16], z[16], deep_alpha[16];
    uint32_t n_fri_layers, n_positions;
    uint8_t fri_roots[16][32];
    uint8_t fri_alphas[16][16];
    uint64_t pow_nonce;
    uint32_t positions[256];
    int32_t comp_degree_ok, _pad;
} zkb_transcript;

/* per-stage device time of the last proof, milliseconds (CUDA events on the context's stream) */
typedef struct {
    float h2d, interpolate, lde, leaf_hash, merkle, constraints, composition, ood, deep, fri, grind, queries, total;
} zkb_stage_times;

/* ---- context ------------------------------------------------------------------------------------ */
/* stream: a cudaStream_t (or NULL for the default stream) the caller wants all work issued on */
int32_t zkb_ctx_create(int32_t device, void* stream, zkb_ctx** out);
/* same, on a private non-blocking stream created and destroyed with the context: what the lanes of zkb_prove_batch should be
 * (contexts that share the default stream are correct but run one after the other) */
int32_t zkb_ctx_create_lane(int32_t device, zkb_ctx** out);
void zkb_ctx_destroy(zkb_ctx* ctx);
const char* zkb_last_error(const zkb_ctx* ctx);
/* number of kernels the context has launched so far (evidence for bench.py's gpu_launches) */
uint64_t zkb_kernel_launches(const zkb_ctx* ctx);
int32_t zkb_last_stage_times(const zkb_ctx* ctx, zkb_stage_times* out);
/* pinned host memory for trace columns (fast H2D); plain malloc'ed memory works too, only slower */
void* zkb_host_alloc(size_t bytes);
void zkb_host_free(void* p);

/* ---- Prover::prove (src/main.rs:228,424,468; src/training/prover.rs:221-301) ------------------------- */
/*
 * cols: trace_width host pointers, column j = trace_len elements (TraceTable columns, column-major).
 * force_nonce: 0 = grind for the smallest valid nonce (non-`concurrent` Winterfell); otherwise use it.
 * proof_out: Proof::to_bytes() layout, allocated by the library; release with zkb_free.
 * The Fiat-Shamir channel runs on the device: the call enqueues every stage without waiting, blocks once, downloads the
 * transcript and the openings in one copy and assembles the proof.  Small proofs (LDE rows x width < 2^22) are replayed from a
 * CUDA graph from the third proof of a shape on; coin seed, assertion values, AIR parameters and the trace are per-proof inputs.
 */
int32_t zkb_prove(zkb_ctx* ctx, const zkb_air_desc* air, const uint8_t* const* cols, uint64_t force_nonce,
                  uint8_t** proof_out, uint64_t* proof_len, zkb_transcript* transcript);
/* same, with the column-major trace [w][n] already resident in device memory */
int32_t zkb_prove_device(zkb_ctx* ctx, const zkb_air_desc* air, const void* d_trace_colmajor, uint64_t force_nonce,
                         uint8_t** proof_out, uint64_t* proof_len, zkb_transcript* transcript);
/*
 * A batch of independent proofs (BASELINE configs[3]: the reference proves its devices one after the other, src/main.rs:160,379):
 * proof i runs on lanes[i % n_lanes]; every lane is a zkb_ctx of its own (device + stream + buffers) driven by its own host thread
 * inside the call, so H2D copies, kernels and Fiat-Shamir round trips of different proofs overlap (create the lanes with
 * zkb_ctx_create_lane or on distinct streams).  Lanes may sit on different devices.  proofs_out[i] / lens_out[i] as in zkb_prove (release each with zkb_free); on failure the first failing proof's status is
 * returned, its message is in that lane's zkb_last_error, and the outputs of proofs that did not complete are NULL / 0.
 */
int32_t zkb_prove_batch(zkb_ctx* const* lanes, uint32_t n_lanes, const zkb_air_desc* const* airs, const uint8_t* const* const* cols,
                        uint32_t count, uint8_t** proofs_out, uint64_t* lens_out);
void zkb_free(void* p);

/* ---- staged surface: the three associated types + the stages inside Prover::prove ------------------------
 * Order: begin -> trace_commit -> constraints_eval -> constraints_commit -> ood_eval -> deep_compose
 *        -> { fri_commit_layer, fri_fold }* -> fri_remainder -> grind -> query -> (next begin)
 */
int32_t zkb_begin(zkb_ctx* ctx, const zkb_air_desc* air);
/* Prover::new_trace_lde -> DefaultTraceLde::new (src/training/prover.rs:273-281): K1-K4 */
int32_t zkb_trace_commit(zkb_ctx* ctx, const uint8_t* const* cols, uint8_t root_out[32]);
int32_t zkb_trace_commit_device(zkb_ctx* ctx, const void* d_trace_colmajor, uint8_t root_out[32]);
/* TraceLde::read_main_trace_frame_into (SURVEY A.4): current and next row of LDE step `lde_step`
 * (next = row lde_step + blowup, wrapping around the LDE domain).  One host round trip per call. */
int32_t zkb_trace_read_frame(zkb_ctx* ctx, uint64_t lde_step, uint8_t* current_out, uint8_t* next_out);
/* the same for `count` steps in ONE round trip: current_out / next_out hold count rows of trace_width elements each.
 * Winterfell's DefaultConstraintEvaluator reads one frame per constraint-evaluation point from rayon threads (TraceLde: Sync);
 * a context is single-threaded and a round trip costs ~20 us, so a caller that keeps the default evaluator must batch its
 * reads through this call — the intended pairing is zkb_constraints_eval, which never moves frames to the host. */
int32_t zkb_trace_read_frames(zkb_ctx* ctx, const uint64_t* lde_steps, uint32_t count, uint8_t* current_out, uint8_t* next_out);
/* TracePolyTable contents, row-major [n][w] coefficients (only needed if the host keeps DEEP) */
int32_t zkb_trace_polys_read(zkb_ctx* ctx, uint8_t* out);
/* Prover::new_evaluator + ConstraintEvaluator::evaluate (src/training/prover.rs:283-290): K5.
 * alpha: the single draw of ConstraintCompositionCoefficients::draw_algebraic.
 * evals_out (optional): CompositionPolyTrace, ce_blowup*trace_len elements. */
int32_t zkb_constraints_eval(zkb_ctx* ctx, const uint8_t alpha[16], uint8_t* evals_out);
/* Prover::build_constraint_commitment -> DefaultConstraintCommitment::new (src/training/prover.rs:292-300): K6 */
int32_t zkb_constraints_commit(zkb_ctx* ctx, uint8_t root_out[32]);
/* TracePolyTable::get_ood_frame + CompositionPoly::evaluate_at: K7.  cur/next: w elements, h: c elements */
int32_t zkb_ood_eval(zkb_ctx* ctx, const uint8_t z[16], uint8_t* cur_out, uint8_t* next_out, uint8_t* h_out);
/* DeepCompositionPoly::{add_trace_polys, add_composition_poly, evaluate}: K8; alpha = the DEEP draw */
int32_t zkb_deep_compose(zkb_ctx* ctx, const uint8_t deep_alpha[16]);
/* FriProver::build_layers, one layer at a time: K9 */
int32_t zkb_fri_num_layers(zkb_ctx* ctx, uint32_t* out);
int32_t zkb_fri_commit_layer(zkb_ctx* ctx, uint8_t root_out[32]);
int32_t zkb_fri_fold(zkb_ctx* ctx, const uint8_t alpha[16]);
/* remainder coefficients in Winterfell's (reversed) order; n_coeffs_out elements */
int32_t zkb_fri_remainder(zkb_ctx* ctx, uint8_t* coeffs_out, uint64_t* n_coeffs_out, uint8_t commitment_out[32]);
/* ProverChannel::grind_query_seed: smallest nonce >= 1 with >= bits trailing zeros: K10 */
int32_t zkb_grind(zkb_ctx* ctx, const uint8_t seed[32], uint32_t bits, uint64_t* nonce_out);
/* TraceLde::query / ConstraintCommitment::query / FriProver::build_proof: K11.
 * which: 0 = trace (any time after zkb_trace_commit), 1 = constraint composition (after zkb_constraints_commit),
 *        2+l = FRI layer l (after zkb_fri_remainder; positions already folded by the caller).
 * rows_out: n_pos rows, row-major; proof_out: BatchMerkleProof::to_bytes(), allocated by the library.
 * After a column-sharded proof (zkb_mg_prove*) the context holds only this rank's share of the trace: ZKB_ERR_STATE. */
int32_t zkb_query(zkb_ctx* ctx, uint32_t which, const uint32_t* positions, uint32_t n_pos, uint8_t* rows_out,
                  uint8_t** proof_out, uint64_t* proof_len);

/* ---- one large proof sharded across the GPUs of a node (SURVEY §8e; BASELINE.json configs[4]) -------------------------
 * One process per GPU.  Rank r owns trace columns [r*w/G, (r+1)*w/G): ingest, interpolation and the coset LDE are column-
 * local; an NCCL all-to-all over NVLink turns column shards into row shards for leaf hashing and the Merkle subtrees, whose
 * roots are all-gathered; constraint evaluation, OOD and DEEP are column-local partial sums combined by an all-gather.
 * `air` describes the WHOLE trace (global width, all assertions); `local_cols` holds this rank's w/G columns.
 * The Fiat-Shamir channel runs replicated on every rank's device (all ranks hold the same commitments, OOD frame and
 * remainder) and the openings are completed by one all-reduce: the host is met once per proof, for the final download.
 * Every rank returns the same proof bytes.  G must be a power of two that divides w (and at most the LDE panel size);
 * the aggregation AIR couples columns i and i+60 and is not shardable. */
int32_t zkb_mg_unique_id(uint8_t out[128]);                                         /* ncclGetUniqueId, on rank 0 */
int32_t zkb_mg_init(zkb_ctx* ctx, int32_t rank, int32_t world, const uint8_t id[128]); /* ncclCommInitRank (collective) */
int32_t zkb_mg_prove(zkb_ctx* ctx, const zkb_air_desc* air, const uint8_t* const* local_cols, uint64_t force_nonce,
                     uint8_t** proof_out, uint64_t* proof_len, zkb_transcript* transcript);
int32_t zkb_mg_prove_device(zkb_ctx* ctx, const zkb_air_desc* air, const void* d_local_trace_colmajor, uint64_t force_nonce,
                            uint8_t** proof_out, uint64_t* proof_len, zkb_transcript* transcript);

/* ---- helpers next to the path (SURVEY §8f) ---------------------------------------------------------- */
/* device-side MiMC chain trace; out_cols_colmajor: w*n elements, host memory */
int32_t zkb_mimc_trace(zkb_ctx* ctx, const uint8_t* seeds, uint32_t w, uint64_t n, const uint8_t* round_constants,
                       uint32_t n_rc, uint8_t* out_colmajor);
/* same, leaving the trace in device memory; returns the device pointer (owned by the context) */
int32_t zkb_mimc_trace_device(zkb_ctx* ctx, const uint8_t* seeds, uint32_t w, uint64_t n, const uint8_t* round_constants,
                              uint32_t n_rc, void** d_out);
/* host-side BLAKE3-256 (Blake3_256::hash); no device needed — used by the CPU verifier of the Python mirror */
int32_t zkb_blake3_host(const uint8_t* data, uint64_t len, uint8_t out[32]);
/* batched mimc_cipher (src/helper.rs:213-220): out[i] = mimc_cipher(inputs[i], round_constants[i], zs[i]); benches/bench_mimc.rs:17-34 */
int32_t zkb_mimc_cipher_batch(zkb_ctx* ctx, const uint8_t* inputs, const uint8_t* round_constants, const uint8_t* zs, uint64_t count,
                              uint8_t* out);
/* batched mimc_hash_matrix (src/helper.rs:222-233; the aggregation digest, src/aggregation/prover.rs:176-178):
 * w = count matrices [ac][fe], b = count vectors [ac]; benches/bench_mimc.rs:39-57 */
int32_t zkb_mimc_hash_matrix_batch(zkb_ctx* ctx, const uint8_t* w, const uint8_t* b, uint32_t ac, uint32_t fe, const uint8_t* round_constants,
                                   uint32_t n_rc, uint64_t count, uint8_t* out);
/* device-side training trace (src/training/prover.rs:90-218 without the PCIe ingest): the caller uploads the n_raw distinct raw
 * state rows (n_raw = batch_size + 1, `half` = 120 values each); rows are [raw + mask || mask] with 64-bit masks generated on the
 * device.  The masks hide the raw model state (the masked first and last rows are public inputs, src/training/air.rs), so they
 * are a ChaCha20 keystream: key32 = 32 key bytes, or NULL to draw the key from OS entropy (getrandom) — what the reference's
 * rand::thread_rng() does (src/training/prover.rs:117-121).  Pass a key only for reproducible tests.  Mask of (row i, column j)
 * = little-endian u64 number (j mod 8) of ChaCha20 block (i * ceil(half/8) + j div 8), nonce 0.
 * Returns the device pointer (context-owned, column-major [2*half][n]) for zkb_prove_device and the first /
 * last trace rows (2*half elements each) that get_pub_inputs needs (src/training/prover.rs:245-246). */
int32_t zkb_training_trace_device(zkb_ctx* ctx, const uint8_t* raw_rows, uint32_t n_raw, uint32_t half, uint64_t n,
                                  const uint8_t* key32, void** d_out, uint8_t* first_row_out, uint8_t* last_row_out);
/* copy `bytes` bytes of context-owned device memory to the host (debugging / tests) */
int32_t zkb_download(zkb_ctx* ctx, const void* d_src, uint64_t bytes, uint8_t* out);
/* upload a column-major host trace into a context-owned device buffer (for device-resident timing) */
int32_t zkb_upload_trace(zkb_ctx* ctx, const uint8_t* const* cols, uint32_t w, uint64_t n, void** d_out);

/* ---- self-test kernels for KATs (field ops and hash_elements on the device) ------------------------------ */
int32_t zkb_test_field(zkb_ctx* ctx, const uint8_t* a, const uint8_t* b, uint32_t n, uint8_t* mul_out, uint8_t* add_out,
                       uint8_t* sub_out, uint8_t* inv_out);
int32_t zkb_test_hash_elements(zkb_ctx* ctx, const uint8_t* rows, uint32_t elems_per_row, uint32_t n_rows,
                               uint8_t* digests_out);
int32_t zkb_test_merkle_root(zkb_ctx* ctx, const uint8_t* leaves, uint64_t n_leaves, uint8_t root_out[32]);
/* LDE of a column-major host matrix: out row-major [n*blowup][w] (for parity tests of K1+K2) */
int32_t zkb_test_lde(zkb_ctx* ctx, const uint8_t* const* cols, uint32_t w, uint64_t n, uint32_t blowup, uint8_t* polys_out,
                     uint8_t* lde_out);

#ifdef __cplusplus
}
#endif
#endif /* ZKB200_H */
