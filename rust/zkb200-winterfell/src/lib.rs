//! zkb200-winterfell — plugs the B200 backend into the reference's `winterfell::Prover` impls.
//!
//! NOT COMPILED IN THIS REPOSITORY (no Rust toolchain in the build image, SURVEY.md D7).  Written against the
//! Winterfell 0.12 surface the reference itself uses (`/root/reference/src/training/prover.rs:3-9,221-301`) plus the
//! trait definitions recalled in SURVEY.md Appendix A.4; items marked VERIFY-FIRST depend on upstream details that
//! could not be read here (Appendix D).  Every value these types hand to Winterfell is checked against the CPU oracle
//! through the same C-ABI calls by `tests/test_gpu_parity2.py::test_staged_values_*`.
//!
//! Two integration levels:
//!
//! 1. **Associated types** (what `BASELINE.json` asks for; `main.rs` untouched).  [`GpuTraceLde`],
//!    [`GpuConstraintEvaluator`] and [`GpuConstraintCommitment`] replace the `Default*` types named at
//!    `src/training/prover.rs:228-233` / `src/aggregation/prover.rs:201-206`, and the three factory methods
//!    (`:273-300`) delegate to [`GpuBackend`].  Winterfell's own `generate_proof` keeps the Fiat-Shamir channel,
//!    OOD/DEEP, FRI and `Proof` serialisation, so only mathematically defined values cross the FFI: LDE rows, trace
//!    polynomials, BLAKE3 digests, constraint evaluations, Merkle openings.  The heavy stages (interpolation, LDE, row
//!    hashing, Merkle trees, constraint evaluation) run on the GPU.
//! 2. **Whole proof** — [`GpuProve::prove_gpu`]: all of `Prover::prove` on the device through `zkb_prove` (what
//!    `bench.py` measures; DEEP, FRI, grinding and the channel on the GPU as well).  Needs `prove` → `prove_gpu` at the
//!    three call sites of `src/main.rs` (`:228,424,468`); the returned bytes are in `Proof::to_bytes()` layout.
pub mod ffi;

use std::ffi::CStr;
use std::marker::PhantomData;
use std::ptr;
use std::sync::{Arc, Mutex};

use winter_utils::Deserializable;
use winterfell::{
    crypto::{hashers::Blake3_256, BatchMerkleProof, ElementHasher, Hasher, MerkleTree},
    math::{fields::f128::BaseElement as Felt, FieldElement, StarkField, ToElements},
    matrix::ColMatrix,
    Air, Assertion, AuxRandElements, CompositionPoly, CompositionPolyTrace, ConstraintCommitment,
    ConstraintCompositionCoefficients, ConstraintEvaluator, EvaluationFrame, PartitionOptions, Proof, ProofOptions, Prover,
    ProverError, Queries, StarkDomain, Trace, TraceInfo, TraceLde, TracePolyTable, TraceTable, VerifierError,
};

type H = Blake3_256<Felt>;
type Digest = <H as Hasher>::Digest;
type VC = MerkleTree<H>;

// ---------------------------------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------------------------------

/// One `zkb_ctx`: a device + stream binding that owns all device memory of the proofs run through it.
/// A context is single-threaded (include/zkb200.h); Winterfell requires `TraceLde: Sync` and may call into it from rayon
/// workers, so every use goes through the mutex of [`GpuBackend`].
pub struct GpuContext {
    raw: *mut ffi::zkb_ctx,
}
unsafe impl Send for GpuContext {}

impl GpuContext {
    pub fn new(device: i32) -> Result<Self, String> {
        let mut raw = ptr::null_mut();
        let rc = unsafe { ffi::zkb_ctx_create(device, ptr::null_mut(), &mut raw) };
        if rc != 0 {
            let msg = unsafe { CStr::from_ptr(ffi::zkb_last_error(ptr::null())) };
            return Err(format!("zkb_ctx_create failed ({rc}): {}", msg.to_string_lossy()));
        }
        Ok(Self { raw })
    }
    fn last_error(&self) -> String {
        unsafe { CStr::from_ptr(ffi::zkb_last_error(self.raw)) }.to_string_lossy().into_owned()
    }
    /// Status → panic.  The reference treats construction errors as panics (`src/training/prover.rs:59-61`,
    /// `tests/integration_tests.rs:219-227`) and `ProverError` (winter-prover 0.12: `UnsatisfiedTransitionConstraintError`,
    /// `MismatchedConstraintPolynomialDegree`, `UnsupportedFieldExtension`) has no variant for a device failure, so a
    /// non-zero `zkb_status` — bad argument, CUDA error, out of memory, call out of order — aborts with the library's message
    /// instead of being squeezed into an unrelated variant.
    fn check(&self, rc: i32, what: &str) {
        if rc != 0 {
            panic!("{what} failed (zkb_status {rc}): {}", self.last_error());
        }
    }
}
impl GpuContext {
    /// `winterfell::verify::<Air, Blake3_256, DefaultRandomCoin, MerkleTree>` for every (proof bytes, AIR) pair in one call
    /// (`src/main.rs:251-257, 430-436, 478-484`), with `AcceptableOptions::OptionSet([air's options])`.  A rejected proof is an
    /// `Err` entry; a bad argument or a device failure panics like every other call of this crate (see `check`).
    pub fn verify_batch(&self, batch: &[(&[u8], &GpuAirDesc)]) -> Vec<Result<(), VerifierError>> {
        let descs: Vec<ffi::zkb_air_desc> = batch.iter().map(|(_, a)| a.0.as_ffi()).collect();
        let airs: Vec<*const ffi::zkb_air_desc> = descs.iter().map(|d| d as *const _).collect();
        let proofs: Vec<*const u8> = batch.iter().map(|(p, _)| p.as_ptr()).collect();
        let lens: Vec<u64> = batch.iter().map(|(p, _)| p.len() as u64).collect();
        let mut verdicts = vec![0i32; batch.len()];
        let rc = unsafe {
            ffi::zkb_verify_batch(self.raw, airs.as_ptr(), proofs.as_ptr(), lens.as_ptr(), batch.len() as u32, verdicts.as_mut_ptr(),
                                  ptr::null_mut())
        };
        self.check(rc, "zkb_verify_batch");
        verdicts.into_iter().map(verifier_error).collect()
    }
}
/// zkb_verdict -> winter-verifier 0.12's `VerifierError` (VERIFY-FIRST: variant names recalled from upstream, not compiled here)
fn verifier_error(v: i32) -> Result<(), VerifierError> {
    use winterfell::{FriVerifierError as F, VerifierError as V};
    match v {
        ffi::ZKB_VERIFY_OK => Ok(()),
        ffi::ZKB_VERIFY_MALFORMED | ffi::ZKB_VERIFY_TRACE_INFO | ffi::ZKB_VERIFY_COMMITMENTS | ffi::ZKB_VERIFY_OOD_FRAME
        | ffi::ZKB_VERIFY_TRACE_VALUES | ffi::ZKB_VERIFY_CONSTRAINT_VALUES => {
            Err(V::ProofDeserializationError(format!("zkb_verdict {v}")))
        }
        ffi::ZKB_VERIFY_OPTIONS => Err(V::UnacceptableProofOptions),
        ffi::ZKB_VERIFY_OOD_CONSISTENCY => Err(V::InconsistentOodConstraintEvaluations),
        ffi::ZKB_VERIFY_POW => Err(V::QuerySeedProofOfWorkVerificationFailed),
        ffi::ZKB_VERIFY_UNIQUE_QUERIES => Err(V::ProofDeserializationError("number of unique queries".into())),
        ffi::ZKB_VERIFY_TRACE_MERKLE => Err(V::TraceQueryDoesNotMatchCommitment),
        ffi::ZKB_VERIFY_CONSTRAINT_MERKLE => Err(V::ConstraintQueryDoesNotMatchCommitment),
        ffi::ZKB_VERIFY_FRI_VALUES => Err(V::FriVerificationFailed(F::InvalidLayerValues)),
        ffi::ZKB_VERIFY_FRI_MERKLE => Err(V::FriVerificationFailed(F::LayerCommitmentMismatch)),
        ffi::ZKB_VERIFY_FRI_FOLDING => Err(V::FriVerificationFailed(F::InvalidLayerFolding(0))),
        ffi::ZKB_VERIFY_FRI_TRUNCATION => Err(V::FriVerificationFailed(F::DegreeTruncation(0, 0, 0))),
        ffi::ZKB_VERIFY_REMAINDER_DEGREE => Err(V::FriVerificationFailed(F::RemainderDegreeMismatch(0))),
        ffi::ZKB_VERIFY_REMAINDER_COMMITMENT => Err(V::FriVerificationFailed(F::RemainderCommitmentMismatch)),
        _ => Err(V::FriVerificationFailed(F::InvalidRemainderFolding)),
    }
}
impl Drop for GpuContext {
    fn drop(&mut self) {
        unsafe { ffi::zkb_ctx_destroy(self.raw) }
    }
}

/// Which of the three AIRs a prover drives, plus the AIR parameters the device function needs.
#[derive(Clone)]
pub enum GpuAir {
    /// src/training/air.rs — all transition evaluations are zero (src/helper.rs:141-146).
    Training,
    /// src/aggregation/air.rs — `k` is `pub_inputs.k` (src/aggregation/air.rs:108).
    Aggregation { k: Felt },
    /// MiMC chains with the periodic round-constant column (src/helper.rs:404-406).
    Mimc { round_constants: Vec<Felt> },
}

fn felts_to_bytes(v: &[Felt]) -> Vec<u8> {
    // f128 is canonical: 16 little-endian bytes per element (SURVEY A.1)
    let mut out = Vec::with_capacity(v.len() * 16);
    for e in v {
        out.extend_from_slice(&e.as_int().to_le_bytes());
    }
    out
}
fn bytes_to_felts(b: &[u8]) -> Vec<Felt> {
    b.chunks_exact(16).map(|c| Felt::new(u128::from_le_bytes(c.try_into().unwrap()))).collect()
}
fn digest_from(b: [u8; 32]) -> Digest {
    // ByteDigest<32>: Deserializable reads the 32 raw bytes
    Digest::read_from_bytes(&b).expect("a 32-byte digest")
}

fn batching_code(m: winterfell::BatchingMethod) -> u32 {
    match m {
        winterfell::BatchingMethod::Linear => 0,
        winterfell::BatchingMethod::Algebraic => 1,
        #[allow(unreachable_patterns)]
        _ => 2,
    }
}

/// The AIR a batch-verified proof is checked against: what `winterfell::verify` receives as the AIR type, the public inputs and
/// `AcceptableOptions::OptionSet([options])`.  Build `air` the way `verify` does, `A::new(trace_info, pub_inputs, options)` with
/// the options the caller accepts (src/main.rs:98-107 for the reference's proofs).
pub struct GpuAirDesc(AirDescriptor);
impl GpuAirDesc {
    pub fn new<A: Air<BaseField = Felt>>(air: &A, kind: &GpuAir, pub_inputs: &A::PublicInputs) -> Self {
        Self(AirDescriptor::new(air, kind, &pub_inputs.to_elements()))
    }
}

/// Owned copy of everything `zkb_air_desc` points to (the C struct borrows these buffers for the duration of a call).
struct AirDescriptor {
    air_id: u32,
    width: u32,
    len: u64,
    options: ProofOptions,
    pub_elems: Vec<u8>,
    cols: Vec<u32>,
    steps: Vec<u64>,
    values: Vec<u8>,
    params: Vec<u8>,
}
impl AirDescriptor {
    fn new<A: Air<BaseField = Felt>>(air: &A, kind: &GpuAir, pub_elems: &[Felt]) -> Self {
        let assertions: Vec<Assertion<Felt>> = air.get_assertions();
        let (air_id, params) = match kind {
            GpuAir::Training => (ffi::ZKB_AIR_ID_TRAINING, vec![]),
            GpuAir::Aggregation { k } => (ffi::ZKB_AIR_ID_AGGREGATION, felts_to_bytes(&[*k])),
            GpuAir::Mimc { round_constants } => (ffi::ZKB_AIR_ID_MIMC, felts_to_bytes(round_constants)),
        };
        Self {
            air_id,
            width: air.trace_info().main_trace_width() as u32,
            len: air.trace_length() as u64,
            options: air.options().clone(),
            pub_elems: felts_to_bytes(pub_elems),
            cols: assertions.iter().map(|a| a.column() as u32).collect(),
            steps: assertions.iter().map(|a| a.first_step() as u64).collect(),
            values: felts_to_bytes(&assertions.iter().map(|a| a.values()[0]).collect::<Vec<_>>()),
            params,
        }
    }
    /// The options pass through unchanged: the library proves every FRI folding factor `ProofOptions::new` accepts
    /// (2, 4, 8 and 16) and returns `ZKB_ERR_INVALID` for options it does not support.
    fn as_ffi(&self) -> ffi::zkb_air_desc {
        let o = &self.options;
        ffi::zkb_air_desc {
            air_id: self.air_id,
            trace_width: self.width,
            trace_len: self.len,
            num_queries: o.num_queries() as u32,
            blowup: o.blowup_factor() as u32,
            grinding_bits: o.grinding_factor(),
            field_extension: o.field_extension() as u32,
            folding: o.to_fri_options().folding_factor() as u32,
            rem_max_degree: o.to_fri_options().remainder_max_degree() as u32,
            batching_constraints: batching_code(o.constraint_batching_method()), // VERIFY-FIRST: accessor names
            batching_deep: batching_code(o.deep_poly_batching_method()),
            pub_elems: self.pub_elems.as_ptr(),
            n_pub_elems: (self.pub_elems.len() / 16) as u64,
            assert_cols: self.cols.as_ptr(),
            assert_steps: self.steps.as_ptr(),
            assert_values: self.values.as_ptr(),
            n_assertions: self.cols.len() as u64,
            params: self.params.as_ptr(),
            n_params: (self.params.len() / 16) as u64,
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// level 1: the three associated types
// ---------------------------------------------------------------------------------------------------------------------

struct BackendState {
    ctx: GpuContext,
    air: Option<AirDescriptor>,
}

/// The prover-side handle: lives in the prover struct (one field), is told the AIR in `get_pub_inputs`, and implements the
/// three factory methods.  Cloning shares the context.
#[derive(Clone)]
pub struct GpuBackend {
    state: Arc<Mutex<BackendState>>,
}

impl GpuBackend {
    pub fn new(device: i32) -> Self {
        let ctx = GpuContext::new(device).unwrap_or_else(|e| panic!("{e}"));
        Self { state: Arc::new(Mutex::new(BackendState { ctx, air: None })) }
    }

    /// Called from the prover's `get_pub_inputs` — the first thing `Prover::prove` does (SURVEY §3.2 step 0) — because
    /// `new_trace_lde` receives neither the AIR nor the public inputs, and the device-side evaluator needs the assertions,
    /// the AIR parameters and the options when the trace is committed.
    pub fn set_air<A>(&self, info: &TraceInfo, pub_inputs: &A::PublicInputs, options: &ProofOptions, kind: GpuAir)
    where
        A: Air<BaseField = Felt>,
        A::PublicInputs: ToElements<Felt> + Clone,
    {
        let air = A::new(info.clone(), pub_inputs.clone(), options.clone());
        let desc = AirDescriptor::new(&air, &kind, &pub_inputs.to_elements());
        self.state.lock().unwrap().air = Some(desc);
    }

    /// `Prover::new_trace_lde` (`src/training/prover.rs:273-281`): K1-K4 on the device.
    pub fn new_trace_lde<E: FieldElement<BaseField = Felt>>(
        &self, info: &TraceInfo, main: &ColMatrix<Felt>, domain: &StarkDomain<Felt>, _po: PartitionOptions,
    ) -> (GpuTraceLde<E>, TracePolyTable<E>) {
        let st = self.state.lock().unwrap();
        let desc = st.air.as_ref().expect("GpuBackend::set_air must be called from get_pub_inputs before proving");
        assert_eq!(desc.width as usize, main.num_cols(), "trace width does not match the AIR given to set_air");
        assert_eq!(desc.len as usize, main.num_rows(), "trace length does not match the AIR given to set_air");
        let ffi_desc = desc.as_ffi();
        st.ctx.check(unsafe { ffi::zkb_begin(st.ctx.raw, &ffi_desc) }, "zkb_begin");
        // TraceTable keeps one Vec<Felt> per column (src/helper.rs:197-211); Felt is repr(transparent) over u128.  The columns
        // are only borrowed for this call, which matches `main: &ColMatrix`.
        let col_ptrs: Vec<*const u8> = (0..main.num_cols()).map(|j| main.get_column(j).as_ptr() as *const u8).collect();
        let mut root = [0u8; 32];
        st.ctx.check(unsafe { ffi::zkb_trace_commit(st.ctx.raw, col_ptrs.as_ptr(), root.as_mut_ptr()) }, "zkb_trace_commit");
        // TracePolyTable: the library keeps the coefficients row-major [n][w]; Winterfell wants one Vec per column
        let (n, w) = (main.num_rows(), main.num_cols());
        let mut raw = vec![0u8; n * w * 16];
        st.ctx.check(unsafe { ffi::zkb_trace_polys_read(st.ctx.raw, raw.as_mut_ptr()) }, "zkb_trace_polys_read");
        let mut columns: Vec<Vec<Felt>> = (0..w).map(|_| Vec::with_capacity(n)).collect();
        for row in raw.chunks_exact(w * 16) {
            for (j, cell) in row.chunks_exact(16).enumerate() {
                columns[j].push(Felt::new(u128::from_le_bytes(cell.try_into().unwrap())));
            }
        }
        let polys = TracePolyTable::new(ColMatrix::new(columns));
        let lde = GpuTraceLde {
            backend: self.clone(),
            root: digest_from(root),
            info: info.clone(),
            blowup: domain.trace_to_lde_blowup(),
            lde_len: domain.lde_domain_size(),
            _e: PhantomData,
        };
        (lde, polys)
    }

    /// `Prover::new_evaluator` (`src/training/prover.rs:283-290`).  Only the single draw of
    /// `ConstraintCompositionCoefficients::draw_algebraic` crosses the boundary: with `BatchingMethod::Algebraic`
    /// (`src/main.rs:105`) the coefficients are alpha^0, alpha^1, ... over the transition constraints and then the assertions
    /// (SURVEY A.5), which is what the device-side evaluator regenerates.
    pub fn new_evaluator<'a, A: Air<BaseField = Felt>, E: FieldElement<BaseField = Felt>>(
        &self, air: &'a A, aux: Option<AuxRandElements<E>>, comp: ConstraintCompositionCoefficients<E>,
    ) -> GpuConstraintEvaluator<'a, A, E> {
        assert!(aux.is_none(), "the reference's AIRs have no auxiliary trace segment");
        let alpha = if comp.transition.len() > 1 { comp.transition[1] } else { comp.boundary[0] };
        // the device regenerates the powers: make sure that is what Winterfell drew (catches Linear batching and any change of
        // the coefficient order upstream)
        let mut p = E::ONE;
        for c in comp.transition.iter().chain(comp.boundary.iter()) {
            assert!(*c == p, "constraint composition coefficients are not consecutive powers of one challenge");
            p *= alpha;
        }
        GpuConstraintEvaluator { air, backend: self.clone(), alpha }
    }

    /// `Prover::build_constraint_commitment` (`src/training/prover.rs:292-300`): the device already holds the evaluations it
    /// produced in `evaluate`; it interpolates, extends, hashes and builds the tree (K6).  `CompositionPoly` — which
    /// Winterfell's `generate_proof` evaluates at the OOD point and feeds into the DEEP polynomial on the host — is built with
    /// Winterfell's own constructor from the same evaluations.
    pub fn build_constraint_commitment<E: FieldElement<BaseField = Felt>>(
        &self, trace: CompositionPolyTrace<E>, num_cols: usize, domain: &StarkDomain<Felt>, _po: PartitionOptions,
    ) -> (GpuConstraintCommitment<E>, CompositionPoly<E>) {
        let mut root = [0u8; 32];
        {
            let st = self.state.lock().unwrap();
            st.ctx.check(unsafe { ffi::zkb_constraints_commit(st.ctx.raw, root.as_mut_ptr()) }, "zkb_constraints_commit");
        }
        let poly = CompositionPoly::new(trace, domain, num_cols);
        (GpuConstraintCommitment { backend: self.clone(), root: digest_from(root), width: num_cols, _e: PhantomData }, poly)
    }

    /// rows + `BatchMerkleProof` of commitment `which` (0 = main trace, 1 = constraint composition) at `positions`
    fn query<E: FieldElement<BaseField = Felt>>(&self, which: u32, width: usize, positions: &[usize]) -> Queries {
        let st = self.state.lock().unwrap();
        let pos: Vec<u32> = positions.iter().map(|&p| p as u32).collect();
        let mut rows = vec![0u8; positions.len() * width * 16];
        let (mut out, mut len) = (ptr::null_mut::<u8>(), 0u64);
        st.ctx.check(
            unsafe { ffi::zkb_query(st.ctx.raw, which, pos.as_ptr(), pos.len() as u32, rows.as_mut_ptr(), &mut out, &mut len) },
            "zkb_query",
        );
        let bytes = unsafe { std::slice::from_raw_parts(out, len as usize) }.to_vec();
        unsafe { ffi::zkb_free(out as *mut _) };
        // the library emits BatchMerkleProof::write_into bytes (depth, then per-index node vectors)
        let opening = BatchMerkleProof::<H>::read_from_bytes(&bytes).expect("zkb_query returned a malformed batch Merkle proof");
        let values: Vec<Vec<E>> = rows.chunks_exact(width * 16).map(|r| bytes_to_felts(r).into_iter().map(E::from).collect()).collect();
        Queries::new::<H, E, VC>(opening, values)
    }
}

/// `Prover::TraceLde` on the GPU: the LDE matrix, its row hashes and the Merkle tree stay in HBM.
pub struct GpuTraceLde<E: FieldElement<BaseField = Felt>> {
    backend: GpuBackend,
    root: Digest,
    info: TraceInfo,
    blowup: usize,
    lde_len: usize,
    _e: PhantomData<E>,
}

impl<E: FieldElement<BaseField = Felt>> TraceLde<E> for GpuTraceLde<E> {
    type HashFn = H;
    type VC = VC;

    fn get_main_trace_commitment(&self) -> Digest {
        self.root
    }

    fn set_aux_trace(&mut self, _aux: &ColMatrix<E>, _domain: &StarkDomain<Felt>) -> (ColMatrix<E>, Digest) {
        unreachable!("the reference's AIRs declare no auxiliary trace segment (TraceInfo::new, src/training/prover.rs:213)")
    }

    /// One host round trip per call (`zkb_trace_read_frame`).  This exists for completeness: it is what Winterfell's
    /// `DefaultConstraintEvaluator` would call `ce_domain_size` times from rayon workers, serialised by the context mutex —
    /// do NOT pair `GpuTraceLde` with the default evaluator.  [`GpuConstraintEvaluator`] never reads frames: it evaluates
    /// on the device.  (A host-side evaluator that insists on frames should fetch them in bulk with
    /// `zkb_trace_read_frames`, thousands of steps per call.)
    fn read_main_trace_frame_into(&self, lde_step: usize, frame: &mut EvaluationFrame<Felt>) {
        let w = self.info.main_trace_width();
        let (mut cur, mut nxt) = (vec![0u8; w * 16], vec![0u8; w * 16]);
        {
            let st = self.backend.state.lock().unwrap();
            st.ctx.check(
                unsafe { ffi::zkb_trace_read_frame(st.ctx.raw, lde_step as u64, cur.as_mut_ptr(), nxt.as_mut_ptr()) },
                "zkb_trace_read_frame",
            );
        }
        frame.current_mut().copy_from_slice(&bytes_to_felts(&cur));
        frame.next_mut().copy_from_slice(&bytes_to_felts(&nxt));
    }

    fn read_aux_trace_frame_into(&self, _lde_step: usize, _frame: &mut EvaluationFrame<E>) {
        unreachable!("no auxiliary trace segment")
    }

    fn read_lagrange_kernel_frame_into(
        &self, _lde_step: usize, _col_idx: usize, _frame: &mut winterfell::LagrangeKernelEvaluationFrame<E>,
    ) {
        unreachable!("no Lagrange kernel column")
    }

    /// `TraceLde::query` → `zkb_query(which = 0)`; one `Queries` per trace segment (only the main one).
    fn query(&self, positions: &[usize]) -> Vec<Queries> {
        vec![self.backend.query::<Felt>(0, self.info.main_trace_width(), positions)]
    }

    fn trace_len(&self) -> usize {
        self.lde_len
    }
    fn blowup(&self) -> usize {
        self.blowup
    }
    fn trace_info(&self) -> &TraceInfo {
        &self.info
    }
}

/// `Prover::ConstraintEvaluator` on the GPU (`k_eval_constraints`): one kernel over the constraint-evaluation domain that
/// evaluates the AIR's transition constraints (`src/training/air.rs:154-287`, `src/aggregation/air.rs:101-119`), the boundary
/// terms, the divisors, and combines them.
pub struct GpuConstraintEvaluator<'a, A: Air<BaseField = Felt>, E: FieldElement<BaseField = Felt>> {
    #[allow(dead_code)]
    air: &'a A,
    backend: GpuBackend,
    alpha: E,
}

impl<'a, A: Air<BaseField = Felt>, E: FieldElement<BaseField = Felt>> ConstraintEvaluator<E> for GpuConstraintEvaluator<'a, A, E> {
    type Air = A;

    /// `trace` is the `GpuTraceLde` created through the same backend: its LDE is already on the device, so it is not read here.
    fn evaluate<T: TraceLde<E>>(self, trace: &T, domain: &StarkDomain<Felt>) -> CompositionPolyTrace<E> {
        assert_eq!(E::EXTENSION_DEGREE, 1, "only FieldExtension::None is supported (src/main.rs:102)");
        assert_eq!(trace.trace_len(), domain.lde_domain_size());
        let n = domain.ce_domain_size();
        let mut raw = vec![0u8; n * 16];
        let alpha_base: Felt = self.alpha.base_element(0);
        let alpha = alpha_base.as_int().to_le_bytes();
        {
            let st = self.backend.state.lock().unwrap();
            st.ctx.check(unsafe { ffi::zkb_constraints_eval(st.ctx.raw, alpha.as_ptr(), raw.as_mut_ptr()) }, "zkb_constraints_eval");
        }
        CompositionPolyTrace::new(bytes_to_felts(&raw).into_iter().map(E::from).collect())
    }
}

/// `Prover::ConstraintCommitment` on the GPU: composition-column LDE, row hashes and Merkle tree stay in HBM.
pub struct GpuConstraintCommitment<E: FieldElement<BaseField = Felt>> {
    backend: GpuBackend,
    root: Digest,
    width: usize,
    _e: PhantomData<E>,
}

impl<E: FieldElement<BaseField = Felt>> ConstraintCommitment<E> for GpuConstraintCommitment<E> {
    type HashFn = H;
    type VC = VC;

    fn commitment(&self) -> Digest {
        self.root
    }
    /// `ConstraintCommitment::query` → `zkb_query(which = 1)`
    fn query(&self, positions: &[usize]) -> Queries {
        self.backend.query::<E>(1, self.width, positions)
    }
}

// The reference's prover then reads (src/training/prover.rs; the aggregation prover is analogous with GpuAir::Aggregation):
//
//     pub struct TrainingUpdateProver { options: ProofOptions, /* ... unchanged ... */ gpu: zkb200_winterfell::GpuBackend }
//     // in new():  gpu: zkb200_winterfell::GpuBackend::new(0),
//
//     impl Prover for TrainingUpdateProver {
//         /* BaseField, Air, Trace, HashFn, VC, RandomCoin unchanged (:222-227) */
//         type TraceLde<E: FieldElement<BaseField = Self::BaseField>> = zkb200_winterfell::GpuTraceLde<E>;
//         type ConstraintEvaluator<'a, E: FieldElement<BaseField = Self::BaseField>> =
//             zkb200_winterfell::GpuConstraintEvaluator<'a, Self::Air, E>;
//         type ConstraintCommitment<E: FieldElement<BaseField = Self::BaseField>> = zkb200_winterfell::GpuConstraintCommitment<E>;
//
//         fn get_pub_inputs(&self, trace: &Self::Trace) -> TrainingUpdateInputs {
//             /* ... unchanged ... */
//             self.gpu.set_air::<TrainingUpdateAir>(trace.info(), &inputs, &self.options, zkb200_winterfell::GpuAir::Training);
//             inputs
//         }
//         fn new_trace_lde<E: ...>(&self, info, main, domain, po) -> (Self::TraceLde<E>, TracePolyTable<E>) {
//             self.gpu.new_trace_lde(info, main, domain, po)
//         }
//         fn new_evaluator<'a, E: ...>(&self, air, aux, comp) -> Self::ConstraintEvaluator<'a, E> {
//             self.gpu.new_evaluator(air, aux, comp)
//         }
//         fn build_constraint_commitment<E: ...>(&self, trace, num_cols, domain, po) -> (Self::ConstraintCommitment<E>, CompositionPoly<E>) {
//             self.gpu.build_constraint_commitment(trace, num_cols, domain, po)
//         }
//     }
//
// src/main.rs, tests/ and benches/ are untouched.

// ---------------------------------------------------------------------------------------------------------------------
// level 2: the whole proof on the device
// ---------------------------------------------------------------------------------------------------------------------

/// Extension trait: `prover.prove_gpu(&ctx, trace)` is a drop-in for `prover.prove(trace)`
/// (src/main.rs:228,424,468) that also runs OOD/DEEP, FRI, grinding and the Fiat-Shamir channel on the GPU.
pub trait GpuProve: Prover<BaseField = Felt, Trace = TraceTable<Felt>>
where
    <Self::Air as Air>::PublicInputs: ToElements<Felt> + Clone,
{
    /// AIR id + parameters for the device-side constraint evaluator.
    fn gpu_air(&self, pub_inputs: &<Self::Air as Air>::PublicInputs) -> GpuAir;

    fn prove_gpu(&self, ctx: &GpuContext, trace: TraceTable<Felt>) -> Result<Proof, ProverError> {
        let pub_inputs = self.get_pub_inputs(&trace);
        let air = Self::Air::new(trace.info().clone(), pub_inputs.clone(), self.options().clone());
        let desc = AirDescriptor::new(&air, &self.gpu_air(&pub_inputs), &pub_inputs.to_elements());
        let ffi_desc = desc.as_ffi();
        let main: &ColMatrix<Felt> = trace.main_segment();
        let col_ptrs: Vec<*const u8> = (0..main.num_cols()).map(|j| main.get_column(j).as_ptr() as *const u8).collect();
        let (mut out, mut len) = (ptr::null_mut::<u8>(), 0u64);
        let mut ts = std::mem::MaybeUninit::<ffi::zkb_transcript>::zeroed();
        let rc = unsafe { ffi::zkb_prove(ctx.raw, &ffi_desc, col_ptrs.as_ptr(), 0, &mut out, &mut len, ts.as_mut_ptr()) };
        ctx.check(rc, "zkb_prove");
        let ts = unsafe { ts.assume_init() };
        if ts.comp_degree_ok == 0 {
            // what Winterfell reports in debug builds when the trace does not satisfy the AIR: the composition polynomial
            // does not fit the declared number of columns (expected degree, actual degree unknown to the host)
            return Err(ProverError::MismatchedConstraintPolynomialDegree(air.context().num_constraint_composition_columns() * trace.length(), usize::MAX));
        }
        let bytes = unsafe { std::slice::from_raw_parts(out, len as usize) }.to_vec();
        unsafe { ffi::zkb_free(out as *mut _) };
        // our own serialiser produced these bytes: a parse failure is a bug in the wire-format restatement (DESIGN.md §6,
        // "not verified against upstream"), not a prover error — say so loudly
        Ok(Proof::from_bytes(&bytes).unwrap_or_else(|e| panic!("libzkb200 returned bytes winterfell::Proof cannot parse: {e}")))
    }
}
