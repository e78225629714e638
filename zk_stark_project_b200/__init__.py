"""zk_stark_project_b200 — B200-native STARK proving backend for FireMines/zk_stark_project.

Host-side mirror (Python, because no Rust toolchain exists in the build image) of the reference's
Winterfell `Prover` surface — `TrainingUpdateProver`, `GlobalUpdateProver` and the newly defined
`MimcProver` — on top of the C ABI of include/zkb200.h (libzkb200.so, hand-written sm_100a kernels).
There is no CPU path: importing works anywhere, proving needs the built library and a CUDA device.
"""
from .field import P, Felt, f64_to_felt
from .options import ProofOptions, FieldExtension, BatchingMethod
from .trace import TraceTable, DeviceTrace
from .prover import Proof, Prover, ProverError
from .verifier import verify, verify_batch, VerifierError
from .training import TrainingUpdateProver, TrainingUpdateInputs, TrainingUpdateAir
from .aggregation import GlobalUpdateProver, GlobalUpdateInputs, GlobalUpdateAir
from .mimc import MimcProver, MimcInputs, MimcAir, mimc_cipher, mimc_hash_matrix, get_round_constants

__all__ = [
    "P", "Felt", "f64_to_felt", "ProofOptions", "FieldExtension", "BatchingMethod", "TraceTable", "DeviceTrace", "Proof", "Prover",
    "ProverError", "verify", "verify_batch", "VerifierError", "TrainingUpdateProver", "TrainingUpdateInputs", "TrainingUpdateAir", "GlobalUpdateProver",
    "GlobalUpdateInputs", "GlobalUpdateAir", "MimcProver", "MimcInputs", "MimcAir", "mimc_cipher", "mimc_hash_matrix",
    "get_round_constants",
]
