"""B200-native batched Groth16/BN254 verifier for the RISC Zero v2.1 and SP1 v5 proof formats: a drop-in
for the verification path of gnosisguild/stylus-zkvm-verifiers (see DESIGN.md).  The compute path is
hand-written sm_100a CUDA behind the C ABI of include/zkv.h; this package is the thin host mirror."""
from . import errors, synth  # noqa: F401
from ._native import (ZKV_INVALID_INITIALIZATION, ZKV_INVALID_PROOF_DATA, ZKV_OK, ZKV_SELECTOR_MISMATCH,  # noqa: F401
                      ZKV_VERIFICATION_FAILED, ZKV_VM_RISC0, ZKV_VM_SP1, ZkvError)
from .verifier import (GpuBackend, Groth16Verifier, RawKeyVerifier, RiscZeroVerifier, RiscZeroVerifierRouter, Sp1Verifier, Sp1VerifierGateway, VerificationKey, VerificationKeySet, device_count, ec_add_batch,  # noqa: F401
                       ec_mul_batch, ec_pairing, ec_pairing_batch, fp12_op_batch, fp_mul_batch, g2_check_batch, g2_mul_batch, imad_peak, launch_count, pairing4_batch, pinned_copy, raw_key_bytes, vk_x_batch, wave_proofs)
