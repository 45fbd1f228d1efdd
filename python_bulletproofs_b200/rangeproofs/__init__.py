from .rangeproof_prover import NIRangeProver
from .rangeproof_verifier import RangeVerifier
from .rangeproof_aggreg_prover import AggregNIRangeProver
from .rangeproof_aggreg_verifier import AggregRangeVerifier
from .batch import (verify_range_proofs_batch, verify_aggreg_range_proofs_batch, verify_mixed_range_proofs_batch,
                    prove_range_proofs_packed, prove_range_proofs_batch)

__all__ = [
    "NIRangeProver",
    "RangeVerifier",
    "AggregNIRangeProver",
    "AggregRangeVerifier",
    "verify_range_proofs_batch",
    "verify_aggreg_range_proofs_batch",
    "verify_mixed_range_proofs_batch",
    "prove_range_proofs_packed",
    "prove_range_proofs_batch",
]
