"""jubjub_schnorr_b200: B200-native (sm_100a) batch verifier for dusk-network/jubjub-schnorr signatures.

Only the verify path of the reference lives here (SURVEY.md section 8): the CUDA library behind the C ABI
of include/jjschnorr_b200.h and a host-side mirror of the reference's key / signature types.
"""
from .batch import (DOUBLE, SINGLE, STATUS_BYTES_ERROR, STATUS_INVALID_POINT, STATUS_INVALID_SIGNATURE, STATUS_OK,  # noqa: F401
                    VARGEN, BatchVerifier, JjsError, KeySet)
