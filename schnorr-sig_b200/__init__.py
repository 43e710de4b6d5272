"""schnorr-sig_b200 -- B200-native Schnorr verification engine (Cheetah curve, Rescue hash).

Drop-in for the verification hot path of toposware/schnorr-sig: `Signature::verify`,
`verify_batch`, `hash_message` (+ the device signer / key generation used to synthesise inputs).
Everything below the API is hand-written sm_100a CUDA behind the C ABI of include/schnorr_b200.h;
there is no CPU fallback.
"""
from .api import (KEYED_SIGNATURE_LENGTH, PUBLIC_KEY_LENGTH, SCALAR_LENGTH, SIGNATURE_LENGTH, KeyedSignature,
                  KeyPair, KeySet, OsRng, PanicError, PrivateKey, PublicKey, Result, Signature, SignatureError,
                  verify_batch, verify_prepared_batch, locate_invalid, verify_batch_keyed, locate_invalid_keyed,
                  ChainCode, ExtendedPrivateKey, ExtendedPublicKey)
from .engine import Engine, EngineError, default_engine, OK, INVALID_PUBLIC_KEY, INVALID_SIGNATURE, MALFORMED
from . import synth, distributed  # noqa: F401
from .distributed import ShardedVerifier, shard_bounds

__all__ = ["Engine", "EngineError", "default_engine", "KeyPair", "KeySet", "PrivateKey", "PublicKey", "Signature",
           "KeyedSignature", "SignatureError", "PanicError", "Result", "OsRng", "verify_batch",
           "verify_prepared_batch", "locate_invalid", "verify_batch_keyed", "locate_invalid_keyed",
           "ChainCode", "ExtendedPrivateKey", "ExtendedPublicKey", "synth", "distributed", "ShardedVerifier", "shard_bounds"]
