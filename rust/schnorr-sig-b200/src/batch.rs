//! Replacement body of `verify_batch` (src/batch.rs:31-50) and the failed-batch localisation the reference lacks.

use cheetah::Scalar;
use rand_core::{CryptoRng, RngCore};
use schnorr_sig::{PublicKey, Signature, SignatureError};

use crate::{public_key_record, ENGINE};

fn records(signatures: &[Signature], public_keys: &[PublicKey]) -> (Vec<[u8; 81]>, Vec<[u8; 96]>, Vec<u8>) {
    let sigs = signatures.iter().map(|s| s.to_bytes()).collect();
    let (pks, infs) = public_keys.iter().map(public_key_record).unzip();
    (sigs, pks, infs)
}

/// One full-width random scalar per signature, drawn exactly where the reference draws it (src/batch.rs:75-78).
fn randomizers(n: usize, mut rng: impl CryptoRng + RngCore) -> Vec<[u8; 32]> {
    (0..n).map(|_| Scalar::random(&mut rng).to_bytes()).collect()
}

/// `verify_batch(signatures, public_keys, messages, rng)`: same asserts, same RNG consumption, same `Result`.
pub fn verify_batch(signatures: &[Signature], public_keys: &[PublicKey], messages: &[&[u8]],
                    rng: impl CryptoRng + RngCore) -> Result<(), SignatureError> {
    assert!(signatures.len() == public_keys.len(), "We should have the same number of signatures than public keys");
    assert!(messages.len() == public_keys.len(), "We should have the same number of messages than public keys");
    let (sigs, pks, infs) = records(signatures, public_keys);
    let rand = randomizers(sigs.len(), rng);
    match ENGINE.with(|e| e.verify_batch(&sigs, &pks, &infs, messages, &rand)) {
        0 => Ok(()),
        2 => Err(SignatureError::InvalidSignature),
        // src/batch.rs:67,104 unwrap a `CtOption` that is `None` for these inputs
        _ => panic!("called `Option::unwrap()` on a `None` value"),
    }
}

/// Indices of the signatures that make a batch fail, in batch semantics (flag byte of `sig.x` honoured, no subgroup
/// check on the keys -- src/batch.rs:102-106).  Empty for a batch that verifies.
pub fn locate_invalid(signatures: &[Signature], public_keys: &[PublicKey], messages: &[&[u8]],
                      rng: impl CryptoRng + RngCore) -> Vec<usize> {
    let (sigs, pks, infs) = records(signatures, public_keys);
    let rand = randomizers(sigs.len(), rng);
    let flags = ENGINE.with(|e| e.locate_invalid(&sigs, &pks, &infs, messages, &rand));
    assert!(flags.iter().all(|&f| f != 3), "called `Option::unwrap()` on a `None` value");
    flags.iter().enumerate().filter(|(_, &f)| f != 0).map(|(i, _)| i).collect()
}

/// `verify_batch` with the randomisers generated on the device from a 32-byte seed instead of drawn from an RNG on the
/// host (`Scalar::random` per signature, src/batch.rs:75-78): the host sends 32 bytes instead of 32 per signature.  The
/// seed must come fresh from a CSPRNG for every batch and stay unknown to the signers until the verdict; a signer who
/// knows it in advance can build a batch whose invalid terms cancel.
pub fn verify_batch_seeded(signatures: &[Signature], public_keys: &[PublicKey], messages: &[&[u8]],
                           seed: &[u8; 32]) -> Result<(), SignatureError> {
    assert!(signatures.len() == public_keys.len(), "We should have the same number of signatures than public keys");
    assert!(messages.len() == public_keys.len(), "We should have the same number of messages than public keys");
    let (sigs, pks, infs) = records(signatures, public_keys);
    match ENGINE.with(|e| e.verify_batch_seeded(&sigs, &pks, &infs, messages, seed)) {
        0 => Ok(()),
        2 => Err(SignatureError::InvalidSignature),
        _ => panic!("called `Option::unwrap()` on a `None` value"),
    }
}

/// `locate_invalid` with the randomisers of `verify_batch_seeded(.., seed)`, generated on the devices: the culprits of
/// that failed batch.
pub fn locate_invalid_seeded(signatures: &[Signature], public_keys: &[PublicKey], messages: &[&[u8]],
                             seed: &[u8; 32]) -> Vec<usize> {
    let (sigs, pks, infs) = records(signatures, public_keys);
    let flags = ENGINE.with(|e| e.locate_invalid_seeded(&sigs, &pks, &infs, messages, seed));
    assert!(flags.iter().all(|&f| f != 3), "called `Option::unwrap()` on a `None` value");
    flags.iter().enumerate().filter(|(_, &f)| f != 0).map(|(i, _)| i).collect()
}
