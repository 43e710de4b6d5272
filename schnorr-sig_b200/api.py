"""Host-side mirror of the reference's public API for the verification path (src/lib.rs:182-195):
same type names, method names, argument meaning and error behaviour, so that parity tests read
like the reference's own tests.  All arithmetic runs in the CUDA engine; nothing here computes on
field or curve elements.

  Signature::verify / to_bytes / from_bytes            src/signature.rs:181-227
  KeyedSignature::verify / to_bytes / from_bytes       src/signature.rs:230-271
  PublicKey::from(&PrivateKey) / verify_signature / to_bytes / from_bytes   src/public.rs:26-56, src/signature.rs:170-176
  PrivateKey::new / sign / to_bytes / from_bytes       src/private.rs:49-82, src/signature.rs:65-80
  KeyPair::new / sign / verify_signature               src/keypair.rs:57-65, src/signature.rs:114-165
  verify_batch                                         src/batch.rs:31-50
  verify_batch_keyed / locate_invalid_keyed            src/signature.rs:237-271, src/batch.rs:31-130
  SignatureError                                       src/error.rs:13-31
"""
import os

import numpy as np

from .engine import default_engine, OK, INVALID_PUBLIC_KEY, INVALID_SIGNATURE, MALFORMED

SCALAR_LENGTH = 32            # src/constants.rs:12
BASEFIELD_LENGTH = 48         # src/constants.rs:18
PUBLIC_KEY_LENGTH = 49        # src/constants.rs:24
SIGNATURE_LENGTH = 81         # src/constants.rs:30
KEYED_SIGNATURE_LENGTH = 130  # src/constants.rs:33

_Q = 0x7AF2599B3B3F22D0563FBF0F990A37B5327AA72330157722D443623EAED4ACCF   # include/cheetah_params.h


class SignatureError(Exception):
    """src/error.rs:13-31"""
    InvalidPublicKey = "InvalidPublicKey"
    InvalidSignature = "InvalidSignature"
    _DISPLAY = {
        "InvalidPublicKey": "The public key is not an element of the prime subgroup.",
        "InvalidSignature": "The signature is invalid or was incorrectly computed.",
    }

    def __init__(self, kind):
        super().__init__(self._DISPLAY[kind])
        self.kind = kind

    def __repr__(self):
        return self.kind

    def __eq__(self, other):
        return isinstance(other, SignatureError) and other.kind == self.kind

    def __hash__(self):
        return hash(self.kind)


class PanicError(Exception):
    """Inputs on which the reference panics (unwrap on a non-canonical encoding, src/signature.rs:186,
    src/batch.rs:67,104)."""


class Result:
    """Result<(), SignatureError>"""

    def __init__(self, err=None):
        self._err = err

    def is_ok(self):
        return self._err is None

    def is_err(self):
        return self._err is not None

    def unwrap(self):
        if self._err is not None:
            raise self._err
        return None

    def unwrap_err(self):
        if self._err is None:
            raise PanicError("called unwrap_err on Ok")
        return self._err

    def __repr__(self):
        return "Ok(())" if self._err is None else "Err(%r)" % self._err

    def __bool__(self):
        return self.is_ok()


def _result_from_verdict(v):
    if v == OK:
        return Result()
    if v == INVALID_PUBLIC_KEY:
        return Result(SignatureError(SignatureError.InvalidPublicKey))
    if v == INVALID_SIGNATURE:
        return Result(SignatureError(SignatureError.InvalidSignature))
    if v == MALFORMED:
        raise PanicError("called `Option::unwrap()` on a `None` value (non-canonical encoding)")
    raise RuntimeError("engine returned an unknown verdict %r" % v)


class OsRng:
    def fill_bytes(self, n):
        return os.urandom(n)


def _random_scalar(rng) -> int:
    """Scalar::random: a uniformly distributed element of Z_q (wide reduction of 64 random bytes)."""
    return int.from_bytes(rng.fill_bytes(64), "little") % _Q


def _pack(msgs):
    off = np.zeros(len(msgs) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(m) for m in msgs])
    blob = np.frombuffer(b"".join(bytes(m) for m in msgs), dtype=np.uint8)
    return (blob.copy() if blob.size else np.zeros(0, dtype=np.uint8)), off


class PublicKey:
    """PublicKey(AffinePoint): affine x||y (96 bytes) + identity flag (src/public.rs:24)."""

    def __init__(self, xy96: bytes, infinity: bool = False):
        xy96 = bytes(xy96)
        assert len(xy96) == 96
        self.xy = bytes(96) if infinity else xy96
        self.infinity = bool(infinity)

    @classmethod
    def from_private(cls, sk: "PrivateKey"):
        pk, inf = default_engine().keygen(np.frombuffer(sk.to_bytes(), dtype=np.uint8).reshape(1, 32))
        return cls(bytes(pk[0]), bool(inf[0]))

    @classmethod
    def from_raw_coordinates(cls, x_limbs, y_limbs):
        """AffinePoint::from_raw_coordinates with Fp6::from_raw_unchecked limbs (src/signature.rs:386-405)."""
        return cls(b"".join(int(c).to_bytes(8, "little") for c in list(x_limbs) + list(y_limbs)))

    def to_bytes(self) -> bytes:
        return bytes(default_engine().compress(np.frombuffer(self.xy, dtype=np.uint8).reshape(1, 96),
                                               np.array([self.infinity], dtype=np.uint8))[0])

    @classmethod
    def from_bytes(cls, b: bytes):
        """CtOption<Self>: None when the encoding does not decode (src/public.rs:54-56)."""
        b = bytes(b)
        assert len(b) == PUBLIC_KEY_LENGTH
        pk, inf, ok = default_engine().decompress(np.frombuffer(b, dtype=np.uint8).reshape(1, 49))
        return cls(bytes(pk[0]), bool(inf[0])) if ok[0] else None

    def verify_signature(self, signature: "Signature", message: bytes) -> Result:
        return signature.verify(message, self)

    def __eq__(self, other):
        return isinstance(other, PublicKey) and (self.xy, self.infinity) == (other.xy, other.infinity)

    def __hash__(self):
        return hash((self.xy, self.infinity))


class Signature:
    """Signature { x: CompressedPoint, e: Scalar } (src/signature.rs:34-40)."""

    def __init__(self, x49: bytes, e: bytes):
        self.x = bytes(x49)
        self.e = e.to_bytes(32, "little") if isinstance(e, int) else bytes(e)
        assert len(self.x) == 49 and len(self.e) == 32

    def to_bytes(self) -> bytes:
        return self.x + self.e

    @classmethod
    def from_bytes(cls, b: bytes):
        """CtOption<Self>: None when the scalar is not canonical (src/signature.rs:217-227)."""
        b = bytes(b)
        assert len(b) == SIGNATURE_LENGTH
        if int.from_bytes(b[49:], "little") >= _Q:
            return None
        return cls(b[:49], b[49:])

    def verify(self, message: bytes, pkey: PublicKey) -> Result:
        sig = np.frombuffer(self.to_bytes(), dtype=np.uint8).reshape(1, 81)
        pk = np.frombuffer(pkey.xy, dtype=np.uint8).reshape(1, 96)
        blob, off = _pack([message])
        v = default_engine().verify_many(sig, pk, np.array([pkey.infinity], dtype=np.uint8), blob, off)
        return _result_from_verdict(int(v[0]))

    def __eq__(self, other):
        return isinstance(other, Signature) and (self.x, self.e) == (other.x, other.e)


class KeySet:
    """Public keys registered once for many verifications (no reference counterpart: the reference verifies each
    signature from scratch).  Registration runs the subgroup check of every key and builds its table on the GPU;
    verify_signature then gives what Signature.verify gives for that key without repeating that per-key work.
    `status[i]`: 0 = key i is in the prime-order subgroup (identity included), 1 = it is not, 3 = non-canonical limb."""

    def __init__(self, public_keys):
        keys = list(public_keys)
        pks = np.frombuffer(b"".join(k.xy for k in keys), dtype=np.uint8).reshape(len(keys), 96)
        inf = np.array([k.infinity for k in keys], dtype=np.uint8)
        self._handle, self.status = default_engine().register_keys(pks, inf)

    def __len__(self):
        return self._handle.n_keys

    @staticmethod
    def _pack_keys(public_keys):
        keys = list(public_keys)
        pks = np.frombuffer(b"".join(k.xy for k in keys), dtype=np.uint8).reshape(len(keys), 96)
        inf = np.array([k.infinity for k in keys], dtype=np.uint8)
        return pks, inf

    def _indices(self, indices):
        idx = [int(i) for i in indices]
        for i in idx:
            if not 0 <= i < len(self):
                raise PanicError("index out of bounds: the len is %d but the index is %d" % (len(self), i))
        return np.array(idx, dtype=np.uint32)

    def append(self, public_keys) -> range:
        """Registers keys in the next slots; returns their indices.  `status` grows with them."""
        pks, inf = self._pack_keys(public_keys)
        first = len(self)
        st = default_engine().keyset_append(self._handle, pks, inf)
        self.status = np.concatenate([self.status, st])
        return range(first, len(self))

    def replace(self, indices, public_keys):
        """Registers public_keys[j] in slot indices[j] (distinct indices inside the set); the slots keep their index."""
        idx = self._indices(indices)
        pks, inf = self._pack_keys(public_keys)
        assert len(idx) == len(pks), "one index per key"
        st = default_engine().keyset_replace(self._handle, idx, pks, inf)
        self.status = self.status.copy()
        self.status[idx] = st

    def remove(self, indices):
        """Removes slots: they keep their index, which then panics as an index outside the set does (status 3)."""
        idx = self._indices(indices)
        default_engine().keyset_remove(self._handle, idx)
        self.status = self.status.copy()
        self.status[idx] = 3

    def verify_signature(self, index: int, signature: Signature, message: bytes) -> Result:
        """Signature::verify(message, &keys[index]); an index outside the set panics, as indexing a slice does."""
        index = int(index)
        idx = np.array([index if 0 <= index < 2**32 else 2**32 - 1], dtype=np.uint32)
        sig = np.frombuffer(signature.to_bytes(), dtype=np.uint8).reshape(1, 81)
        blob, off = _pack([message])
        v = default_engine().verify_registered_many(self._handle, sig, idx, blob, off)
        return _result_from_verdict(int(v[0]))

    def index_of(self, public_key):
        """Index of `public_key` (a PublicKey or its 49-byte encoding) in the set: the smallest index of a key whose
        encoding is exactly those bytes and which decompresses to its registered record; None when there is none."""
        b = public_key.to_bytes() if isinstance(public_key, PublicKey) else bytes(public_key)
        assert len(b) == PUBLIC_KEY_LENGTH
        k = int(default_engine().keyset_lookup(self._handle, np.frombuffer(b, dtype=np.uint8).reshape(1, 49))[0])
        return None if k == 0xFFFFFFFF else k

    def verify_keyed(self, keyed, message: bytes) -> Result:
        """KeyedSignature::verify(message) for a KeyedSignature or its 130 bytes: the registered path when the key is in
        the set, what KeyedSignature.verify gives otherwise; a record whose key or scalar does not decode panics."""
        b = keyed.to_bytes() if isinstance(keyed, KeyedSignature) else bytes(keyed)
        assert len(b) == KEYED_SIGNATURE_LENGTH
        blob, off = _pack([message])
        v = default_engine().verify_keyed_registered_many(self._handle, np.frombuffer(b, dtype=np.uint8).reshape(1, 130),
                                                           blob, off)
        return _result_from_verdict(int(v[0]))

    def _batch_inputs(self, indices, signatures, messages, rng):
        n = len(signatures)
        assert len(indices) == n, "We should have the same number of signatures than public keys"
        assert len(messages) == n, "We should have the same number of messages than public keys"
        idx = np.array([int(i) if 0 <= int(i) < 2**32 else 2**32 - 1 for i in indices], dtype=np.uint32)
        sigs = np.frombuffer(b"".join(s.to_bytes() for s in signatures), dtype=np.uint8).reshape(n, 81)
        blob, off = _pack(messages)
        rng = rng or OsRng()
        rand = np.zeros((n, 32), dtype=np.uint8)
        for i in range(n):
            rand[i] = np.frombuffer(_random_scalar(rng).to_bytes(32, "little"), dtype=np.uint8)
        return sigs, idx, blob, off, rand

    def verify_batch(self, indices, signatures, messages, rng=None) -> Result:
        """verify_batch(signatures, [keys[i] for i in indices], messages, rng) (src/batch.rs:31-130) with the key side of
        the batch equation summed per key of the set; an index outside the set gives the malformed-batch error."""
        sigs, idx, blob, off, rand = self._batch_inputs(indices, signatures, messages, rng)
        v, _lhs, _rhs = default_engine().verify_batch_registered(self._handle, sigs, idx, blob, off, rand)
        return _result_from_verdict(v)

    def locate_invalid(self, indices, signatures, messages, rng=None):
        """locate_invalid(signatures, [keys[i] for i in indices], messages, rng): [(index, SignatureError), ...] in batch
        semantics; a malformed item or an index outside the set panics."""
        if len(signatures) == 0:
            assert len(indices) == 0 and len(messages) == 0
            return []
        sigs, idx, blob, off, rand = self._batch_inputs(indices, signatures, messages, rng)
        flags = default_engine().locate_invalid_registered(self._handle, sigs, idx, blob, off, rand)
        out = []
        for i in np.nonzero(flags)[0]:
            if flags[i] == MALFORMED:
                raise PanicError("item %d has a key index outside the set or a non-canonical or undecodable encoding" % i)
            out.append((int(i), SignatureError(SignatureError.InvalidSignature)))
        return out

    def verify_batch_keyed(self, keyed_signatures, messages, rng=None) -> Result:
        """verify_batch_keyed (below) with the records whose key is in the set taking its registered record and the
        key side summed per key: the same result."""
        recs, blob, off, rand = _keyed_batch_inputs(keyed_signatures, messages, rng)
        v, _lhs, _rhs = default_engine().verify_batch_keyed_registered(self._handle, recs, blob, off, rand)
        return _result_from_verdict(v)

    def locate_invalid_keyed(self, keyed_signatures, messages, rng=None):
        """locate_invalid_keyed (below) with the records whose key is in the set taking its registered record."""
        if len(keyed_signatures) == 0:
            assert len(messages) == 0
            return []
        recs, blob, off, rand = _keyed_batch_inputs(keyed_signatures, messages, rng)
        return _keyed_located(default_engine().locate_invalid_keyed_registered(self._handle, recs, blob, off, rand))


class KeyedSignature:
    def __init__(self, public_key: PublicKey, signature: Signature):
        self.public_key = public_key
        self.signature = signature

    def verify(self, message: bytes) -> Result:
        return self.signature.verify(message, self.public_key)

    def to_bytes(self) -> bytes:
        return self.public_key.to_bytes() + self.signature.to_bytes()

    @classmethod
    def from_bytes(cls, b: bytes):
        b = bytes(b)
        assert len(b) == KEYED_SIGNATURE_LENGTH
        pk = PublicKey.from_bytes(b[:49])
        sig = Signature.from_bytes(b[49:])
        return None if pk is None or sig is None else cls(pk, sig)


class PrivateKey:
    """PrivateKey(Scalar) (src/private.rs:25); the secret scalar never leaves the host except as the
    32-byte input of the device signer."""

    def __init__(self, scalar: int):
        self._k = int(scalar) % _Q

    @classmethod
    def new(cls, rng=None):
        rng = rng or OsRng()
        while True:
            k = _random_scalar(rng)
            if k:
                return cls(k)

    @classmethod
    def from_bytes(cls, b: bytes):
        k = int.from_bytes(bytes(b), "little")
        return None if (k >= _Q or k == 0) else cls(k)

    def to_bytes(self) -> bytes:
        return self._k.to_bytes(32, "little")

    def sign(self, message: bytes, rng=None) -> Signature:
        return KeyPair(self, PublicKey.from_private(self)).sign(message, rng)

    def sign_and_bind_pkey(self, message: bytes, rng=None) -> KeyedSignature:
        return KeyPair(self, PublicKey.from_private(self)).sign_and_bind_pkey(message, rng)


class KeyPair:
    def __init__(self, private_key: PrivateKey, public_key: PublicKey):
        self.private_key = private_key
        self.public_key = public_key

    @classmethod
    def new(cls, rng=None):
        sk = PrivateKey.new(rng)
        return cls(sk, PublicKey.from_private(sk))

    def sign(self, message: bytes, rng=None) -> Signature:
        rng = rng or OsRng()
        r = _random_scalar(rng)
        blob, off = _pack([message])
        out = default_engine().sign_many(
            np.frombuffer(self.private_key.to_bytes(), dtype=np.uint8).reshape(1, 32),
            np.frombuffer(self.public_key.xy, dtype=np.uint8).reshape(1, 96),
            np.array([self.public_key.infinity], dtype=np.uint8), blob, off,
            np.frombuffer(r.to_bytes(32, "little"), dtype=np.uint8).reshape(1, 32))
        b = bytes(out[0])
        return Signature(b[:49], b[49:])

    def sign_and_bind_pkey(self, message: bytes, rng=None) -> KeyedSignature:
        return KeyedSignature(self.public_key, self.sign(message, rng))

    def verify_signature(self, signature: Signature, message: bytes) -> Result:
        return signature.verify(message, self.public_key)


# ---- hierarchical deterministic derivation (src/derivation.rs) -----------------------------------------------------
CHAIN_CODE_LENGTH = 32
EXTENDED_PRIVATE_KEY_LENGTH = 64
EXTENDED_PUBLIC_KEY_LENGTH = 81


class ChainCode:
    """BIP32-like chain code (src/derivation.rs:30-32)."""

    def __init__(self, b: bytes):
        b = bytes(b)
        assert len(b) == CHAIN_CODE_LENGTH
        self.bytes = b

    def __eq__(self, other):
        return isinstance(other, ChainCode) and self.bytes == other.bytes

    def __hash__(self):
        return hash(self.bytes)


def _index_u32(i) -> int:
    """The reference takes the index as `&[u8; 4]`, little-endian (src/derivation.rs:86-90); ints are accepted too."""
    return int.from_bytes(bytes(i), "little") if isinstance(i, (bytes, bytearray, list, tuple)) else int(i)


class ExtendedPrivateKey:
    """A derivable private key and its chain code (src/derivation.rs:46-53).  Methods return None where the reference
    returns a `CtOption` that is none."""

    def __init__(self, key: PrivateKey, chaincode: ChainCode):
        self.key, self.chaincode = key, chaincode

    @classmethod
    def generate_master_key(cls, seed: bytes):
        seed = bytes(seed)
        assert len(seed) == 32
        out, ok = default_engine().derive_master_keys(np.frombuffer(seed, dtype=np.uint8).reshape(1, 32))
        return cls._from_record(out[0]) if ok[0] else None

    @classmethod
    def _from_record(cls, rec):
        rec = bytes(rec)
        return cls(PrivateKey(int.from_bytes(rec[:32], "little")), ChainCode(rec[32:]))

    def to_bytes(self) -> bytes:
        return self.key.to_bytes() + self.chaincode.bytes

    @classmethod
    def from_bytes(cls, b: bytes):
        b = bytes(b)
        assert len(b) == EXTENDED_PRIVATE_KEY_LENGTH
        key = PrivateKey.from_bytes(b[:32])
        return None if key is None else cls(key, ChainCode(b[32:]))

    def derive_private_many(self, indices):
        """Children for many indices in one device call -> list of ExtendedPrivateKey / None."""
        idx = np.array([_index_u32(i) for i in indices], dtype=np.uint32)
        out, ok = default_engine().derive_private_children(self.to_bytes(), idx)
        return [self._from_record(out[k]) if ok[k] else None for k in range(len(idx))]

    def derive_private(self, i):
        return self.derive_private_many([i])[0]

    def derive_hardened_private(self, i):
        return self.derive_private(i) if _index_u32(i) >> 31 else None          # src/derivation.rs:121-123

    def derive_normal_private(self, i):
        return None if _index_u32(i) >> 31 else self.derive_private(i)          # src/derivation.rs:149-151

    def derive_public(self, i):
        child = self.derive_private(i)
        return None if child is None else ExtendedPublicKey.from_extended_private_key(child)

    def __eq__(self, other):
        return isinstance(other, ExtendedPrivateKey) and self.to_bytes() == other.to_bytes()


class ExtendedPublicKey:
    """A derivable public key and its chain code (src/derivation.rs:204-211)."""

    def __init__(self, key: PublicKey, chaincode: ChainCode):
        self.key, self.chaincode = key, chaincode

    @classmethod
    def from_extended_private_key(cls, xsk: ExtendedPrivateKey):
        return cls(PublicKey.from_private(xsk.key), xsk.chaincode)

    def to_bytes(self) -> bytes:
        return self.key.to_bytes() + self.chaincode.bytes

    @classmethod
    def from_bytes(cls, b: bytes):
        b = bytes(b)
        assert len(b) == EXTENDED_PUBLIC_KEY_LENGTH
        key = PublicKey.from_bytes(b[:49])
        return None if key is None or key.infinity else cls(key, ChainCode(b[49:]))

    def derive_normal_public_many(self, indices):
        """Non-hardened public children for many indices in one device call (HMAC-SHA512 + one fixed-base
        multiplication per child on the GPU) -> list of ExtendedPublicKey / None."""
        idx = np.array([_index_u32(i) for i in indices], dtype=np.uint32)
        out, ok = default_engine().derive_public_children(self.to_bytes(), idx)
        res = []
        for k in range(len(idx)):
            key = PublicKey.from_bytes(bytes(out[k, :49])) if ok[k] else None
            res.append(None if key is None else ExtendedPublicKey(key, ChainCode(bytes(out[k, 49:]))))
        return res

    def derive_normal_public(self, i):
        return self.derive_normal_public_many([i])[0]

    def __eq__(self, other):
        return isinstance(other, ExtendedPublicKey) and (self.key, self.chaincode) == (other.key, other.chaincode)


def verify_batch(signatures, public_keys, messages, rng=None) -> Result:
    """src/batch.rs:31-50: asserts equal lengths, draws one full-width random scalar per signature,
    checks  sum s_i R_i - sum s_i h_i P_i == (sum s_i e_i) G  on the GPU."""
    assert len(signatures) == len(public_keys), "We should have the same number of signatures than public keys"
    assert len(messages) == len(public_keys), "We should have the same number of messages than public keys"
    rng = rng or OsRng()
    n = len(signatures)
    rand = np.zeros((n, 32), dtype=np.uint8)
    for i in range(n):
        rand[i] = np.frombuffer(_random_scalar(rng).to_bytes(32, "little"), dtype=np.uint8)
    return verify_prepared_batch(rand, signatures, public_keys, messages)


def locate_invalid(signatures, public_keys, messages, rng=None):
    """Failed-batch localisation (SURVEY.md 8 f3).  The reference returns one Err for the whole batch
    (src/batch.rs:125-129); this returns [(index, SignatureError), ...] for every item whose own term of the batch
    equation fails -- BATCH semantics (src/batch.rs:102-106): the signature's point is decompressed with its flag byte,
    public keys are not subgroup-checked.  A signature with a flipped y-sign flag is therefore reported here (it makes
    verify_batch fail) although Signature::verify accepts it.  Runs on the device: bisection over partial MSMs, then an
    exact per-item check of the failing slices (schnorr_b200_locate_invalid).  Malformed encodings panic as in
    verify_batch."""
    n = len(signatures)
    assert len(public_keys) == n and len(messages) == n
    if n == 0:
        return []
    rng = rng or OsRng()
    sigs = np.frombuffer(b"".join(s.to_bytes() for s in signatures), dtype=np.uint8).reshape(n, 81)
    pks = np.frombuffer(b"".join(k.xy for k in public_keys), dtype=np.uint8).reshape(n, 96)
    inf = np.array([k.infinity for k in public_keys], dtype=np.uint8)
    blob, off = _pack(messages)
    rand = np.zeros((n, 32), dtype=np.uint8)
    for i in range(n):
        rand[i] = np.frombuffer(_random_scalar(rng).to_bytes(32, "little"), dtype=np.uint8)
    flags = default_engine().locate_invalid(sigs, pks, inf, blob, off, rand)
    out = []
    for i in np.nonzero(flags)[0]:
        if flags[i] == MALFORMED:
            raise PanicError("signature %d has a non-canonical or undecodable encoding" % i)
        out.append((int(i), SignatureError(SignatureError.InvalidSignature)))
    return out


def _keyed_batch_inputs(keyed_signatures, messages, rng):
    n = len(keyed_signatures)
    assert len(messages) == n, "We should have the same number of messages than signatures"
    recs = [k.to_bytes() if isinstance(k, KeyedSignature) else bytes(k) for k in keyed_signatures]
    assert all(len(b) == KEYED_SIGNATURE_LENGTH for b in recs)
    recs = np.frombuffer(b"".join(recs), dtype=np.uint8).reshape(n, KEYED_SIGNATURE_LENGTH)
    blob, off = _pack(messages)
    rng = rng or OsRng()
    rand = np.zeros((n, 32), dtype=np.uint8)
    for i in range(n):
        rand[i] = np.frombuffer(_random_scalar(rng).to_bytes(32, "little"), dtype=np.uint8)
    return recs, blob, off, rand


def _keyed_located(flags):
    out = []
    for i in np.nonzero(flags)[0]:
        if flags[i] == MALFORMED:
            raise PanicError("record %d has an undecodable key or a non-canonical or undecodable signature" % i)
        out.append((int(i), SignatureError(SignatureError.InvalidSignature)))
    return out


def verify_batch_keyed(keyed_signatures, messages, rng=None) -> Result:
    """verify_batch over KeyedSignature objects or their 130-byte records (src/signature.rs:237-271,
    src/batch.rs:31-130): verify_batch([k.signature ...], [k.public_key ...], messages, rng) with the keys decoded on
    the device.  A record whose key does not decode panics, as unwrapping KeyedSignature::from_bytes does."""
    recs, blob, off, rand = _keyed_batch_inputs(keyed_signatures, messages, rng)
    v, _lhs, _rhs = default_engine().verify_batch_keyed(recs, blob, off, rand)
    return _result_from_verdict(v)


def locate_invalid_keyed(keyed_signatures, messages, rng=None):
    """locate_invalid over KeyedSignature objects or their 130-byte records: [(index, SignatureError), ...] in batch
    semantics; a record whose key or signature does not decode panics."""
    if len(keyed_signatures) == 0:
        assert len(messages) == 0
        return []
    recs, blob, off, rand = _keyed_batch_inputs(keyed_signatures, messages, rng)
    return _keyed_located(default_engine().locate_invalid_keyed(recs, blob, off, rand))


def verify_prepared_batch(randomizers32, signatures, public_keys, messages) -> Result:
    """The reference's seam for caller-supplied randomisers (src/batch.rs:84-130)."""
    n = len(signatures)
    sigs = np.frombuffer(b"".join(s.to_bytes() for s in signatures), dtype=np.uint8).reshape(n, 81)
    pks = np.frombuffer(b"".join(k.xy for k in public_keys), dtype=np.uint8).reshape(n, 96)
    inf = np.array([k.infinity for k in public_keys], dtype=np.uint8)
    blob, off = _pack(messages)
    v, _lhs, _rhs = default_engine().verify_batch(sigs, pks, inf, blob, off, randomizers32)
    return _result_from_verdict(v)
