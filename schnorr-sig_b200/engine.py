"""Array-level host API over the C ABI: one `Engine` = one `schnorr_b200_ctx` on one GPU, or -- given a list of
devices -- one multi-device context (`schnorr_b200_create_multi`) whose host entry points shard every call.

Buffers may be numpy arrays (host), torch tensors (host-pinned or CUDA) or raw integer addresses.
The `*_dev` methods take device buffers, enqueue on the engine's stream and do not synchronise;
the plain methods take host buffers and run the same kernels with the copies inside the call.
Layouts are those of include/schnorr_b200.h (the reference's own byte encodings).
"""
import ctypes as C

import numpy as np

from . import _lib

OK, INVALID_PUBLIC_KEY, INVALID_SIGNATURE, MALFORMED = 0, 1, 2, 3


class EngineError(RuntimeError):
    pass


def _ptr(x):
    if x is None:
        return None
    if isinstance(x, int):
        return C.c_void_p(x)
    if isinstance(x, np.ndarray):
        if not x.flags["C_CONTIGUOUS"]:
            raise ValueError("buffers must be C-contiguous")
        return C.c_void_p(x.ctypes.data)
    if hasattr(x, "data_ptr"):  # torch tensor
        if not x.is_contiguous():
            raise ValueError("buffers must be contiguous")
        return C.c_void_p(x.data_ptr())
    raise TypeError("unsupported buffer type %r" % type(x))


def _u8(a, cols=None):
    a = np.ascontiguousarray(a, dtype=np.uint8)
    if cols is not None and (a.ndim != 2 or a.shape[1] != cols):
        raise ValueError("expected an [n,%d] uint8 array, got %r" % (cols, a.shape))
    return a


class Engine:
    def __init__(self, device=0):
        """device: a CUDA device index, or a list of indices for a multi-device context (a device may repeat)."""
        self._L = _lib.lib()
        h = C.c_void_p()
        if isinstance(device, (list, tuple)):
            devs = (C.c_int * len(device))(*[int(d) for d in device])
            rc = self._L.schnorr_b200_create_multi(devs, len(device), C.byref(h))
            self.devices = [int(d) for d in device]
        else:
            rc = self._L.schnorr_b200_create(int(device), C.byref(h))
            self.devices = [int(device)]
        if rc != 0 or not h.value:
            raise EngineError("schnorr_b200_create(device=%r) failed with %d: a CUDA device is required "
                              "(there is no CPU fallback)" % (device, rc))
        self._h = h
        self.device = self.devices[0]

    @property
    def device_count(self) -> int:
        return int(self._L.schnorr_b200_device_count(self._h))

    # ---- lifecycle -----------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._L.schnorr_b200_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            msg = self._L.schnorr_b200_last_error(self._h)
            raise EngineError("%s failed (%d): %s" % (what, rc, msg.decode() if msg else ""))

    def set_stream(self, cuda_stream_ptr):
        self._check(self._L.schnorr_b200_set_stream(self._h, C.c_void_p(cuda_stream_ptr or 0)), "set_stream")

    def synchronize(self):
        self._check(self._L.schnorr_b200_synchronize(self._h), "synchronize")

    @property
    def launch_count(self) -> int:
        return int(self._L.schnorr_b200_launch_count(self._h))

    def last_kernel_ms(self) -> float:
        ms = C.c_float(0)
        self._check(self._L.schnorr_b200_last_kernel_ms(self._h, C.byref(ms)), "last_kernel_ms")
        return float(ms.value)

    def set_exact_only(self, flag: bool):
        """True: every verification goes through the exact Jacobian kernel (A/B measurements, tests)."""
        self._check(self._L.schnorr_b200_set_exact_only(self._h, 1 if flag else 0), "set_exact_only")

    def set_msm_geometry(self, window_bits: int = 0, segment_len: int = 0):
        """Test hook: force the Pippenger window width / segment length of the batch path (0 = automatic)."""
        self._check(self._L.schnorr_b200_set_msm_geometry(self._h, int(window_bits), int(segment_len)), "set_msm_geometry")

    def last_batch_plan(self):
        """(window bits c, windows K, buckets per window B, segment length T) of the last batch call."""
        c, k, t = C.c_int(0), C.c_int(0), C.c_uint(0)
        self._check(self._L.schnorr_b200_last_batch_plan(self._h, C.byref(c), C.byref(k), C.byref(t)), "last_batch_plan")
        return c.value, k.value, (1 << (c.value - 1)) if c.value else 0, t.value

    def set_dist_threshold(self, max_signatures: int):
        """Calls up to this many signatures use the six-lanes-per-signature kernel (0 = never, 2**62 = always)."""
        self._check(self._L.schnorr_b200_set_dist_threshold(self._h, int(max_signatures)), "set_dist_threshold")

    def set_one_threshold(self, max_signatures: int):
        """Calls up to this many signatures use the block-per-signature kernel (0 = never)."""
        self._check(self._L.schnorr_b200_set_one_threshold(self._h, int(max_signatures)), "set_one_threshold")

    def set_batch_small_threshold(self, max_signatures: int):
        """Batches up to this size run one thread block per signature (0 = never: always the Pippenger pipeline)."""
        self._check(self._L.schnorr_b200_set_batch_small_threshold(self._h, int(max_signatures)), "set_batch_small_threshold")

    def set_batch_dist_threshold(self, max_signatures: int):
        """Batches up to this size hash their challenges on six lanes per signature (0 = never)."""
        self._check(self._L.schnorr_b200_set_batch_dist_threshold(self._h, int(max_signatures)), "set_batch_dist_threshold")

    def last_batch_points(self) -> int:
        """MSM points of the last batch call: 2n for verify_batch, n for a registered batch summed per key, 0 for the
        block-per-signature form of small batches; keyed records summed per key: n + m (host form, m misses) or 2n
        (_dev form)."""
        c = C.c_uint64(0)
        self._check(self._L.schnorr_b200_last_batch_points(self._h, C.byref(c)), "last_batch_points")
        return int(c.value)

    def set_registered_batch_threshold(self, min_signatures_per_key: int):
        """Registered batches sum the key side per key from this many signatures per key of the set (0 = always)."""
        self._check(self._L.schnorr_b200_set_registered_batch_threshold(self._h, int(min_signatures_per_key)),
                    "set_registered_batch_threshold")

    def set_keyset_block_threshold(self, max_keys: int):
        """Registrations of up to this many keys run one thread block per key (0 = never, 2**64 - 1 = always)."""
        self._check(self._L.schnorr_b200_set_keyset_block_threshold(self._h, int(max_keys)), "set_keyset_block_threshold")

    def last_exact_count(self) -> int:
        """Items of the last verify_many* call that the fast path handed to the exact kernel."""
        c = C.c_uint64(0)
        self._check(self._L.schnorr_b200_last_exact_count(self._h, C.byref(c)), "last_exact_count")
        return int(c.value)

    # ---- host-buffer entry points --------------------------------------------------------
    def hash_messages(self, rx48, pk96, msgs, off):
        rx48, pk96, msgs = _u8(rx48, 48), _u8(pk96, 96), _u8(msgs)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        n = rx48.shape[0]
        self._check_offsets(n, pk96.shape[0], off, msgs)
        out = np.zeros((n, 32), dtype=np.uint8)
        self._check(self._L.schnorr_b200_hash_messages(self._h, n, _ptr(rx48), _ptr(pk96), _ptr(msgs), _ptr(off),
                                                       _ptr(out)), "hash_messages")
        return out

    @staticmethod
    def _check_inf(n, inf):
        if inf is not None and inf.shape[0] != n:
            raise AssertionError("pk_inf must hold one flag per public key")

    @staticmethod
    def _check_offsets(n, npk, off, msgs):
        # the reference asserts equal lengths (src/batch.rs:37-44)
        if npk != n:
            raise AssertionError("We should have the same number of signatures than public keys")
        if off.shape[0] != n + 1:
            raise AssertionError("We should have the same number of messages than public keys")
        if n and (int(off[-1]) > msgs.size or np.any(off[1:] < off[:-1])):
            raise ValueError("message offsets out of range")

    def verify_many(self, sigs81, pk96, pk_inf, msgs, off):
        sigs81, pk96, msgs = _u8(sigs81, 81), _u8(pk96, 96), _u8(msgs)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        n = sigs81.shape[0]
        self._check_offsets(n, pk96.shape[0], off, msgs)
        inf = None if pk_inf is None else _u8(pk_inf)
        self._check_inf(n, inf)
        out = np.full(n, 255, dtype=np.uint8)
        self._check(self._L.schnorr_b200_verify_many(self._h, n, _ptr(sigs81), _ptr(pk96), _ptr(inf), _ptr(msgs),
                                                     _ptr(off), _ptr(out)), "verify_many")
        return out

    def verify_keyed_many(self, keyed130, msgs, off):
        """KeyedSignature wire records (49-byte compressed key || 81-byte signature) -> verdicts."""
        keyed130, msgs = _u8(keyed130, 130), _u8(msgs)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        n = keyed130.shape[0]
        self._check_offsets(n, n, off, msgs)
        out = np.full(n, 255, dtype=np.uint8)
        self._check(self._L.schnorr_b200_verify_keyed_many(self._h, n, _ptr(keyed130), _ptr(msgs), _ptr(off), _ptr(out)),
                    "verify_keyed_many")
        return out

    # ---- registered key sets -------------------------------------------------------------
    def register_keys(self, pk96, pk_inf=None):
        """Registers public keys (subgroup check + per-key table on every device) -> (KeySetHandle, status uint8[n_keys]):
        status 0 = in the prime-order subgroup (identity included), 1 = not, 3 = non-canonical limb."""
        pk96 = _u8(pk96, 96)
        n = pk96.shape[0]
        inf = None if pk_inf is None else _u8(pk_inf)
        self._check_inf(n, inf)
        status = np.full(n, 255, dtype=np.uint8)
        h = C.c_void_p()
        self._check(self._L.schnorr_b200_keyset_create(self._h, n, _ptr(pk96), _ptr(inf), _ptr(status), C.byref(h)),
                    "keyset_create")
        return KeySetHandle(self, h, n), status

    def keyset_append(self, keyset, pk96, pk_inf=None):
        """Registers keys in the next slots of `keyset` (indices n_keys, n_keys + 1, ...) -> status uint8[n]."""
        pk96 = _u8(pk96, 96)
        n = pk96.shape[0]
        inf = None if pk_inf is None else _u8(pk_inf)
        self._check_inf(n, inf)
        status = np.full(n, 255, dtype=np.uint8)
        self._check(self._L.schnorr_b200_keyset_append(self._h, keyset.handle, n, _ptr(pk96), _ptr(inf), _ptr(status)),
                    "keyset_append")
        keyset.n_keys += n
        return status

    def keyset_replace(self, keyset, key_idx, pk96, pk_inf=None):
        """Registers pk96[j] in slot key_idx[j] of `keyset` (distinct indices inside the set) -> status uint8[n]."""
        pk96 = _u8(pk96, 96)
        key_idx = np.ascontiguousarray(key_idx, dtype=np.uint32)
        n = pk96.shape[0]
        if key_idx.ndim != 1 or key_idx.shape[0] != n:
            raise ValueError("one key index per key")
        inf = None if pk_inf is None else _u8(pk_inf)
        self._check_inf(n, inf)
        status = np.full(n, 255, dtype=np.uint8)
        self._check(self._L.schnorr_b200_keyset_replace(self._h, keyset.handle, n, _ptr(key_idx), _ptr(pk96), _ptr(inf),
                                                        _ptr(status)), "keyset_replace")
        return status

    def keyset_remove(self, keyset, key_idx):
        """Removes slots of `keyset`: they keep their index and behave like an index outside the set (status 3)."""
        key_idx = np.ascontiguousarray(key_idx, dtype=np.uint32).reshape(-1)
        self._check(self._L.schnorr_b200_keyset_remove(self._h, keyset.handle, key_idx.shape[0], _ptr(key_idx)),
                    "keyset_remove")

    def keyset_debug_export(self, keyset, device_index=0, first=0, count=None, tables=True):
        """Test hook: one device's copy of the set -> dict(pk96, inf, status, tables [count, 32, 129, 12] uint64 or
        None, lut [n_lut, 64] uint8)."""
        count = keyset.n_keys - first if count is None else int(count)
        pk = np.zeros((count, 96), dtype=np.uint8)
        inf = np.zeros(count, dtype=np.uint8)
        status = np.zeros(count, dtype=np.uint8)
        tab = np.zeros((count, 32, 129, 12), dtype=np.uint64) if tables else None
        lut = np.zeros((max(keyset.n_keys, 1), 64), dtype=np.uint8)
        n_lut = C.c_uint32(0)
        self._check(self._L.schnorr_b200_keyset_debug_export(self._h, keyset.handle, int(device_index), int(first), count,
                                                             _ptr(pk), _ptr(inf), _ptr(status), _ptr(tab), _ptr(lut),
                                                             C.byref(n_lut)), "keyset_debug_export")
        return dict(pk96=pk, inf=inf, status=status, tables=tab, lut=lut[:n_lut.value].copy())

    def verify_registered_many(self, keyset, sigs81, key_idx, msgs, off):
        """Signature::verify of sigs81[i] over message i under key key_idx[i] of `keyset` -> verdicts (those of
        verify_many; 3 for an index outside the set)."""
        sigs81, msgs = _u8(sigs81, 81), _u8(msgs)
        key_idx = np.ascontiguousarray(key_idx, dtype=np.uint32)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        n = sigs81.shape[0]
        if key_idx.ndim != 1:
            raise ValueError("key_idx must be one-dimensional")
        self._check_offsets(n, key_idx.shape[0], off, msgs)
        out = np.full(n, 255, dtype=np.uint8)
        self._check(self._L.schnorr_b200_verify_registered_many(self._h, keyset.handle, n, _ptr(sigs81), _ptr(key_idx),
                                                                _ptr(msgs), _ptr(off), _ptr(out)), "verify_registered_many")
        return out

    def verify_registered_many_dev(self, keyset, n, sigs81, key_idx, msgs, off, verdicts):
        """Device buffers (key_idx: n uint32), enqueued on the engine's stream, no synchronisation."""
        self._check(self._L.schnorr_b200_verify_registered_many_dev(self._h, keyset.handle, n, _ptr(sigs81), _ptr(key_idx),
                                                                    _ptr(msgs), _ptr(off), _ptr(verdicts)),
                    "verify_registered_many_dev")

    def keyset_lookup(self, keyset, keys49):
        """49-byte compressed keys -> uint32 indices into `keyset`: the smallest index of a registered key whose encoding
        is exactly those bytes and which decompresses to its registered record, else 0xFFFFFFFF."""
        keys49 = _u8(keys49, 49)
        n = keys49.shape[0]
        out = np.full(n, 0xFFFFFFFF, dtype=np.uint32)
        self._check(self._L.schnorr_b200_keyset_lookup(self._h, keyset.handle, n, _ptr(keys49), _ptr(out)), "keyset_lookup")
        return out

    def keyset_lookup_dev(self, keyset, n, keys49, key_idx):
        """Device buffers (key_idx: n uint32), enqueued on the engine's stream, no synchronisation."""
        self._check(self._L.schnorr_b200_keyset_lookup_dev(self._h, keyset.handle, n, _ptr(keys49), _ptr(key_idx)),
                    "keyset_lookup_dev")

    def verify_keyed_registered_many(self, keyset, keyed130, msgs, off):
        """KeyedSignature wire records against a registered key set -> verdicts (those of verify_keyed_many)."""
        keyed130, msgs = _u8(keyed130, 130), _u8(msgs)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        n = keyed130.shape[0]
        self._check_offsets(n, n, off, msgs)
        out = np.full(n, 255, dtype=np.uint8)
        self._check(self._L.schnorr_b200_verify_keyed_registered_many(self._h, keyset.handle, n, _ptr(keyed130), _ptr(msgs),
                                                                      _ptr(off), _ptr(out)), "verify_keyed_registered_many")
        return out

    def verify_keyed_registered_many_dev(self, keyset, n, keyed130, msgs, off, verdicts):
        """Device buffers, enqueued on the engine's stream, no synchronisation (always the lookup path)."""
        self._check(self._L.schnorr_b200_verify_keyed_registered_many_dev(self._h, keyset.handle, n, _ptr(keyed130),
                                                                          _ptr(msgs), _ptr(off), _ptr(verdicts)),
                    "verify_keyed_registered_many_dev")

    def verify_batch(self, sigs81, pk96, pk_inf, msgs, off, rand32):
        """-> (verdict, lhs97, rhs97)"""
        sigs81, pk96, msgs, rand32 = _u8(sigs81, 81), _u8(pk96, 96), _u8(msgs), _u8(rand32, 32)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        n = sigs81.shape[0]
        self._check_offsets(n, pk96.shape[0], off, msgs)
        if rand32.shape[0] != n:
            raise AssertionError("one randomiser per signature")
        inf = None if pk_inf is None else _u8(pk_inf)
        verdict = C.c_int(-1)
        lhs = np.zeros(97, dtype=np.uint8)
        rhs = np.zeros(97, dtype=np.uint8)
        self._check(self._L.schnorr_b200_verify_batch(self._h, n, _ptr(sigs81), _ptr(pk96), _ptr(inf), _ptr(msgs),
                                                      _ptr(off), _ptr(rand32), C.byref(verdict), _ptr(lhs), _ptr(rhs)),
                    "verify_batch")
        return verdict.value, lhs, rhs

    def _registered_batch_args(self, sigs81, key_idx, msgs, off, rand32):
        sigs81, msgs, rand32 = _u8(sigs81, 81), _u8(msgs), _u8(rand32, 32)
        key_idx = np.ascontiguousarray(key_idx, dtype=np.uint32)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        n = sigs81.shape[0]
        if key_idx.ndim != 1:
            raise ValueError("key_idx must be one-dimensional")
        self._check_offsets(n, key_idx.shape[0], off, msgs)
        if rand32.shape[0] != n:
            raise AssertionError("one randomiser per signature")
        return n, sigs81, key_idx, msgs, off, rand32

    def verify_batch_registered(self, keyset, sigs81, key_idx, msgs, off, rand32):
        """verify_batch of sigs81[i] over message i under key key_idx[i] of `keyset` -> (verdict, lhs97, rhs97), those of
        verify_batch on the gathered keys (3 when an index is outside the set)."""
        n, sigs81, key_idx, msgs, off, rand32 = self._registered_batch_args(sigs81, key_idx, msgs, off, rand32)
        verdict = C.c_int(-1)
        lhs = np.zeros(97, dtype=np.uint8)
        rhs = np.zeros(97, dtype=np.uint8)
        self._check(self._L.schnorr_b200_verify_batch_registered(self._h, keyset.handle, n, _ptr(sigs81), _ptr(key_idx),
                                                                 _ptr(msgs), _ptr(off), _ptr(rand32), C.byref(verdict),
                                                                 _ptr(lhs), _ptr(rhs)), "verify_batch_registered")
        return verdict.value, lhs, rhs

    def locate_invalid_registered(self, keyset, sigs81, key_idx, msgs, off, rand32):
        """locate_invalid against a registered key set -> uint8[n] (3 for an index outside the set)."""
        n, sigs81, key_idx, msgs, off, rand32 = self._registered_batch_args(sigs81, key_idx, msgs, off, rand32)
        flags = np.zeros(n, dtype=np.uint8)
        nb = C.c_uint64(0)
        self._check(self._L.schnorr_b200_locate_invalid_registered(self._h, keyset.handle, n, _ptr(sigs81), _ptr(key_idx),
                                                                   _ptr(msgs), _ptr(off), _ptr(rand32), _ptr(flags),
                                                                   C.byref(nb)), "locate_invalid_registered")
        assert int(nb.value) == int(np.count_nonzero(flags))
        return flags

    def _keyed_batch_args(self, keyed130, msgs, off, rand32):
        keyed130, msgs, rand32 = _u8(keyed130, 130), _u8(msgs), _u8(rand32, 32)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        n = keyed130.shape[0]
        self._check_offsets(n, n, off, msgs)
        if rand32.shape[0] != n:
            raise AssertionError("one randomiser per signature")
        return n, keyed130, msgs, off, rand32

    def verify_batch_keyed(self, keyed130, msgs, off, rand32):
        """verify_batch over 130-byte KeyedSignature records -> (verdict, lhs97, rhs97), those of verify_batch on the
        decoded keys (3 when a key does not decode)."""
        return self._batch_keyed(None, keyed130, msgs, off, rand32)

    def verify_batch_keyed_registered(self, keyset, keyed130, msgs, off, rand32):
        """verify_batch_keyed against a registered key set -> (verdict, lhs97, rhs97), those of verify_batch_keyed."""
        return self._batch_keyed(keyset, keyed130, msgs, off, rand32)

    def _batch_keyed(self, keyset, keyed130, msgs, off, rand32):
        n, keyed130, msgs, off, rand32 = self._keyed_batch_args(keyed130, msgs, off, rand32)
        verdict = C.c_int(-1)
        lhs = np.zeros(97, dtype=np.uint8)
        rhs = np.zeros(97, dtype=np.uint8)
        if keyset is None:
            rc = self._L.schnorr_b200_verify_batch_keyed(self._h, n, _ptr(keyed130), _ptr(msgs), _ptr(off), _ptr(rand32),
                                                         C.byref(verdict), _ptr(lhs), _ptr(rhs))
        else:
            rc = self._L.schnorr_b200_verify_batch_keyed_registered(self._h, keyset.handle, n, _ptr(keyed130), _ptr(msgs),
                                                                    _ptr(off), _ptr(rand32), C.byref(verdict), _ptr(lhs),
                                                                    _ptr(rhs))
        self._check(rc, "verify_batch_keyed" if keyset is None else "verify_batch_keyed_registered")
        return verdict.value, lhs, rhs

    def locate_invalid_keyed(self, keyed130, msgs, off, rand32):
        """locate_invalid over KeyedSignature records -> uint8[n] (3 where a key does not decode)."""
        return self._locate_keyed(None, keyed130, msgs, off, rand32)

    def locate_invalid_keyed_registered(self, keyset, keyed130, msgs, off, rand32):
        """locate_invalid_keyed against a registered key set -> the flags of locate_invalid_keyed."""
        return self._locate_keyed(keyset, keyed130, msgs, off, rand32)

    def _locate_keyed(self, keyset, keyed130, msgs, off, rand32):
        n, keyed130, msgs, off, rand32 = self._keyed_batch_args(keyed130, msgs, off, rand32)
        flags = np.zeros(n, dtype=np.uint8)
        nb = C.c_uint64(0)
        if keyset is None:
            rc = self._L.schnorr_b200_locate_invalid_keyed(self._h, n, _ptr(keyed130), _ptr(msgs), _ptr(off), _ptr(rand32),
                                                           _ptr(flags), C.byref(nb))
        else:
            rc = self._L.schnorr_b200_locate_invalid_keyed_registered(self._h, keyset.handle, n, _ptr(keyed130), _ptr(msgs),
                                                                      _ptr(off), _ptr(rand32), _ptr(flags), C.byref(nb))
        self._check(rc, "locate_invalid_keyed" if keyset is None else "locate_invalid_keyed_registered")
        assert int(nb.value) == int(np.count_nonzero(flags))
        return flags

    def locate_invalid(self, sigs81, pk96, pk_inf, msgs, off, rand32):
        """Failed-batch localisation in batch semantics -> uint8[n]: 0 clean, 2 bad, 3 malformed (see the header)."""
        sigs81, pk96, msgs, rand32 = _u8(sigs81, 81), _u8(pk96, 96), _u8(msgs), _u8(rand32, 32)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        n = sigs81.shape[0]
        self._check_offsets(n, pk96.shape[0], off, msgs)
        if rand32.shape[0] != n:
            raise AssertionError("one randomiser per signature")
        inf = None if pk_inf is None else _u8(pk_inf)
        self._check_inf(n, inf)
        flags = np.zeros(n, dtype=np.uint8)
        nb = C.c_uint64(0)
        self._check(self._L.schnorr_b200_locate_invalid(self._h, n, _ptr(sigs81), _ptr(pk96), _ptr(inf), _ptr(msgs), _ptr(off),
                                                        _ptr(rand32), _ptr(flags), C.byref(nb)), "locate_invalid")
        return flags

    def batch_partial(self, sigs81, pk96, pk_inf, msgs, off, rand32):
        """This rank's share of a batch: host arrays in, the 192-byte partial out (multi-GPU form).
        torch is used only to hold the device buffers."""
        import torch
        sigs81, pk96, msgs, rand32 = _u8(sigs81, 81), _u8(pk96, 96), _u8(msgs), _u8(rand32, 32)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        n = sigs81.shape[0]
        self._check_offsets(n, pk96.shape[0], off, msgs)
        dev = torch.device("cuda", self.device)
        part = torch.zeros(192, dtype=torch.uint8, device=dev)
        if n == 0:
            self.batch_partial_dev(0, None, None, None, None, None, None, part)
        else:
            def up(a):
                return torch.from_numpy(np.ascontiguousarray(a)).to(dev) if a.size else torch.zeros(16, dtype=torch.uint8, device=dev)
            t = [up(sigs81), up(pk96), None if pk_inf is None else up(_u8(pk_inf)), up(msgs),
                 torch.from_numpy(off.view(np.int64)).to(dev), up(rand32)]
            torch.cuda.synchronize(dev)
            self.batch_partial_dev(n, t[0], t[1], t[2], t[3], t[4], t[5], part)
        self.synchronize()
        return part.cpu().numpy()

    def batch_finish(self, partials192):
        partials192 = _u8(partials192, 192)
        verdict = C.c_int(-1)
        lhs = np.zeros(97, dtype=np.uint8)
        rhs = np.zeros(97, dtype=np.uint8)
        self._check(self._L.schnorr_b200_batch_finish(self._h, partials192.shape[0], _ptr(partials192),
                                                      C.byref(verdict), _ptr(lhs), _ptr(rhs)), "batch_finish")
        return verdict.value, lhs, rhs

    def keygen(self, sk32):
        sk32 = _u8(sk32, 32)
        n = sk32.shape[0]
        pk = np.zeros((n, 96), dtype=np.uint8)
        inf = np.zeros(n, dtype=np.uint8)
        self._check(self._L.schnorr_b200_keygen(self._h, n, _ptr(sk32), _ptr(pk), _ptr(inf)), "keygen")
        return pk, inf

    def sign_many(self, sk32, pk96, pk_inf, msgs, off, nonce32):
        sk32, pk96, msgs, nonce32 = _u8(sk32, 32), _u8(pk96, 96), _u8(msgs), _u8(nonce32, 32)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        n = sk32.shape[0]
        self._check_offsets(n, pk96.shape[0], off, msgs)
        inf = None if pk_inf is None else _u8(pk_inf)
        out = np.zeros((n, 81), dtype=np.uint8)
        self._check(self._L.schnorr_b200_sign_many(self._h, n, _ptr(sk32), _ptr(pk96), _ptr(inf), _ptr(msgs), _ptr(off),
                                                   _ptr(nonce32), _ptr(out)), "sign_many")
        return out

    # ---- hierarchical deterministic derivation (src/derivation.rs) -------------------------------------------------
    def derive_master_keys(self, seeds32):
        seeds32 = _u8(seeds32, 32)
        n = seeds32.shape[0]
        out, ok = np.zeros((n, 64), dtype=np.uint8), np.zeros(n, dtype=np.uint8)
        self._check(self._L.schnorr_b200_derive_master_keys(self._h, n, _ptr(seeds32), _ptr(out), _ptr(ok)), "derive_master_keys")
        return out, ok

    def derive_private_children(self, parent_xsk64, indices):
        parent = np.ascontiguousarray(np.frombuffer(bytes(parent_xsk64), dtype=np.uint8))
        assert parent.size == 64
        idx = np.ascontiguousarray(indices, dtype=np.uint32)
        n = idx.shape[0]
        out, ok = np.zeros((n, 64), dtype=np.uint8), np.zeros(n, dtype=np.uint8)
        self._check(self._L.schnorr_b200_derive_private_children(self._h, n, _ptr(parent), _ptr(idx), _ptr(out), _ptr(ok)),
                    "derive_private_children")
        return out, ok

    def derive_public_children(self, parent_xpk81, indices):
        parent = np.ascontiguousarray(np.frombuffer(bytes(parent_xpk81), dtype=np.uint8))
        assert parent.size == 81
        idx = np.ascontiguousarray(indices, dtype=np.uint32)
        n = idx.shape[0]
        out, ok = np.zeros((n, 81), dtype=np.uint8), np.zeros(n, dtype=np.uint8)
        self._check(self._L.schnorr_b200_derive_public_children(self._h, n, _ptr(parent), _ptr(idx), _ptr(out), _ptr(ok)),
                    "derive_public_children")
        return out, ok

    def decompress(self, in49):
        in49 = _u8(in49, 49)
        n = in49.shape[0]
        pk = np.zeros((n, 96), dtype=np.uint8)
        inf = np.zeros(n, dtype=np.uint8)
        ok = np.zeros(n, dtype=np.uint8)
        self._check(self._L.schnorr_b200_decompress(self._h, n, _ptr(in49), _ptr(pk), _ptr(inf), _ptr(ok)), "decompress")
        return pk, inf, ok

    def compress(self, pk96, pk_inf=None):
        pk96 = _u8(pk96, 96)
        n = pk96.shape[0]
        inf = None if pk_inf is None else _u8(pk_inf)
        out = np.zeros((n, 49), dtype=np.uint8)
        self._check(self._L.schnorr_b200_compress(self._h, n, _ptr(pk96), _ptr(inf), _ptr(out)), "compress")
        return out

    def debug_field_ops(self, a6, b6):
        """Test hook: device field operations on n pairs of Fp6 elements -> [n, 8, 6] uint64."""
        a6 = np.ascontiguousarray(a6, dtype=np.uint64).reshape(-1, 6)
        b6 = np.ascontiguousarray(b6, dtype=np.uint64).reshape(-1, 6)
        out = np.zeros((a6.shape[0], 8, 6), dtype=np.uint64)
        self._check(self._L.schnorr_b200_debug_field_ops(self._h, a6.shape[0], _ptr(a6), _ptr(b6), _ptr(out)), "debug_field_ops")
        return out

    def debug_lazy_ops(self, a6, b6):
        """Test hook: lazily reduced fast-path building blocks (a6 may hold non-canonical limbs) -> [n, 8, 6] uint64."""
        a6 = np.ascontiguousarray(a6, dtype=np.uint64).reshape(-1, 6)
        b6 = np.ascontiguousarray(b6, dtype=np.uint64).reshape(-1, 6)
        out = np.zeros((a6.shape[0], 8, 6), dtype=np.uint64)
        self._check(self._L.schnorr_b200_debug_lazy_ops(self._h, a6.shape[0], _ptr(a6), _ptr(b6), _ptr(out)), "debug_lazy_ops")
        return out

    def imad_peak(self, iters=1 << 16):
        w = C.c_double(0)
        ms = C.c_double(0)
        self._check(self._L.schnorr_b200_imad_peak(self._h, int(iters), C.byref(w), C.byref(ms)), "imad_peak")
        return w.value, ms.value

    # ---- raw-pointer entry points (host-pinned or device buffers; no shape checks) -------------
    def verify_many_raw(self, n, sigs81, pk96, pk_inf, msgs, off, verdicts):
        """Host variant on raw buffers (e.g. pinned torch tensors): copies + kernels + copy back."""
        self._check(self._L.schnorr_b200_verify_many(self._h, n, _ptr(sigs81), _ptr(pk96), _ptr(pk_inf), _ptr(msgs),
                                                     _ptr(off), _ptr(verdicts)), "verify_many")

    def verify_many_dev(self, n, sigs81, pk96, pk_inf, msgs, off, verdicts):
        self._check(self._L.schnorr_b200_verify_many_dev(self._h, n, _ptr(sigs81), _ptr(pk96), _ptr(pk_inf), _ptr(msgs),
                                                         _ptr(off), _ptr(verdicts)), "verify_many_dev")

    def verify_keyed_many_dev(self, n, keyed130, msgs, off, verdicts):
        self._check(self._L.schnorr_b200_verify_keyed_many_dev(self._h, n, _ptr(keyed130), _ptr(msgs), _ptr(off),
                                                               _ptr(verdicts)), "verify_keyed_many_dev")

    def hash_messages_dev(self, n, rx48, pk96, msgs, off, digests):
        self._check(self._L.schnorr_b200_hash_messages_dev(self._h, n, _ptr(rx48), _ptr(pk96), _ptr(msgs), _ptr(off),
                                                           _ptr(digests)), "hash_messages_dev")

    def keygen_dev(self, n, sk32, pk96, pk_inf):
        self._check(self._L.schnorr_b200_keygen_dev(self._h, n, _ptr(sk32), _ptr(pk96), _ptr(pk_inf)), "keygen_dev")

    def sign_many_dev(self, n, sk32, pk96, pk_inf, msgs, off, nonce32, sigs81):
        self._check(self._L.schnorr_b200_sign_many_dev(self._h, n, _ptr(sk32), _ptr(pk96), _ptr(pk_inf), _ptr(msgs),
                                                       _ptr(off), _ptr(nonce32), _ptr(sigs81)), "sign_many_dev")

    def verify_batch_dev(self, n, sigs81, pk96, pk_inf, msgs, off, rand32, result216):
        """Whole single-device batch on device buffers; result216 (device) = verdict | lhs97 | rhs97 (see the header)."""
        self._check(self._L.schnorr_b200_verify_batch_dev(self._h, n, _ptr(sigs81), _ptr(pk96), _ptr(pk_inf), _ptr(msgs),
                                                          _ptr(off), _ptr(rand32), _ptr(result216)), "verify_batch_dev")

    def verify_batch_registered_dev(self, keyset, n, sigs81, key_idx, msgs, off, rand32, result216):
        """Registered batch on device buffers (key_idx: n uint32), enqueued on the engine's stream, no synchronisation;
        result216 as in verify_batch_dev."""
        self._check(self._L.schnorr_b200_verify_batch_registered_dev(self._h, keyset.handle, n, _ptr(sigs81), _ptr(key_idx),
                                                                     _ptr(msgs), _ptr(off), _ptr(rand32), _ptr(result216)),
                    "verify_batch_registered_dev")

    def verify_batch_keyed_dev(self, n, keyed130, msgs, off, rand32, result216):
        """Batch over KeyedSignature records on device buffers, enqueued on the engine's stream, no synchronisation;
        result216 as in verify_batch_dev."""
        self._check(self._L.schnorr_b200_verify_batch_keyed_dev(self._h, n, _ptr(keyed130), _ptr(msgs), _ptr(off),
                                                                _ptr(rand32), _ptr(result216)), "verify_batch_keyed_dev")

    def verify_batch_keyed_registered_dev(self, keyset, n, keyed130, msgs, off, rand32, result216):
        """verify_batch_keyed_dev against a registered key set (MSM planned for 2n points)."""
        self._check(self._L.schnorr_b200_verify_batch_keyed_registered_dev(self._h, keyset.handle, n, _ptr(keyed130),
                                                                           _ptr(msgs), _ptr(off), _ptr(rand32),
                                                                           _ptr(result216)),
                    "verify_batch_keyed_registered_dev")

    def batch_partial_dev(self, n, sigs81, pk96, pk_inf, msgs, off, rand32, partial192):
        self._check(self._L.schnorr_b200_batch_partial_dev(self._h, n, _ptr(sigs81), _ptr(pk96), _ptr(pk_inf),
                                                           _ptr(msgs), _ptr(off), _ptr(rand32), _ptr(partial192)),
                    "batch_partial_dev")

    def batch_finish_dev(self, n_partials, partials192, result216):
        self._check(self._L.schnorr_b200_batch_finish_dev(self._h, n_partials, _ptr(partials192), _ptr(result216)),
                    "batch_finish_dev")


class KeySetHandle:
    """A registered key set (schnorr_b200_keyset) of one Engine; keeps the engine alive and frees the tables on close."""

    def __init__(self, engine, handle, n_keys):
        self.engine, self._h, self.n_keys = engine, handle, n_keys

    @property
    def handle(self):
        if self._h is None or not self._h.value:
            raise ValueError("the key set has been closed")
        return self._h

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.engine._L.schnorr_b200_keyset_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_DEFAULT = {}


def default_engine(device: int = 0) -> Engine:
    if device not in _DEFAULT:
        _DEFAULT[device] = Engine(device)
    return _DEFAULT[device]
