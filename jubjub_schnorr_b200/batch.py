"""Batch entry points over numpy / raw device buffers (thin wrappers of the C ABI, include/jjschnorr_b200.h)."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native

STATUS_OK, STATUS_INVALID_SIGNATURE, STATUS_INVALID_POINT, STATUS_BYTES_ERROR = 0, 1, 2, 3
SINGLE, DOUBLE, VARGEN, AGGREGATE = 0, 1, 2, 3
PK_SIZE = {SINGLE: 32, DOUBLE: 64, VARGEN: 64, AGGREGATE: 32}
SIG_SIZE = {SINGLE: 64, DOUBLE: 96, VARGEN: 64, AGGREGATE: 64}


class JjsError(RuntimeError):
    pass


class KeySet:
    """A key set registered with BatchVerifier.keyset_create: its handle in the context, kind (SINGLE or DOUBLE), number of keys,
    per-key status (0 valid, 2 InvalidPoint, 3 BytesError), and what jjs_keyset_info reports: the key-window width of its tables
    (8..4, 0 for decoded points only) and the bytes it holds on each device."""

    def __init__(self, handle, kind, n_keys, key_status, key_window_bits=None, bytes_per_device=None):
        self.handle, self.kind, self.n_keys, self.key_status = handle, kind, n_keys, key_status
        self.key_window_bits, self.bytes_per_device = key_window_bits, bytes_per_device


def _u8(a, width, name):
    a = np.ascontiguousarray(a, dtype=np.uint8)
    if a.size % width:
        raise ValueError(f"{name}: byte length {a.size} is not a multiple of {width}")
    return a.reshape(-1, width)


class BatchVerifier:
    """Owns a jjs_ctx over one or more CUDA devices.  One host thread at a time."""

    def __init__(self, devices=None, memory_limit=None):
        """memory_limit: bytes of device memory the context may hold on each device (jjs_init_limited); None: jjs_init."""
        self._lib = _native.lib()
        self._ctx = C.c_void_p()
        if devices is None:
            devices = [0]
        arr = (C.c_int * len(devices))(*devices)
        if memory_limit is None:
            name, rc = "jjs_init", self._lib.jjs_init(arr, len(devices), C.byref(self._ctx))
        else:
            name, rc = "jjs_init_limited", self._lib.jjs_init_limited(arr, len(devices), int(memory_limit), C.byref(self._ctx))
        if rc != 0:
            msg = self._lib.jjs_last_error(self._ctx).decode() if self._ctx else "allocation failed"
            if self._ctx:
                self._lib.jjs_destroy(self._ctx)
                self._ctx = C.c_void_p()
            raise JjsError(f"{name} failed ({rc}): {msg}")
        self.devices = list(devices)

    def close(self):
        if getattr(self, "_ctx", None):
            self._lib.jjs_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, rc, what):
        if rc != 0:
            raise JjsError(f"{what} failed ({rc}): {self._lib.jjs_last_error(self._ctx).decode()}")

    def memory_info(self, device_index=0):
        """{"bytes_held", "fb_window_bits", "items_in_flight"} of the context on one of its devices (jjs_memory_info)."""
        held, items, bits = C.c_uint64(), C.c_uint64(), C.c_int()
        self._check(self._lib.jjs_memory_info(self._ctx, device_index, C.byref(held), C.byref(bits), C.byref(items)), "jjs_memory_info")
        return {"bytes_held": int(held.value), "fb_window_bits": int(bits.value), "items_in_flight": int(items.value)}

    @property
    def launch_count(self) -> int:
        return int(self._lib.jjs_launch_count(self._ctx))

    STAGES = ("decode", "challenge", "aggregate", "equation", "status", "rtest")

    def profile(self, on: bool):
        self._lib.jjs_profile_enable(self._ctx, int(on))

    def profile_collect(self):
        """{stage: (total_ms, launches)} since the last collect (waits for the recorded events)."""
        ms = (C.c_double * len(self.STAGES))()
        cnt = (C.c_uint64 * len(self.STAGES))()
        self._check(self._lib.jjs_profile_collect(self._ctx, ms, cnt), "jjs_profile_collect")
        return {name: (float(ms[i]), int(cnt[i])) for i, name in enumerate(self.STAGES)}

    # ---- host buffers ---------------------------------------------------------------------------
    def _verify_host(self, variant, fn, name, pk, sig, msg, want_challenge):
        pk, sig, msg = _u8(pk, PK_SIZE[variant], "pk"), _u8(sig, SIG_SIZE[variant], "sig"), _u8(msg, 32, "msg")
        n = msg.shape[0]
        if pk.shape[0] != n or sig.shape[0] != n:
            raise ValueError("pk, sig and msg must describe the same number of items")
        status = np.empty(n, dtype=np.uint8)
        c = np.empty((n, 32), dtype=np.uint8) if want_challenge else None
        self._check(fn(self._ctx, pk.ctypes.data, sig.ctypes.data, msg.ctypes.data, n, status.ctypes.data,
                       c.ctypes.data if want_challenge else None), name)
        return (status, c) if want_challenge else status

    def verify_single(self, pk32, sig64, msg32, want_challenge=False):
        return self._verify_host(SINGLE, self._lib.jjs_verify_single, "jjs_verify_single", pk32, sig64, msg32, want_challenge)

    def verify_batch(self, pk32, sig64, msg32):
        """verify_batch(&[(PublicKey, Signature, BlsScalar)]) -> Vec<bool> as a packed bitmap (uint32 words, bit i % 32 of
        word i // 32) straight from jjs_verify_batch; `unpack_bitmap` turns it into a bool array."""
        pk, sig, msg = _u8(pk32, 32, "pk"), _u8(sig64, 64, "sig"), _u8(msg32, 32, "msg")
        n = msg.shape[0]
        if pk.shape[0] != n or sig.shape[0] != n:
            raise ValueError("pk, sig and msg must describe the same number of items")
        words = np.zeros((n + 31) // 32, dtype=np.uint32)
        self._check(self._lib.jjs_verify_batch(self._ctx, pk.ctypes.data, sig.ctypes.data, msg.ctypes.data, n, words.ctypes.data), "jjs_verify_batch")
        return words

    def _verify_bitmap(self, variant, fn, name, pk, sig, msg):
        pk, sig, msg = _u8(pk, PK_SIZE[variant], "pk"), _u8(sig, SIG_SIZE[variant], "sig"), _u8(msg, 32, "msg")
        n = msg.shape[0]
        if pk.shape[0] != n or sig.shape[0] != n:
            raise ValueError("pk, sig and msg must describe the same number of items")
        words = np.zeros((n + 31) // 32, dtype=np.uint32)
        self._check(fn(self._ctx, pk.ctypes.data, sig.ctypes.data, msg.ctypes.data, n, words.ctypes.data), name)
        return words

    def verify_batch_double(self, pk64, sig96, msg32):
        return self._verify_bitmap(DOUBLE, self._lib.jjs_verify_batch_double, "jjs_verify_batch_double", pk64, sig96, msg32)

    def verify_batch_vargen(self, pk64, sig64, msg32):
        return self._verify_bitmap(VARGEN, self._lib.jjs_verify_batch_vargen, "jjs_verify_batch_vargen", pk64, sig64, msg32)

    def verify_batch_aggregate(self, pks32, offsets, sig64, msg32):
        pks, sig, msg = _u8(pks32, 32, "pks"), _u8(sig64, 64, "sig"), _u8(msg32, 32, "msg")
        offsets = np.ascontiguousarray(offsets, dtype=np.uint32)
        n = msg.shape[0]
        if offsets.shape[0] != n + 1 or sig.shape[0] != n or int(offsets[-1]) != pks.shape[0] or int(offsets[0]) != 0:
            raise ValueError("offsets must have n + 1 entries covering pks32 exactly")
        words = np.zeros((n + 31) // 32, dtype=np.uint32)
        self._check(self._lib.jjs_verify_batch_aggregate(self._ctx, pks.ctypes.data, offsets.ctypes.data, sig.ctypes.data, msg.ctypes.data, n,
                                                         words.ctypes.data), "jjs_verify_batch_aggregate")
        return words

    def verify_mixed(self, parts, want_challenge=False, want_bitmap=False):
        """Several batches of different kinds in one call (jjs_verify_mixed).  parts: iterable of (kind, pk, sig, msg) or, for
        AGGREGATE, (kind, pks, sig, msg, offsets).  Returns one dict per part: status, and c / aggpk / bitmap when asked for."""
        arr, keep, out = self._mixed_parts(parts, want_challenge, want_bitmap)
        self._check(self._lib.jjs_verify_mixed(self._ctx, arr, len(out)), "jjs_verify_mixed")
        return out

    def verify_grouped(self, parts, seed=None, want_challenge=False, want_bitmap=False):
        """Per-item results as verify_mixed returns them, by one random linear combination per group of consecutive items and
        the per-item equations only in groups whose combination fails (jjs_verify_grouped): an item whose equation fails is
        reported valid with probability at most 2^-128.  Returns (results, fallback_items), fallback_items = the items verified
        one by one.  seed: as for verify_all."""
        arr, keep, out = self._mixed_parts(parts, want_challenge, want_bitmap)
        keep_seed, sp = self._seed_ptr(seed)
        fb = C.c_uint64(0)
        self._check(self._lib.jjs_verify_grouped(self._ctx, arr, len(out), sp, C.byref(fb)), "jjs_verify_grouped")
        return out, int(fb.value)

    def verify_grouped_device(self, parts, d_fallback=None, seed=None, stream=None, device_index=0):
        """jjs_verify_grouped_device on raw device pointers: parts = iterable of (kind, pk_ptr, sig_ptr, msg_ptr, n, status_ptr,
        c_ptr_or_None, aggpk_ptr_or_None, bitmap_ptr_or_None) or, for AGGREGATE, the same followed by d_offsets_ptr and h_offsets
        (the host copy of the offsets).  The uint64 fallback count is written to d_fallback (if given) on `stream`."""
        structs, hosts, keep = [], [], []
        for part in parts:
            kind, pk, sig, msg, n, st, c, agg, bm = part[:9]
            d_off, h_off = (part[9], np.ascontiguousarray(part[10], dtype=np.uint32)) if kind == AGGREGATE else (None, None)
            structs.append(_native.Part(kind, pk, d_off, sig, msg, n, st, c, agg, bm))
            hosts.append(h_off.ctypes.data if h_off is not None else None)
            keep.append(h_off)
        arr = (_native.Part * max(len(structs), 1))(*structs)
        harr = (C.c_void_p * max(len(hosts), 1))(*hosts)
        keep_seed, sp = self._seed_ptr(seed)
        self._check(self._lib.jjs_verify_grouped_device(self._ctx, device_index, arr, len(structs), harr, sp, d_fallback, stream),
                    "jjs_verify_grouped_device")

    @staticmethod
    def _mixed_parts(parts, want_challenge, want_bitmap):
        """jjs_part array and output arrays of verify_mixed / verify_grouped"""
        structs, keep, out = [], [], []
        for part in parts:
            kind, pk, sig, msg = part[0], part[1], part[2], part[3]
            pk, sig, msg = _u8(pk, PK_SIZE[kind], "pk"), _u8(sig, SIG_SIZE[kind], "sig"), _u8(msg, 32, "msg")
            n = msg.shape[0]
            off = None
            if kind == AGGREGATE:
                off = np.ascontiguousarray(part[4], dtype=np.uint32)
                if off.shape[0] != n + 1 or int(off[-1]) != pk.shape[0] or int(off[0]) != 0:
                    raise ValueError("offsets must have n + 1 entries covering pks32 exactly")
            elif pk.shape[0] != n:
                raise ValueError("pk, sig and msg must describe the same number of items")
            if sig.shape[0] != n:
                raise ValueError("pk, sig and msg must describe the same number of items")
            res = {"status": np.empty(n, dtype=np.uint8)}
            if want_challenge:
                res["c"] = np.empty((n, 32), dtype=np.uint8)
            if kind == AGGREGATE:
                res["aggpk"] = np.empty((n, 32), dtype=np.uint8)
            if want_bitmap:
                res["bitmap"] = np.zeros((n + 31) // 32, dtype=np.uint32)
            ptr = lambda a: a.ctypes.data if a is not None else None  # noqa: E731
            structs.append(_native.Part(kind, ptr(pk), ptr(off), ptr(sig), ptr(msg), n, ptr(res["status"]), ptr(res.get("c")), ptr(res.get("aggpk")),
                                        ptr(res.get("bitmap"))))
            keep.append((pk, sig, msg, off))
            out.append(res)
        arr = (_native.Part * max(len(structs), 1))(*structs)
        return arr, keep, out

    def verify_mixed_ptr(self, parts):
        """jjs_verify_mixed on raw host pointers (e.g. pinned torch tensors): parts = iterable of
        (kind, pk_ptr, offsets_ptr_or_None, sig_ptr, msg_ptr, n, status_ptr, c_ptr_or_None, aggpk_ptr_or_None, bitmap_ptr_or_None)."""
        structs = [_native.Part(*p) for p in parts]
        arr = (_native.Part * len(structs))(*structs)
        self._check(self._lib.jjs_verify_mixed(self._ctx, arr, len(structs)), "jjs_verify_mixed")

    @staticmethod
    def unpack_bitmap(words, n):
        return np.unpackbits(np.ascontiguousarray(words, dtype="<u4").view(np.uint8), bitorder="little")[:n].astype(bool)

    def status_bitmap_device(self, d_status, n, d_bitmap, stream=None, device_index=0):
        self._check(self._lib.jjs_status_bitmap_device(self._ctx, device_index, d_status, n, d_bitmap, stream), "jjs_status_bitmap_device")

    def verify_double(self, pk64, sig96, msg32, want_challenge=False):
        return self._verify_host(DOUBLE, self._lib.jjs_verify_double, "jjs_verify_double", pk64, sig96, msg32, want_challenge)

    def verify_vargen(self, pk64, sig64, msg32, want_challenge=False):
        return self._verify_host(VARGEN, self._lib.jjs_verify_vargen, "jjs_verify_vargen", pk64, sig64, msg32, want_challenge)

    def verify_aggregate(self, pks32, offsets, sig64, msg32, want_challenge=False, want_aggregate_key=False):
        pks, sig, msg = _u8(pks32, 32, "pks"), _u8(sig64, 64, "sig"), _u8(msg32, 32, "msg")
        offsets = np.ascontiguousarray(offsets, dtype=np.uint32)
        n = msg.shape[0]
        if offsets.shape[0] != n + 1 or sig.shape[0] != n or int(offsets[-1]) != pks.shape[0] or int(offsets[0]) != 0:
            raise ValueError("offsets must have n + 1 entries covering pks32 exactly")
        status = np.empty(n, dtype=np.uint8)
        c = np.empty((n, 32), dtype=np.uint8) if want_challenge else None
        agg = np.empty((n, 32), dtype=np.uint8) if want_aggregate_key else None
        self._check(self._lib.jjs_verify_aggregate(self._ctx, pks.ctypes.data, offsets.ctypes.data, sig.ctypes.data, msg.ctypes.data, n,
                                                   status.ctypes.data, c.ctypes.data if want_challenge else None,
                                                   agg.ctypes.data if want_aggregate_key else None), "jjs_verify_aggregate")
        out = [status]
        if want_challenge:
            out.append(c)
        if want_aggregate_key:
            out.append(agg)
        return out[0] if len(out) == 1 else tuple(out)

    def verify_ext(self, variant, points_ext160, u32, msg32, want_challenge=False):
        """Typed inputs: points as JubJubExtended Montgomery coordinates (160 bytes each, item-major), see jjs_verify_ext."""
        slots = {SINGLE: 2, DOUBLE: 4, VARGEN: 3}[variant]
        pts, u, msg = _u8(points_ext160, 160 * slots, "points"), _u8(u32, 32, "u"), _u8(msg32, 32, "msg")
        n = msg.shape[0]
        if pts.shape[0] != n or u.shape[0] != n:
            raise ValueError("points, u and msg must describe the same number of items")
        status = np.empty(n, dtype=np.uint8)
        c = np.empty((n, 32), dtype=np.uint8) if want_challenge else None
        self._check(self._lib.jjs_verify_ext(self._ctx, variant, pts.ctypes.data, u.ctypes.data, msg.ctypes.data, n, status.ctypes.data,
                                             c.ctypes.data if want_challenge else None), "jjs_verify_ext")
        return (status, c) if want_challenge else status

    def points_to_ext(self, points32, z_mont32):
        pts, z = _u8(points32, 32, "points"), _u8(z_mont32, 32, "z")
        out = np.empty((pts.shape[0], 160), dtype=np.uint8)
        self._check(self._lib.jjs_points_to_ext(self._ctx, pts.ctypes.data, z.ctypes.data, pts.shape[0], out.ctypes.data), "jjs_points_to_ext")
        return out

    def multisig_combine(self, pks32, R32, S32, z32, offsets, msg32):
        """multisig::combine per session: (status[n], bad_index[n], sig[n,64], share_ok[K]); see jjs_multisig_combine."""
        pks, Rs, Ss, zs, msg = _u8(pks32, 32, "pks"), _u8(R32, 32, "R"), _u8(S32, 32, "S"), _u8(z32, 32, "z"), _u8(msg32, 32, "msg")
        offsets = np.ascontiguousarray(offsets, dtype=np.uint32)
        n, K = msg.shape[0], pks.shape[0]
        if offsets.shape[0] != n + 1 or int(offsets[0]) != 0 or int(offsets[-1]) != K or not (Rs.shape[0] == Ss.shape[0] == zs.shape[0] == K):
            raise ValueError("offsets must have n + 1 entries covering the participant arrays exactly")
        status = np.empty(n, dtype=np.uint8)
        bad = np.empty(n, dtype=np.uint32)
        sig = np.empty((n, 64), dtype=np.uint8)
        ok = np.empty(K, dtype=np.uint8)
        self._check(self._lib.jjs_multisig_combine(self._ctx, pks.ctypes.data, Rs.ctypes.data, Ss.ctypes.data, zs.ctypes.data, offsets.ctypes.data,
                                                   msg.ctypes.data, n, ok.ctypes.data, status.ctypes.data, bad.ctypes.data, sig.ctypes.data),
                    "jjs_multisig_combine")
        return status, bad, sig, ok

    def challenge_only(self, variant, pk, sig, msg32):
        pk, sig, msg = _u8(pk, PK_SIZE[variant], "pk"), _u8(sig, SIG_SIZE[variant], "sig"), _u8(msg32, 32, "msg")
        n = msg.shape[0]
        c = np.empty((n, 32), dtype=np.uint8)
        self._check(self._lib.jjs_challenge_only(self._ctx, variant, pk.ctypes.data, sig.ctypes.data, msg.ctypes.data, n, c.ctypes.data),
                    "jjs_challenge_only")
        return c

    def subgroup_check(self, points32, method=0):
        """is_torsion_free per point (1 / 0, 0xff = undecodable); method 0 Tate pairing, 1 scalar multiplication by r."""
        pts = _u8(points32, 32, "points")
        out = np.empty(pts.shape[0], dtype=np.uint8)
        self._check(self._lib.jjs_subgroup_check(self._ctx, pts.ctypes.data, pts.shape[0], method, out.ctypes.data), "jjs_subgroup_check")
        return out

    def fb_table_check(self, which, entries):
        """Number of the given fixed-base table entries (flat indices) that differ from their definition; which: 0 G, 1 G'."""
        idx = np.ascontiguousarray(entries, dtype=np.uint32)
        bad = np.zeros(1, dtype=np.uint32)
        self._check(self._lib.jjs_fb_table_check(self._ctx, int(which), idx.ctypes.data, idx.shape[0], bad.ctypes.data), "jjs_fb_table_check")
        return int(bad[0])

    def sign_batch(self, variant, sk32, rnd32, msg32, gen_scalar32=None):
        """(pk bytes, sig bytes) for n items; mirrors PublicKey::from(&sk) + sk.sign(rng, msg) of the reference."""
        sk, rnd, msg = _u8(sk32, 32, "sk"), _u8(rnd32, 32, "rnd"), _u8(msg32, 32, "msg")
        n = msg.shape[0]
        gsc = _u8(gen_scalar32, 32, "gen_scalar") if gen_scalar32 is not None else None
        if variant == VARGEN and gsc is None:
            raise ValueError("var-generator signing needs gen_scalar32")
        pk = np.empty((n, PK_SIZE[variant]), dtype=np.uint8)
        sig = np.empty((n, SIG_SIZE[variant]), dtype=np.uint8)
        self._check(self._lib.jjs_sign_batch(self._ctx, variant, sk.ctypes.data, rnd.ctypes.data, gsc.ctypes.data if gsc is not None else None,
                                             msg.ctypes.data, n, pk.ctypes.data, sig.ctypes.data), "jjs_sign_batch")
        return pk, sig

    def sign_aggregate_batch(self, sk32, offsets, rnd32, msg32):
        """(signer keys [K,32], signatures [n,64]) for ragged signer sets; see jjs_sign_aggregate_batch."""
        sk, rnd, msg = _u8(sk32, 32, "sk"), _u8(rnd32, 32, "rnd"), _u8(msg32, 32, "msg")
        offsets = np.ascontiguousarray(offsets, dtype=np.uint32)
        n = msg.shape[0]
        if offsets.shape[0] != n + 1 or int(offsets[-1]) != sk.shape[0] or int(offsets[0]) != 0:
            raise ValueError("offsets must have n + 1 entries covering sk32 exactly")
        pks = np.empty((sk.shape[0], 32), dtype=np.uint8)
        sig = np.empty((n, 64), dtype=np.uint8)
        self._check(self._lib.jjs_sign_aggregate_batch(self._ctx, sk.ctypes.data, offsets.ctypes.data, rnd.ctypes.data, msg.ctypes.data, n,
                                                       pks.ctypes.data, sig.ctypes.data), "jjs_sign_aggregate_batch")
        return pks, sig

    def verify_aggregate_device(self, d_pks, d_offsets, h_offsets, d_sig, d_msg, n, d_status, d_c=None, d_agg=None, stream=None, device_index=0):
        h_offsets = np.ascontiguousarray(h_offsets, dtype=np.uint32)
        self._check(self._lib.jjs_verify_aggregate_device(self._ctx, device_index, d_pks, d_offsets, h_offsets.ctypes.data, d_sig, d_msg, n,
                                                          d_status, d_c, d_agg, stream), "jjs_verify_aggregate_device")

    # ---- registered key sets ---------------------------------------------------------------------
    def keyset_create(self, kind, pks, memory_limit=None):
        """Register keys of kind SINGLE (pks: n x 32 bytes) or DOUBLE (n x 64) on every device: 8-bit key tables
        (jjs_keyset_create), or with memory_limit the widest tables, else the decoded points only, that fit in that many bytes
        per device (jjs_keyset_create_limited)."""
        if kind not in (SINGLE, DOUBLE):
            raise ValueError("key sets hold SINGLE or DOUBLE keys")
        pk = _u8(pks, PK_SIZE[kind], "pks")
        status = np.empty(pk.shape[0], dtype=np.uint8)
        handle = C.c_int(-1)
        if memory_limit is None:
            self._check(self._lib.jjs_keyset_create(self._ctx, kind, pk.ctypes.data, pk.shape[0], status.ctypes.data, C.byref(handle)), "jjs_keyset_create")
        else:
            self._check(self._lib.jjs_keyset_create_limited(self._ctx, kind, pk.ctypes.data, pk.shape[0], int(memory_limit), status.ctypes.data,
                                                            C.byref(handle)), "jjs_keyset_create_limited")
        bits, held = C.c_int(-1), C.c_uint64(0)
        self._check(self._lib.jjs_keyset_info(self._ctx, handle.value, C.byref(bits), C.byref(held)), "jjs_keyset_info")
        return KeySet(handle.value, kind, pk.shape[0], status, bits.value, held.value)

    def keyset_destroy(self, ks):
        self._check(self._lib.jjs_keyset_destroy(self._ctx, ks.handle), "jjs_keyset_destroy")

    def verify_keyed(self, ks, key_index, sig, msg32, want_challenge=False, want_bitmap=False):
        """Item i under key key_index[i] of the key set (jjs_verify_keyed).  Returns status, plus c and / or the accept bitmap
        when asked for (in that order)."""
        idx = np.ascontiguousarray(key_index, dtype=np.uint32).reshape(-1)
        sig, msg = _u8(sig, SIG_SIZE[ks.kind], "sig"), _u8(msg32, 32, "msg")
        n = msg.shape[0]
        if idx.shape[0] != n or sig.shape[0] != n:
            raise ValueError("key_index, sig and msg must describe the same number of items")
        status = np.empty(n, dtype=np.uint8)
        c = np.empty((n, 32), dtype=np.uint8) if want_challenge else None
        words = np.zeros((n + 31) // 32, dtype=np.uint32) if want_bitmap else None
        self._check(self._lib.jjs_verify_keyed(self._ctx, ks.handle, idx.ctypes.data, sig.ctypes.data, msg.ctypes.data, n, status.ctypes.data,
                                               c.ctypes.data if want_challenge else None, words.ctypes.data if want_bitmap else None),
                    "jjs_verify_keyed")
        out = [status] + ([c] if want_challenge else []) + ([words] if want_bitmap else [])
        return out[0] if len(out) == 1 else tuple(out)

    def verify_keyed_device(self, ks, d_key_index, d_sig, d_msg, n, d_status, d_c=None, stream=None, device_index=0):
        """jjs_verify_keyed_device on raw device pointers (uint32 key indices), enqueued on `stream`."""
        self._check(self._lib.jjs_verify_keyed_device(self._ctx, device_index, ks.handle, d_key_index, d_sig, d_msg, n, d_status, d_c, stream),
                    "jjs_verify_keyed_device")

    def keyset_table_check(self, ks, entries):
        """Number of the given key-table entries (flat indices, see jjs_keyset_table_check) that differ from their definition."""
        idx = np.ascontiguousarray(entries, dtype=np.uint32)
        bad = np.zeros(1, dtype=np.uint32)
        self._check(self._lib.jjs_keyset_table_check(self._ctx, ks.handle, idx.ctypes.data, idx.shape[0], bad.ctypes.data), "jjs_keyset_table_check")
        return int(bad[0])

    # ---- whole-batch verification ----------------------------------------------------------------
    @staticmethod
    def _seed_ptr(seed):
        if seed is None:
            return None, None
        s = np.ascontiguousarray(np.frombuffer(bytes(seed), dtype=np.uint8))
        if s.size != 32:
            raise ValueError("seed must be 32 bytes")
        return s, s.ctypes.data

    def verify_all(self, kind, pk, sig, msg32, seed=None) -> bool:
        """True iff every item (kind SINGLE or DOUBLE) would verify, by one random linear combination of all the equations
        (jjs_verify_all): a batch with a failing equation passes with probability at most 2^-128.  seed: None draws a fresh
        secret seed from the operating system for every call; 32 given bytes make the call deterministic (tests only)."""
        if kind not in (SINGLE, DOUBLE):
            raise ValueError("verify_all takes SINGLE or DOUBLE items")
        pk, sig, msg = _u8(pk, PK_SIZE[kind], "pk"), _u8(sig, SIG_SIZE[kind], "sig"), _u8(msg32, 32, "msg")
        n = msg.shape[0]
        if pk.shape[0] != n or sig.shape[0] != n:
            raise ValueError("pk, sig and msg must describe the same number of items")
        keep, sp = self._seed_ptr(seed)
        ok = C.c_int(0)
        self._check(self._lib.jjs_verify_all(self._ctx, kind, pk.ctypes.data, sig.ctypes.data, msg.ctypes.data, n, sp, C.byref(ok)), "jjs_verify_all")
        return bool(ok.value)

    def verify_all_device(self, kind, d_pk, d_sig, d_msg, n, d_all_valid, seed=None, stream=None, device_index=0):
        """jjs_verify_all_device on raw device pointers: the int32 verdict is written to d_all_valid on `stream`."""
        keep, sp = self._seed_ptr(seed)
        self._check(self._lib.jjs_verify_all_device(self._ctx, device_index, kind, d_pk, d_sig, d_msg, n, sp, d_all_valid, stream),
                    "jjs_verify_all_device")

    def verify_all_mixed(self, parts, seed=None) -> bool:
        """True iff every item of every part would verify (jjs_verify_mixed status 0), by one random linear combination over all
        the parts (jjs_verify_all_mixed).  parts: as for verify_mixed, (kind, pk, sig, msg) or, for AGGREGATE, (kind, pks, sig,
        msg, offsets), any of the four kinds.  seed: as for verify_all."""
        structs, keep = [], []
        for part in parts:
            kind, pk, sig, msg = part[0], part[1], part[2], part[3]
            if kind not in PK_SIZE:
                raise ValueError("unknown kind %r" % (kind,))
            pk, sig, msg = _u8(pk, PK_SIZE[kind], "pk"), _u8(sig, SIG_SIZE[kind], "sig"), _u8(msg, 32, "msg")
            n = msg.shape[0]
            off = None
            if kind == AGGREGATE:
                off = np.ascontiguousarray(part[4], dtype=np.uint32)
                if off.shape[0] != n + 1 or int(off[-1]) != pk.shape[0] or int(off[0]) != 0:
                    raise ValueError("offsets must have n + 1 entries covering pks32 exactly")
            elif pk.shape[0] != n:
                raise ValueError("pk, sig and msg must describe the same number of items")
            if sig.shape[0] != n:
                raise ValueError("pk, sig and msg must describe the same number of items")
            structs.append(_native.Part(kind, pk.ctypes.data, off.ctypes.data if off is not None else None, sig.ctypes.data, msg.ctypes.data, n,
                                        None, None, None, None))
            keep.append((pk, sig, msg, off))
        arr = (_native.Part * max(len(structs), 1))(*structs)
        keep_seed, sp = self._seed_ptr(seed)
        ok = C.c_int(0)
        self._check(self._lib.jjs_verify_all_mixed(self._ctx, arr, len(structs), sp, C.byref(ok)), "jjs_verify_all_mixed")
        return bool(ok.value)

    def verify_all_mixed_device(self, parts, d_all_valid, seed=None, stream=None, device_index=0):
        """jjs_verify_all_mixed_device on raw device pointers: parts = iterable of (kind, pk_ptr, sig_ptr, msg_ptr, n) or, for
        AGGREGATE, (kind, pks_ptr, sig_ptr, msg_ptr, n, d_offsets_ptr, h_offsets) with h_offsets the host copy of the offsets.
        The int32 verdict is written to d_all_valid on `stream`."""
        structs, hosts, keep = [], [], []
        for part in parts:
            kind, pk, sig, msg, n = part[:5]
            d_off, h_off = (part[5], np.ascontiguousarray(part[6], dtype=np.uint32)) if kind == AGGREGATE else (None, None)
            structs.append(_native.Part(kind, pk, d_off, sig, msg, n, None, None, None, None))
            hosts.append(h_off.ctypes.data if h_off is not None else None)
            keep.append(h_off)
        arr = (_native.Part * max(len(structs), 1))(*structs)
        harr = (C.c_void_p * max(len(hosts), 1))(*hosts)
        keep_seed, sp = self._seed_ptr(seed)
        self._check(self._lib.jjs_verify_all_mixed_device(self._ctx, device_index, arr, len(structs), harr, sp, d_all_valid, stream),
                    "jjs_verify_all_mixed_device")

    # ---- raw host / device pointers (pinned torch tensors, device tensors: pass .data_ptr()) ----------
    def verify_host_ptr(self, variant, pk_ptr, sig_ptr, msg_ptr, n, status_ptr, c_ptr=None):
        fn = {SINGLE: self._lib.jjs_verify_single, DOUBLE: self._lib.jjs_verify_double, VARGEN: self._lib.jjs_verify_vargen}[variant]
        self._check(fn(self._ctx, pk_ptr, sig_ptr, msg_ptr, n, status_ptr, c_ptr), "jjs_verify (host pointers)")

    def verify_device(self, variant, d_pk, d_sig, d_msg, n, d_status, d_c=None, stream=None, device_index=0):
        fn = {SINGLE: self._lib.jjs_verify_single_device, DOUBLE: self._lib.jjs_verify_double_device,
              VARGEN: self._lib.jjs_verify_vargen_device}[variant]
        self._check(fn(self._ctx, device_index, d_pk, d_sig, d_msg, n, d_status, d_c, stream), "jjs_verify (device pointers)")
