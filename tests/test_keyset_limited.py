"""Key sets within a byte budget (jjs_keyset_create_limited / jjs_keyset_info): key-window widths 8..4 and points-only sets return,
item for item, the status and challenge bytes of jjs_verify_single / jjs_verify_double with the keys written out, and the budget
picks the widest layout whose peak footprint fits.  The CPU part runs the twin (tests/hostsim/keyset_limited_twin.cpp) at every
width; the `gpu` part runs the library."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import __graft_entry__ as entry
from oracle import c_oracle as co
from tests import adversarial as adv
from tests.test_keyset import UNDECODABLE, _p, _register, _repeat_keys

LAYOUTS = [8, 7, 6, 5, 4, 0]     # key-window widths, widest first; 0: decoded points only
SMALL_LIMIT = 50_000_000          # the limited context of tests/test_memory_limit.py: ~16 MB left for key sets


def windows(kw):
    return (251 + kw - 1) // kw


def peak_bytes(kind, n_keys, kw):
    """What a key set holds on a device while it is built (include/jjschnorr_b200.h): 65 B of decoded point and flags and 32 B of
    wire key per key point, plus with tables 96 B per entry and 128 B of window base per window."""
    npts = (kind + 1) * n_keys
    return npts * (65 + 32 + (windows(kw) * (96 << (kw - 1)) + 128 * windows(kw) if kw else 0))


def held_bytes(kind, n_keys, kw):
    """What the key set keeps once built: the points, their flags and the tables."""
    npts = (kind + 1) * n_keys
    return npts * (65 + (windows(kw) * (96 << (kw - 1)) if kw else 0))


def expected_layout(bv, kind, n_keys, budget):
    """The layout jjs_keyset_create_limited picks on bv for `budget`: the widest whose peak fits the budget and what the context's
    limit leaves; None if not even the points fit."""
    room = budget if bv.test_limit is None else min(budget, bv.test_limit - bv.memory_info()["bytes_held"])
    return next((kw for kw in LAYOUTS if peak_bytes(kind, n_keys, kw) <= room), None)


def test_layout_sizes():
    """The per-key-point table sizes the header documents."""
    assert [held_bytes(0, 1, kw) - 65 for kw in LAYOUTS] == [393_216, 221_184, 129_024, 78_336, 48_384, 0]


# ---- CPU: the twin at every width -----------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def L(tmp_path_factory):
    """tests/hostsim/keyset_limited_twin.cpp (the host simulator plus the keyed stages at every width), built into a temporary
    directory."""
    src = os.path.join(entry.ROOT, "tests", "hostsim", "keyset_limited_twin.cpp")
    out = str(tmp_path_factory.mktemp("keyset_limited_twin") / "libkeyset_limited_twin.so")
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-o", out, src])
    return C.CDLL(out)


def _twin_keyed(L, kind, kw, keys, idx, sig, msg):
    n = msg.shape[0]
    ks_status = np.zeros(keys.shape[0], np.uint8)
    L.hs_keyset_build_w(kind, kw, _p(keys), C.c_size_t(keys.shape[0]), _p(ks_status))
    st, c = np.zeros(n, np.uint8), np.zeros((n, 32), np.uint8)
    L.hs_verify_keyed(_p(idx), _p(sig), _p(msg), C.c_size_t(n), _p(st), _p(c))
    return st, c, ks_status


@pytest.mark.parametrize("kw", LAYOUTS)
@pytest.mark.parametrize("vi,kind", [(0, "single"), (1, "double")])
def test_twin_at_every_width_equals_unkeyed(L, vi, kind, kw):
    """The adversarial batches of test_keyed_twin_equals_unkeyed_on_adversarial_batches (every point class on keys and signature
    points, torsion-shifted and mixed-order R, invalid and undecodable keys, unknown indices) under a key set of each layout: the
    statuses and challenges of hs_verify with the keys written out, and of the C oracle."""
    gen = {"single": co.gen_single, "double": co.gen_double}[kind]
    ver = {"single": co.verify_single, "double": co.verify_double}[kind]
    rng = np.random.default_rng(21 + vi)
    pk, sig, msg = gen(0x4E1, 96)
    pk, sig, msg, _, _ = adv.make_adversarial(kind, pk, sig, msg, seed=5, frac=0.5)
    tpk, tsig, tmsg, _ = adv.torsion_shifted_signatures(kind, 12, seed=13)
    pk, sig, msg = _repeat_keys(np.concatenate([pk, tpk]), np.concatenate([sig, tsig]), np.concatenate([msg, tmsg]), rng)
    keys, idx, written = _register(pk, rng, n_out_of_range=9)
    n = msg.shape[0]
    st, c, ks_status = _twin_keyed(L, vi, kw, keys, idx, sig, msg)
    hst, hc = np.zeros(n, np.uint8), np.zeros((n, 32), np.uint8)
    L.hs_verify(vi, _p(written), _p(sig), _p(msg), C.c_size_t(n), _p(hst), _p(hc))
    ost, oc = ver(written, sig, msg)
    assert np.array_equal(st, hst) and np.array_equal(c, hc)
    assert np.array_equal(st, ost) and np.array_equal(c, oc)
    assert (st[idx >= keys.shape[0]] == 3).all() and not c[idx >= keys.shape[0]].any()
    assert {0, 1, 2, 3} <= set(st.tolist()) and {0, 2, 3} <= set(ks_status.tolist())


@pytest.mark.parametrize("kw", [7, 6, 5, 4])
def test_twin_settles_r_by_the_equation(L, kw):
    """With tables of any width, the equation of a valid item establishes R's subgroup membership: no deferred test runs."""
    pk, sig, msg = co.gen_single(0x4E2, 24)
    pk, sig, msg = _repeat_keys(pk, sig, msg, np.random.default_rng(3), reps=2)
    keys, idx, _ = _register(pk, np.random.default_rng(4), n_out_of_range=0)
    eqs, rts = C.c_int(), C.c_int()
    L.hs_rtest_counters(C.byref(eqs), C.byref(rts))
    st, _, _ = _twin_keyed(L, 0, kw, keys, idx, sig, msg)
    L.hs_rtest_counters(C.byref(eqs), C.byref(rts))
    assert not st.any() and eqs.value == msg.shape[0] and rts.value == 0


@pytest.mark.parametrize("kw", [7, 6, 5, 4])
def test_twin_tables_equal_definition(L, kw):
    """Every entry of the tables of a valid single key and of one that fails is_valid() (the identity's table) equals
    keyed_table_entry at that width."""
    pk, _, _ = co.gen_single(0x4E3, 1)
    keys = np.ascontiguousarray(np.concatenate([pk, np.frombuffer(adv.torsion()[4], np.uint8)[None, :]]))
    status = np.zeros(2, np.uint8)
    L.hs_keyset_build_w(0, kw, _p(keys), C.c_size_t(2), _p(status))
    assert status.tolist() == [0, 2]
    a, b = (C.c_uint32 * 24)(), (C.c_uint32 * 24)()
    for p in range(2):
        for w in range(windows(kw)):
            for j in range(1, (1 << (kw - 1)) + 1):
                L.hs_keyed_entry(C.c_size_t(p), w, j, a, b)
                assert list(a) == list(b), (p, w, j)


def test_new_entry_points_on_an_inert_context():
    """jjs_init without a usable device: jjs_keyset_create_limited and jjs_keyset_info answer JJS_ERR_CUDA like every other one."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    entry.build_cuda()
    from jubjub_schnorr_b200 import _native
    lib = _native.lib()
    ctx = C.c_void_p()
    assert lib.jjs_init(None, 1, C.byref(ctx)) == -2 and ctx
    buf = (C.c_uint8 * 4096)()
    h, bits, held = C.c_int(-1), C.c_int(-7), C.c_uint64(7)
    assert lib.jjs_keyset_create_limited(ctx, 0, buf, 4, 1 << 30, buf, C.byref(h)) == -2
    assert lib.jjs_keyset_info(ctx, 0, C.byref(bits), C.byref(held)) == -2
    assert h.value == -1 and bits.value == -7 and held.value == 7
    assert lib.jjs_keyset_info(None, 0, None, None) == -1
    lib.jjs_destroy(ctx)


# ---- GPU --------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module", params=[None, 256 << 20], ids=["init", "limited"])
def bv(request):
    """A jjs_init context and a 256 MiB limited one (about 110 MB left for key sets: 8-bit tables for some 270 key points)."""
    from jubjub_schnorr_b200 import BatchVerifier
    with BatchVerifier([0], memory_limit=request.param) as v:
        v.test_limit = request.param
        yield v


def _adversarial_keyed(bv, vi, kind, n_keys, n, seed):
    """n adversarial items signed by n_keys keys plus torsion-shifted commitments, registered with their distinct keys, and unknown
    indices: (keys, idx, sig, msg, keys written out per item)."""
    from tests.test_keyset import _signed_under
    rng = np.random.default_rng(seed)
    pk, sig, msg = _signed_under(bv, vi, n_keys, n, seed=seed)
    pk, sig, msg, _, _ = adv.make_adversarial(kind, pk, sig, msg, seed=seed + 1, frac=0.4)
    tpk, tsig, tmsg, _ = adv.torsion_shifted_signatures(kind, 24, seed=seed + 2)
    pk, sig, msg = np.concatenate([pk, tpk]), np.concatenate([sig, tsig]), np.concatenate([msg, tmsg])
    keys, idx, written = _register(pk, rng, n_out_of_range=100)
    return keys, idx, sig, msg, written


@pytest.mark.gpu
@pytest.mark.parametrize("vi,kind", [(0, "single"), (1, "double")])
def test_every_layout_equals_unkeyed(bv, vi, kind):
    """Each layout, forced through a budget equal to its peak (on the limited context, the widest that its limit leaves room for):
    jjs_keyset_info reports it, bytes_held grows by its bytes and jjs_keyset_destroy returns them, and the host and device entry
    points (status, challenge, bitmap) equal the unkeyed call with the keys written out, on an adversarial batch."""
    import torch
    ver = {"single": bv.verify_single, "double": bv.verify_double}[kind]
    keys, idx, sig, msg, written = _adversarial_keyed(bv, vi, kind, 32, 1 << 11, seed=0x51 + vi)
    n = msg.shape[0]
    ust, uc = ver(written, sig, msg, True)
    assert {0, 1, 2, 3} <= set(ust.tolist())
    d_idx, d_sig, d_msg = (torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (idx.view(np.int32), sig, msg))
    seen = set()
    for kw in LAYOUTS:
        held = bv.memory_info()["bytes_held"]
        budget = peak_bytes(vi, keys.shape[0], kw)
        want = expected_layout(bv, vi, keys.shape[0], budget)
        ks = bv.keyset_create(vi, keys, memory_limit=budget)
        seen.add(ks.key_window_bits)
        try:
            assert (ks.key_window_bits, ks.bytes_per_device) == (want, held_bytes(vi, keys.shape[0], want))
            assert bv.memory_info()["bytes_held"] - held == ks.bytes_per_device
            st, c, words = bv.verify_keyed(ks, idx, sig, msg, want_challenge=True, want_bitmap=True)
            assert np.array_equal(st, ust) and np.array_equal(c, uc), kw
            assert np.array_equal(bv.unpack_bitmap(words, n), st == 0)
            d_st = torch.full((n,), 0xEE, dtype=torch.uint8, device="cuda")
            d_c = torch.full((n, 32), 0xEE, dtype=torch.uint8, device="cuda")
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            bv.verify_keyed_device(ks, d_idx.data_ptr(), d_sig.data_ptr(), d_msg.data_ptr(), n, d_st.data_ptr(), d_c.data_ptr(), stream=s.cuda_stream)
            s.synchronize()
            assert np.array_equal(d_st.cpu().numpy(), st) and np.array_equal(d_c.cpu().numpy(), c), kw
        finally:
            bv.keyset_destroy(ks)
        assert bv.memory_info()["bytes_held"] == held
    assert bv.test_limit or seen == set(LAYOUTS)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1])
def test_a_large_budget_is_keyset_create(bv, kind):
    """A budget at least the 8-bit peak gives 8-bit tables: the bytes_held delta and the outputs of jjs_keyset_create."""
    from jubjub_schnorr_b200 import workload as wl
    pks, idx, sig, msg, expected, _ = wl.make_keyed_batch(bv, kind, 100, 20_000, 0.1, seed=0x52 + kind)
    outs, deltas = [], []
    for limit in (None, peak_bytes(kind, pks.shape[0], 8), 1 << 40):
        held = bv.memory_info()["bytes_held"]
        ks = bv.keyset_create(kind, pks, memory_limit=limit)
        deltas.append(bv.memory_info()["bytes_held"] - held)
        assert (ks.key_window_bits, ks.bytes_per_device) == (8, deltas[-1])
        outs.append((ks.key_status, *bv.verify_keyed(ks, idx, sig, msg, want_challenge=True, want_bitmap=True)))
        bv.keyset_destroy(ks)
    assert np.array_equal(outs[0][1], expected) and len(set(deltas)) == 1
    for o in outs[1:]:
        assert all(np.array_equal(a, b) for a, b in zip(o, outs[0]))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1])
def test_budget_sweep(bv, kind):
    """One byte below each layout's peak picks the next narrower layout; below the points-only peak the call returns
    JJS_ERR_NOMEM, holds nothing, and the context still verifies."""
    from jubjub_schnorr_b200 import JjsError
    from jubjub_schnorr_b200 import workload as wl
    pks, idx, sig, msg, expected, _ = wl.make_keyed_batch(bv, kind, 40, 5_000, 0.1, seed=0x53 + kind)
    n_keys = pks.shape[0]
    held = bv.memory_info()["bytes_held"]
    for kw, narrower in zip(LAYOUTS[:-1], LAYOUTS[1:]):
        ks = bv.keyset_create(kind, pks, memory_limit=peak_bytes(kind, n_keys, kw) - 1)
        try:
            assert ks.key_window_bits == narrower == expected_layout(bv, kind, n_keys, peak_bytes(kind, n_keys, kw) - 1), kw
            assert bv.memory_info()["bytes_held"] - held == ks.bytes_per_device == held_bytes(kind, n_keys, narrower)
            assert np.array_equal(bv.verify_keyed(ks, idx, sig, msg), expected)
        finally:
            bv.keyset_destroy(ks)
        assert bv.memory_info()["bytes_held"] == held
    for limit in (peak_bytes(kind, n_keys, 0) - 1, 1):
        with pytest.raises(JjsError, match=r"\(-3\).*%d bytes" % peak_bytes(kind, n_keys, 0)):
            bv.keyset_create(kind, pks, memory_limit=limit)
        assert bv.memory_info()["bytes_held"] == held
    ks = bv.keyset_create(kind, pks)
    assert np.array_equal(bv.verify_keyed(ks, idx, sig, msg), expected)
    bv.keyset_destroy(ks)


@pytest.mark.gpu
@pytest.mark.parametrize("kw", LAYOUTS)
@pytest.mark.parametrize("kind", [0, 1])
def test_tables_equal_definition(bv, kind, kw):
    """jjs_keyset_table_check at every width: 10^5 random entries and one full window of each key point equal j 2^(KW w) PK
    recomputed by double-and-add (the identity's table for the invalid keys); a points-only set has no table to check."""
    from jubjub_schnorr_b200 import JjsError
    from jubjub_schnorr_b200 import workload as wl
    pks, _, _, _, _, _ = wl.make_keyed_batch(bv, kind, 100, 64, 0.0, seed=0x4E7)
    assert expected_layout(bv, kind, pks.shape[0], peak_bytes(kind, pks.shape[0], kw)) == kw
    ks = bv.keyset_create(kind, pks, memory_limit=peak_bytes(kind, pks.shape[0], kw))
    try:
        assert ks.key_window_bits == kw
        if kw == 0:
            with pytest.raises(JjsError, match=r"\(-1\).*no table"):
                bv.keyset_table_check(ks, np.zeros(4, np.uint32))
            return
        e, nw = 1 << (kw - 1), windows(kw)
        npts = pks.shape[0] * (kind + 1)
        rng = np.random.default_rng(8 + kw)
        assert bv.keyset_table_check(ks, rng.integers(0, npts * nw * e, size=100_000).astype(np.uint32)) == 0
        last = (np.arange(npts)[:, None] * (nw * e) + (nw - 1) * e + np.arange(e)[None, :]).reshape(-1)
        assert bv.keyset_table_check(ks, last.astype(np.uint32)) == 0
    finally:
        bv.keyset_destroy(ks)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1])
def test_small_limited_context(kind):
    """On the limited context of test_keyed_parity_and_refusal, the 200-key set that jjs_keyset_create refuses registers within a
    budget, verifies like the unkeyed call, and keeps bytes_held within the limit."""
    from jubjub_schnorr_b200 import BatchVerifier, JjsError
    from jubjub_schnorr_b200 import workload as wl
    with BatchVerifier([0], memory_limit=SMALL_LIMIT) as small:
        pks, idx, sig, msg, expected, _ = wl.make_keyed_batch(small, kind, 196, 3 * 4096 + 17, 0.2, seed=0x54 + kind)
        assert pks.shape[0] >= 200
        with pytest.raises(JjsError, match=r"\(-3\).*memory limit"):
            small.keyset_create(kind, pks)
        held = small.memory_info()["bytes_held"]
        ks = small.keyset_create(kind, pks, memory_limit=SMALL_LIMIT)
        assert small.memory_info()["bytes_held"] == held + ks.bytes_per_device <= SMALL_LIMIT
        assert ks.key_window_bits == next(kw for kw in LAYOUTS if peak_bytes(kind, pks.shape[0], kw) <= SMALL_LIMIT - held)
        st, c = small.verify_keyed(ks, idx, sig, msg, want_challenge=True)
        written = pks[np.minimum(idx, pks.shape[0] - 1)].copy()
        written[idx >= pks.shape[0], :32] = UNDECODABLE
        st_u, c_u = (small.verify_single if kind == 0 else small.verify_double)(written, sig, msg, True)
        assert np.array_equal(st, expected) and np.array_equal(st, st_u) and np.array_equal(c, c_u)
        small.keyset_destroy(ks)
        assert small.memory_info()["bytes_held"] == held


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [4, 0])
def test_many_keys_at_full_size(kw):
    """2^16 single keys at KW = 4 and points-only, make_keyed_batch at 2^20 items: the statuses known by construction."""
    from jubjub_schnorr_b200 import BatchVerifier
    from jubjub_schnorr_b200 import workload as wl
    with BatchVerifier([0]) as g:
        pks, idx, sig, msg, expected, _ = wl.make_keyed_batch(g, wl.SINGLE, 1 << 16, 1 << 20, 0.10, seed=0x55)
        ks = g.keyset_create(wl.SINGLE, pks, memory_limit=peak_bytes(0, pks.shape[0], kw))
        assert ks.key_window_bits == kw
        st, words = g.verify_keyed(ks, idx, sig, msg, want_bitmap=True)
        assert np.array_equal(st, expected) and np.array_equal(g.unpack_bitmap(words, msg.shape[0]), st == 0)
        g.keyset_destroy(ks)


@pytest.mark.gpu
def test_argument_errors(bv):
    """Kind 2 or 3, n_keys = 0, a budget of 0, NULL pointers, and an unknown handle to jjs_keyset_info return JJS_ERR_ARGUMENT and
    hold nothing; NULL outputs of jjs_keyset_info are allowed."""
    from jubjub_schnorr_b200 import workload as wl
    lib, ctx = bv._lib, bv._ctx
    pks, idx, sig, msg, expected, _ = wl.make_keyed_batch(bv, 0, 8, 256, 0.2, seed=0x56)
    held = bv.memory_info()["bytes_held"]
    h = C.c_int(-1)
    status = np.zeros(pks.shape[0], np.uint8)
    big = 1 << 40
    for kind in (2, 3):
        assert lib.jjs_keyset_create_limited(ctx, kind, pks.ctypes.data, 4, big, status.ctypes.data, C.byref(h)) == -1
    assert lib.jjs_keyset_create_limited(ctx, 0, pks.ctypes.data, 0, big, status.ctypes.data, C.byref(h)) == -1
    assert lib.jjs_keyset_create_limited(ctx, 0, pks.ctypes.data, 4, 0, status.ctypes.data, C.byref(h)) == -1
    assert lib.jjs_keyset_create_limited(ctx, 0, None, 4, big, status.ctypes.data, C.byref(h)) == -1
    assert lib.jjs_keyset_create_limited(ctx, 0, pks.ctypes.data, 4, big, status.ctypes.data, None) == -1
    assert lib.jjs_keyset_create_limited(None, 0, pks.ctypes.data, 4, big, status.ctypes.data, C.byref(h)) == -1
    assert h.value == -1 and bv.memory_info()["bytes_held"] == held
    bits, nbytes = C.c_int(-7), C.c_uint64(7)
    for handle in (12345, -1):
        assert lib.jjs_keyset_info(ctx, handle, C.byref(bits), C.byref(nbytes)) == -1
    ks = bv.keyset_create(0, pks, memory_limit=big)
    assert lib.jjs_keyset_info(ctx, ks.handle, None, None) == 0
    bv.keyset_destroy(ks)
    assert lib.jjs_keyset_info(ctx, ks.handle, C.byref(bits), C.byref(nbytes)) == -1
    assert (bits.value, nbytes.value) == (-7, 7)
    ks = bv.keyset_create(0, pks, memory_limit=peak_bytes(0, pks.shape[0], 0))   # the context still registers and verifies
    try:
        assert ks.key_window_bits == 0 and np.array_equal(bv.verify_keyed(ks, idx, sig, msg), expected)
    finally:
        bv.keyset_destroy(ks)


@pytest.mark.gpu
def test_two_devices():
    """A budgeted key set on a context over two devices: one width on both, and the results of the one-device layout.  Needs two
    GPUs; skipped on a one-GPU box."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from jubjub_schnorr_b200 import BatchVerifier
    from jubjub_schnorr_b200 import workload as wl
    with BatchVerifier([0, 1]) as g:
        for kind, n in ((0, 300_001), (1, 70_001)):
            pks, idx, sig, msg, expected, _ = wl.make_keyed_batch(g, kind, 512, n, 0.2, seed=0x57 + kind)
            for kw in (5, 0):
                held = [g.memory_info(k)["bytes_held"] for k in (0, 1)]
                ks = g.keyset_create(kind, pks, memory_limit=peak_bytes(kind, pks.shape[0], kw))
                assert ks.key_window_bits == kw
                assert [g.memory_info(k)["bytes_held"] - held[k] for k in (0, 1)] == [ks.bytes_per_device] * 2
                st, words = g.verify_keyed(ks, idx, sig, msg, want_bitmap=True)
                assert np.array_equal(st, expected) and np.array_equal(g.unpack_bitmap(words, n), st == 0)
                d_idx, d_sig, d_msg = (torch.from_numpy(np.ascontiguousarray(a)).to("cuda:1") for a in (idx.view(np.int32), sig, msg))
                d_st = torch.zeros(n, dtype=torch.uint8, device="cuda:1")
                with torch.cuda.device(1):
                    g.verify_keyed_device(ks, d_idx.data_ptr(), d_sig.data_ptr(), d_msg.data_ptr(), n, d_st.data_ptr(), device_index=1,
                                          stream=torch.cuda.current_stream().cuda_stream)
                    torch.cuda.synchronize()
                assert np.array_equal(d_st.cpu().numpy(), st)
                g.keyset_destroy(ks)
