"""Registered key sets (jjs_keyset_create / jjs_verify_keyed): for every item, the keyed path returns the status byte and challenge
bytes that jjs_verify_single / jjs_verify_double return for the same item with its key written out, on valid and adversarial
inputs; an index out of range behaves like a key that does not decode.  The CPU part runs the twin of the keyed pipeline
(tests/hostsim/keyset_twin.cpp, built from the kernels' stage functions); the `gpu` part runs the library."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import __graft_entry__ as entry
from oracle import c_oracle as co
from tests import adversarial as adv

UNDECODABLE = np.frombuffer(adv.noncanonical_v_encoding(np.random.default_rng(0)), np.uint8)   # what an unknown index stands for


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _register(pk_items, rng, n_out_of_range):
    """Key set made of the distinct keys of a batch (in a shuffled order) and each item's index into it; n_out_of_range items get
    an index past the end.  Returns (keys, key_index, keys written out per item with UNDECODABLE for the unknown indices)."""
    uniq, inv = np.unique(pk_items, axis=0, return_inverse=True)
    perm = rng.permutation(uniq.shape[0])
    keys = np.ascontiguousarray(uniq[perm])
    idx = np.argsort(perm)[inv.reshape(-1)].astype(np.uint32)
    out = rng.choice(idx.shape[0], size=n_out_of_range, replace=False)
    idx[out] = keys.shape[0] + rng.integers(0, 1 << 31, size=n_out_of_range).astype(np.uint32)
    written = keys[np.minimum(idx, keys.shape[0] - 1)].copy()
    written[out, :32] = UNDECODABLE
    return keys, idx, written


def _repeat_keys(pk, sig, msg, rng, reps=3):
    """Items repeated `reps` times in a random order, so that keys recur within the batch."""
    order = rng.permutation(np.repeat(np.arange(msg.shape[0]), reps))
    return pk[order], sig[order], msg[order]


# ---- CPU: the twin ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def L(tmp_path_factory):
    """tests/hostsim/keyset_twin.cpp (the host simulator plus the keyed stages), built into a temporary directory."""
    src = os.path.join(entry.ROOT, "tests", "hostsim", "keyset_twin.cpp")
    out = str(tmp_path_factory.mktemp("keyset_twin") / "libkeyset_twin.so")
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-o", out, src])
    return C.CDLL(out)


def _twin_keyed(L, kind, keys, idx, sig, msg):
    n = msg.shape[0]
    ks_status = np.zeros(keys.shape[0], np.uint8)
    L.hs_keyset_build(kind, _p(keys), C.c_size_t(keys.shape[0]), _p(ks_status))
    st, c = np.zeros(n, np.uint8), np.zeros((n, 32), np.uint8)
    L.hs_verify_keyed(_p(idx), _p(sig), _p(msg), C.c_size_t(n), _p(st), _p(c))
    return st, c, ks_status


@pytest.mark.parametrize("vi,kind", [(0, "single"), (1, "double")])
def test_keyed_twin_equals_unkeyed_on_adversarial_batches(L, vi, kind):
    """Adversarial items (every point class on keys and signature points, torsion-shifted commitments, mixed-order R) under a key
    set of their distinct keys, valid, invalid and undecodable alike, plus unknown indices: the keyed twin gives the statuses
    and challenges of hs_verify with the keys written out, and of the C oracle."""
    gen = {"single": co.gen_single, "double": co.gen_double}[kind]
    ver = {"single": co.verify_single, "double": co.verify_double}[kind]
    rng = np.random.default_rng(21 + vi)
    pk, sig, msg = gen(0x4E1, 96)
    pk, sig, msg, _, _ = adv.make_adversarial(kind, pk, sig, msg, seed=5, frac=0.5)
    tpk, tsig, tmsg, _ = adv.torsion_shifted_signatures(kind, 12, seed=13)
    pk, sig, msg = _repeat_keys(np.concatenate([pk, tpk]), np.concatenate([sig, tsig]), np.concatenate([msg, tmsg]), rng)
    keys, idx, written = _register(pk, rng, n_out_of_range=9)
    n = msg.shape[0]
    st, c, ks_status = _twin_keyed(L, vi, keys, idx, sig, msg)
    hst, hc = np.zeros(n, np.uint8), np.zeros((n, 32), np.uint8)
    L.hs_verify(vi, _p(written), _p(sig), _p(msg), C.c_size_t(n), _p(hst), _p(hc))
    ost, oc = ver(written, sig, msg)
    assert np.array_equal(st, hst) and np.array_equal(c, hc)
    assert np.array_equal(st, ost) and np.array_equal(c, oc)
    assert (st[idx >= keys.shape[0]] == 3).all() and not c[idx >= keys.shape[0]].any()
    assert {0, 1, 2, 3} <= set(st.tolist())
    assert {0, 2, 3} <= set(ks_status.tolist())


def test_keyed_twin_settles_r_by_the_equation(L):
    """On valid items the equation establishes R's subgroup membership: no deferred test is run."""
    pk, sig, msg = co.gen_single(0x4E2, 24)
    pk, sig, msg = _repeat_keys(pk, sig, msg, np.random.default_rng(3), reps=2)
    keys, idx, _ = _register(pk, np.random.default_rng(4), n_out_of_range=0)
    eqs, rts = C.c_int(), C.c_int()
    L.hs_rtest_counters(C.byref(eqs), C.byref(rts))
    st, _, _ = _twin_keyed(L, 0, keys, idx, sig, msg)
    L.hs_rtest_counters(C.byref(eqs), C.byref(rts))
    assert not st.any() and eqs.value == msg.shape[0] and rts.value == 0


def test_keyed_twin_tables_equal_definition(L):
    """Every entry of the tables of two keys (a valid single key, and one that fails is_valid(), whose table is the
    identity's) equals keyed_table_entry."""
    pk, _, _ = co.gen_single(0x4E3, 1)
    keys = np.ascontiguousarray(np.concatenate([pk, np.frombuffer(adv.torsion()[4], np.uint8)[None, :]]))
    status = np.zeros(2, np.uint8)
    L.hs_keyset_build(0, _p(keys), C.c_size_t(2), _p(status))
    assert status.tolist() == [0, 2]
    a, b = (C.c_uint32 * 24)(), (C.c_uint32 * 24)()
    for p in range(2):
        for w in range(32):
            for j in range(1, 129):
                L.hs_keyed_entry(C.c_size_t(p), w, j, a, b)
                assert list(a) == list(b), (p, w, j)


def test_keyset_entry_points_on_an_inert_context():
    """jjs_init without a usable device: the key-set entry points answer JJS_ERR_CUDA like every other one."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    entry.build_cuda()
    from jubjub_schnorr_b200 import _native
    lib = _native.lib()
    ctx = C.c_void_p()
    assert lib.jjs_init(None, 1, C.byref(ctx)) == -2 and ctx
    buf = (C.c_uint8 * 4096)()
    h = C.c_int(-1)
    calls = [
        lambda: lib.jjs_keyset_create(ctx, 0, buf, 4, buf, C.byref(h)),
        lambda: lib.jjs_keyset_destroy(ctx, 0),
        lambda: lib.jjs_verify_keyed(ctx, 0, buf, buf, buf, 4, buf, None, None),
        lambda: lib.jjs_verify_keyed_device(ctx, 0, 0, buf, buf, buf, 4, buf, None, None),
        lambda: lib.jjs_keyset_table_check(ctx, 0, buf, 4, buf),
    ]
    for i, call in enumerate(calls):
        assert call() == -2, i
    assert h.value == -1
    assert b"no CUDA device" in lib.jjs_last_error(ctx)
    lib.jjs_destroy(ctx)


# ---- GPU --------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def bv():
    from jubjub_schnorr_b200 import BatchVerifier
    with BatchVerifier([0]) as v:
        yield v


def _signed_under(bv, kind, n_keys, n, seed):
    """n valid items signed by n_keys keys (drawn uniformly): (per-item keys, sig, msg)."""
    from jubjub_schnorr_b200 import workload as wl
    rng = np.random.default_rng(seed)
    sk = wl.random_scalars(rng, n_keys, 251)
    sk[:, 0] |= 1
    idx = rng.integers(0, n_keys, size=n)
    rnd, msg = wl.random_scalars(rng, n, 251), wl.random_scalars(rng, n, 254)
    pk, sig = bv.sign_batch(kind, sk[idx], rnd, msg)
    return pk, sig, msg


@pytest.mark.gpu
@pytest.mark.parametrize("vi,kind", [(0, "single"), (1, "double")])
def test_keyed_equals_unkeyed_on_adversarial_batches(bv, vi, kind):
    """2^16 adversarial items signed by 1 024 keys, registered with every tampered key they carry, plus torsion-shifted
    commitments and unknown indices: status and challenge bytes identical to the unkeyed call with the keys written out, and a
    sample identical to the C oracle."""
    ver = {"single": bv.verify_single, "double": bv.verify_double}[kind]
    over = {"single": co.verify_single, "double": co.verify_double}[kind]
    rng = np.random.default_rng(31 + vi)
    pk, sig, msg = _signed_under(bv, vi, 1024, 1 << 16, seed=vi)
    pk, sig, msg, _, _ = adv.make_adversarial(kind, pk, sig, msg, seed=6, frac=0.4)
    tpk, tsig, tmsg, _ = adv.torsion_shifted_signatures(kind, 48, seed=17)
    pk, sig, msg = np.concatenate([pk, tpk]), np.concatenate([sig, tsig]), np.concatenate([msg, tmsg])
    keys, idx, written = _register(pk, rng, n_out_of_range=300)
    ks = bv.keyset_create(vi, keys)
    try:
        st, c = bv.verify_keyed(ks, idx, sig, msg, want_challenge=True)
        ust, uc = ver(written, sig, msg, True)
        assert np.array_equal(st, ust) and np.array_equal(c, uc)
        assert (st[idx >= keys.shape[0]] == 3).all() and (st[-48:] >= 2).all()
        assert {0, 1, 2, 3} <= set(st.tolist()) and {0, 2, 3} <= set(ks.key_status.tolist())
        sample = np.concatenate([np.nonzero(idx >= keys.shape[0])[0], rng.choice(msg.shape[0], size=4000, replace=False),
                                 np.arange(msg.shape[0] - 48, msg.shape[0])])
        ost, oc = over(written[sample], sig[sample], msg[sample])
        assert np.array_equal(st[sample], ost) and np.array_equal(c[sample], oc)
    finally:
        bv.keyset_destroy(ks)


@pytest.mark.gpu
def test_keyed_workload_at_full_size(bv):
    """make_keyed_batch at 2^20 + 7 items (several sub-chunks, n not a multiple of 32): statuses equal the expectation known by
    construction, challenges equal the unkeyed call's, the bitmap is status == 0 packed; n = 0 and 1 work."""
    from jubjub_schnorr_b200 import workload as wl
    n = (1 << 20) + 7
    pks, idx, sig, msg, expected, cls = wl.make_keyed_batch(bv, wl.SINGLE, 1024, n, 0.10, seed=0x4E5)
    assert set(np.unique(cls).tolist()) == set(range(-1, len(wl.KEYED_CLASSES)))
    ks = bv.keyset_create(wl.SINGLE, pks)
    try:
        assert ks.key_status[:1025].tolist() == [0] * 1025 and (ks.key_status[1025:] != 0).all()
        st, c, words = bv.verify_keyed(ks, idx, sig, msg, want_challenge=True, want_bitmap=True)
        assert np.array_equal(st, expected)
        assert np.array_equal(bv.unpack_bitmap(words, n), st == 0) and int(words[-1]) >> (n % 32) == 0
        written = pks[np.minimum(idx, pks.shape[0] - 1)].copy()
        written[idx >= pks.shape[0]] = UNDECODABLE
        ust, uc = bv.verify_single(written, sig, msg, True)
        assert np.array_equal(st, ust) and np.array_equal(c, uc)
        for m in (0, 1, 33):
            st_m, c_m = bv.verify_keyed(ks, idx[:m], sig[:m], msg[:m], want_challenge=True)
            assert np.array_equal(st_m, st[:m]) and np.array_equal(c_m, c[:m])
        assert np.array_equal(bv.verify_keyed(ks, idx[:0], sig[:0], msg[:0], want_bitmap=True)[1], np.zeros(0, np.uint32))
    finally:
        bv.keyset_destroy(ks)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1])
def test_keyed_device_entry_on_a_side_stream(bv, kind):
    """jjs_verify_keyed_device on torch tensors, enqueued on a non-default stream: the bytes of the host-buffer call."""
    import torch
    from jubjub_schnorr_b200 import workload as wl
    n = 600_001 if kind == 0 else 300_001
    pks, idx, sig, msg, expected, _ = wl.make_keyed_batch(bv, kind, 64, n, 0.10, seed=0x4E6 + kind)
    ks = bv.keyset_create(kind, pks)
    try:
        st, c = bv.verify_keyed(ks, idx, sig, msg, want_challenge=True)
        assert np.array_equal(st, expected)
        d_idx, d_sig, d_msg = (torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (idx.view(np.int32), sig, msg))
        d_st = torch.full((n,), 0xEE, dtype=torch.uint8, device="cuda")
        d_c = torch.full((n, 32), 0xEE, dtype=torch.uint8, device="cuda")
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        bv.verify_keyed_device(ks, d_idx.data_ptr(), d_sig.data_ptr(), d_msg.data_ptr(), n, d_st.data_ptr(), d_c.data_ptr(), stream=s.cuda_stream)
        s.synchronize()
        assert np.array_equal(d_st.cpu().numpy(), st) and np.array_equal(d_c.cpu().numpy(), c)
    finally:
        bv.keyset_destroy(ks)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1])
def test_keyset_tables_equal_definition(bv, kind):
    """jjs_keyset_table_check: 10^5 random entries of the built tables, and every entry of one window of each key point, equal
    j 2^(8 w) PK recomputed by double-and-add (the identity's table for the invalid keys)."""
    from jubjub_schnorr_b200 import workload as wl
    pks, _, _, _, _, _ = wl.make_keyed_batch(bv, kind, 100, 64, 0.0, seed=0x4E7)
    ks = bv.keyset_create(kind, pks)
    try:
        total = pks.shape[0] * (kind + 1) * 4096
        rng = np.random.default_rng(8)
        assert bv.keyset_table_check(ks, rng.integers(0, total, size=100_000).astype(np.uint32)) == 0
        window = (np.arange(pks.shape[0] * (kind + 1))[:, None] * 4096 + 31 * 128 + np.arange(128)[None, :]).reshape(-1)
        assert bv.keyset_table_check(ks, window.astype(np.uint32)) == 0
    finally:
        bv.keyset_destroy(ks)


@pytest.mark.gpu
def test_keyset_argument_errors(bv):
    """A destroyed or unknown handle, kind VARGEN and n_keys = 0 return JJS_ERR_ARGUMENT; the context stays usable."""
    from jubjub_schnorr_b200 import JjsError, KeySet
    from jubjub_schnorr_b200 import workload as wl
    lib, ctx = bv._lib, bv._ctx
    pks, idx, sig, msg, expected, _ = wl.make_keyed_batch(bv, 0, 8, 256, 0.2, seed=0x4E8)
    h = C.c_int(-1)
    status = np.zeros(pks.shape[0], np.uint8)
    assert lib.jjs_keyset_create(ctx, 2, pks.ctypes.data, 4, status.ctypes.data, C.byref(h)) == -1
    assert lib.jjs_keyset_create(ctx, 0, pks.ctypes.data, 0, status.ctypes.data, C.byref(h)) == -1 and h.value == -1
    ks = bv.keyset_create(0, pks)
    bv.keyset_destroy(ks)
    out = np.zeros(256, np.uint8)
    bad = np.zeros(1, np.uint32)
    for handle in (ks.handle, 12345, -1):
        assert lib.jjs_verify_keyed(ctx, handle, idx.ctypes.data, sig.ctypes.data, msg.ctypes.data, 256, out.ctypes.data, None, None) == -1
        assert lib.jjs_verify_keyed_device(ctx, 0, handle, idx.ctypes.data, sig.ctypes.data, msg.ctypes.data, 256, out.ctypes.data, None, None) == -1
        assert lib.jjs_keyset_table_check(ctx, handle, idx.ctypes.data, 4, bad.ctypes.data) == -1
        assert lib.jjs_keyset_destroy(ctx, handle) == -1
    with pytest.raises(JjsError):
        bv.verify_keyed(KeySet(ks.handle, 0, ks.n_keys, ks.key_status), idx, sig, msg)
    ks = bv.keyset_create(0, pks)      # a fresh handle still works, and so do the unkeyed calls
    try:
        assert np.array_equal(bv.verify_keyed(ks, idx, sig, msg), expected)
    finally:
        bv.keyset_destroy(ks)


@pytest.mark.gpu
def test_keyed_on_two_devices():
    """A key set on a context over two devices: the batch is sharded and each device uses its own copy of the tables.  Needs two
    GPUs; skipped on a one-GPU box."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from jubjub_schnorr_b200 import BatchVerifier
    from jubjub_schnorr_b200 import workload as wl
    with BatchVerifier([0, 1]) as g:
        for kind, n in ((0, 300_001), (1, 70_001)):
            pks, idx, sig, msg, expected, _ = wl.make_keyed_batch(g, kind, 512, n, 0.2, seed=0x4E9 + kind)
            ks = g.keyset_create(kind, pks)
            st, c, words = g.verify_keyed(ks, idx, sig, msg, want_challenge=True, want_bitmap=True)
            assert np.array_equal(st, expected) and np.array_equal(g.unpack_bitmap(words, n), st == 0)
            d_idx, d_sig, d_msg = (torch.from_numpy(np.ascontiguousarray(a)).to("cuda:1") for a in (idx.view(np.int32), sig, msg))
            d_st = torch.zeros(n, dtype=torch.uint8, device="cuda:1")
            with torch.cuda.device(1):
                g.verify_keyed_device(ks, d_idx.data_ptr(), d_sig.data_ptr(), d_msg.data_ptr(), n, d_st.data_ptr(), device_index=1,
                                      stream=torch.cuda.current_stream().cuda_stream)
                torch.cuda.synchronize()
            assert np.array_equal(d_st.cpu().numpy(), st)
            g.keyset_destroy(ks)
