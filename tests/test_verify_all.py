"""Whole-batch verification (jjs_verify_all / jjs_verify_all_device): one random linear combination of all the equations of a
batch decides "every item is valid".  The CPU part runs the twin (tests/hostsim/rlc_twin.cpp, built from the same rlc.cuh
functions as the kernels) against RFC 8439, the host simulator and the oracle's big-integer curve arithmetic; the `gpu` part
runs the library against its own per-item verification."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import __graft_entry__ as entry
from oracle import c_oracle as co
from oracle import jjs_oracle as o
from tests import adversarial as adv

KINDS = [(0, "single"), (1, "double")]


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _seed(k):
    return np.frombuffer(np.random.default_rng([0x5EED, k]).bytes(32), np.uint8).copy()


# ---- CPU: the twin ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def L(tmp_path_factory):
    """tests/hostsim/rlc_twin.cpp (the host simulator plus the combination's stages), built into a temporary directory."""
    src = os.path.join(entry.ROOT, "tests", "hostsim", "rlc_twin.cpp")
    out = str(tmp_path_factory.mktemp("rlc_twin") / "librlc_twin.so")
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-o", out, src])
    lib = C.CDLL(out)
    lib.hs_chacha20_block.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
    lib.hs_rlc_msm.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_uint32, C.c_void_p]
    lib.hs_rlc_msm.restype = C.c_int
    lib.hs_verify_all.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int)]
    lib.hs_verify.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
    return lib


def _twin_all(L, vi, pk, sig, msg, seed, c=6, seg=4):
    ok = C.c_int(-1)
    L.hs_verify_all(vi, _p(pk), _p(sig), _p(msg), msg.shape[0], _p(seed), c, seg, C.byref(ok))
    return ok.value


def test_twin_chacha20_matches_rfc8439_block_vector(L):
    """RFC 8439 section 2.3.2: key 00..1f, nonce 00:00:00:09:00:00:00:4a:00:00:00:00, block counter 1."""
    key = np.frombuffer(bytes(range(32)), "<u4").copy()
    nonce = np.frombuffer(bytes.fromhex("000000090000004a00000000"), "<u4").copy()
    out = np.zeros(16, np.uint32)
    L.hs_chacha20_block(_p(key), 1, _p(nonce), _p(out))
    assert out.astype("<u4").tobytes().hex() == (
        "10f1e7e4d13b5915500fdd1fa32071c4c7d1f4c733c068030422aa9ac3d46c4e"
        "d2826446079faa0914c2d705d98b02a2b5129cd1de164eb9cbd083e8a2503c4e")


@pytest.mark.parametrize("n,c,seg", [(1, 6, 4), (7, 6, 4), (33, 7, 5), (64, 8, 4), (64, 16, 32)])
def test_twin_msm_equals_term_by_term_sum(L, n, c, seg):
    """sum k_i P_i through digits, sort, segments with their merge levels, running-sum slices and Horner equals the sum of
    pmul(P_i, k_i) with the oracle's big integers.  Repeated points and scalars make buckets that span many segments."""
    rng = np.random.default_rng([n, c, seg])
    pts, ks, ref = [], [], o.IDENTITY
    for i in range(n):
        P = o.pmul(o.G, int(rng.integers(1, 1 << 62))) if i % 5 else o.pmul(o.G_NUMS, 3)
        k = int.from_bytes(rng.bytes(32), "little") % (1 << 252) if i % 3 else (1 << 251) - 1
        pts.append(o.point_to_bytes(P))
        ks.append(k.to_bytes(32, "little"))
        ref = o.padd(ref, o.pmul(P, k))
    out = np.zeros(32, np.uint8)
    pa, ka = np.frombuffer(b"".join(pts), np.uint8).copy(), np.frombuffer(b"".join(ks), np.uint8).copy()
    assert L.hs_rlc_msm(_p(pa), _p(ka), n, c, seg, 32, _p(out)) == 0
    assert out.tobytes() == o.point_to_bytes(ref)


def _adversarial_items(kind, seed):
    """One item per class of tests/adversarial.py (make_adversarial over exactly as many items as it has classes, every
    item tampered) plus torsion-shifted commitments of order 2, 4 and 8."""
    gen = {"single": co.gen_single, "double": co.gen_double}[kind]
    n_classes = len(adv.POINT_CLASSES) * (2 if kind == "single" else 4) + 8
    pk, sig, msg = gen(0xA11 + seed, n_classes)
    pk, sig, msg, _, _ = adv.make_adversarial(kind, pk, sig, msg, seed=seed, frac=1.0)
    tpk, tsig, tmsg, _ = adv.torsion_shifted_signatures(kind, 6, seed=seed + 1)
    return np.concatenate([pk, tpk]), np.concatenate([sig, tsig]), np.concatenate([msg, tmsg])


@pytest.mark.parametrize("vi,kind", KINDS)
def test_twin_verify_all_equals_all_statuses_zero(L, vi, kind):
    """Every adversarial class planted singly at the first, middle and last position of an otherwise valid batch, for several
    seeds: the twin's verdict is all(hs_verify status == 0) (and the oracle's); valid batches pass for every seed."""
    gen = {"single": co.gen_single, "double": co.gen_double}[kind]
    ver = {"single": co.verify_single, "double": co.verify_double}[kind]
    bpk, bsig, bmsg = _adversarial_items(kind, seed=3)
    vpk, vsig, vmsg = gen(0xB0B + vi, 9)
    for s in range(3):
        assert _twin_all(L, vi, vpk, vsig, vmsg, _seed(s)) == 1
    rejected = 0
    for j in range(bmsg.shape[0]):
        for pos, s in ((0, 0), (4, 1), (8, 2)):
            pk, sig, msg = vpk.copy(), vsig.copy(), vmsg.copy()
            pk[pos], sig[pos], msg[pos] = bpk[j], bsig[j], bmsg[j]
            hst, hc = np.zeros(9, np.uint8), np.zeros((9, 32), np.uint8)
            L.hs_verify(vi, _p(pk), _p(sig), _p(msg), 9, _p(hst), _p(hc))
            ost, _ = ver(pk, sig, msg)
            assert np.array_equal(hst, ost)
            want = int(bool(np.all(hst == 0)))
            assert _twin_all(L, vi, pk, sig, msg, _seed(10 * j + s)) == want, (j, pos)
            rejected += 1 - want
    assert rejected == 3 * bmsg.shape[0]   # every planted item is invalid


def test_twin_cancelling_errors_are_rejected(L):
    """u_1 + d and u_2 - d leave errors dG and -dG, which cancel in a plain sum but not under independent weights."""
    pk, sig, msg = co.gen_single(0xCA, 5)
    d = 0x1234567
    for i, sgn in ((1, 1), (3, -1)):
        u = (int.from_bytes(sig[i, :32].tobytes(), "little") + sgn * d) % o.R_ORDER
        sig[i, :32] = np.frombuffer(o.le32(u), np.uint8)
    for s in range(5):
        assert _twin_all(L, 0, pk, sig, msg, _seed(100 + s)) == 0


def test_twin_empty_batch_is_valid(L):
    e = np.zeros((0, 32), np.uint8)
    assert _twin_all(L, 0, e, np.zeros((0, 64), np.uint8), e, _seed(0)) == 1


def test_new_entry_points_refuse_an_inert_context_and_other_kinds():
    """Without a usable device jjs_init hands back an inert context: both entry points answer JJS_ERR_CUDA for single and
    double items and JJS_ERR_ARGUMENT for kinds 2 and 3, and the reason of the failed init survives."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    entry.build_cuda()
    from jubjub_schnorr_b200 import _native
    lib = _native.lib()
    ctx = C.c_void_p()
    assert lib.jjs_init(None, 1, C.byref(ctx)) == -2 and ctx
    buf = (C.c_uint8 * 4096)()
    ok = C.c_int(7)
    for kind, want in ((0, -2), (1, -2), (2, -1), (3, -1)):
        assert lib.jjs_verify_all(ctx, kind, buf, buf, buf, 4, None, C.byref(ok)) == want, kind
        assert lib.jjs_verify_all_device(ctx, 0, kind, buf, buf, buf, 4, None, buf, None) == want, kind
    assert b"no CUDA device" in lib.jjs_last_error(ctx)
    lib.jjs_destroy(ctx)


# ---- GPU ----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def bv():
    from jubjub_schnorr_b200 import BatchVerifier
    with BatchVerifier([0]) as b:
        yield b


@pytest.fixture(scope="module")
def small():
    """A limited context at the floor: 2^12 items per pass, 2^11 per scratch half."""
    from jubjub_schnorr_b200 import BatchVerifier
    with BatchVerifier([0], memory_limit=50_000_000) as b:
        assert b.memory_info()["items_in_flight"] == 1 << 12
        yield b


_VALID = {}


def _valid(bv, vi, n):
    from jubjub_schnorr_b200 import workload as wl
    if (vi, n) not in _VALID:
        _VALID[(vi, n)] = wl.make_valid(bv, vi, n, seed=0xA11 + n)
    return _VALID[(vi, n)]


def _plant(batch, items, j, pos):
    pk, sig, msg = (a.copy() for a in batch)
    pk[pos], sig[pos], msg[pos] = items[0][j], items[1][j], items[2][j]
    return pk, sig, msg


@pytest.mark.gpu
@pytest.mark.parametrize("vi,kind", KINDS)
def test_valid_batches_are_accepted(bv, vi, kind):
    for n in (0, 1, 2, 33, 4097, 3 * (1 << 12) + 5, 1 << 20):
        pk, sig, msg = _valid(bv, vi, n)
        assert bv.verify_all(vi, pk, sig, msg, seed=_seed(n).tobytes()) is True, n
        assert bv.verify_all(vi, pk, sig, msg) is True, n


@pytest.mark.gpu
@pytest.mark.parametrize("vi,kind", KINDS)
def test_any_bad_item_is_rejected(bv, small, vi, kind):
    """Each adversarial class planted at the first and last position; a sample across the first-slice / sub-chunk boundary of a
    jjs_init context (2^17) and across a pass boundary of a limited context at the floor (2^11)."""
    bad = _adversarial_items(kind, seed=7)
    nb = bad[2].shape[0]
    base = _valid(bv, vi, 4097)
    for j in range(nb):
        for pos in (0, 4096):
            assert bv.verify_all(vi, *_plant(base, bad, j, pos), seed=_seed(j).tobytes()) is False, (j, pos)
    big = _valid(bv, vi, (1 << 17) + 1024)
    for j in range(0, nb, 5):
        for pos in ((1 << 17) - 1, 1 << 17):
            assert bv.verify_all(vi, *_plant(big, bad, j, pos)) is False, (j, pos)
    mid = _valid(bv, vi, 3 * (1 << 12) + 5)
    assert small.verify_all(vi, *mid) is True
    for j in range(nb):
        pos = ((1 << 11) - 1, 1 << 11, 1 << 12)[j % 3]
        assert small.verify_all(vi, *_plant(mid, bad, j, pos)) is False, (j, pos)


def _same_key_pair(bv, delta):
    """Two single items signed with one secret key, their u shifted by +delta and -delta (errors delta G and -delta G)."""
    from jubjub_schnorr_b200 import workload as wl
    rng = np.random.default_rng(0xCA)
    sk = np.repeat(wl.random_scalars(rng, 1, 251), 2, axis=0)
    sk[:, 0] |= 1
    rnd, msg = wl.random_scalars(rng, 2, 251), wl.random_scalars(rng, 2, 250)
    pk, sig = bv.sign_batch(0, sk, rnd, msg)
    for i, sgn in ((0, 1), (1, -1)):
        u = (int.from_bytes(sig[i, :32].tobytes(), "little") + sgn * delta) % o.R_ORDER
        sig[i, :32] = np.frombuffer(o.le32(u), np.uint8)
    return pk, sig, msg


@pytest.mark.gpu
def test_cancelling_errors_are_rejected(bv):
    pk, sig, msg = _same_key_pair(bv, 0xD17A)
    assert not np.any(bv.verify_single(pk, sig, msg) == 0)
    vpk, vsig, vmsg = _valid(bv, 0, 33)
    pk, sig, msg = np.concatenate([vpk, pk]), np.concatenate([vsig, sig]), np.concatenate([vmsg, msg])
    for s in range(20):
        assert bv.verify_all(0, pk, sig, msg, seed=_seed(200 + s).tobytes()) is False, s


@pytest.mark.gpu
def test_torsion_shifted_and_mixed_order_commitments_are_rejected(bv):
    from jubjub_schnorr_b200 import workload as wl
    for vi, kind in KINDS:
        tpk, tsig, tmsg, _ = adv.torsion_shifted_signatures(kind, 6, seed=41)
        base = _valid(bv, vi, 33)
        for j in range(6):
            assert bv.verify_all(vi, *_plant(base, (tpk, tsig, tmsg), j, 17), seed=_seed(j).tobytes()) is False
    pk, sig, msg = (a.copy() for a in _valid(bv, 1, 33))
    for enc in wl.MIXED_ORDER:
        s2 = sig.copy()
        s2[5, 64:96] = np.frombuffer(enc.tobytes(), np.uint8)
        assert bv.verify_all(1, pk, s2, msg) is False


@pytest.mark.gpu
@pytest.mark.parametrize("vi,kind", KINDS)
def test_agrees_with_the_per_item_path(bv, vi, kind):
    from jubjub_schnorr_b200 import workload as wl
    ver = {0: bv.verify_single, 1: bv.verify_double}[vi]
    for k, frac in enumerate((0.0, None, 0.1)):
        pk, sig, msg = _valid(bv, vi, 20000)
        if frac is None:
            pk, sig, msg, _, _ = wl.invalidate(vi, pk, sig, msg, 1 / 20000, seed=k)
        elif frac:
            pk, sig, msg, _, _ = wl.invalidate(vi, pk, sig, msg, frac, seed=k)
        want = bool(np.all(ver(pk, sig, msg) == 0))
        assert want == (frac == 0.0)
        assert bv.verify_all(vi, pk, sig, msg, seed=_seed(k).tobytes()) is want


@pytest.mark.gpu
def test_no_memory_growth(bv, small):
    for b in (small, bv):
        pk, sig, msg = _valid(bv, 1, 4097)
        b.verify_double(pk, sig, msg)   # a jjs_init context has its scratch after its first verification
        before = b.memory_info()
        assert b.verify_all(1, pk, sig, msg) is True
        assert b.memory_info() == before


@pytest.mark.gpu
@pytest.mark.parametrize("vi,kind", KINDS)
def test_device_entry_point_on_a_side_stream(bv, vi, kind):
    import torch
    dev = torch.device("cuda:0")
    for n, bad in ((0, False), (5000, False), ((1 << 19) + 77, False), ((1 << 19) + 77, True)):
        pk, sig, msg = (a.copy() for a in _valid(bv, vi, max(n, 1)))
        if n == 0:
            pk, sig, msg = pk[:0], sig[:0], msg[:0]
        if bad:
            sig[n - 1, 0] ^= 1
        want = bv.verify_all(vi, pk, sig, msg, seed=_seed(n).tobytes())
        assert want is (not bad)
        tp, ts, tm = (torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (pk, sig, msg))
        out = torch.full((1,), -1, dtype=torch.int32, device=dev)
        s = torch.cuda.Stream(device=dev)
        s.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(s):
            bv.verify_all_device(vi, tp.data_ptr(), ts.data_ptr(), tm.data_ptr(), n, out.data_ptr(), seed=_seed(n).tobytes(),
                                 stream=s.cuda_stream)
        s.synchronize()
        assert int(out.item()) == int(want), n


@pytest.mark.gpu
def test_two_devices():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from jubjub_schnorr_b200 import BatchVerifier
    with BatchVerifier([0, 1]) as g:
        pk, sig, msg = _valid(g, 0, 40000)
        assert g.verify_all(0, pk, sig, msg) is True
        sig = sig.copy()
        sig[39999, 0] ^= 1
        assert g.verify_all(0, pk, sig, msg) is False
