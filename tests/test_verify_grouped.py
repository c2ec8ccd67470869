"""Grouped verification (jjs_verify_grouped / jjs_verify_grouped_device): per-item results from one random linear combination
per group of consecutive items, with the per-item equations only in groups whose combination fails.

The CPU part runs the twin (tests/hostsim/rlc_group_twin.cpp) against the C oracle item by item; the `gpu` part runs the library
against its own per-item verification (jjs_verify_mixed) and the oracle."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import __graft_entry__ as entry
from oracle import c_oracle as co
from oracle import jjs_oracle as o
from tests import adversarial as adv
from tests.test_verify_all_mixed import (AGGREGATE, DOUBLE, SINGLE, VARGEN, _agg_items, _agg_part, _bad_aggregate_items, _bad_wire_items, _le, _p,
                                         _plant, _seed, _valid_parts)

GROUP_MAX = 1 << 16   # the header's bound on a group


# ---- CPU: the twin ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def L(tmp_path_factory):
    src = os.path.join(entry.ROOT, "tests", "hostsim", "rlc_group_twin.cpp")
    out = str(tmp_path_factory.mktemp("rlc_group_twin") / "librlc_group_twin.so")
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-o", out, src])
    lib = C.CDLL(out)
    vp = C.c_void_p
    lib.hs_verify_grouped.argtypes = [C.c_size_t, vp, vp, vp, vp, vp, vp, vp, C.c_size_t, C.c_int, C.c_int, vp, vp, vp, vp]
    lib.hs_verify_grouped.restype = C.c_long
    lib.hs_verify_all_mixed.argtypes = [C.c_size_t, vp, vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.POINTER(C.c_int)]
    return lib


def _twin(L, parts, seed, g, c=6, seg=4):
    """(status, c32, verdicts, fallback) of the twin, all parts concatenated"""
    k = len(parts)
    keep = [tuple(np.ascontiguousarray(a) for a in p[1:]) for p in parts]
    ptrs = lambda i: (C.c_void_p * max(k, 1))(*[keep[j][i].ctypes.data if i < len(keep[j]) else None for j in range(k)])  # noqa: E731
    kinds = (C.c_int * max(k, 1))(*[p[0] for p in parts])
    ns = (C.c_size_t * max(k, 1))(*[p[3].shape[0] for p in parts])
    n = sum(p[3].shape[0] for p in parts)
    st, cw, vd = np.full(n, 0xFF, np.uint8), np.zeros((n, 32), np.uint8), np.zeros(n + 1, np.uint8)
    fb = C.c_uint64(0)
    groups = L.hs_verify_grouped(k, kinds, ptrs(0), ptrs(1), ptrs(2), ptrs(3), ns, _p(seed), g, c, seg, _p(st), _p(cw), _p(vd), C.byref(fb))
    assert groups >= 0, "a one-group pass differs from the whole-batch combination"
    return st, cw, vd[:groups], fb.value


def _oracle(parts):
    st, cw = [], []
    for p in parts:
        if p[0] == AGGREGATE:
            s, c, _ = co.verify_aggregate(p[1], p[4], p[2], p[3])
        else:
            s, c = {SINGLE: co.verify_single, DOUBLE: co.verify_double, VARGEN: co.verify_vargen}[p[0]](p[1], p[2], p[3])
        st.append(s)
        cw.append(c)
    return np.concatenate(st), np.concatenate(cw)


def _break_eq(parts, p, pos, d=1):
    """u + d of item pos of part p: its equation fails, everything else stays valid"""
    parts = list(parts)
    q = [a.copy() if isinstance(a, np.ndarray) else a for a in parts[p]]
    q[2][pos, :32] = _le((int.from_bytes(q[2][pos, :32].tobytes(), "little") + d) % o.R_ORDER)
    parts[p] = tuple(q)
    return parts


def _check_twin(L, parts, seed, g):
    st, cw, vd, fb = _twin(L, parts, seed, g)
    want_st, want_c = _oracle(parts)
    assert np.array_equal(st, want_st)
    assert np.array_equal(cw, want_c)
    return st, vd, fb


@pytest.mark.parametrize("kinds", [(SINGLE, AGGREGATE), (DOUBLE, VARGEN)])
def test_twin_equals_the_oracle_on_every_class_at_group_and_part_edges(L, kinds):
    """Every adversarial class of every kind planted at the first and last item of a group (g = 4: items 3 and 4) and of a part
    (0 and 7 of 8): statuses and challenges equal the oracle's item by item; only the failing group's items are redone."""
    g = 4
    base = []
    for i, k in enumerate(kinds):
        if k == AGGREGATE:
            base.append(_agg_part(_agg_items(*co.gen_aggregate(0x6A0 + i, [2, 3, 4, 1, 2, 3, 1, 2]))))
        else:
            base.append((k, *{SINGLE: co.gen_single, DOUBLE: co.gen_double, VARGEN: co.gen_vargen}[k](0x6A0 + i, 8)))
    st, vd, fb = _check_twin(L, base, _seed(0), g)
    assert np.all(st == 0) and np.all(vd == 1) and fb == 0
    for p, kind in enumerate(kinds):
        bad = _bad_aggregate_items(p) if kind == AGGREGATE else _bad_wire_items(kind, p)
        for j, item in enumerate(bad):
            for pos in (0, 3, 4, 7):
                parts = _plant(base, p, pos, item)
                st, vd, fb = _check_twin(L, parts, _seed(10 * j + pos), g)
                assert fb <= g, (p, j, pos)
                # a fallback happens only in the planted item's group, and only when the item entered with a failing equation
                assert (fb > 0) == (_oracle(parts)[0][sum(q[3].shape[0] for q in base[:p]) + pos] == 1), (p, j, pos)


def test_twin_two_bad_items_in_one_group_and_in_different_groups(L):
    g = 4
    (k, pk, sig, msg), = _valid_parts((SINGLE,), 0x2B)
    pk, sig, msg = (np.concatenate([a, a, a]) for a in (pk, sig, msg))   # 15 items, 4 groups
    parts = [(k, pk, sig, msg)]
    for a, b in ((4, 6), (3, 4), (0, 14)):
        bad = _break_eq(_break_eq(parts, 0, a), 0, b, 2)
        st, vd, fb = _check_twin(L, bad, _seed(a + b), g)
        assert list(np.nonzero(st)[0]) == [a, b]
        groups = {a // g, b // g}
        assert fb == sum(min(g, 15 - q * g) for q in groups)
        assert [q for q in range(len(vd)) if not vd[q]] == sorted(groups)


def test_twin_cancelling_errors_inside_one_group(L):
    """u + d on one item and u - d on another item with the same key and message cancel in a plain sum of the group, not under
    independent weights: both are found and reported 1."""
    (k, pk, sig, msg), = _valid_parts((SINGLE,), 0xCC)
    pk[3], msg[3] = pk[2], msg[2]
    sig[3] = sig[2]
    parts = _break_eq(_break_eq([(k, pk, sig, msg)], 0, 2, 0x1234567), 0, 3, o.R_ORDER - 0x1234567)
    for s in range(4):
        st, vd, fb = _check_twin(L, parts, _seed(500 + s), 8)
        assert list(st) == [0, 0, 1, 1, 0] and list(vd) == [0] and fb == 5


def test_twin_torsion_and_mixed_order_commitments_and_a_torsion_generator(L):
    """R shifted by a point of order 8, R of mixed order (R + T4), and a var-generator item over Gen + T: each fails only a
    subgroup test, which every point passes before it enters; the statuses are the oracle's."""
    (k, pk, sig, msg), = _valid_parts((SINGLE,), 0x70)
    for t in (8, 4, 2):
        s = sig.copy()
        s[1, 32:] = np.frombuffer(co.point_add(s[1, 32:].tobytes(), adv.torsion()[t]), np.uint8)
        st, vd, fb = _check_twin(L, [(k, pk, s, msg)], _seed(t), 2)
        assert st[1] == 2 and fb == 0
    T = o.point_from_bytes(adv.torsion()[8])
    gen = o.padd(o.pmul(o.G, 0x1357), T)
    sk, m = 0x2468ACE, 0x1111
    u, R = o.sign_var_gen(sk, gen, 0x99, m)
    vpk = np.frombuffer(o.point_to_bytes(o.pmul(gen, sk)) + o.point_to_bytes(gen), np.uint8).reshape(1, 64).copy()
    vsig = np.frombuffer(o.le32(u) + o.point_to_bytes(R), np.uint8).reshape(1, 64).copy()
    vmsg = _le(m).reshape(1, 32).copy()
    base = _valid_parts((VARGEN,), 0x71)[0]
    parts = [(VARGEN, *(np.concatenate([a, b]) for a, b in zip(base[1:4], (vpk, vsig, vmsg))))]
    st, vd, fb = _check_twin(L, parts, _seed(9), 2)
    assert st[-1] == 2 and np.all(st[:-1] == 0) and fb == 0


@pytest.mark.parametrize("kinds", [(SINGLE,), (DOUBLE,), (VARGEN,), (AGGREGATE,), (VARGEN, AGGREGATE, SINGLE, DOUBLE)])
def test_twin_one_group_is_the_whole_batch_combination(L, kinds):
    """g >= every part: the twin's grouped keys and point equal the whole-batch ones (checked inside the twin) and, on parts
    whose items all enter, each part's verdict is hs_verify_all_mixed's on that part."""
    base = _valid_parts(kinds, 0x1F)
    for j, parts in enumerate([base, _break_eq(base, len(base) - 1, 1)]):
        for c in (6, 9):
            st, cw, vd, fb = _twin(L, parts, _seed(j), 1 << 16, c=c)
            assert len(vd) == len(parts) and list(vd) == [1] * (len(parts) - j) + [0] * j
            if len(parts) == 1:
                ok = C.c_int(-1)
                keep = [np.ascontiguousarray(a) for a in parts[0][1:]] + [None] * (5 - len(parts[0]))
                ptr = lambda i: (C.c_void_p * 1)(keep[i].ctypes.data if keep[i] is not None else None)  # noqa: E731
                L.hs_verify_all_mixed(1, (C.c_int * 1)(parts[0][0]), ptr(0), ptr(1), ptr(2), ptr(3), (C.c_size_t * 1)(parts[0][3].shape[0]),
                                      _p(_seed(j)), c, 4, C.byref(ok))
                assert vd[0] == ok.value == 1 - j, (j, c)


def test_new_entry_points_refuse_an_inert_context():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    entry.build_cuda()
    from jubjub_schnorr_b200 import _native
    lib = _native.lib()
    ctx = C.c_void_p()
    assert lib.jjs_init(None, 1, C.byref(ctx)) == -2 and ctx
    buf = (C.c_uint8 * 4096)()
    a = C.addressof(buf)
    part = _native.Part(SINGLE, a, None, a, a, 4, a, None, None, None)
    fb = C.c_uint64(7)
    assert lib.jjs_verify_grouped(ctx, C.byref(part), 1, None, C.byref(fb)) == -2
    assert lib.jjs_verify_grouped_device(ctx, 0, C.byref(part), 1, None, None, None, None) == -2
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


_CACHE = {}


def _part(bv, kind, n, seed=0, frac=0.0):
    from jubjub_schnorr_b200 import workload as wl
    key = (kind, n, seed, frac)
    if key not in _CACHE:
        if kind == AGGREGATE:
            pks, off, sig, msg, _, _ = wl.make_aggregate_batch(bv, n, frac, seed=0xA66 + n + seed)
            _CACHE[key] = (AGGREGATE, pks, sig, msg, off)
        else:
            _CACHE[key] = (kind, *wl.make_batch(bv, kind, n, frac, seed=0xA11 + n + seed)[:3])
    return _CACHE[key]


def _same(a, b, what=""):
    assert len(a) == len(b)
    for q, (x, y) in enumerate(zip(a, b)):
        assert x.keys() == y.keys(), (what, q)
        for f in x:
            assert np.array_equal(x[f], y[f]), (what, q, f, np.nonzero(np.asarray(x[f]) != np.asarray(y[f]))[0][:8])


def _grouped_vs_mixed(b, parts, seed=None):
    got, fb = b.verify_grouped(parts, seed=seed, want_challenge=True, want_bitmap=True)
    want = b.verify_mixed(parts, want_challenge=True, want_bitmap=True)
    _same(got, want)
    return got, fb


@pytest.mark.gpu
def test_parity_with_verify_mixed_at_ten_percent_invalid(bv):
    """make_batch / make_aggregate_batch at 10 % invalid (the bench's classes) for every kind, and the configs[3] / [4] mixes:
    status, challenges, aggregate keys and bitmaps equal jjs_verify_mixed's item by item."""
    for kind in (SINGLE, DOUBLE, VARGEN, AGGREGATE):
        _, fb = _grouped_vs_mixed(bv, [_part(bv, kind, 100_000, frac=0.1)])
        assert 0 < fb <= 100_000
    half = 1 << 18
    _grouped_vs_mixed(bv, [_part(bv, VARGEN, half, frac=0.1), _part(bv, AGGREGATE, half, frac=0.1)])
    _grouped_vs_mixed(bv, [_part(bv, SINGLE, half, frac=0.1), _part(bv, DOUBLE, half, frac=0.1)])


@pytest.mark.gpu
def test_against_the_oracle(bv):
    for kind in (SINGLE, DOUBLE, VARGEN, AGGREGATE):
        parts = [_part(bv, kind, 1 << 14, 1, frac=0.1)]
        (got,), _ = bv.verify_grouped(parts, want_challenge=True)
        st, cw = _oracle(parts)
        assert np.array_equal(got["status"], st), kind
        assert np.array_equal(got["c"], cw), kind
        if kind == AGGREGATE:
            agg = co.verify_aggregate(parts[0][1], parts[0][4], parts[0][2], parts[0][3])[2]
            ok = st != 3   # the oracle leaves the aggregate unset when some field fails to decode
            assert np.array_equal(got["aggpk"][ok], agg[ok])


@pytest.mark.gpu
def test_valid_batches_need_no_fallback(bv):
    for kind in (SINGLE, DOUBLE, VARGEN, AGGREGATE):
        for n in (1, 33, 4097, 1 << 20):
            (r,), fb = bv.verify_grouped([_part(bv, kind, n)])
            assert np.all(r["status"] == 0) and fb == 0, (kind, n)
    half = 1 << 19
    for parts in ([_part(bv, VARGEN, half), _part(bv, AGGREGATE, half)], [_part(bv, SINGLE, half), _part(bv, DOUBLE, half)]):
        res, fb = bv.verify_grouped(parts, want_bitmap=True)
        assert fb == 0 and all(np.all(r["status"] == 0) for r in res)
        assert all(np.all(bv.unpack_bitmap(r["bitmap"], p[3].shape[0])) for r, p in zip(res, parts))
    assert bv.verify_grouped([]) == ([], 0)


@pytest.mark.gpu
def test_one_failing_item_at_every_edge(bv):
    """One equation-failing item at a group edge (2^12, 2^14, 2^16), the first-slice edge (2^17), the sub-chunk edge (2^19) and the
    first and last item of each part: exactly that item gets status 1, and at most one group is redone."""
    n = (1 << 19) + 100
    kinds = (SINGLE, VARGEN, AGGREGATE, DOUBLE)
    parts = [_part(bv, k, n if k in (SINGLE, AGGREGATE) else 70_000) for k in kinds]
    for p in range(len(parts)):
        m = parts[p][3].shape[0]
        for pos in sorted({0, (1 << 12) - 1, 1 << 12, (1 << 14) - 1, 1 << 14, (1 << 16) - 1, 1 << 16, (1 << 17) - 1, 1 << 17, (1 << 19) - 1, 1 << 19, m - 1}):
            if pos >= m:
                continue
            bad = _break_eq(parts, p, pos)
            res, fb = bv.verify_grouped(bad)
            for q, r in enumerate(res):
                want = np.zeros(bad[q][3].shape[0], np.uint8)
                if q == p:
                    want[pos] = 1
                assert np.array_equal(r["status"], want), (p, pos, q)
            assert 1 <= fb <= GROUP_MAX, (p, pos, fb)


@pytest.mark.gpu
def test_every_item_failing(bv):
    """Every item of every part tampered (10 % invalid classes plus the rest with broken equations): exact parity, and every item
    that passed decoding and validity is redone."""
    for kind in (SINGLE, DOUBLE, VARGEN, AGGREGATE):
        part = _part(bv, kind, 5000, 2, frac=0.1)
        q = list(part)
        q[2] = q[2].copy()
        u = [(int.from_bytes(q[2][i, :32].tobytes(), "little") + 1) % o.R_ORDER for i in range(q[3].shape[0])]
        q[2][:, :32] = np.stack([_le(x) for x in u])
        parts = [tuple(q)]
        want = bv.verify_mixed(parts)
        assert np.all(want[0]["status"] != 0)
        _, fb = _grouped_vs_mixed(bv, parts)
        assert fb == int(np.sum(want[0]["status"] == 1)), kind


@pytest.mark.gpu
def test_statuses_do_not_depend_on_the_seed(bv):
    parts = [_part(bv, SINGLE, 30_000, 3, frac=0.1), _part(bv, AGGREGATE, 20_000, 3, frac=0.1)]
    runs = [bv.verify_grouped(parts, seed=s, want_challenge=True) for s in (_seed(1).tobytes(), _seed(2).tobytes(), None)]
    for res, fb in runs[1:]:
        _same(res, runs[0][0])
        assert fb == runs[0][1]


@pytest.mark.gpu
def test_limited_context_at_the_floor(bv, small):
    """Many passes of a context at C = 2^12 (groups cut at the passes): parity with jjs_verify_mixed, memory_info unchanged."""
    parts = [_part(bv, AGGREGATE, 10_000, 4, frac=0.1), _part(bv, VARGEN, 9000, 4, frac=0.1), _part(bv, DOUBLE, 5000, 4)]
    parts = _break_eq(parts, 2, 4999)
    small.verify_mixed(parts)
    before = small.memory_info()
    _grouped_vs_mixed(small, parts)
    assert small.memory_info() == before
    bv.verify_mixed(parts)
    before = bv.memory_info()
    _grouped_vs_mixed(bv, parts)
    assert bv.memory_info() == before


@pytest.mark.gpu
def test_both_halves_run_fallback_equations_at_once(bv):
    """2^20 singles and 2^19 var-generator items with failing items in every sub-chunk (consecutive sub-chunks run side by side on
    the two scratch halves): each half's fallback equations keep to its own pass scratch, so the results are exact."""
    rng = np.random.default_rng(0xFA11)
    for kind, n in ((SINGLE, 1 << 20), (VARGEN, 1 << 19)):
        parts = [_part(bv, kind, n)]
        for pos in rng.choice(n, 64, replace=False):
            parts = _break_eq(parts, 0, int(pos))
        _, fb = _grouped_vs_mixed(bv, parts)
        assert 64 <= fb <= 64 * GROUP_MAX


def _to_dev(parts, dev):
    import torch
    dparts, keep, outs = [], [], []
    for p in parts:
        n = p[3].shape[0]
        t = [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in p[1:4]]
        o_ = {"status": torch.full((n,), 0xFF, dtype=torch.uint8, device=dev), "c": torch.zeros((n, 32), dtype=torch.uint8, device=dev),
              "bitmap": torch.zeros(((n + 31) // 32,), dtype=torch.int32, device=dev)}
        if p[0] == AGGREGATE:
            o_["aggpk"] = torch.zeros((n, 32), dtype=torch.uint8, device=dev)
        keep += t
        outs.append(o_)
        e = (p[0], t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), n, o_["status"].data_ptr(), o_["c"].data_ptr(),
             o_["aggpk"].data_ptr() if "aggpk" in o_ else None, o_["bitmap"].data_ptr())
        if p[0] == AGGREGATE:
            off = torch.from_numpy(np.ascontiguousarray(p[4])).to(dev)
            keep.append(off)
            e += (off.data_ptr(), p[4])
        dparts.append(e)
    return dparts, keep, outs


@pytest.mark.gpu
def test_device_entry_point_on_a_side_stream(bv):
    import torch
    dev = torch.device("cuda:0")
    n = (1 << 18) + 77
    parts = [_part(bv, VARGEN, n, frac=0.1), _part(bv, AGGREGATE, n, frac=0.1), _part(bv, SINGLE, 5000)]
    want, want_fb = bv.verify_grouped(parts, seed=_seed(3).tobytes(), want_challenge=True, want_bitmap=True)
    dparts, keep, outs = _to_dev(parts, dev)
    fb = torch.full((1,), -1, dtype=torch.int64, device=dev)
    s = torch.cuda.Stream(device=dev)
    s.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(s):
        bv.verify_grouped_device(dparts, fb.data_ptr(), seed=_seed(3).tobytes(), stream=s.cuda_stream)
    s.synchronize()
    assert int(fb.item()) == want_fb > 0
    for w, g in zip(want, outs):
        assert np.array_equal(g["status"].cpu().numpy(), w["status"])
        assert np.array_equal(g["c"].cpu().numpy(), w["c"])
        assert np.array_equal(g["bitmap"].cpu().numpy().view(np.uint32), w["bitmap"])
        if "aggpk" in w:
            assert np.array_equal(g["aggpk"].cpu().numpy(), w["aggpk"])


@pytest.mark.gpu
def test_argument_errors(bv):
    from jubjub_schnorr_b200 import _native
    lib, ctx = bv._lib, bv._ctx
    buf = (C.c_uint8 * 4096)()
    off = (C.c_uint32 * 5)(0, 1, 2, 3, 4)
    a = C.addressof(buf)
    fb = C.c_uint64(7)

    def call(part, harr=None):
        rh = lib.jjs_verify_grouped(ctx, C.byref(part), 1, None, C.byref(fb))
        rd = lib.jjs_verify_grouped_device(ctx, 0, C.byref(part), 1, harr, None, None, None)
        return rh, rd
    assert call(_native.Part(4, a, None, a, a, 4, a, None, None, None)) == (-1, -1)            # unknown kind
    assert call(_native.Part(-1, a, None, a, a, 4, a, None, None, None)) == (-1, -1)
    assert call(_native.Part(AGGREGATE, a, None, a, a, 4, a, None, None, None)) == (-1, -1)    # aggregate without offsets
    assert call(_native.Part(SINGLE, a, None, a, a, 4, None, a, None, None)) == (-1, -1)       # neither status nor bitmap
    assert lib.jjs_verify_grouped(ctx, None, 2, None, C.byref(fb)) == -1                        # NULL parts
    assert lib.jjs_verify_grouped_device(ctx, 0, None, 2, None, None, None, None) == -1
    agg = _native.Part(AGGREGATE, a, C.addressof(off), a, a, 4, a, None, None, None)            # device call without host offsets
    assert lib.jjs_verify_grouped_device(ctx, 0, C.byref(agg), 1, None, None, None, None) == -1
    assert lib.jjs_verify_grouped(ctx, None, 0, None, C.byref(fb)) == 0 and fb.value == 0


@pytest.mark.gpu
def test_cpp_verify_grouped(bv, tmp_path):
    """Gpu::verify_grouped of include/jubjub_schnorr.hpp (tests/cpp/test_grouped.cpp): the statuses and challenges of
    jjs_verify_mixed, and a fallback count."""
    kind, pk, sig, msg = _part(bv, DOUBLE, 20_000, 5, frac=0.1)
    (want,) = bv.verify_mixed([(kind, pk, sig, msg)], want_challenge=True)
    n = msg.shape[0]
    src = tmp_path / "in.bin"
    src.write_bytes(np.int32(kind).tobytes() + np.uint64(n).tobytes() + pk.tobytes() + sig.tobytes() + msg.tobytes())
    exe = str(tmp_path / "test_grouped")
    libdir = os.path.join(entry.ROOT, "jubjub_schnorr_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(entry.ROOT, "include"), "-o", exe,
                           os.path.join(entry.ROOT, "tests", "cpp", "test_grouped.cpp"), "-L", libdir, "-ljjschnorr_b200", "-Wl,-rpath," + libdir])
    out = subprocess.run([exe, str(src), str(tmp_path / "out.bin")], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "cpp grouped ok" in out.stdout, out.stderr
    got = (tmp_path / "out.bin").read_bytes()
    assert np.array_equal(np.frombuffer(got[:n], np.uint8), want["status"])
    assert np.array_equal(np.frombuffer(got[n:33 * n], np.uint8).reshape(n, 32), want["c"])
    assert 0 < int(np.frombuffer(got[33 * n:], np.uint64)[0]) <= n


@pytest.mark.gpu
def test_two_devices(bv):
    """Parts split into shards over two devices, a failing item on each side of the shard edge: parity and a summed fallback."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from jubjub_schnorr_b200 import BatchVerifier
    parts = [_part(bv, VARGEN, 40_000, frac=0.1), _part(bv, AGGREGATE, 40_000, frac=0.1), _part(bv, DOUBLE, 20_000)]
    parts = _break_eq(_break_eq(parts, 2, 9999), 2, 10_000)
    with BatchVerifier([0, 1]) as g2:
        got, fb = g2.verify_grouped(parts, want_challenge=True, want_bitmap=True)
        _same(got, bv.verify_mixed(parts, want_challenge=True, want_bitmap=True))
        assert fb >= 2
