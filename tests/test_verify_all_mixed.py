"""Whole-batch verification across the parts of a mixed call (jjs_verify_all_mixed / jjs_verify_all_mixed_device): one random
linear combination over items of every kind -- single, double, var-generator and aggregate-key -- decides "every item is valid".
The CPU part runs the twin (tests/hostsim/rlc_mixed_twin.cpp) against the C oracle and against the one-kind twin of
jjs_verify_all; the `gpu` part runs the library against its own per-item verification."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import __graft_entry__ as entry
from oracle import c_oracle as co
from oracle import jjs_oracle as o
from tests import adversarial as adv

SINGLE, DOUBLE, VARGEN, AGGREGATE = 0, 1, 2, 3


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _seed(k):
    return np.frombuffer(np.random.default_rng([0x5EED, 0xA11, k]).bytes(32), np.uint8).copy()


def _le(x):
    return np.frombuffer(o.le32(x), np.uint8)


# ---- CPU: the twin ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def L(tmp_path_factory):
    """tests/hostsim/rlc_mixed_twin.cpp (rlc_twin.cpp, the host simulator and the mixed combination), built into a temporary
    directory."""
    src = os.path.join(entry.ROOT, "tests", "hostsim", "rlc_mixed_twin.cpp")
    out = str(tmp_path_factory.mktemp("rlc_mixed_twin") / "librlc_mixed_twin.so")
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-o", out, src])
    lib = C.CDLL(out)
    vp = C.c_void_p
    lib.hs_verify_all_mixed.argtypes = [C.c_size_t, vp, vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.POINTER(C.c_int)]
    lib.hs_verify_all.argtypes = [C.c_int, vp, vp, vp, C.c_size_t, vp, C.c_int, C.c_int, C.POINTER(C.c_int)]
    return lib


def _twin_mixed(L, parts, seed, c=6, seg=4):
    """parts: (kind, pk, sig, msg) or (AGGREGATE, pks, sig, msg, offsets)"""
    k = len(parts)
    keep = [tuple(np.ascontiguousarray(a) for a in p[1:]) for p in parts]
    ptrs = lambda i: (C.c_void_p * max(k, 1))(*[keep[j][i].ctypes.data if i < len(keep[j]) else None for j in range(k)])  # noqa: E731
    kinds = (C.c_int * max(k, 1))(*[p[0] for p in parts])
    ns = (C.c_size_t * max(k, 1))(*[p[3].shape[0] for p in parts])
    ok = C.c_int(-1)
    L.hs_verify_all_mixed(k, kinds, ptrs(0), ptrs(1), ptrs(2), ptrs(3), ns, _p(seed), c, seg, C.byref(ok))
    return ok.value


def _oracle_all(parts):
    for p in parts:
        if p[3].shape[0] == 0:
            continue
        if p[0] == AGGREGATE:
            st = co.verify_aggregate(p[1], p[4], p[2], p[3])[0]
        else:
            st = {SINGLE: co.verify_single, DOUBLE: co.verify_double, VARGEN: co.verify_vargen}[p[0]](p[1], p[2], p[3])[0]
        if np.any(st != 0):
            return 0
    return 1


def _agg_items(pks, offsets, sig, msg):
    return [(pks[offsets[i]:offsets[i + 1]].copy(), sig[i].copy(), msg[i].copy()) for i in range(msg.shape[0])]


def _agg_part(items):
    counts = [it[0].shape[0] for it in items]
    offsets = np.zeros(len(items) + 1, np.uint32)
    np.cumsum(counts, out=offsets[1:])
    pks = np.concatenate([it[0] for it in items]) if items else np.zeros((0, 32), np.uint8)
    return (AGGREGATE, pks.reshape(-1, 32), np.stack([it[1] for it in items]), np.stack([it[2] for it in items]), offsets)


def _bad_aggregate_items(seed):
    """The aggregate classes: a tampered signer key, a key that does not decode, no signers, a tampered u, R shifted by a
    point of order 8."""
    rng = np.random.default_rng(seed)
    items = _agg_items(*co.gen_aggregate(0xA66 + seed, [3, 2, 1, 4, 2]))
    items[0][0][1] = np.frombuffer(o.point_to_bytes(o.pmul(o.G, 1 + int(rng.integers(1, 1 << 40)))), np.uint8)
    items[1][0][0] = np.frombuffer(adv.off_curve_encoding(rng), np.uint8)
    items[2] = (np.zeros((0, 32), np.uint8), items[2][1], items[2][2])
    items[3][1][:32] = _le((int.from_bytes(items[3][1][:32].tobytes(), "little") + 1) % o.R_ORDER)
    items[4][1][32:] = np.frombuffer(co.point_add(items[4][1][32:].tobytes(), adv.torsion()[8]), np.uint8)
    return items


def _bad_wire_items(kind, seed):
    """One item per class of tests/adversarial.py for the kind (every item tampered)."""
    gen = {SINGLE: co.gen_single, DOUBLE: co.gen_double, VARGEN: co.gen_vargen}[kind]
    name = {SINGLE: "single", DOUBLE: "double", VARGEN: "vargen"}[kind]
    slots = {SINGLE: 2, DOUBLE: 4, VARGEN: 3}[kind]
    n = len(adv.POINT_CLASSES) * slots + 8
    pk, sig, msg = gen(0xBAD + seed, n)
    pk, sig, msg, _, _ = adv.make_adversarial(name, pk, sig, msg, seed=seed, frac=1.0)
    return [(pk[j], sig[j], msg[j]) for j in range(n)]


def _valid_parts(kinds, seed):
    out = []
    for i, k in enumerate(kinds):
        if k == AGGREGATE:
            out.append(_agg_part(_agg_items(*co.gen_aggregate(seed + i, [2, 3, 4, 1, 2]))))
        else:
            gen = {SINGLE: co.gen_single, DOUBLE: co.gen_double, VARGEN: co.gen_vargen}[k]
            out.append((k, *gen(seed + i, 5)))
    return out


def _plant(parts, p, pos, item):
    parts = list(parts)
    if parts[p][0] == AGGREGATE:
        items = _agg_items(parts[p][1], parts[p][4], parts[p][2], parts[p][3])
        items[pos] = item
        parts[p] = _agg_part(items)
    else:
        k, pk, sig, msg = (a.copy() if isinstance(a, np.ndarray) else a for a in parts[p])
        pk[pos], sig[pos], msg[pos] = item
        parts[p] = (k, pk, sig, msg)
    return parts


@pytest.mark.parametrize("kinds", [(VARGEN, SINGLE, AGGREGATE), (DOUBLE, AGGREGATE, VARGEN)])
def test_twin_verdict_equals_the_oracle_on_every_class_in_every_part(L, kinds):
    """Every adversarial class planted singly at the first, middle and last position of each part of a valid three-part call:
    the twin's verdict is all(status == 0) of the oracle, over several seeds; the valid call passes for every seed."""
    base = _valid_parts(kinds, 0x3A0)
    for s in range(3):
        assert _twin_mixed(L, base, _seed(s)) == 1
    for p, kind in enumerate(kinds):
        bad = _bad_aggregate_items(p) if kind == AGGREGATE else _bad_wire_items(kind, p)
        for j, item in enumerate(bad):
            for pos in (0, 2, 4):
                parts = _plant(base, p, pos, item)
                want = _oracle_all(parts)
                assert want == 0, (p, j)
                assert _twin_mixed(L, parts, _seed(100 * j + pos)) == want, (p, j, pos)


def test_twin_cancelling_errors_across_parts_are_rejected(L):
    """+d G in a single item and -d G in a var-generator item whose generator is G cancel in a plain sum, not under
    independent weights."""
    d = 0x1234567
    pk, sig, msg = co.gen_single(0xCA, 3)
    sig[1, :32] = _le((int.from_bytes(sig[1, :32].tobytes(), "little") + d) % o.R_ORDER)
    sk, m = 0x5EC12E7, 0xABCDEF
    u, R = o.sign_var_gen(sk, o.G, 0x77, m)
    vpk = np.frombuffer(o.point_to_bytes(o.pmul(o.G, sk)) + o.point_to_bytes(o.G), np.uint8).reshape(1, 64).copy()
    vsig = np.frombuffer(o.le32((u - d) % o.R_ORDER) + o.point_to_bytes(R), np.uint8).reshape(1, 64).copy()
    vmsg = _le(m).reshape(1, 32).copy()
    parts = [(SINGLE, pk, sig, msg), (VARGEN, vpk, vsig, vmsg)]
    assert _oracle_all(parts) == 0
    for s in range(5):
        assert _twin_mixed(L, parts, _seed(300 + s)) == 0
    vsig[0, :32] = _le(u)
    sig[1, :32] = _le((int.from_bytes(sig[1, :32].tobytes(), "little") - d) % o.R_ORDER)
    assert _oracle_all(parts) == 1 and _twin_mixed(L, parts, _seed(0)) == 1


def test_twin_rejects_a_generator_with_a_torsion_component(L):
    """A var-generator item signed over Gen + T (T of order 8) satisfies its equation exactly; only the generator's subgroup
    test rejects it (the reference: InvalidPoint)."""
    T = o.point_from_bytes(adv.torsion()[8])
    gen = o.padd(o.pmul(o.G, 0x1357), T)
    sk, m = 0x2468ACE, 0x1111
    u, R = o.sign_var_gen(sk, gen, 0x99, m)
    pk = np.frombuffer(o.point_to_bytes(o.pmul(gen, sk)) + o.point_to_bytes(gen), np.uint8).reshape(1, 64).copy()
    sig = np.frombuffer(o.le32(u) + o.point_to_bytes(R), np.uint8).reshape(1, 64).copy()
    msg = _le(m).reshape(1, 32).copy()
    assert list(co.verify_vargen(pk, sig, msg)[0]) == [2]
    base = _valid_parts((VARGEN, SINGLE), 0x70)
    parts = [(VARGEN, np.concatenate([base[0][1], pk]), np.concatenate([base[0][2], sig]), np.concatenate([base[0][3], msg])), base[1]]
    for s in range(3):
        assert _twin_mixed(L, parts, _seed(400 + s)) == 0


@pytest.mark.parametrize("kind", [SINGLE, DOUBLE])
def test_twin_one_part_call_is_jjs_verify_all(L, kind):
    """A one-part call is exactly jjs_verify_all's combination: same verdict as the one-kind twin for the same seed, on a
    valid batch and with each bad item planted, at several window widths."""
    (_, pk, sig, msg), = _valid_parts((kind,), 0x1F)
    bad = _bad_wire_items(kind, 9)
    for j, item in enumerate([None] + bad[::3]):
        p, s, m = pk.copy(), sig.copy(), msg.copy()
        if item is not None:
            p[2], s[2], m[2] = item
        for c in (6, 9):
            ok = C.c_int(-1)
            L.hs_verify_all(kind, _p(p), _p(s), _p(m), 5, _p(_seed(j)), c, 4, C.byref(ok))
            assert _twin_mixed(L, [(kind, p, s, m)], _seed(j), c=c) == ok.value == (item is None), (j, c)


def test_twin_empty_call_is_valid(L):
    e = np.zeros((0, 32), np.uint8)
    assert _twin_mixed(L, [], _seed(0)) == 1
    assert _twin_mixed(L, [(SINGLE, e, np.zeros((0, 64), np.uint8), e), (AGGREGATE, e, np.zeros((0, 64), np.uint8), e, np.zeros(1, np.uint32))],
                       _seed(0)) == 1


def test_new_entry_points_refuse_an_inert_context():
    """Without a usable device jjs_init hands back an inert context: both new entry points answer JJS_ERR_CUDA, and the
    reason of the failed init survives."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    entry.build_cuda()
    from jubjub_schnorr_b200 import _native
    lib = _native.lib()
    ctx = C.c_void_p()
    assert lib.jjs_init(None, 1, C.byref(ctx)) == -2 and ctx
    buf = (C.c_uint8 * 4096)()
    part = _native.Part(SINGLE, C.addressof(buf), None, C.addressof(buf), C.addressof(buf), 4, None, None, None, None)
    ok = C.c_int(7)
    assert lib.jjs_verify_all_mixed(ctx, C.byref(part), 1, None, C.byref(ok)) == -2
    assert lib.jjs_verify_all_mixed_device(ctx, 0, C.byref(part), 1, None, None, buf, None) == -2
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
    """A limited context at the floor: 2^12 items per pass, 2^11 per scratch half, 512 aggregate items per pass."""
    from jubjub_schnorr_b200 import BatchVerifier
    with BatchVerifier([0], memory_limit=50_000_000) as b:
        assert b.memory_info()["items_in_flight"] == 1 << 12
        yield b


_CACHE = {}


def _part(bv, kind, n, seed=0):
    """A valid part of n items (cached)."""
    from jubjub_schnorr_b200 import workload as wl
    key = (kind, n, seed)
    if key not in _CACHE:
        if kind == AGGREGATE:
            pks, off, sig, msg, _, _ = wl.make_aggregate_batch(bv, n, 0.0, seed=0xA66 + n + seed)
            _CACHE[key] = (AGGREGATE, pks, sig, msg, off)
        else:
            _CACHE[key] = (kind, *wl.make_valid(bv, kind, n, seed=0xA11 + n + seed))
    return _CACHE[key]


def _bad_item(kind, j=0):
    """A bad item of the kind, (pk, sig, msg) -- for aggregate items (keys, sig, msg) -- whose keys all decode."""
    if kind == AGGREGATE:
        return _bad_aggregate_items(j)[(0, 3, 4)[j % 3]]
    return _bad_wire_items(kind, j)[-8 + j % 8]


def _per_item_all(bv, parts):
    res = bv.verify_mixed(parts)
    return all(bool(np.all(r["status"] == 0)) for r in res)


@pytest.mark.gpu
def test_valid_batches_of_every_kind_and_mix_are_accepted(bv):
    for kind in (SINGLE, DOUBLE, VARGEN, AGGREGATE):
        for n in (0, 1, 33, 4097, 1 << 20):
            assert bv.verify_all_mixed([_part(bv, kind, n)], seed=_seed(n).tobytes()) is True, (kind, n)
    half = 1 << 19
    assert bv.verify_all_mixed([_part(bv, VARGEN, half), _part(bv, AGGREGATE, half)]) is True      # configs[3]-style
    assert bv.verify_all_mixed([_part(bv, SINGLE, half), _part(bv, DOUBLE, half)]) is True         # configs[4]-style
    assert bv.verify_all_mixed([]) is True


@pytest.mark.gpu
def test_one_bad_item_across_boundaries_is_rejected(bv, small):
    """A bad item at the first and last item of every part, across the first-slice / sub-chunk boundary (2^17) of a jjs_init
    context, and across the pass boundaries of a limited context at the floor (2^11 wire items, 512 aggregate items)."""
    kinds = (VARGEN, AGGREGATE, SINGLE, DOUBLE)
    parts = [_part(bv, k, (1 << 17) + 100) for k in kinds]
    assert bv.verify_all_mixed(parts) is True
    for p, k in enumerate(kinds):
        for pos in (0, (1 << 17) - 1, 1 << 17, (1 << 17) + 99):
            assert bv.verify_all_mixed(_plant(parts, p, pos, _bad_item(k, pos))) is False, (p, pos)
    parts = [_part(bv, k, 3 * (1 << 11) + 5) for k in kinds]
    assert small.verify_all_mixed(parts) is True
    for p, k in enumerate(kinds):
        for pos in (0, 511, 512, (1 << 11) - 1, 1 << 11, 3 * (1 << 11) + 4):
            assert small.verify_all_mixed(_plant(parts, p, pos, _bad_item(k, pos))) is False, (p, pos)


@pytest.mark.gpu
def test_agrees_with_per_item_verification(bv):
    """Random mixes with a few invalid items: the verdict is all(status == 0) of jjs_verify_mixed, over random seeds."""
    from jubjub_schnorr_b200 import workload as wl
    rng = np.random.default_rng(0xA9)
    for t in range(8):
        parts = []
        for k in rng.permutation(4)[: 1 + t % 4]:
            n = int(rng.integers(1, 30000))
            if k == AGGREGATE:
                pks, off, sig, msg, _, _ = wl.make_aggregate_batch(bv, n, 0.0 if t % 2 else 2.0 / n, seed=t)
                parts.append((AGGREGATE, pks, sig, msg, off))
            else:
                pk, sig, msg = wl.make_valid(bv, int(k), n, seed=t)
                if t % 2 == 0:
                    pk, sig, msg, _, _ = wl.invalidate(int(k), pk, sig, msg, 1.0 / n, seed=t)
                parts.append((int(k), pk, sig, msg))
        want = _per_item_all(bv, parts)
        for s in range(2):
            assert bv.verify_all_mixed(parts, seed=_seed(10 * t + s).tobytes()) is want, t


@pytest.mark.gpu
def test_one_part_call_agrees_with_verify_all(bv):
    for kind in (SINGLE, DOUBLE):
        k, pk, sig, msg = _part(bv, kind, 20000)
        for bad in (False, True):
            s = sig.copy()
            if bad:
                s[12345, 0] ^= 1
            want = bv.verify_all(kind, pk, s, msg, seed=_seed(7).tobytes())
            assert want is (not bad)
            assert bv.verify_all_mixed([(kind, pk, s, msg)], seed=_seed(7).tobytes()) is want


@pytest.mark.gpu
def test_limited_context_at_the_floor(bv, small):
    """Aggregate and var-generator parts spanning many passes of a context at C = 2^12: the verdicts of a jjs_init context, and
    memory_info unchanged (the accumulators of both halves survive every aggregation pass)."""
    parts = [_part(bv, AGGREGATE, 10000, 1), _part(bv, VARGEN, 9000, 1), _part(bv, SINGLE, 3000, 1)]
    small.verify_mixed(parts)
    before = small.memory_info()
    for b in (small, bv):
        assert b.verify_all_mixed(parts, seed=_seed(1).tobytes()) is True
        for p in range(len(parts)):
            pos = parts[p][3].shape[0] - 1
            assert b.verify_all_mixed(_plant(parts, p, pos, _bad_item(parts[p][0], p))) is False, p
    assert small.memory_info() == before
    bv.verify_mixed(parts)
    before = bv.memory_info()
    assert bv.verify_all_mixed(parts) is True
    assert bv.memory_info() == before


def _to_dev(parts, dev):
    import torch
    dparts, keep = [], []
    for p in parts:
        t = [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in p[1:4]]
        keep += t
        entry_ = (p[0], t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), p[3].shape[0])
        if p[0] == AGGREGATE:
            off = torch.from_numpy(np.ascontiguousarray(p[4])).to(dev)
            keep.append(off)
            entry_ += (off.data_ptr(), p[4])
        dparts.append(entry_)
    return dparts, keep


@pytest.mark.gpu
def test_device_entry_point_on_a_side_stream(bv):
    import torch
    dev = torch.device("cuda:0")
    n = (1 << 18) + 77
    parts = [_part(bv, VARGEN, n), _part(bv, AGGREGATE, n), _part(bv, SINGLE, 5000)]
    for case in ("empty", "valid", "bad"):
        use = [] if case == "empty" else (parts if case == "valid" else _plant(parts, 1, n - 1, _bad_item(AGGREGATE, 1)))
        want = bv.verify_all_mixed(use, seed=_seed(3).tobytes())
        assert want is (case != "bad")
        dparts, keep = _to_dev(use, dev)
        out = torch.full((1,), -1, dtype=torch.int32, device=dev)
        s = torch.cuda.Stream(device=dev)
        s.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(s):
            bv.verify_all_mixed_device(dparts, out.data_ptr(), seed=_seed(3).tobytes(), stream=s.cuda_stream)
        s.synchronize()
        assert int(out.item()) == int(want), case


@pytest.mark.gpu
def test_argument_errors(bv):
    from jubjub_schnorr_b200 import _native
    lib, ctx = bv._lib, bv._ctx
    buf = (C.c_uint8 * 4096)()
    off = (C.c_uint32 * 5)(0, 1, 2, 3, 4)
    a = C.addressof(buf)
    ok = C.c_int(7)

    def call(part, harr=None):
        rh = lib.jjs_verify_all_mixed(ctx, C.byref(part), 1, None, C.byref(ok))
        rd = lib.jjs_verify_all_mixed_device(ctx, 0, C.byref(part), 1, harr, None, a, None)
        return rh, rd
    assert call(_native.Part(4, a, None, a, a, 4, None, None, None, None)) == (-1, -1)          # unknown kind
    assert call(_native.Part(-1, a, None, a, a, 4, None, None, None, None)) == (-1, -1)
    assert call(_native.Part(AGGREGATE, a, None, a, a, 4, None, None, None, None)) == (-1, -1)  # aggregate without offsets
    for field in range(4):                                                                        # an output field
        outs = [None] * 4
        outs[field] = a
        assert call(_native.Part(SINGLE, a, None, a, a, 4, *outs)) == (-1, -1), field
    part = _native.Part(SINGLE, a, None, a, a, 0, None, None, None, None)
    assert lib.jjs_verify_all_mixed(ctx, C.byref(part), 1, None, None) == -1                      # NULL all_valid
    assert lib.jjs_verify_all_mixed_device(ctx, 0, C.byref(part), 1, None, None, None, None) == -1
    agg = _native.Part(AGGREGATE, a, C.addressof(off), a, a, 4, None, None, None, None)          # device call without host offsets
    assert lib.jjs_verify_all_mixed_device(ctx, 0, C.byref(agg), 1, None, None, a, None) == -1
    assert lib.jjs_verify_all_mixed(ctx, None, 0, None, C.byref(ok)) == 0 and ok.value == 1


@pytest.mark.gpu
def test_two_devices(bv):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from jubjub_schnorr_b200 import BatchVerifier
    parts = [_part(bv, VARGEN, 40000), _part(bv, AGGREGATE, 40000), _part(bv, DOUBLE, 20000)]
    with BatchVerifier([0, 1]) as g:
        assert g.verify_all_mixed(parts) is True
        for p in range(3):
            assert g.verify_all_mixed(_plant(parts, p, parts[p][3].shape[0] - 1, _bad_item(parts[p][0], p))) is False, p
