"""Memory-limited contexts (jjs_init_limited / jjs_memory_info): the configuration the policy picks for a device memory limit, and
item-for-item parity of every entry point on a limited context with the C oracle and with a jjs_init context.  The parity tests
use a limit that gives the smallest capacity, C = 2^12 items per pass with 12-bit fixed-base tables, and batch sizes that are not
multiples of C and span several passes and several host staging windows."""
import ctypes as C

import numpy as np
import pytest

import __graft_entry__ as entry
from oracle import c_oracle as co
from tests import adversarial as adv

MiB, GiB = 1 << 20, 1 << 30
SMALL_LIMIT = 50_000_000            # capacity 2^12, 12-bit tables, ~16 MB left for growth and key sets
N = 3 * 4096 + 17                   # items of the parity batches: four passes of C = 2^12, the last one partial


def _policy(limit):
    """(width, capacity, bytes) the policy of include/jjschnorr_b200.h implies, restated from the allocation sizes: constant tables,
    two fixed-base tables of W-bit windows, 1 024 SAFE tags, and per item of capacity the pipeline scratch (4 points, flags,
    challenge, work and retest lists), the table scratch (3 x 36 field elements), the aggregate scratch (two halves of C / 8 items
    with 4 keys each) and 320 B of staging.  None below the floor."""
    def fb(w):
        return 2 * 96 * ((252 + w - 1) // w) * (1 << w)

    def total(w, c):
        consts = 6 * 256 * 32 + (1 << 13) + 32 * 1024
        pipeline = 2 * 32 * 4 * c + 4 * c + c + 2 * c + 32 * c + 8 * c + 32 + 8 * c + 32 * 108 * c
        agg_items = c // 8
        agg = 2 * (4 * agg_items * (32 + 32 + 1 + 32 + 4 + 4) + 4 * agg_items + 65 * 5 * 4 + 4)
        return consts + fb(w) + pipeline + agg + 320 * c

    c = 1 << 20
    while c >= 1 << 12:
        if total(12, c) <= limit:
            w = 21 if total(21, c) <= limit else 12
            return w, c, total(w, c)
        c //= 2
    return None


# ---- without a GPU ----------------------------------------------------------------------------------------------------
def test_limit_of_zero_is_an_argument_error():
    entry.build_cuda()
    from jubjub_schnorr_b200 import _native
    lib = _native.lib()
    ctx = C.c_void_p()
    assert lib.jjs_init_limited(None, 1, 0, C.byref(ctx)) == -1 and not ctx


def test_limited_init_without_a_device_leaves_an_inert_context():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    entry.build_cuda()
    from jubjub_schnorr_b200 import _native
    lib = _native.lib()
    ctx = C.c_void_p()
    assert lib.jjs_init_limited(None, 1, 256 * MiB, C.byref(ctx)) == -2 and ctx
    assert b"no CUDA device" in lib.jjs_last_error(ctx)
    held, bits, items = C.c_uint64(), C.c_int(), C.c_uint64()
    assert lib.jjs_memory_info(ctx, 0, C.byref(held), C.byref(bits), C.byref(items)) == -2
    buf = (C.c_uint8 * 256)()
    assert lib.jjs_verify_single(ctx, buf, buf, buf, 1, buf, None) == -2
    lib.jjs_destroy(ctx)


def test_policy_restatement():
    """The documented configurations: 256 MiB -> 2^15 items, 1 GiB -> 2^17, 8 GiB -> 2^20 with 12-bit tables, 16 GiB -> 2^20 with
    the 21-bit tables; the floor is about 40 MB."""
    assert _policy(256 * MiB)[:2] == (12, 1 << 15)
    assert _policy(1 * GiB)[:2] == (12, 1 << 17)
    assert _policy(8 * GiB)[:2] == (12, 1 << 20)
    assert _policy(16 * GiB)[:2] == (21, 1 << 20)
    assert _policy(SMALL_LIMIT)[:2] == (12, 1 << 12)
    assert _policy(30_000_000) is None and 30e6 < _policy(SMALL_LIMIT)[2] < 40e6


# ---- on the GPU -------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def full():
    from jubjub_schnorr_b200 import BatchVerifier
    with BatchVerifier([0]) as bv:
        yield bv


@pytest.fixture(scope="module")
def small():
    from jubjub_schnorr_b200 import BatchVerifier
    with BatchVerifier([0], memory_limit=SMALL_LIMIT) as bv:
        yield bv


@pytest.mark.gpu
@pytest.mark.parametrize("limit", [256 * MiB, 1 * GiB, 8 * GiB, 16 * GiB, 100_000_000, SMALL_LIMIT])
def test_configuration_for_a_limit(limit):
    from jubjub_schnorr_b200 import BatchVerifier
    w, c, total = _policy(limit)
    with BatchVerifier([0], memory_limit=limit) as bv:
        info = bv.memory_info()
        assert (info["fb_window_bits"], info["items_in_flight"]) == (w, c)
        assert info["bytes_held"] == total <= limit
        if c == 1 << 14:
            assert info["bytes_held"] < 256 * MiB
        # a first verification allocates nothing more
        pk, sig, msg = co.gen_single(0x11, 1000)
        st = bv.verify_single(pk, sig, msg)
        assert (st == 0).all() and bv.memory_info()["bytes_held"] == total


@pytest.mark.gpu
def test_jjs_init_context_reports_its_configuration(full):
    info = full.memory_info()
    assert info["fb_window_bits"] == 21 and info["items_in_flight"] == 1 << 20
    assert info["bytes_held"] >= 2 * 96 * 12 * (1 << 21)


@pytest.mark.gpu
def test_limit_below_the_floor():
    from jubjub_schnorr_b200 import _native
    lib = _native.lib()
    ctx = C.c_void_p()
    assert lib.jjs_init_limited(None, 1, 30_000_000, C.byref(ctx)) == -3 and ctx
    assert b"below the smallest configuration" in lib.jjs_last_error(ctx)
    assert lib.jjs_memory_info(ctx, 0, None, None, None) == -2
    buf = (C.c_uint8 * 256)()
    assert lib.jjs_verify_single(ctx, buf, buf, buf, 1, buf, None) == -2
    lib.jjs_destroy(ctx)


@pytest.mark.gpu
def test_reference_kats_on_a_limited_context(small):
    from tests import test_gpu_parity as parity
    parity.test_reference_kats_on_gpu(small)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["single", "double", "vargen"])
def test_adversarial_parity(full, small, kind):
    """Adversarial items (every point class, torsion-shifted commitments) over several passes: statuses, challenges and accept
    bitmaps equal the C oracle's and the jjs_init context's."""
    from jubjub_schnorr_b200 import SINGLE, DOUBLE, VARGEN
    gen = {"single": co.gen_single, "double": co.gen_double, "vargen": co.gen_vargen}[kind]
    cver = {"single": co.verify_single, "double": co.verify_double, "vargen": co.verify_vargen}[kind]
    variant = {"single": SINGLE, "double": DOUBLE, "vargen": VARGEN}[kind]
    pk, sig, msg = gen(0x3A1, N - 48)
    pk, sig, msg, _, _ = adv.make_adversarial(kind, pk, sig, msg, seed=3, frac=0.4)
    if kind != "vargen":
        tpk, tsig, tmsg, _ = adv.torsion_shifted_signatures(kind, 48, seed=9)
        pk, sig, msg = np.concatenate([pk, tpk]), np.concatenate([sig, tsig]), np.concatenate([msg, tmsg])
    st_o, c_o = cver(pk, sig, msg)
    outs = []
    for bv in (small, full):
        ver = {SINGLE: bv.verify_single, DOUBLE: bv.verify_double, VARGEN: bv.verify_vargen}[variant]
        bm = {SINGLE: bv.verify_batch, DOUBLE: bv.verify_batch_double, VARGEN: bv.verify_batch_vargen}[variant]
        st, c = ver(pk, sig, msg, True)
        outs.append((st, c, bm(pk, sig, msg)))
    (st, c, words), (st_f, c_f, words_f) = outs
    assert np.array_equal(st, st_o) and np.array_equal(c, c_o)
    assert np.array_equal(st, st_f) and np.array_equal(c, c_f) and np.array_equal(words, words_f)
    assert set(st.tolist()) == {0, 1, 2, 3}


def _aggregate_items(n_small):
    rng = np.random.default_rng(0xA66)
    signers = np.concatenate([rng.integers(1, 9, size=n_small), [600]]).astype(np.uint32)
    pks, offsets, sig, msg = co.gen_aggregate(0xA67, signers)
    bad = rng.choice(signers.shape[0], size=signers.shape[0] // 5, replace=False)
    sig[bad, 0] ^= 1
    return pks, offsets, sig, msg


@pytest.mark.gpu
def test_aggregate_parity(full, small):
    """Aggregate-key items with 1-8 signers and one of 600 (a tag table larger than the initial one) over several passes."""
    pks, offsets, sig, msg = _aggregate_items(N)
    st_o, c_o, agg_o = co.verify_aggregate(pks, offsets, sig, msg)
    st, c, agg = small.verify_aggregate(pks, offsets, sig, msg, want_challenge=True, want_aggregate_key=True)
    st_f, c_f, agg_f = full.verify_aggregate(pks, offsets, sig, msg, want_challenge=True, want_aggregate_key=True)
    assert np.array_equal(st, st_o) and np.array_equal(c, c_o) and np.array_equal(agg, agg_o)
    assert np.array_equal(st, st_f) and np.array_equal(c, c_f) and np.array_equal(agg, agg_f)
    assert np.array_equal(small.verify_batch_aggregate(pks, offsets, sig, msg), full.verify_batch_aggregate(pks, offsets, sig, msg))
    assert small.memory_info()["bytes_held"] <= SMALL_LIMIT


@pytest.mark.gpu
def test_mixed_parity(full, small):
    """One jjs_verify_mixed call of all four kinds."""
    from jubjub_schnorr_b200 import SINGLE, DOUBLE, VARGEN
    from jubjub_schnorr_b200.batch import AGGREGATE
    parts = []
    for kind, gen, n in ((SINGLE, co.gen_single, N), (DOUBLE, co.gen_double, 5001), (VARGEN, co.gen_vargen, 3001)):
        pk, sig, msg = gen(0x5E0 + kind, n)
        sig[::7, 0] ^= 1
        parts.append((kind, pk, sig, msg))
    pks, offsets, sig, msg = _aggregate_items(2000)
    parts.append((AGGREGATE, pks, sig, msg, offsets))
    res = small.verify_mixed(parts, want_challenge=True, want_bitmap=True)
    ref = full.verify_mixed(parts, want_challenge=True, want_bitmap=True)
    for r, f in zip(res, ref):
        assert r.keys() == f.keys()
        for k in r:
            assert np.array_equal(r[k], f[k]), k
    st_o, c_o = co.verify_single(*parts[0][1:4])
    assert np.array_equal(res[0]["status"], st_o) and np.array_equal(res[0]["c"], c_o)


@pytest.mark.gpu
def test_device_entry_points_on_a_side_stream(full, small):
    import torch
    from jubjub_schnorr_b200 import SINGLE, DOUBLE, VARGEN
    side = torch.cuda.Stream()
    for variant, gen in ((SINGLE, co.gen_single), (DOUBLE, co.gen_double), (VARGEN, co.gen_vargen)):
        pk, sig, msg = gen(0xDE0 + variant, N)
        sig[::5, 0] ^= 1
        d_pk, d_sig, d_msg = (torch.from_numpy(a).cuda() for a in (pk, sig, msg))
        outs = []
        for bv in (small, full):
            d_st = torch.full((N,), 0xEE, dtype=torch.uint8, device="cuda")
            d_c = torch.zeros((N, 32), dtype=torch.uint8, device="cuda")
            d_bm = torch.zeros((N + 31) // 32, dtype=torch.int32, device="cuda")
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                bv.verify_device(variant, d_pk.data_ptr(), d_sig.data_ptr(), d_msg.data_ptr(), N, d_st.data_ptr(), d_c.data_ptr(), stream=side.cuda_stream)
                bv.status_bitmap_device(d_st.data_ptr(), N, d_bm.data_ptr(), stream=side.cuda_stream)
            side.synchronize()
            outs.append((d_st.cpu().numpy(), d_c.cpu().numpy(), d_bm.cpu().numpy()))
        for a, b in zip(*outs):
            assert np.array_equal(a, b)
    pks, offsets, sig, msg = _aggregate_items(N)
    n = msg.shape[0]
    outs = []
    for bv in (small, full):
        d = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (pks, offsets.view(np.int32), sig, msg)]
        d_st = torch.zeros(n, dtype=torch.uint8, device="cuda")
        d_agg = torch.zeros((n, 32), dtype=torch.uint8, device="cuda")
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            bv.verify_aggregate_device(d[0].data_ptr(), d[1].data_ptr(), offsets, d[2].data_ptr(), d[3].data_ptr(), n, d_st.data_ptr(), d_agg=d_agg.data_ptr(),
                                       stream=side.cuda_stream)
        side.synchronize()
        outs.append((d_st.cpu().numpy(), d_agg.cpu().numpy()))
    assert np.array_equal(outs[0][0], outs[1][0]) and np.array_equal(outs[0][1], outs[1][1])


@pytest.mark.gpu
def test_typed_parity(full, small):
    from jubjub_schnorr_b200 import workload as wl
    pts, u, msg, expected = wl.make_typed_single_batch(full, N, 0.3, seed=0x7E)
    st, c = small.verify_ext(0, pts, u, msg, True)
    st_f, c_f = full.verify_ext(0, pts, u, msg, True)
    assert np.array_equal(st, expected) and np.array_equal(st, st_f) and np.array_equal(c, c_f)


@pytest.mark.gpu
def test_multisig_combine_parity(full, small):
    """Sessions of 1-4 participants (more than one chunk of sessions) and a few invalid shares."""
    rng = np.random.default_rng(0x5E5)
    signers = rng.integers(1, 5, size=2500)
    pks, Rs, Ss, zs, offsets, msg = co.gen_multisig(0x5E6, signers)
    bad = rng.choice(zs.shape[0], size=50, replace=False)
    zs[bad, 1] ^= 1
    res = small.multisig_combine(pks, Rs, Ss, zs, offsets, msg)
    ref = full.multisig_combine(pks, Rs, Ss, zs, offsets, msg)
    orc = co.multisig_combine(pks, Rs, Ss, zs, offsets, msg)
    for a, b, o in zip(res, ref, orc):
        assert np.array_equal(a, b) and np.array_equal(a, o)


@pytest.mark.gpu
def test_fixed_base_tables_of_12_bits(small):
    """Random entries of both 12-bit tables and every entry of the last window equal their definition."""
    assert small.memory_info()["fb_window_bits"] == 12
    rng = np.random.default_rng(0xFB)
    last = np.arange(20 * 4096, 21 * 4096, dtype=np.uint32)
    entries = np.concatenate([rng.integers(0, 21 * 4096, size=4096).astype(np.uint32), last])
    for which in (0, 1):
        assert small.fb_table_check(which, entries) == 0


@pytest.mark.gpu
def test_signing_parity(full, small):
    from jubjub_schnorr_b200 import workload as wl
    rng = np.random.default_rng(0x516)
    n = 5000
    sk, rnd, gsc = (wl.random_scalars(rng, n, 250) for _ in range(3))
    msg = wl.random_scalars(rng, n, 250)
    for variant in (0, 1, 2):
        g = gsc if variant == 2 else None
        a = small.sign_batch(variant, sk, rnd, msg, g)
        b = full.sign_batch(variant, sk, rnd, msg, g)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    offsets = np.concatenate([[0], np.cumsum(rng.integers(1, 9, size=1000))]).astype(np.uint32)
    ask = wl.random_scalars(rng, int(offsets[-1]), 250)
    arnd, amsg = wl.random_scalars(rng, 1000, 250), wl.random_scalars(rng, 1000, 250)
    a = small.sign_aggregate_batch(ask, offsets, arnd, amsg)
    b = full.sign_aggregate_batch(ask, offsets, arnd, amsg)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1])
def test_keyed_parity_and_refusal(small, kind):
    """Keyed verification on a limited context equals the unkeyed path with the keys written out; a key set that would cross the
    limit is refused with JJS_ERR_NOMEM, holds nothing, and the context keeps verifying."""
    from jubjub_schnorr_b200 import JjsError
    from jubjub_schnorr_b200 import workload as wl
    pks, idx, sig, msg, expected, _ = wl.make_keyed_batch(small, kind, 4, N, 0.2, seed=0x4E0 + kind)
    ks = small.keyset_create(kind, pks)
    st, c, words = small.verify_keyed(ks, idx, sig, msg, want_challenge=True, want_bitmap=True)
    written = pks[np.minimum(idx, pks.shape[0] - 1)].copy()
    out = idx >= pks.shape[0]
    written[out, :32] = np.frombuffer(adv.noncanonical_v_encoding(np.random.default_rng(0)), np.uint8)
    ver = small.verify_single if kind == 0 else small.verify_double
    st_u, c_u = ver(written, sig, msg, True)
    assert np.array_equal(st, expected) and np.array_equal(st, st_u) and np.array_equal(c, c_u)
    assert np.array_equal(small.unpack_bitmap(words, N), st == 0)
    held = small.memory_info()["bytes_held"]
    big = np.repeat(pks[:1], 200, axis=0)
    with pytest.raises(JjsError, match=r"\(-3\).*memory limit"):
        small.keyset_create(kind, big)
    assert small.memory_info()["bytes_held"] == held
    assert np.array_equal(small.verify_keyed(ks, idx, sig, msg), st)
    small.keyset_destroy(ks)


def test_two_device_limited_context():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from jubjub_schnorr_b200 import BatchVerifier
    pk, sig, msg = co.gen_double(0x2D, 40_001)
    sig[::9, 0] ^= 1
    st_o, c_o = co.verify_double(pk, sig, msg)
    with BatchVerifier([0, 1], memory_limit=256 * MiB) as g:
        for k in (0, 1):
            assert g.memory_info(k)["items_in_flight"] == 1 << 15 and g.memory_info(k)["bytes_held"] <= 256 * MiB
        st, c = g.verify_double(pk, sig, msg, True)
    assert np.array_equal(st, st_o) and np.array_equal(c, c_o)
