"""GPU parity: the CUDA path (through the C ABI) against the pinned oracle, item by item."""
import json
import os

import numpy as np
import pytest

from oracle import c_oracle as co
from oracle import jjs_oracle as o
from tests import adversarial as adv
from tests.test_oracle_kat import legacy_double_fixture

pytestmark = pytest.mark.gpu

KAT = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "reference_kat.json")))


@pytest.fixture(scope="module")
def bv():
    from jubjub_schnorr_b200 import BatchVerifier
    with BatchVerifier([0]) as v:
        yield v


def _a(b):
    return np.frombuffer(bytes(b), dtype=np.uint8)


def test_reference_kats_on_gpu(bv):
    k, s = KAT["multisig_kat"], KAT["serde_kat"]
    st, c = bv.verify_single(_a(bytes.fromhex(k["AGGREGATE_PUBLIC_KEY"])), _a(bytes.fromhex(k["SIGNATURE"])), _a(o.le32(31)), True)
    assert st[0] == 0 and c.tobytes().hex() == k["CHALLENGE"]
    m = bytes.fromhex("6dfe107145b1cba63d5f5ed0c410c09441fbc0d70c9bfea970949499aa128214")
    st, c = bv.verify_single(_a(o.b58decode(s["serde_public_key"], 32)), _a(o.b58decode(s["serde_signature"], 64)), _a(m), True)
    assert st[0] == 0 and c.tobytes().hex() == "7ad531e479fe4f1d2c1858c180e18f57e549d7eda93c85f46344f4716de67e02"
    st, c = bv.verify_double(_a(o.b58decode(s["serde_public_key_double"], 64)), _a(o.b58decode(s["serde_signature_double"], 96)), _a(m), True)
    assert st[0] == 0 and c.tobytes().hex() == "b706ff0423cbdff51e73ee23985e66a5f827343f03ecf4e9ecd7f32fc9791901"
    rng = o.StdRng(s["_seed"]); rng.random_fr(); rng.random_fr()
    mv = o.le32(rng.random_fq())
    st, c = bv.verify_vargen(_a(o.b58decode(s["serde_public_key_var_gen"], 64)), _a(o.b58decode(s["serde_signature_var_gen"], 64)), _a(mv), True)
    assert st[0] == 0 and c.tobytes().hex() == "648cf37f901b93870bec5cb3d7339934efd8307d7c667a3718cd14643a677603"
    pkb, sig, mb = legacy_double_fixture()
    assert bv.verify_double(_a(pkb), _a(sig), _a(mb))[0] == 1


@pytest.mark.parametrize("kind,n", [("single", 4096), ("double", 2048), ("vargen", 2048)])
def test_adversarial_batch_matches_oracle(bv, kind, n):
    gen = {"single": co.gen_single, "double": co.gen_double, "vargen": co.gen_vargen}[kind]
    cver = {"single": co.verify_single, "double": co.verify_double, "vargen": co.verify_vargen}[kind]
    gver = {"single": bv.verify_single, "double": bv.verify_double, "vargen": bv.verify_vargen}[kind]
    pk, sig, msg = gen(0xB200, n)
    pk, sig, msg, expected, names = adv.make_adversarial(kind, pk, sig, msg, seed=11, frac=0.4)
    st_o, c_o = cver(pk, sig, msg)
    st_g, c_g = gver(pk, sig, msg, True)
    bad = np.nonzero(st_g != st_o)[0]
    assert bad.size == 0, [(int(i), names[i], int(st_g[i]), int(st_o[i])) for i in bad[:10]]
    assert np.array_equal(st_o, expected)
    assert np.array_equal(c_g, c_o)
    assert set(st_g.tolist()) == {0, 1, 2, 3}


SPECIAL_U = [0, 1, 2, 7, 8, o.R_ORDER - 1, o.R_ORDER - 2, o.R_ORDER // 2, o.R_ORDER // 3, 1 << 84, 1 << 126, (1 << 126) - 1, 1 << 127, 1 << 168,
             (1 << 170) - 1, 1 << 250, (1 << 251) + 12345]


@pytest.mark.parametrize("kind", ["single", "double", "vargen"])
def test_special_response_scalars(bv, kind):
    """Response scalars u at the edges of the scalar decompositions (0, 1, r - 1, powers of two around the half-size and the
    three-scalar bounds) in otherwise valid items: the equation must simply fail, exactly as in the oracle, next to untouched
    valid items in the same warps."""
    gen = {"single": co.gen_single, "double": co.gen_double, "vargen": co.gen_vargen}[kind]
    cver = {"single": co.verify_single, "double": co.verify_double, "vargen": co.verify_vargen}[kind]
    gver = {"single": bv.verify_single, "double": bv.verify_double, "vargen": bv.verify_vargen}[kind]
    n = 4 * len(SPECIAL_U)
    pk, sig, msg = gen(0xB207, n)
    for j, u in enumerate(SPECIAL_U):
        sig[4 * j, :32] = np.frombuffer(u.to_bytes(32, "little"), dtype=np.uint8)
    st_o, c_o = cver(pk, sig, msg)
    st_g, c_g = gver(pk, sig, msg, True)
    assert (st_o[0::4] == 1).all() and not st_o[1::4].any()
    assert np.array_equal(st_g, st_o) and np.array_equal(c_g, c_o)


@pytest.mark.parametrize("kind", ["single", "double", "vargen"])
def test_torsion_shifted_signatures_are_invalid_points(bv, kind):
    """R = r*B + T (T of order 2, 4, 8) signed by the key holder: the equation holds up to torsion, so only the
    (deferred) subgroup test of R rejects them -- mixed into valid items so both branches share warps."""
    gen = {"single": co.gen_single, "double": co.gen_double, "vargen": co.gen_vargen}[kind]
    cver = {"single": co.verify_single, "double": co.verify_double, "vargen": co.verify_vargen}[kind]
    gver = {"single": bv.verify_single, "double": bv.verify_double, "vargen": bv.verify_vargen}[kind]
    n = 192
    fpk, fsig, fmsg, exp = adv.torsion_shifted_signatures(kind, n, seed=3)
    vpk, vsig, vmsg = gen(0xB201, n)
    pk, sig, msg = np.empty((2 * n, fpk.shape[1]), np.uint8), np.empty((2 * n, fsig.shape[1]), np.uint8), np.empty((2 * n, 32), np.uint8)
    pk[0::2], pk[1::2], sig[0::2], sig[1::2], msg[0::2], msg[1::2] = fpk, vpk, fsig, vsig, fmsg, vmsg
    st_o, c_o = cver(pk, sig, msg)
    st_g, c_g = gver(pk, sig, msg, True)
    assert np.array_equal(st_o[0::2], exp) and not st_o[1::2].any()
    assert np.array_equal(st_g, st_o) and np.array_equal(c_g, c_o)


@pytest.mark.parametrize("kind,n", [("single", 8192), ("double", 4096), ("vargen", 4096)])
def test_bitflip_fuzz_matches_oracle(bv, kind, n):
    """Random single-bit flips in keys, signatures and messages (half of them in the top byte of a field): statuses
    and challenges equal the oracle's on every item."""
    gen = {"single": co.gen_single, "double": co.gen_double, "vargen": co.gen_vargen}[kind]
    cver = {"single": co.verify_single, "double": co.verify_double, "vargen": co.verify_vargen}[kind]
    gver = {"single": bv.verify_single, "double": bv.verify_double, "vargen": bv.verify_vargen}[kind]
    pk, sig, msg = gen(0xF022, n)
    pk, sig, msg = adv.bitflip_fuzz(pk, sig, msg, seed=99)
    st_o, c_o = cver(pk, sig, msg)
    st_g, c_g = gver(pk, sig, msg, True)
    bad = np.nonzero(st_g != st_o)[0]
    assert bad.size == 0, [(int(i), int(st_g[i]), int(st_o[i])) for i in bad[:10]]
    assert np.array_equal(c_g, c_o)
    assert len(set(st_o.tolist())) >= 3      # the fuzz reaches decode failures, invalid points and bad signatures


def test_config0_2p16_valid_singles_item_by_item(bv):
    """BASELINE.json configs[0]: 2^16 random valid single signatures (the reference's CPU-runnable case), every status
    and every challenge scalar against the oracle, through the host entry point and through verify_batch's bitmap."""
    n = 1 << 16
    pk, sig, msg = co.gen_single(0xB200, n)
    st_o, c_o = co.verify_single(pk, sig, msg)
    assert not st_o.any()
    st_g, c_g = bv.verify_single(pk, sig, msg, True)
    assert np.array_equal(st_g, st_o) and np.array_equal(c_g, c_o)
    assert bv.unpack_bitmap(bv.verify_batch(pk, sig, msg), n).all()


def test_challenge_only_matches_oracle(bv):
    pk, sig, msg = co.gen_single(3, 512)
    _, c_o = co.verify_single(pk, sig, msg)
    assert np.array_equal(bv.challenge_only(0, pk, sig, msg), c_o)


def test_ragged_and_empty(bv):
    for n in (0, 1, 31, 33, 129):
        pk, sig, msg = co.gen_single(5, n)
        st = bv.verify_single(pk, sig, msg)
        assert st.shape == (n,) and (st == 0).all()


def test_fixed_base_tables_match_their_definition(bv):
    """The window tables for G and G' are built in two passes with shared inversions (csrc/curve.cuh, fb_combine_entries); a sample
    of entries -- the first and last digit of every window, batch boundaries, random ones -- is recomputed on the GPU by plain
    double-and-add from the definition digit * 2^(width * window) * B and must agree exactly.  (The tables are exercised end to end
    by every signing and verification test as well; this one localises a fault.)"""
    rng = np.random.default_rng(21)
    size = 12 << 21   # 12 windows of 2^21 entries (the device default, JJS_FB_W = 21)
    edges = [w * (1 << 21) + d for w in range(12) for d in (0, 1, 7, 8, 9, (1 << 11) - 1, 1 << 11, (1 << 11) + 1, (1 << 21) - 9, (1 << 21) - 8, (1 << 21) - 1)]
    idx = np.concatenate([np.asarray(edges, dtype=np.uint32), rng.integers(0, size, size=20000, dtype=np.uint32)])
    for which in (0, 1):
        assert bv.fb_table_check(which, idx) == 0


def test_subgroup_tate_equals_scalar_mul_definition(bv):
    """The production subgroup test (order-8 Tate pairing) against [r]P == identity on the GPU, over random curve
    points in every torsion coset, the torsion points themselves and undecodable strings."""
    rng = np.random.default_rng(17)
    n = 1 << 15
    pk, _, _ = co.gen_single(23, n // 8)
    t8 = adv.torsion()[8]
    pts = [pk]
    cur = pk
    for _ in range(7):  # P + j * T8
        cur = np.stack([_a(co.point_add(cur[i].tobytes(), t8)) for i in range(cur.shape[0])])
        pts.append(cur)
    rand = rng.integers(0, 256, size=(4096, 32), dtype=np.uint8)  # arbitrary strings: ~half decode, any coset
    tors = [o.point_to_bytes(o.IDENTITY)]
    for _ in range(7):
        tors.append(co.point_add(tors[-1], t8))
    allp = np.concatenate(pts + [rand, np.stack([_a(x) for x in tors])])
    a = bv.subgroup_check(allp, method=0)
    b = bv.subgroup_check(allp, method=1)
    assert np.array_equal(a, b)
    assert (a[: n // 8] == 1).all() and (a[n // 8: n] == 0).all()
    assert a[-8:].tolist() == [1, 0, 0, 0, 0, 0, 0, 0]
    ref = np.array([co.point_is_valid(allp[i].tobytes()) for i in range(n, n + 256)])  # oracle: -1 undecodable else is_valid
    got = a[n: n + 256].astype(np.int64)
    got[got == 255] = -1
    assert np.array_equal(got, ref)


def test_aggregate_key_verify_matches_oracle(bv):
    """multisig::aggregate_pk + PublicKey::verify (reference src/multisig.rs:154-156, 416-429): KAT, ragged signer
    counts, a tampered signature, a small-order signer key (not validated by aggregate_pk) and an undecodable key."""
    k = KAT["multisig_kat"]
    pks = _a(b"".join(bytes.fromhex(x) for x in k["PUBLIC_KEYS"]))
    st, c, agg = bv.verify_aggregate(pks, [0, 3], _a(bytes.fromhex(k["SIGNATURE"])), _a(o.le32(31)), True, True)
    assert st[0] == 0 and c.tobytes().hex() == k["CHALLENGE"] and agg.tobytes().hex() == k["AGGREGATE_PUBLIC_KEY"]
    rng = np.random.default_rng(3)
    signers = rng.integers(1, 6, size=600)
    signers[7] = 0  # empty signer set: the aggregate is the identity -> InvalidPoint
    pks, off, sig, msg = co.gen_aggregate(29, signers)
    sig[2, 0] ^= 1
    pks[off[3]] = _a(adv.torsion()[4])
    pks[off[4]] = _a(adv.off_curve_encoding(rng))
    sig[5, 32:] = _a(o.point_to_bytes(o.IDENTITY))
    msg[6] = 0xFF
    st_o, c_o, agg_o = co.verify_aggregate(pks, off, sig, msg)
    st_g, c_g, agg_g = bv.verify_aggregate(pks, off, sig, msg, True, True)
    assert np.array_equal(st_g, st_o) and np.array_equal(c_g, c_o)
    ok = st_o != 3  # the oracle leaves the aggregate unset when some field fails to decode
    assert np.array_equal(agg_g[ok], agg_o[ok])
    assert st_o[:8].tolist() == [0, 0, 1, 2, 3, 2, 3, 2]


def test_aggregate_key_has_no_signer_limit(bv):
    """aggregate_pk over 65 and 200 signers (reference src/multisig.rs:393-429 has no limit; round 1 stopped at 64): bit-exact
    status, challenge and aggregate key; then a batch whose signer counts straddle every bucket of the device-side ordering
    (the CPU oracle needs seconds per many-signer item: n hashes of 2 + 2 n elements each)."""
    signers = np.array([65, 200, 0, 64, 66, 1, 63], dtype=np.uint32)
    pks, off, sig, msg = co.gen_aggregate(31, signers)
    sig[4, 1] ^= 4
    st_o, c_o, agg_o = co.verify_aggregate(pks, off, sig, msg)
    assert st_o.tolist() == [0, 0, 2, 0, 1, 0, 0]
    st_g, c_g, agg_g = bv.verify_aggregate(pks, off, sig, msg, True, True)
    assert np.array_equal(st_g, st_o) and np.array_equal(c_g, c_o) and np.array_equal(agg_g, agg_o)
    rng = np.random.default_rng(5)
    signers = rng.integers(0, 70, size=300).astype(np.uint32)
    pks, off, sig, msg = co.gen_aggregate(37, signers)
    sig[::9, 0] ^= 1
    st_o, c_o, agg_o = co.verify_aggregate(pks, off, sig, msg)
    st_g, c_g, agg_g = bv.verify_aggregate(pks, off, sig, msg, True, True)
    assert np.array_equal(st_g, st_o) and np.array_equal(c_g, c_o) and np.array_equal(agg_g, agg_o)
    assert np.array_equal(bv.unpack_bitmap(bv.verify_batch_aggregate(pks, off, sig, msg), len(signers)), st_o == 0)


def test_multisig_combine_has_no_participant_limit(bv):
    """Sessions of 32, 40 and 100 participants (round 1 reported InvalidMultisigTranscript above 31): the reference's combine() result."""
    signers = np.array([32, 40, 3, 100, 31], dtype=np.uint32)
    pks, Rs, Ss, zs, off, msg = co.gen_multisig(47, signers)
    zs[off[3] + 57, 0] ^= 1
    st_o, bad_o, sig_o, ok_o = co.multisig_combine(pks, Rs, Ss, zs, off, msg)
    assert st_o.tolist() == [0, 0, 0, 5, 0] and bad_o[3] == 57
    st_g, bad_g, sig_g, ok_g = bv.multisig_combine(pks, Rs, Ss, zs, off, msg)
    assert np.array_equal(st_g, st_o) and np.array_equal(bad_g, bad_o) and np.array_equal(sig_g, sig_o) and np.array_equal(ok_g, ok_o)


def test_mixed_call_matches_separate_calls_and_oracle(bv):
    """jjs_verify_mixed: four kinds in one call (BASELINE configs[3] / [4] shape) against the oracle, item by item; bitmaps per part."""
    from jubjub_schnorr_b200 import batch as B
    n = 3000
    parts, oracle = [], []
    for kind, gen, ver in ((B.SINGLE, co.gen_single, co.verify_single), (B.DOUBLE, co.gen_double, co.verify_double), (B.VARGEN, co.gen_vargen, co.verify_vargen)):
        pk, sig, msg = gen(0xA0 + kind, n + 17 * kind)
        name = {B.SINGLE: "single", B.DOUBLE: "double", B.VARGEN: "vargen"}[kind]
        pk, sig, msg, _, _ = adv.make_adversarial(name, pk, sig, msg, seed=kind, frac=0.3)
        parts.append((kind, pk, sig, msg))
        oracle.append(ver(pk, sig, msg))
    signers = np.random.default_rng(2).integers(1, 6, size=n // 2).astype(np.uint32)
    pks, off, sig, msg = co.gen_aggregate(53, signers)
    sig[::5, 2] ^= 8
    parts.append((B.AGGREGATE, pks, sig, msg, off))
    st_a, c_a, agg_a = co.verify_aggregate(pks, off, sig, msg)
    parts.append((B.SINGLE, np.zeros((0, 32), np.uint8), np.zeros((0, 64), np.uint8), np.zeros((0, 32), np.uint8)))   # an empty part is fine
    res = bv.verify_mixed(parts, want_challenge=True, want_bitmap=True)
    for r, (st_o, c_o) in zip(res[:3], oracle):
        assert np.array_equal(r["status"], st_o) and np.array_equal(r["c"], c_o)
        assert np.array_equal(bv.unpack_bitmap(r["bitmap"], len(st_o)), st_o == 0)
    assert np.array_equal(res[3]["status"], st_a) and np.array_equal(res[3]["c"], c_a) and np.array_equal(res[3]["aggpk"], agg_a)
    assert res[4]["status"].size == 0
    # bitmap entry points of the other kinds
    assert np.array_equal(bv.unpack_bitmap(bv.verify_batch_double(*parts[1][1:4]), len(oracle[1][0])), oracle[1][0] == 0)
    assert np.array_equal(bv.unpack_bitmap(bv.verify_batch_vargen(*parts[2][1:4]), len(oracle[2][0])), oracle[2][0] == 0)


def test_gpu_signing_matches_reference_vectors(bv):
    """jjs_sign_batch reproduces the pinned signatures of reference tests/serde.rs (seed 2321) bit for bit."""
    s = KAT["serde_kat"]
    rng = o.StdRng(s["_seed"])
    sk, m, rnd = rng.random_fr(), rng.random_fq(), rng.random_fr()
    pk, sig = bv.sign_batch(0, _a(o.le32(sk)), _a(o.le32(rnd)), _a(o.le32(m)))
    assert o.b58encode(pk.tobytes()) == s["serde_public_key"] and o.b58encode(sig.tobytes()) == s["serde_signature"]
    pk, sig = bv.sign_batch(1, _a(o.le32(sk)), _a(o.le32(rnd)), _a(o.le32(m)))
    assert o.b58encode(pk.tobytes()) == s["serde_public_key_double"] and o.b58encode(sig.tobytes()) == s["serde_signature_double"]
    rng = o.StdRng(s["_seed"])
    sk, g, m, rnd = rng.random_fr(), rng.random_fr(), rng.random_fq(), rng.random_fr()
    pk, sig = bv.sign_batch(2, _a(o.le32(sk)), _a(o.le32(rnd)), _a(o.le32(m)), _a(o.le32(g)))
    assert o.b58encode(pk.tobytes()) == s["serde_public_key_var_gen"] and o.b58encode(sig.tobytes()) == s["serde_signature_var_gen"]


@pytest.mark.parametrize("vi,kind", [(0, "single"), (1, "double"), (2, "vargen")])
def test_typed_inputs_match_oracle(bv, vi, kind):
    """jjs_verify_ext (SURVEY 8(f) row 1): JubJubExtended coordinates in, same statuses and challenges as the wire path,
    plus the typed-only failure modes."""
    from tests import typed_inputs as ti
    gen = {"single": co.gen_single, "double": co.gen_double, "vargen": co.gen_vargen}[kind]
    gver = {"single": bv.verify_single, "double": bv.verify_double, "vargen": bv.verify_vargen}[kind]
    n = 1500
    pk, sig, msg = gen(0x7E, n)
    pk, sig, msg, _, _ = adv.make_adversarial(kind, pk, sig, msg, seed=3, frac=0.4)
    st_wire, c_wire = gver(pk, sig, msg, True)
    pts, u, keep = ti.to_typed(vi, pk, sig, msg, seed=4)
    pts, u, msg_k = pts[keep], u[keep], msg[keep]
    st_g, c_g = bv.verify_ext(vi, pts, u, msg_k, True)
    assert np.array_equal(st_g, st_wire[keep]) and np.array_equal(c_g, c_wire[keep])
    bad, expected = ti.corrupt_typed(pts, st_g, seed=5)
    st_o, c_o = co.verify_ext(vi, bad, u, msg_k)
    st_b, c_b = bv.verify_ext(vi, bad, u, msg_k, True)
    assert np.array_equal(st_b, st_o) and np.array_equal(c_b, c_o)
    assert set(st_b.tolist()) == {0, 1, 2, 3}


def test_multisig_combine_matches_oracle(bv):
    """jjs_multisig_combine (SURVEY 8(f) row 2): the pinned KAT, then 6000 generated sessions with tampered shares,
    swapped commitments, undecodable fields and empty sessions, item by item against the oracle; every combined
    signature is then verified under its aggregate key by the GPU verify path."""
    import json as _json
    import time
    k = KAT["multisig_kat"]
    arr = lambda xs: _a(b"".join(bytes.fromhex(x) for x in xs))
    st, bad, sig, ok = bv.multisig_combine(arr(k["PUBLIC_KEYS"]), arr(k["R_POINTS"]), arr(k["S_POINTS"]), arr(k["INDIVIDUAL_SHARES"]), [0, 3], _a(o.le32(31)))
    assert st[0] == 0 and sig.tobytes().hex() == k["SIGNATURE"] and ok.tolist() == [1, 1, 1]
    rng = np.random.default_rng(8)
    n = 6000
    signers = rng.integers(1, 6, size=n)
    signers[::97] = 0
    pks, Rs, Ss, zs, off, msg = co.gen_multisig(41, signers)
    for i in range(0, n, 7):
        if signers[i] == 0:
            continue
        j = off[i] + int(rng.integers(0, signers[i]))
        kind = (i // 7) % 5
        if kind == 0:
            zs[j, 0] ^= 1
        elif kind == 1:
            Rs[j] = Ss[j]
        elif kind == 2:
            pks[j] = _a(adv.off_curve_encoding(rng))
        elif kind == 3:
            zs[j] = 0xFF
        else:
            msg[i, 0] ^= 1
    st_o, bad_o, sig_o, ok_o = co.multisig_combine(pks, Rs, Ss, zs, off, msg)
    t0 = time.perf_counter()
    st_g, bad_g, sig_g, ok_g = bv.multisig_combine(pks, Rs, Ss, zs, off, msg)
    dt = time.perf_counter() - t0
    assert np.array_equal(st_g, st_o) and np.array_equal(bad_g, bad_o) and np.array_equal(sig_g, sig_o) and np.array_equal(ok_g, ok_o)
    assert set(st_o.tolist()) == {0, 3, 4, 5}
    good = np.nonzero(st_g == 0)[0]
    keys = np.concatenate([pks[off[i]:off[i + 1]] for i in good])
    goff = np.zeros(len(good) + 1, dtype=np.uint32)
    np.cumsum(signers[good], out=goff[1:])
    assert (bv.verify_aggregate(keys, goff, sig_g[good], msg[good]) == 0).all()
    # throughput on a larger batch of valid 3-party sessions (oracle spot check on a sample)
    nb = 1 << 16
    pks, Rs, Ss, zs, off, msg = co.gen_multisig(43, np.full(nb, 3))
    bv.multisig_combine(pks, Rs, Ss, zs, off, msg)
    t0 = time.perf_counter()
    st_b, _, sig_b, ok_b = bv.multisig_combine(pks, Rs, Ss, zs, off, msg)
    dt = time.perf_counter() - t0
    assert (st_b == 0).all() and (ok_b == 1).all()
    st_s, _, sig_s, _ = co.multisig_combine(pks[:3 * 256], Rs[:3 * 256], Ss[:3 * 256], zs[:3 * 256], off[:257], msg[:256])
    assert np.array_equal(st_s, st_b[:256]) and np.array_equal(sig_s, sig_b[:256])
    print(_json.dumps({"path": "jjs_multisig_combine (host buffers, 3 participants per session)", "sessions": nb, "participants": int(off[-1]),
                       "seconds": dt, "sessions_per_s": nb / dt, "shares_per_s": int(off[-1]) / dt}))


def test_fp64_pipe_multiplier_equals_integer_multiplier_on_device():
    """csrc/fq_fp.cuh (DFMA, 52-bit limbs) against csrc/fq.cuh (IMAD.WIDE) on 14.5 M random products on the GPU;
    the CPU twin of the same header is checked against big integers in tests/test_hostsim.py."""
    import subprocess
    import __graft_entry__ as entry
    entry.build_tools()
    out = subprocess.run([os.path.join(entry.ROOT, "tools", "microbench_fqfp")], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    res = json.loads(out.stdout)
    assert res["mismatches"] == 0 and res["checked"] > 10_000_000
