"""Synthetic batches for the bench (SURVEY.md section 8(d)): random keys / messages / signatures produced on the
GPU by jjs_sign_batch, then a fixed fraction of items is invalidated by byte-level edits whose result under
the reference's semantics is known by construction.  No oracle code is involved here.

Seed convention: numpy PCG64 seeded with (seed, rank, variant).  Scalars are 251 random bits (< r) and
messages 254 random bits (< q): enough entropy for a throughput workload, documented as such.
"""
from __future__ import annotations

import numpy as np

from .batch import DOUBLE, PK_SIZE, SIG_SIZE, SINGLE, VARGEN, BatchVerifier

Q_INT = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
R_INT = 0x0E7DB4EA6533AFA906673B0101343B00A6682093CCC81082D0970E5ED6F72CB7


def _le(x: int) -> np.ndarray:
    return np.frombuffer(x.to_bytes(32, "little"), dtype=np.uint8)


IDENTITY = _le(1)
ORDER2 = _le(Q_INT - 1)                      # (0, -1)
ORDER4 = _le(0)                              # (sqrt(-1) with even parity, 0)
ORDER8 = np.frombuffer(bytes.fromhex("dd96f4ef68200dffa1a484f390ee069166724dad3530a1162e986619b2bd58c9"), dtype=np.uint8)
OFF_CURVE = np.frombuffer(bytes.fromhex("0035c5bf742a2ff6de23941764d58bb90aa10b4bdcd78d8ab947c8ec8957e246"), dtype=np.uint8)
V_GE_Q = _le(Q_INT + 5)                      # non-canonical v
U_GE_R = _le(R_INT + 7)
M_GE_Q = _le(Q_INT + 11)
# Points of MIXED order, k * G + T with T of order 2, 4 or 8 (SURVEY 8(c): "PK = P + T", "R = valid R + T"): they decode, lie on
# the curve and are not the identity, so only is_torsion_free() rejects them.  Constants made once with the oracle's point
# arithmetic (tools/extract_golden.py documents the recipe: (1000003 (j + 1) + 17) * G + m * T_order); tests/test_abi.py checks them.
MIXED_ORDER = [np.frombuffer(bytes.fromhex(h), dtype=np.uint8) for h in (
    "f3f480af970d8742264b534b585c5c3ffda90b19a31f5287b0a533ee44cc4e18", "ebf0e228dff8472ef13783db34384a284bab12f45b0097b4c1937fefc4b0d999",
    "6553baa30b49ed3ffcbf2c3cee5f2224a56b0862e62478ebe324cfd61ef787f3", "d52dfe7fd1a7a00ae9a3362ab56b698eae104f00a0bea2c79dff9a71bae6bbec",
    "3879814d0e65f7fd2b4e628d8bbf7175d2b68f9f8fad8461eeb31d2879b23891", "3506cbd4a95aad5688e3d580b9da7310cf89c9a41a0e7759827abaeb39213ce1",
    "863ff5766785670f205a1becfe28b55d68c61ee4c5bf2f2d5cade46a7744aba8", "2cadc2aee2583016fa0a9e5e4b871aaa718819e8555667b0429898d3200c763b")]

# (name, status under the reference's semantics)
CLASSES = [
    ("u_plus_one", 1), ("u_ge_r", 3), ("msg_bit_flip", 1), ("msg_ge_q", 3), ("R_from_next_item", 1), ("R_sign_flip", 1),
    ("pk_from_next_item", 1), ("pk_identity", 2), ("R_identity", 2), ("pk_order2", 2), ("pk_order4", 2), ("R_order8", 2),
    ("pk_v_ge_q", 3), ("R_v_ge_q", 3), ("R_off_curve", 3), ("pk_off_curve", 3), ("pk_mixed_order", 2), ("R_mixed_order", 2),
]


def random_scalars(rng, n, bits):
    a = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    full, rem = divmod(bits, 8)
    a[:, full + (1 if rem else 0):] = 0
    if rem:
        a[:, full] &= (1 << rem) - 1
    return a


def make_valid(bv: BatchVerifier, variant: int, n: int, seed: int, rank: int = 0):
    rng = np.random.default_rng([seed, rank, variant])
    sk = random_scalars(rng, n, 251)
    sk[:, 0] |= 1  # never zero
    rnd = random_scalars(rng, n, 251)
    msg = random_scalars(rng, n, 254)
    gsc = None
    if variant == VARGEN:
        gsc = random_scalars(rng, n, 251)
        gsc[:, 0] |= 1
    pk, sig = bv.sign_batch(variant, sk, rnd, msg, gsc)
    return pk, sig, msg


def invalidate(variant: int, pk, sig, msg, frac: float, seed: int, rank: int = 0):
    """Tamper round(frac * n) items, classes in rotation.  Returns (pk, sig, msg, expected_status, class_index)."""
    rng = np.random.default_rng([seed, rank, variant, 99])
    n = msg.shape[0]
    pk, sig, msg = pk.copy(), sig.copy(), msg.copy()
    expected = np.zeros(n, dtype=np.uint8)
    cls = np.full(n, -1, dtype=np.int16)
    k = int(round(frac * n))
    idx = np.sort(rng.choice(n, size=k, replace=False)) if k else np.zeros(0, dtype=np.int64)
    chosen = np.zeros(n, dtype=bool)
    chosen[idx] = True
    orig_pk, orig_sig = pk.copy(), sig.copy()
    for j, i in enumerate(idx):
        c = j % len(CLASSES)
        name, st = CLASSES[c]
        nxt = (i + 1) % n
        if name == "u_plus_one":
            u = (int.from_bytes(sig[i, :32].tobytes(), "little") + 1) % R_INT
            sig[i, :32] = _le(u)
        elif name == "u_ge_r":
            sig[i, :32] = U_GE_R
        elif name == "msg_bit_flip":
            msg[i, 0] ^= 1
        elif name == "msg_ge_q":
            msg[i] = M_GE_Q
        elif name == "R_from_next_item":
            sig[i, 32:64] = orig_sig[nxt, 32:64]
        elif name == "R_sign_flip":
            sig[i, 63] ^= 0x80
        elif name == "pk_from_next_item":
            pk[i, :32] = orig_pk[nxt, :32]
        elif name == "pk_identity":
            pk[i, :32] = IDENTITY
        elif name == "R_identity":
            sig[i, 32:64] = IDENTITY
        elif name == "pk_order2":
            pk[i, :32] = ORDER2
        elif name == "pk_order4":
            pk[i, :32] = ORDER4
        elif name == "R_order8":
            sig[i, 32:64] = ORDER8
        elif name == "pk_v_ge_q":
            pk[i, :32] = V_GE_Q
        elif name == "R_v_ge_q":
            sig[i, 32:64] = V_GE_Q
        elif name == "R_off_curve":
            sig[i, 32:64] = OFF_CURVE
        elif name == "pk_off_curve":
            pk[i, :32] = OFF_CURVE
        elif name == "pk_mixed_order":
            pk[i, :32] = MIXED_ORDER[j % len(MIXED_ORDER)]
        elif name == "R_mixed_order":
            sig[i, 32:64] = MIXED_ORDER[j % len(MIXED_ORDER)]
        expected[i] = st
        cls[i] = c
    return pk, sig, msg, expected, cls


AGG_CLASSES = [
    ("u_plus_one", 1), ("u_ge_r", 3), ("msg_bit_flip", 1), ("msg_ge_q", 3), ("R_from_next_item", 1), ("R_sign_flip", 1),
    ("R_identity", 2), ("R_order8", 2), ("R_v_ge_q", 3), ("R_off_curve", 3), ("signer_key_from_next_item", 1),
    ("signer_key_off_curve", 3), ("signer_key_v_ge_q", 3), ("R_mixed_order", 2),
]


def make_aggregate_batch(bv: BatchVerifier, n: int, invalid_frac: float, seed: int = 0xB200, rank: int = 0, signers=(2, 3, 4)):
    """Aggregate-key items (SURVEY 8(d) config 4): signer counts uniform over `signers`, signed on the GPU, then a
    fraction invalidated.  Returns (pks[K,32], offsets[n+1], sig, msg, expected_status, class_index)."""
    rng = np.random.default_rng([seed, rank, 7])
    counts = rng.choice(np.asarray(signers, dtype=np.uint32), size=n)
    offsets = np.zeros(n + 1, dtype=np.uint32)
    np.cumsum(counts, out=offsets[1:])
    K = int(offsets[-1])
    sk = random_scalars(rng, K, 251)
    sk[:, 0] |= 1
    rnd = random_scalars(rng, n, 251)
    msg = random_scalars(rng, n, 254)
    pks, sig = bv.sign_aggregate_batch(sk, offsets, rnd, msg)
    expected = np.zeros(n, dtype=np.uint8)
    cls = np.full(n, -1, dtype=np.int16)
    k = int(round(invalid_frac * n))
    idx = np.sort(rng.choice(n, size=k, replace=False)) if k else np.zeros(0, dtype=np.int64)
    orig_sig, orig_pks = sig.copy(), pks.copy()
    for j, i in enumerate(idx):
        c = j % len(AGG_CLASSES)
        name, st = AGG_CLASSES[c]
        nxt = (i + 1) % n
        if name == "u_plus_one":
            sig[i, :32] = _le((int.from_bytes(sig[i, :32].tobytes(), "little") + 1) % R_INT)
        elif name == "u_ge_r":
            sig[i, :32] = U_GE_R
        elif name == "msg_bit_flip":
            msg[i, 0] ^= 1
        elif name == "msg_ge_q":
            msg[i] = M_GE_Q
        elif name == "R_from_next_item":
            sig[i, 32:] = orig_sig[nxt, 32:]
        elif name == "R_sign_flip":
            sig[i, 63] ^= 0x80
        elif name == "R_identity":
            sig[i, 32:] = IDENTITY
        elif name == "R_order8":
            sig[i, 32:] = ORDER8
        elif name == "R_v_ge_q":
            sig[i, 32:] = V_GE_Q
        elif name == "R_off_curve":
            sig[i, 32:] = OFF_CURVE
        elif name == "signer_key_from_next_item":
            pks[offsets[i]] = orig_pks[offsets[nxt]]
        elif name == "signer_key_off_curve":
            pks[offsets[i + 1] - 1] = OFF_CURVE
        elif name == "signer_key_v_ge_q":
            pks[offsets[i]] = V_GE_Q
        elif name == "R_mixed_order":
            sig[i, 32:] = MIXED_ORDER[j % len(MIXED_ORDER)]
        expected[i] = st
        cls[i] = c
    return pks, offsets, sig, msg, expected, cls


def make_typed_single_batch(bv: BatchVerifier, n: int, invalid_frac: float, seed: int = 0xB200, rank: int = 0):
    """Typed single-signature items (jjs_verify_ext): a wire batch whose point fields all decode, converted on the GPU
    to JubJubExtended coordinates with random z.  Returns (points[n,320], u[n,32], msg, expected_status)."""
    decodable = [i for i, (name, _) in enumerate(CLASSES) if name not in ("pk_v_ge_q", "R_v_ge_q", "R_off_curve", "pk_off_curve")]
    pk, sig, msg = make_valid(bv, SINGLE, n, seed, rank)
    pk, sig, msg, expected, cls = invalidate(SINGLE, pk, sig, msg, invalid_frac, seed, rank)
    undec = (cls >= 0) & ~np.isin(cls, decodable)
    # undecodable encodings cannot be typed: restore those items to their valid form
    pk0, sig0, msg0 = make_valid(bv, SINGLE, n, seed, rank)
    pk[undec], sig[undec], msg[undec], expected[undec] = pk0[undec], sig0[undec], msg0[undec], 0
    rng = np.random.default_rng([seed, rank, 31])
    z = random_scalars(rng, 2 * n, 254)
    z[:, 0] |= 1
    pts = bv.points_to_ext(np.concatenate([pk, sig[:, 32:]]), z)
    points = np.concatenate([pts[:n], pts[n:]], axis=1)
    return np.ascontiguousarray(points), np.ascontiguousarray(sig[:, :32]), msg, expected


# Invalid keys registered after the valid ones in make_keyed_batch: (class name, encoding of the key's first point)
KEYED_BAD_KEYS = [("pk_identity", IDENTITY), ("pk_order2", ORDER2), ("pk_order4", ORDER4), ("pk_v_ge_q", V_GE_Q), ("pk_off_curve", OFF_CURVE)] + \
    [("pk_mixed_order", m) for m in MIXED_ORDER]
KEYED_CLASSES = CLASSES + [("key_index_out_of_range", 3)]


def make_keyed_batch(bv: BatchVerifier, kind: int, n_keys: int, n: int, invalid_frac: float, seed: int = 0xB200, rank: int = 0):
    """Items under a registered key set (jjs_verify_keyed): n_keys signing keys, each item signed by one drawn uniformly, then a
    fraction invalidated with the classes of `invalidate` plus an out-of-range key index.  The key classes become indices:
    the set holds the n_keys signing keys, then one valid key that signs nothing (what `pk_from_next_item` points to when the
    next item has the same key) and the invalid keys of KEYED_BAD_KEYS (for DOUBLE their second point is a valid pk').
    Returns (pks[n_keys + 1 + len(KEYED_BAD_KEYS), PK_SIZE], key_index[n], sig, msg, expected_status, class_index)."""
    rng = np.random.default_rng([seed, rank, kind, 17])
    sk = random_scalars(rng, n_keys + 1, 251)
    sk[:, 0] |= 1
    idx = rng.integers(0, n_keys, size=n, dtype=np.int64).astype(np.uint32)
    rnd = random_scalars(rng, n_keys + 1 + n, 251)
    msg = random_scalars(rng, n_keys + 1 + n, 254)
    pk_all, sig_all = bv.sign_batch(kind, np.concatenate([sk, sk[idx]]), rnd, msg)
    good, sig, msg = pk_all[:n_keys + 1], sig_all[n_keys + 1:].copy(), msg[n_keys + 1:].copy()
    bad = np.repeat(good[:1], len(KEYED_BAD_KEYS), axis=0)
    for b, (_, enc) in enumerate(KEYED_BAD_KEYS):
        bad[b, :32] = enc
    pks = np.ascontiguousarray(np.concatenate([good, bad]))
    bad_of = {}
    for b, (name, _) in enumerate(KEYED_BAD_KEYS):
        bad_of.setdefault(name, []).append(n_keys + 1 + b)
    expected = np.zeros(n, dtype=np.uint8)
    cls = np.full(n, -1, dtype=np.int16)
    k = int(round(invalid_frac * n))
    chosen = np.sort(rng.choice(n, size=k, replace=False)) if k else np.zeros(0, dtype=np.int64)
    orig_sig, orig_idx = sig.copy(), idx.copy()
    for j, i in enumerate(chosen):
        c = j % len(KEYED_CLASSES)
        name, st = KEYED_CLASSES[c]
        nxt = (i + 1) % n
        if name == "u_plus_one":
            sig[i, :32] = _le((int.from_bytes(sig[i, :32].tobytes(), "little") + 1) % R_INT)
        elif name == "u_ge_r":
            sig[i, :32] = U_GE_R
        elif name == "msg_bit_flip":
            msg[i, 0] ^= 1
        elif name == "msg_ge_q":
            msg[i] = M_GE_Q
        elif name == "R_from_next_item":
            sig[i, 32:64] = orig_sig[nxt, 32:64]
        elif name == "R_sign_flip":
            sig[i, 63] ^= 0x80
        elif name == "pk_from_next_item":
            idx[i] = orig_idx[nxt] if orig_idx[nxt] != orig_idx[i] else n_keys
        elif name in ("R_identity", "R_order8", "R_v_ge_q", "R_off_curve", "R_mixed_order"):
            sig[i, 32:64] = {"R_identity": IDENTITY, "R_order8": ORDER8, "R_v_ge_q": V_GE_Q, "R_off_curve": OFF_CURVE,
                             "R_mixed_order": MIXED_ORDER[j % len(MIXED_ORDER)]}[name]
        elif name == "key_index_out_of_range":
            idx[i] = pks.shape[0] + j
        else:
            choices = bad_of[name]
            idx[i] = choices[j % len(choices)]
        expected[i] = st
        cls[i] = c
    return pks, idx, sig, msg, expected, cls


def make_batch(bv: BatchVerifier, variant: int, n: int, invalid_frac: float, seed: int = 0xB200, rank: int = 0):
    pk, sig, msg = make_valid(bv, variant, n, seed, rank)
    assert pk.shape == (n, PK_SIZE[variant]) and sig.shape == (n, SIG_SIZE[variant])
    return invalidate(variant, pk, sig, msg, invalid_frac, seed, rank)


__all__ = ["make_batch", "make_aggregate_batch", "make_keyed_batch", "make_valid", "invalidate", "CLASSES", "AGG_CLASSES", "KEYED_CLASSES", "SINGLE",
           "DOUBLE", "VARGEN"]
