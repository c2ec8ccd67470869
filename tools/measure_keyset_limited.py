#!/usr/bin/env python3
"""Key sets within a byte budget (jjs_keyset_create_limited): every layout (key-window widths 8..4 and decoded points only) against
the 8-bit set of jjs_keyset_create and the unkeyed call, on one GPU, in one process.  Per configuration (key kind, number of keys
K): 2^20 items from workload.make_keyed_batch with 10 % invalid items; each layout is forced through the budget (a budget equal
to its peak footprint, the width read back with jjs_keyset_info); rates device-resident (CUDA events around the calls) and from
pinned host buffers (host clock around synchronous calls), all layouts and the unkeyed call alternated round by round, medians
over the rounds; outputs checked against the unkeyed call; create time and bytes per layout; the per-stage breakdown from a
profiled pass.  Also a 256 MiB limited context with 2^10 single keys and a 1 GiB one with 2^16 keys.  Prints one JSON line
(kept in profiles/)."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from jubjub_schnorr_b200 import BatchVerifier, JjsError  # noqa: E402
from jubjub_schnorr_b200 import workload as wl  # noqa: E402

LAYOUTS = [8, 7, 6, 5, 4, 0]


def gpu_info():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = (x.strip() for x in out.split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def peak_bytes(kind, n_keys, kw):
    """The peak footprint of a key set (include/jjschnorr_b200.h): 65 B of point and flags and 32 B of wire key per key point, with
    tables 96 B per entry and 128 B of window base per window."""
    nw = (251 + kw - 1) // kw if kw else 0
    return (kind + 1) * n_keys * (97 + (nw * (96 << (kw - 1)) + 128 * nw if kw else 0))


def timed_device(calls, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out = []
    for call in calls:
        e0.record()
        for _ in range(steps):
            call()
        e1.record()
        e1.synchronize()
        out.append(e0.elapsed_time(e1) / steps)
    return out


def timed_host(calls, steps):
    out = []
    for call in calls:
        t0 = time.perf_counter()
        for _ in range(steps):
            call()
        out.append(1e3 * (time.perf_counter() - t0) / steps)
    return out


def stages(bv, call, steps):
    bv.profile(True)
    for _ in range(steps):
        call()
    bv.profile(False)
    return {k: round(v[0] / steps, 3) for k, v in bv.profile_collect().items()}


def create(bv, kind, pks, limit):
    torch.cuda.synchronize()
    held = bv.memory_info()["bytes_held"]
    t0 = time.perf_counter()
    ks = bv.keyset_create(kind, pks, memory_limit=limit)
    ms = 1e3 * (time.perf_counter() - t0)
    assert bv.memory_info()["bytes_held"] - held == ks.bytes_per_device
    return ks, {"budget": limit, "key_window_bits": ks.key_window_bits, "bytes_per_device": ks.bytes_per_device, "create_ms": round(ms, 2)}


def measure(bv, kind, K, n, steps, rounds, seed, budgets):
    """A key set per entry of `budgets` ((bytes, expected width); bytes None: jjs_keyset_create) and the unkeyed call, alternated."""
    pks, idx, sig, msg, expected, _ = wl.make_keyed_batch(bv, kind, K, n, 0.10, seed=seed)
    written = pks[np.minimum(idx, pks.shape[0] - 1)].copy()
    written[idx >= pks.shape[0], :32] = wl.V_GE_Q      # an unknown index reports like a key that does not decode
    unkeyed = bv.verify_single if kind == wl.SINGLE else bv.verify_double
    ust, uc = unkeyed(written, sig, msg, True)
    assert np.array_equal(ust, expected)
    sets, info = [], []
    try:
        for budget, kw in budgets:
            ks, row = create(bv, kind, pks, budget)
            sets.append(ks)
            assert kw is None or ks.key_window_bits == kw
            st, c = bv.verify_keyed(ks, idx, sig, msg, want_challenge=True)
            assert np.array_equal(st, ust) and np.array_equal(c, uc)
            info.append(row)
        h_idx, h_sig, h_msg, h_pk = (torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy() for a in (idx, sig, msg, written))
        d_idx, d_sig, d_msg, d_pk = (torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (idx.view(np.int32), sig, msg, written))
        d_st = torch.empty(n, dtype=torch.uint8, device="cuda")
        s = torch.cuda.current_stream().cuda_stream
        dev_calls = [(lambda ks=ks: bv.verify_keyed_device(ks, d_idx.data_ptr(), d_sig.data_ptr(), d_msg.data_ptr(), n, d_st.data_ptr(), stream=s))
                     for ks in sets]
        dev_calls.append(lambda: bv.verify_device(kind, d_pk.data_ptr(), d_sig.data_ptr(), d_msg.data_ptr(), n, d_st.data_ptr(), stream=s))
        host_calls = [(lambda ks=ks: bv.verify_keyed(ks, h_idx, h_sig, h_msg)) for ks in sets] + [lambda: unkeyed(h_pk, h_sig, h_msg)]
        timed_device(dev_calls, 2)   # warm-up of every shape
        timed_host(host_calls, 1)
        dev, host = [], []
        for _ in range(rounds):      # alternated: every layout, then the unkeyed call, round after round
            dev.append(timed_device(dev_calls, steps))
            host.append(timed_host(host_calls, steps))
        for call in dev_calls:
            call()
            torch.cuda.synchronize()
            assert np.array_equal(d_st.cpu().numpy(), ust)
        st_prof = [stages(bv, call, steps) for call in dev_calls]
    finally:
        for ks in sets:
            bv.keyset_destroy(ks)

    def rate(rows, j):
        ms = float(np.median([r[j] for r in rows]))
        return {"per_s": round(n / ms * 1e3), "median_ms": round(ms, 3), "ms": [round(r[j], 3) for r in rows]}
    out = []
    for j, row in enumerate(info):
        row.update({"device_resident": rate(dev, j), "host_buffers": rate(host, j), "stage_ms_per_step": st_prof[j]})
        out.append(row)
    u = len(info)
    return {"kind": "single" if kind == wl.SINGLE else "double", "keys": K, "registered_keys": int(pks.shape[0]), "layouts": out,
            "unkeyed": {"device_resident": rate(dev, u), "host_buffers": rate(host, u), "stage_ms_per_step": st_prof[u]},
            "outputs_match_unkeyed": True}


def limited(limit, K, n, steps, rounds):
    """A jjs_init_limited context of `limit` bytes with K single keys: what jjs_keyset_create does, then the layout a budget of the
    whole limit gets and its rate against the unkeyed call on the same context."""
    with BatchVerifier([0], memory_limit=limit) as bv:
        held0 = bv.memory_info()["bytes_held"]
        pks = wl.make_keyed_batch(bv, wl.SINGLE, K, 1, 0.0, seed=7)[0]
        try:
            bv.keyset_destroy(bv.keyset_create(wl.SINGLE, pks))
            plain = "registered"
        except JjsError as e:
            plain = str(e)
        r = measure(bv, wl.SINGLE, K, n, steps, rounds, seed=0xB2A0 + K, budgets=[(limit, None)])
        r.update({"limit": limit, "context_bytes_held": held0, "keyset_create": plain})
        return r


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--items", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--configs", default="single:1024,single:65536,double:1024", help="kind:keys,...")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("measure_keyset_limited.py needs a CUDA device")
    info = gpu_info()
    configs = []
    with BatchVerifier([0]) as bv:
        for spec in a.configs.split(","):
            kind, K = spec.split(":")
            kind = {"single": wl.SINGLE, "double": wl.DOUBLE}[kind]
            n_keys = int(K) + 1 + len(wl.KEYED_BAD_KEYS)   # what make_keyed_batch registers
            configs.append(measure(bv, kind, int(K), a.items, a.steps, a.rounds, seed=0xB200 + len(configs),
                                   budgets=[(peak_bytes(kind, n_keys, kw), kw) for kw in LAYOUTS]))
    ctxs = [limited(256 << 20, 1 << 10, a.items, a.steps, a.rounds), limited(1 << 30, 1 << 16, a.items, a.steps, a.rounds)]
    line = json.dumps({"metric": "keyset_layouts_verifications_per_second", "gpu": info, "items": a.items, "invalid_frac": 0.10, "steps": a.steps,
                       "rounds": a.rounds, "configs": configs, "limited_contexts": ctxs})
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
