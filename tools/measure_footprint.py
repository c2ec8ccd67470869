#!/usr/bin/env python3
"""Memory-limited contexts (jjs_init_limited) against a jjs_init context, on one GPU, in one process.  Per context (jjs_init, and
limits of 8 GiB, 1 GiB and 256 MiB): the configuration it picked (fixed-base window width, items per pass), the device memory it
holds, the time of jjs_init / jjs_init_limited and of its first verification (1 024 singles, host buffers); the rates
device-resident (CUDA events around the calls) and from pinned host buffers (host clock around synchronous calls) on 2^20
singles and 2^20 doubles (10 % invalid) and on 2^20 keyed singles (2^10 keys), each alternated round by round with the same call
on the jjs_init context; and the host wall time of jjs_verify_single for n = 1 and n = 1 024.  Prints one JSON line (kept in
profiles/)."""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from jubjub_schnorr_b200 import BatchVerifier, JjsError  # noqa: E402
from jubjub_schnorr_b200 import workload as wl  # noqa: E402
from measure_keyed import gpu_info, timed_device, timed_host  # noqa: E402

LIMITS = [("jjs_init", None), ("8GiB", 8 << 30), ("1GiB", 1 << 30), ("256MiB", 256 << 20)]


def workloads(gen, n):
    """(name, variant or key-set keys, pinned host inputs, device inputs, expected status) per workload."""
    out = []
    for name, variant in (("single", wl.SINGLE), ("double", wl.DOUBLE)):
        pk, sig, msg, expected, _ = wl.make_batch(gen, variant, n, 0.10, seed=0xF0 + variant)
        h = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy() for a in (pk, sig, msg)]
        d = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (pk, sig, msg)]
        out.append((name, variant, h, d, expected))
    pks, idx, sig, msg, expected, _ = wl.make_keyed_batch(gen, wl.SINGLE, 1 << 10, n, 0.10, seed=0xF7)
    h = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy() for a in (idx, sig, msg)]
    d = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (idx.view(np.int32), sig, msg)]
    out.append(("keyed_single_1024", pks, h, d, expected))
    return out


def calls(bv, w, n, d_st, ks):
    name, arg, h, d, _ = w
    s = torch.cuda.current_stream().cuda_stream
    if name.startswith("keyed"):
        return (lambda: bv.verify_keyed(ks, *h),
                lambda: bv.verify_keyed_device(ks, d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), n, d_st.data_ptr(), stream=s))
    ver = bv.verify_single if arg == wl.SINGLE else bv.verify_double
    return (lambda: ver(*h), lambda: bv.verify_device(arg, d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), n, d_st.data_ptr(), stream=s))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--items", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("measure_footprint.py needs a CUDA device")
    info = gpu_info()
    n = a.items
    rows = []
    full = None
    for label, limit in LIMITS:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        bv = BatchVerifier([0], memory_limit=limit)
        init_ms = 1e3 * (time.perf_counter() - t0)
        if full is None:
            full = bv
            works = workloads(full, n)
            p1, s1, m1, _, _ = wl.make_batch(full, wl.SINGLE, 1024, 0.0, seed=0xF9)
        t0 = time.perf_counter()
        bv.verify_single(p1, s1, m1)
        first_ms = 1e3 * (time.perf_counter() - t0)
        mem = bv.memory_info()
        row = {"context": label, "limit_bytes": limit, "fb_window_bits": mem["fb_window_bits"], "items_in_flight": mem["items_in_flight"],
               "bytes_held_after_init_and_first_call": mem["bytes_held"], "init_ms": round(init_ms, 1), "first_verification_ms": round(first_ms, 2),
               "workloads": {}}
        for w in works:
            name, arg, _, _, expected = w
            ks = [None, None]
            if name.startswith("keyed"):
                try:   # 2^10 + 14 key tables take 408 MB: more than a 256 MiB context may hold
                    ks = [c.keyset_create(wl.SINGLE, arg) for c in (bv, full)]
                except JjsError as e:
                    if ks[0] is not None:
                        bv.keyset_destroy(ks[0])
                    row["workloads"][name] = {"refused": str(e)}
                    continue
            d_st = torch.empty(n, dtype=torch.uint8, device="cuda")
            (h_lim, d_lim), (h_full, d_full) = calls(bv, w, n, d_st, ks[0]), calls(full, w, n, d_st, ks[1])
            st = h_lim()
            st = st[0] if isinstance(st, tuple) else st
            assert np.array_equal(st, expected), name
            timed_device([d_lim, d_full], 1)
            timed_host([h_lim, h_full], 1)
            dev, host = [], []
            for _ in range(a.rounds):   # alternated: limited, jjs_init, limited, ...
                dev.append(timed_device([d_lim, d_full], a.steps))
                host.append(timed_host([h_lim, h_full], a.steps))
            d_lim()
            torch.cuda.synchronize()
            assert np.array_equal(d_st.cpu().numpy(), expected), name
            med = lambda rs, i: float(np.median([r[i] for r in rs]))  # noqa: E731
            row["workloads"][name] = {
                "device_resident_per_s": n / med(dev, 0) * 1e3, "device_resident_jjs_init_per_s": n / med(dev, 1) * 1e3,
                "device_ratio": med(dev, 1) / med(dev, 0),
                "host_pinned_per_s": n / med(host, 0) * 1e3, "host_pinned_jjs_init_per_s": n / med(host, 1) * 1e3,
                "host_ratio": med(host, 1) / med(host, 0),
                "device_ms": [[round(x, 3) for x in r] for r in dev], "host_ms": [[round(x, 3) for x in r] for r in host]}
            for c, k in zip((bv, full), ks):
                if k is not None:
                    c.keyset_destroy(k)
        lat = {}
        for m in (1, 1024):
            pk, sig, msg = p1[:m].copy(), s1[:m].copy(), m1[:m].copy()
            bv.verify_single(pk, sig, msg)
            t = timed_host([lambda: bv.verify_single(pk, sig, msg)], 50)[0]
            lat[str(m)] = round(t, 4)
        row["verify_single_host_ms"] = lat
        row["bytes_held_at_end"] = bv.memory_info()["bytes_held"]
        rows.append(row)
        if bv is not full:
            bv.close()
    full.close()
    print(json.dumps({"metric": "memory_limited_context_footprint_and_rates", "gpu": info, "items": n, "invalid_frac": 0.10, "steps": a.steps,
                      "rounds": a.rounds, "contexts": rows}))


if __name__ == "__main__":
    main()
