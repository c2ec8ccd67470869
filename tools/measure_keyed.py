#!/usr/bin/env python3
"""Registered key sets (jjs_verify_keyed) against the same items with their keys written out (jjs_verify_single /
jjs_verify_double), on one GPU, in one process.  Per configuration (key kind, number of keys K): 2^20 items from
workload.make_keyed_batch with 10 % invalid items; the rates device-resident (device buffers, CUDA events around the calls)
and from pinned host buffers (host clock around synchronous calls), keyed and unkeyed runs alternated round by round; the
per-stage breakdown of both from a profiled second pass; the key-set build time and size.  Also the time to register 10 000
single keys.  Prints one JSON line (kept in profiles/)."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from jubjub_schnorr_b200 import BatchVerifier  # noqa: E402
from jubjub_schnorr_b200 import workload as wl  # noqa: E402

TABLE_BYTES_PER_POINT = 32 * 128 * 96


def gpu_info():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = (x.strip() for x in out.split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def timed_device(calls, steps):
    """ms per call of each callable, CUDA events around `steps` back-to-back calls on the current stream."""
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


def measure(bv, kind, K, n, steps, rounds, seed):
    pks, idx, sig, msg, expected, _ = wl.make_keyed_batch(bv, kind, K, n, 0.10, seed=seed)
    written = pks[np.minimum(idx, pks.shape[0] - 1)].copy()
    written[idx >= pks.shape[0], :32] = wl.V_GE_Q      # an unknown index reports like a key that does not decode
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ks = bv.keyset_create(kind, pks)
    build_ms = 1e3 * (time.perf_counter() - t0)
    try:
        unkeyed = bv.verify_single if kind == wl.SINGLE else bv.verify_double
        st, c = bv.verify_keyed(ks, idx, sig, msg, want_challenge=True)
        ust, uc = unkeyed(written, sig, msg, True)
        assert np.array_equal(st, expected) and np.array_equal(st, ust) and np.array_equal(c, uc)
        # host buffers (pinned)
        h_idx, h_sig, h_msg, h_pk = (torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy() for a in (idx, sig, msg, written))
        host_calls = [lambda: bv.verify_keyed(ks, h_idx, h_sig, h_msg), lambda: unkeyed(h_pk, h_sig, h_msg)]
        # device buffers
        d_idx, d_sig, d_msg, d_pk = (torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (idx.view(np.int32), sig, msg, written))
        d_st = torch.empty(n, dtype=torch.uint8, device="cuda")
        s = torch.cuda.current_stream().cuda_stream
        dev_calls = [lambda: bv.verify_keyed_device(ks, d_idx.data_ptr(), d_sig.data_ptr(), d_msg.data_ptr(), n, d_st.data_ptr(), stream=s),
                     lambda: bv.verify_device(kind, d_pk.data_ptr(), d_sig.data_ptr(), d_msg.data_ptr(), n, d_st.data_ptr(), stream=s)]
        timed_device(dev_calls, 2)   # warm-up of every shape
        timed_host(host_calls, 1)
        dev, host = [], []
        for _ in range(rounds):      # alternated: keyed, unkeyed, keyed, ...
            dev.append(timed_device(dev_calls, steps))
            host.append(timed_host(host_calls, steps))
        torch.cuda.synchronize()
        assert np.array_equal(d_st.cpu().numpy(), ust)   # the last call was the unkeyed device call
        dev_calls[0]()
        torch.cuda.synchronize()
        assert np.array_equal(d_st.cpu().numpy(), st)
        sk, su = stages(bv, dev_calls[0], steps), stages(bv, dev_calls[1], steps)
    finally:
        bv.keyset_destroy(ks)

    def rates(rows):
        k, u = float(np.median([r[0] for r in rows])), float(np.median([r[1] for r in rows]))
        return {"keyed_per_s": n / k * 1e3, "unkeyed_per_s": n / u * 1e3, "speedup": u / k, "keyed_ms": [round(r[0], 3) for r in rows],
                "unkeyed_ms": [round(r[1], 3) for r in rows]}
    return {"kind": "single" if kind == wl.SINGLE else "double", "keys": K, "registered_keys": int(pks.shape[0]),
            "table_bytes_per_key": TABLE_BYTES_PER_POINT * (kind + 1), "keyset_bytes": TABLE_BYTES_PER_POINT * (kind + 1) * int(pks.shape[0]),
            "keyset_create_ms": round(build_ms, 2), "device_resident": rates(dev), "host_buffers": rates(host),
            "stage_ms_per_step": {"keyed": sk, "unkeyed": su}, "equation_stage_ratio": round(sk["equation"] / su["equation"], 4),
            "outputs_match_unkeyed": True}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--items", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--configs", default="single:1,single:1024,single:65536,double:1024", help="kind:keys,...")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("measure_keyed.py needs a CUDA device")
    info = gpu_info()
    bv = BatchVerifier([0])
    # registration time of 10 000 single keys (after a small warm-up registration that loads the kernels)
    pks = wl.make_keyed_batch(bv, wl.SINGLE, 10_000, 1, 0.0, seed=1)[0][:10_000]
    bv.keyset_destroy(bv.keyset_create(wl.SINGLE, pks[:16]))
    create_ms = []
    for _ in range(3):
        t0 = time.perf_counter()
        ks = bv.keyset_create(wl.SINGLE, pks)
        create_ms.append(round(1e3 * (time.perf_counter() - t0), 2))
        bv.keyset_destroy(ks)
    configs = []
    for spec in a.configs.split(","):
        kind, K = spec.split(":")
        configs.append(measure(bv, {"single": wl.SINGLE, "double": wl.DOUBLE}[kind], int(K), a.items, a.steps, a.rounds, seed=0xB200 + len(configs)))
    bv.close()
    print(json.dumps({"metric": "keyed_vs_unkeyed_verifications_per_second", "gpu": info, "items": a.items, "invalid_frac": 0.10,
                      "steps": a.steps, "rounds": a.rounds, "keyset_create_10k_single_ms": create_ms, "configs": configs}))


if __name__ == "__main__":
    main()
