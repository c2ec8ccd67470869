"""Whole-batch verification (jjs_verify_all) against per-item verification plus an all() on a B200, in one process.

For 2^20 all-valid single and double items, device-resident and from pinned host buffers, alternating the two in each of three
rounds (median reported):
  all     jjs_verify_all_device / jjs_verify_all
  items   jjs_verify_single_device / _double_device + (status == 0).all() on the device, read back;
          jjs_verify_single / _double from pinned buffers + numpy all() on the host
plus the time of a batch with one bad item (what a caller pays before falling back to per-item verification), the per-stage
split of one profiled jjs_verify_all pass, and the registers and spills of the k_rlc_* kernels from `-Xptxas -v`.
Writes JSON to --out (default gpu_out/measure_verify_all.json under the working directory).

    python tools/measure_verify_all.py [--n 1048576] [--rounds 3] [--out path]
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def ptxas_rlc():
    """registers / spill bytes of the whole-batch kernels, from a compile of kernels.cu with -Xptxas -v"""
    import __graft_entry__ as entry
    with tempfile.TemporaryDirectory() as d:
        r = subprocess.run([os.environ.get("NVCC", "nvcc"), *entry.NVCC_FLAGS, "-Xptxas", "-v", "-o", os.path.join(d, "lib.so"),
                            os.path.join(entry.CSRC, "kernels.cu")], capture_output=True, text=True)
    out, cur = {}, None
    for line in r.stderr.splitlines():
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            k = re.search(r"(k_rlc_\w+?)(?:I|E|P)", m.group(1))
            cur = None
            if k:
                cur = k.group(1) + ("<12>" if "ILi12E" in m.group(1) else "<21>" if "ILi21E" in m.group(1) else "")
            continue
        if cur is None:
            continue
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m:
            out.setdefault(cur, {})["spill_bytes"] = int(m.group(1)) + int(m.group(2))
        m = re.search(r"Used (\d+) registers", line)
        if m:
            out.setdefault(cur, {})["registers"] = int(m.group(1))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join("gpu_out", "measure_verify_all.json"))
    args = ap.parse_args()
    import torch

    from jubjub_schnorr_b200 import BatchVerifier
    from jubjub_schnorr_b200 import workload as wl
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    res = {"card": card(), "n": args.n, "rounds": args.rounds, "unit": "ms per call, median of the rounds",
           "estimate_from_issue": {"single_all_valid_ms": "mid-30s against ~49 per step", "gain": "+30-40 %"}}
    seed = bytes(range(32))
    with BatchVerifier([0]) as bv:
        for vi, name in ((wl.SINGLE, "single"), (wl.DOUBLE, "double")):
            pk, sig, msg = wl.make_valid(bv, vi, args.n, seed=0x11 + vi)
            bad_sig = sig.copy()
            bad_sig[args.n // 2, 0] ^= 1
            pins = [torch.from_numpy(a).pin_memory() for a in (pk, sig, msg, bad_sig)]
            dts = [p.to(dev) for p in pins]
            st_h = torch.empty(args.n, dtype=torch.uint8).pin_memory()
            st_d = torch.empty(args.n, dtype=torch.uint8, device=dev)
            out_d = torch.empty(1, dtype=torch.int32, device=dev)
            stream = torch.cuda.current_stream(dev).cuda_stream

            def t(fn):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                r = fn()
                torch.cuda.synchronize()
                return (time.perf_counter() - t0) * 1e3, r

            def all_dev(s_i=1):
                bv.verify_all_device(vi, dts[0].data_ptr(), dts[s_i].data_ptr(), dts[2].data_ptr(), args.n, out_d.data_ptr(), stream=stream)
                return bool(out_d.item())

            def items_dev(s_i=1):
                bv.verify_device(vi, dts[0].data_ptr(), dts[s_i].data_ptr(), dts[2].data_ptr(), args.n, st_d.data_ptr(), stream=stream)
                return bool((st_d == 0).all().item())

            def all_host(s_i=1):
                ok = C_all_host(s_i)
                return ok

            def C_all_host(s_i):
                import ctypes as C
                okv = C.c_int(0)
                rc = bv._lib.jjs_verify_all(bv._ctx, vi, pins[0].data_ptr(), pins[s_i].data_ptr(), pins[2].data_ptr(), args.n, None, C.byref(okv))
                assert rc == 0, bv._lib.jjs_last_error(bv._ctx)
                return bool(okv.value)

            def items_host(s_i=1):
                bv.verify_host_ptr(vi, pins[0].data_ptr(), pins[s_i].data_ptr(), pins[2].data_ptr(), args.n, st_h.data_ptr())
                return bool(np.all(st_h.numpy() == 0))

            fns = {"all_device": all_dev, "items_device": items_dev, "all_host": all_host, "items_host": items_host}
            for f in fns.values():   # warm-up (scratch allocation, module load, sort-algorithm choice)
                assert f() is True
            times = {k: [] for k in fns}
            for _ in range(args.rounds):
                for k, f in fns.items():
                    ms, ok = t(f)
                    assert ok is True
                    times[k].append(ms)
            r = {k: float(np.median(v)) for k, v in times.items()}
            r["all_rounds"] = times
            r["speedup_device"] = r["items_device"] / r["all_device"]
            r["speedup_host"] = r["items_host"] / r["all_host"]
            bad = [t(lambda: all_dev(3)) for _ in range(args.rounds)]
            assert all(ok is False for _, ok in bad)
            r["one_bad_item_all_device"] = float(np.median([ms for ms, _ in bad]))
            badi = [t(lambda: items_dev(3)) for _ in range(args.rounds)]
            assert all(ok is False for _, ok in badi)
            r["one_bad_item_items_device"] = float(np.median([ms for ms, _ in badi]))
            bv.profile(True)
            bv.profile_collect()
            assert all_dev() is True
            r["stages_all_device_profiled"] = bv.profile_collect()
            assert items_dev() is True
            r["stages_items_device_profiled"] = bv.profile_collect()
            bv.profile(False)
            res[name] = r
            print(name, json.dumps({k: v for k, v in r.items() if not isinstance(v, dict)}), flush=True)
    res["ptxas"] = ptxas_rlc()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["ptxas"]))


if __name__ == "__main__":
    main()
