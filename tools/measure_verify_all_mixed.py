"""Whole-batch verification across kinds (jjs_verify_all_mixed) against per-item verification plus an all() on a B200, in one
process.

For 2^20 all-valid items of each workload -- var-generator, aggregate-key (2-4 signers), a configs[3] mix (half var-generator,
half aggregate) and a configs[4] mix (half single, half double) -- device-resident and from pinned host buffers, alternating
the two in each of three rounds (median reported):
  all     jjs_verify_all_mixed_device / jjs_verify_all_mixed
  items   the per-kind *_device entry points on one stream + (status == 0).all() on the device, read back;
          jjs_verify_mixed from pinned buffers + numpy all() on the host
plus the time of a call with one bad item, a one-part single call against jjs_verify_all (both device-resident, alternated),
the per-stage split of one profiled call of each, and the card's name, power limit and clock read in the same run.
Writes JSON to --out (default gpu_out/measure_verify_all_mixed.json under the working directory).

    python tools/measure_verify_all_mixed.py [--n 1048576] [--rounds 3] [--out path]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from measure_verify_all import card, ptxas_rlc  # noqa: E402

SINGLE, DOUBLE, VARGEN, AGGREGATE = 0, 1, 2, 3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join("gpu_out", "measure_verify_all_mixed.json"))
    args = ap.parse_args()
    import torch

    from jubjub_schnorr_b200 import BatchVerifier, _native
    from jubjub_schnorr_b200 import workload as wl
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    n, half = args.n, args.n // 2
    res = {"card": card(), "n": n, "rounds": args.rounds, "unit": "ms per call, median of the rounds",
           "estimate_from_issue": {"vargen": "1.3-1.4x", "aggregate": "~1.1x"}}

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3, r

    with BatchVerifier([0]) as bv:
        stream = torch.cuda.current_stream(dev).cuda_stream

        def make(kind, m, seed):
            if kind == AGGREGATE:
                pks, off, sig, msg, _, _ = wl.make_aggregate_batch(bv, m, 0.0, seed=seed)
                return (AGGREGATE, pks, sig, msg, off)
            return (kind, *wl.make_valid(bv, kind, m, seed=seed))

        workloads = {
            "vargen": [make(VARGEN, n, 0x21)],
            "aggregate": [make(AGGREGATE, n, 0x22)],
            "configs3_vargen_aggregate": [make(VARGEN, half, 0x23), make(AGGREGATE, n - half, 0x24)],
            "configs4_single_double": [make(SINGLE, half, 0x25), make(DOUBLE, n - half, 0x26)],
        }
        for name, parts in workloads.items():
            # pinned host copies, device copies, and the same with one bad item (the last item of the last part)
            pins, devs, bad_pins, bad_devs = [], [], [], []
            for p in parts:
                arrs = [np.ascontiguousarray(a) for a in p[1:]]
                pins.append([torch.from_numpy(a).pin_memory() for a in arrs])
                devs.append([t.to(dev) for t in pins[-1]])
            bsig = parts[-1][2].copy()
            bsig[-1, 0] ^= 1
            bad_pin = torch.from_numpy(bsig).pin_memory()
            bad_dev = bad_pin.to(dev)
            st_d = [torch.empty(p[3].shape[0], dtype=torch.uint8, device=dev) for p in parts]
            st_h = [torch.empty(p[3].shape[0], dtype=torch.uint8).pin_memory() for p in parts]
            out_d = torch.empty(1, dtype=torch.int32, device=dev)

            def sig_of(i, host, bad):
                if bad and i == len(parts) - 1:
                    return bad_pin if host else bad_dev
                return (pins if host else devs)[i][1]

            def all_dev(bad=False):
                dp = []
                for i, p in enumerate(parts):
                    d = devs[i]
                    e = (p[0], d[0].data_ptr(), sig_of(i, False, bad).data_ptr(), d[2].data_ptr(), p[3].shape[0])
                    if p[0] == AGGREGATE:
                        e += (d[3].data_ptr(), p[4])
                    dp.append(e)
                bv.verify_all_mixed_device(dp, out_d.data_ptr(), stream=stream)
                return bool(out_d.item())

            def items_dev(bad=False):
                for i, p in enumerate(parts):
                    d, m = devs[i], p[3].shape[0]
                    if p[0] == AGGREGATE:
                        bv.verify_aggregate_device(d[0].data_ptr(), d[3].data_ptr(), p[4], sig_of(i, False, bad).data_ptr(), d[2].data_ptr(), m,
                                                   st_d[i].data_ptr(), stream=stream)
                    else:
                        bv.verify_device(p[0], d[0].data_ptr(), sig_of(i, False, bad).data_ptr(), d[2].data_ptr(), m, st_d[i].data_ptr(), stream=stream)
                return bool(all((s == 0).all().item() for s in st_d))

            def host_parts(with_status):
                out = []
                for i, p in enumerate(parts):
                    h = pins[i]
                    out.append(_native.Part(p[0], h[0].data_ptr(), h[3].data_ptr() if p[0] == AGGREGATE else None, h[1].data_ptr(), h[2].data_ptr(),
                                            p[3].shape[0], st_h[i].data_ptr() if with_status else None, None, None, None))
                return (_native.Part * len(out))(*out)

            def all_host():
                ok = C.c_int(0)
                rc = bv._lib.jjs_verify_all_mixed(bv._ctx, host_parts(False), len(parts), None, C.byref(ok))
                assert rc == 0, bv._lib.jjs_last_error(bv._ctx)
                return bool(ok.value)

            def items_host():
                rc = bv._lib.jjs_verify_mixed(bv._ctx, host_parts(True), len(parts))
                assert rc == 0, bv._lib.jjs_last_error(bv._ctx)
                return bool(all(np.all(s.numpy() == 0) for s in st_h))

            fns = {"all_device": all_dev, "items_device": items_dev, "all_host": all_host, "items_host": items_host}
            for f in fns.values():   # warm-up (scratch growth, module load, sort-algorithm choice)
                assert f() is True
            times = {k: [] for k in fns}
            for _ in range(args.rounds):
                for k, f in fns.items():
                    ms, ok = timed(f)
                    assert ok is True, (name, k)
                    times[k].append(ms)
            r = {k: float(np.median(v)) for k, v in times.items()}
            r["all_rounds"] = times
            r["speedup_device"] = r["items_device"] / r["all_device"]
            r["speedup_host"] = r["items_host"] / r["all_host"]
            bad = [timed(lambda: all_dev(True)) for _ in range(args.rounds)]
            assert all(ok is False for _, ok in bad)
            r["one_bad_item_all_device"] = float(np.median([ms for ms, _ in bad]))
            bv.profile(True)
            bv.profile_collect()
            assert all_dev() is True
            r["stages_all_device_profiled"] = bv.profile_collect()
            assert items_dev() is True
            r["stages_items_device_profiled"] = bv.profile_collect()
            bv.profile(False)
            res[name] = r
            print(name, json.dumps({k: v for k, v in r.items() if not isinstance(v, dict)}), flush=True)
            del pins, devs, st_d, st_h
            torch.cuda.empty_cache()

        # a one-part single call against jjs_verify_all on the same items, alternated
        pk, sig, msg = wl.make_valid(bv, SINGLE, n, seed=0x27)
        d = [torch.from_numpy(a).to(dev) for a in (pk, sig, msg)]
        out_d = torch.empty(1, dtype=torch.int32, device=dev)
        fns = {
            "verify_all_device": lambda: (bv.verify_all_device(SINGLE, d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), n, out_d.data_ptr(), stream=stream),
                                          bool(out_d.item()))[1],
            "verify_all_mixed_device": lambda: (bv.verify_all_mixed_device([(SINGLE, d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), n)], out_d.data_ptr(),
                                                                           stream=stream), bool(out_d.item()))[1],
        }
        for f in fns.values():
            assert f() is True
        times = {k: [] for k in fns}
        for _ in range(max(args.rounds, 5)):
            for k, f in fns.items():
                ms, ok = timed(f)
                assert ok is True
                times[k].append(ms)
        r = {k: float(np.median(v)) for k, v in times.items()}
        r["all_rounds"] = times
        res["one_part_single"] = r
        print("one_part_single", json.dumps({k: v for k, v in r.items() if not isinstance(v, dict)}), flush=True)
    res["ptxas"] = ptxas_rlc()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["ptxas"]))


if __name__ == "__main__":
    main()
