"""Grouped verification (jjs_verify_grouped) against per-item verification on a B200, in one process plus one child process per
A/B library.

For 2^20 items of each workload -- single, double, var-generator, aggregate-key (2-4 signers), a configs[3] mix (half
var-generator, half aggregate) and a configs[4] mix (half single, half double) -- with 0, 1, 16 and 256 equation-failing items
at random positions and with the bench's 10 % invalid classes, device-resident and from pinned host buffers, alternating the two
paths in each of three rounds (median reported):
  grouped  jjs_verify_grouped_device / jjs_verify_grouped
  items    the per-kind *_device entry points on one stream / jjs_verify_mixed
The outputs of both paths are compared item by item at every timed size.  Also: the crossover (the first failing-item count at
which the grouped call is slower), the per-stage split of one profiled call, and the card's name, power limit and clock read in
the same run.
--ab-dir: the group-size sweep (2^20 singles, 16 failing items, device-resident) over libraries built with -DJJS_GROUP_LOG2 =
12, 14, 16 and 0 (one group per pass), built there if missing.  --parent-lib: a library of the parent commit, whose one-part
jjs_verify_all_device on 2^20 singles is timed against this tree's, alternated in one child process each.
Writes JSON to --out (default gpu_out/measure_verify_grouped.json under the working directory).

    python tools/measure_verify_grouped.py [--n 1048576] [--rounds 3] [--ab-dir DIR] [--parent-lib PATH] [--out path]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from measure_verify_all import card  # noqa: E402

SINGLE, DOUBLE, VARGEN, AGGREGATE = 0, 1, 2, 3
R_ORDER = 0x0E7DB4EA6533AFA906673B0101343B00A6682093CCC81082D0970E5ED6F72CB7
GROUP_LOG2 = (12, 14, 16, 0)


def timed(torch, fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, r


def break_eq(sig, positions):
    """u + 1 mod r at the given items: their equations fail, nothing else changes"""
    sig = sig.copy()
    for i in positions:
        u = (int.from_bytes(sig[i, :32].tobytes(), "little") + 1) % R_ORDER
        sig[i, :32] = np.frombuffer(u.to_bytes(32, "little"), np.uint8)
    return sig


def child(args):
    """--child grouped|all: time one call shape on the library named by JJS_B200_LIB; prints one JSON line"""
    import types

    import torch

    class Lib(C.CDLL):   # a parent-commit library predates jjs_verify_grouped, whose prototypes _native sets
        def __getattr__(self, name):
            try:
                return super().__getattr__(name)
            except AttributeError:
                if name.startswith("jjs_verify_grouped"):
                    return types.SimpleNamespace()
                raise
    C.CDLL = Lib
    from jubjub_schnorr_b200 import BatchVerifier
    from jubjub_schnorr_b200 import workload as wl
    dev = torch.device("cuda:0")
    n = args.n
    with BatchVerifier([0]) as bv:
        stream = torch.cuda.current_stream(dev).cuda_stream
        pk, sig, msg = wl.make_valid(bv, SINGLE, n, seed=0x31)
        if args.child == "grouped":
            sig = break_eq(sig, np.random.default_rng(0x16).choice(n, 16, replace=False))
        d = [torch.from_numpy(a).to(dev) for a in (pk, sig, msg)]
        st = torch.empty(n, dtype=torch.uint8, device=dev)
        fb = torch.zeros(1, dtype=torch.int64, device=dev)
        out = torch.empty(1, dtype=torch.int32, device=dev)

        def grouped():
            bv.verify_grouped_device([(SINGLE, d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), n, st.data_ptr(), None, None, None)], fb.data_ptr(),
                                     stream=stream)
            return int((st != 0).sum().item())

        def whole():
            bv.verify_all_device(SINGLE, d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), n, out.data_ptr(), stream=stream)
            return int(out.item())
        fn = grouped if args.child == "grouped" else whole
        want = fn()
        times = []
        for _ in range(max(args.rounds, 5)):
            ms, r = timed(torch, fn)
            assert r == want
            times.append(ms)
        kernels = {}
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        for e in prof.key_averages():
            if e.device_type == torch.autograd.DeviceType.CUDA:
                kernels[e.key[:60]] = round(e.device_time_total / 1e3, 4)
        print(json.dumps({"ms": float(np.median(times)), "rounds": times, "result": want, "fallback_items": int(fb.item()),
                          "kernel_ms_profiled": kernels}), flush=True)


def run_child(mode, lib, args):
    env = dict(os.environ, JJS_B200_LIB=lib)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", mode, "--n", str(args.n), "--rounds", str(args.rounds)], env=env,
                       capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stderr[-4000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def sweep(args):
    import __graft_entry__ as entry
    os.makedirs(args.ab_dir, exist_ok=True)   # the one-group build is the A/B baseline, not a shipped option
    libs = {g: os.path.join(args.ab_dir, "libjjs_g%d.so" % g) for g in GROUP_LOG2}
    procs = [subprocess.Popen([os.environ.get("NVCC", "nvcc"), *entry.NVCC_FLAGS, "-DJJS_GROUP_LOG2=%d" % g, "-o", lib, os.path.join(entry.CSRC, "kernels.cu")])
             for g, lib in libs.items() if not os.path.exists(lib)]
    assert all(p.wait() == 0 for p in procs)
    out = {}
    for rnd in range(2):   # two passes over the variants, alternated
        for g, lib in libs.items():
            r = run_child("grouped", lib, args)
            out.setdefault("g=2^%d" % g if g else "one group per pass", []).append(r)
            print("sweep", g, json.dumps(r)[:200], flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--ab-dir", default=None)
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--child", default=None)
    ap.add_argument("--workloads", default="single,double,vargen,aggregate,configs3_vargen_aggregate,configs4_single_double")
    ap.add_argument("--out", default=os.path.join("gpu_out", "measure_verify_grouped.json"))
    args = ap.parse_args()
    if args.child:
        return child(args)
    import torch

    from jubjub_schnorr_b200 import BatchVerifier, _native
    from jubjub_schnorr_b200 import workload as wl
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    n, half = args.n, args.n // 2
    res = {"card": card(), "n": n, "rounds": args.rounds, "unit": "ms per call, median of the rounds"}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    if args.ab_dir:
        res["group_size_sweep_2^20_singles_16_failing_device"] = sweep(args)
    if args.parent_lib:
        this = os.path.join(ROOT, "jubjub_schnorr_b200", "libjjschnorr_b200.so")
        reg = {}
        for _ in range(2):
            for name, lib in (("parent", args.parent_lib), ("this", this)):
                reg.setdefault(name, []).append(run_child("all", lib, args))
        res["verify_all_device_one_part_single_vs_parent"] = reg
        print("parent", json.dumps({k: [r["ms"] for r in v] for k, v in reg.items()}), flush=True)

    with BatchVerifier([0]) as bv:
        stream = torch.cuda.current_stream(dev).cuda_stream

        def make(kind, m, seed, frac=0.0):
            if kind == AGGREGATE:
                pks, off, sig, msg, _, _ = wl.make_aggregate_batch(bv, m, frac, seed=seed)
                return (AGGREGATE, pks, sig, msg, off)
            return (kind, *wl.make_batch(bv, kind, m, frac, seed=seed)[:3])

        shapes = {
            "single": [(SINGLE, n)], "double": [(DOUBLE, n)], "vargen": [(VARGEN, n)], "aggregate": [(AGGREGATE, n)],
            "configs3_vargen_aggregate": [(VARGEN, half), (AGGREGATE, n - half)],
            "configs4_single_double": [(SINGLE, half), (DOUBLE, n - half)],
        }
        for name, shape in shapes.items():
            if name not in args.workloads.split(","):
                continue
            valid = [make(k, m, 0x40 + i) for i, (k, m) in enumerate(shape)]
            cases = {}
            rng = np.random.default_rng(0xBAD)
            for bad in (0, 1, 16, 256):
                pos = rng.choice(n, bad, replace=False)
                parts, lo = [], 0
                for p in valid:
                    m = p[3].shape[0]
                    here = [int(x) - lo for x in pos if lo <= x < lo + m]
                    parts.append((p[0], p[1], break_eq(p[2], here) if here else p[2], *p[3:]))
                    lo += m
                cases["%d_failing" % bad] = parts
            cases["10pct_invalid"] = [make(k, m, 0x50 + i, 0.1) for i, (k, m) in enumerate(shape)]
            rcase = {}
            for cname, parts in cases.items():
                pins = [[torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in p[1:]] for p in parts]
                devs = [[t.to(dev) for t in pp] for pp in pins]
                ms_ = [p[3].shape[0] for p in parts]
                st_d = {k: [torch.empty(m, dtype=torch.uint8, device=dev) for m in ms_] for k in ("g", "i")}
                st_h = {k: [torch.empty(m, dtype=torch.uint8).pin_memory() for m in ms_] for k in ("g", "i")}
                fb_d = torch.zeros(1, dtype=torch.int64, device=dev)
                fb_h = C.c_uint64(0)

                def grouped_dev():
                    dp = []
                    for i, p in enumerate(parts):
                        d = devs[i]
                        e = (p[0], d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), ms_[i], st_d["g"][i].data_ptr(), None, None, None)
                        if p[0] == AGGREGATE:
                            e += (d[3].data_ptr(), p[4])
                        dp.append(e)
                    bv.verify_grouped_device(dp, fb_d.data_ptr(), stream=stream)

                def items_dev():
                    for i, p in enumerate(parts):
                        d = devs[i]
                        if p[0] == AGGREGATE:
                            bv.verify_aggregate_device(d[0].data_ptr(), d[3].data_ptr(), p[4], d[1].data_ptr(), d[2].data_ptr(), ms_[i],
                                                       st_d["i"][i].data_ptr(), stream=stream)
                        else:
                            bv.verify_device(p[0], d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), ms_[i], st_d["i"][i].data_ptr(), stream=stream)

                def host_parts(key):
                    out = []
                    for i, p in enumerate(parts):
                        h = pins[i]
                        out.append(_native.Part(p[0], h[0].data_ptr(), h[3].data_ptr() if p[0] == AGGREGATE else None, h[1].data_ptr(), h[2].data_ptr(),
                                                ms_[i], st_h[key][i].data_ptr(), None, None, None))
                    return (_native.Part * len(out))(*out)

                def grouped_host():
                    assert bv._lib.jjs_verify_grouped(bv._ctx, host_parts("g"), len(parts), None, C.byref(fb_h)) == 0, bv._lib.jjs_last_error(bv._ctx)

                def items_host():
                    assert bv._lib.jjs_verify_mixed(bv._ctx, host_parts("i"), len(parts)) == 0, bv._lib.jjs_last_error(bv._ctx)

                fns = {"grouped_device": grouped_dev, "items_device": items_dev, "grouped_host": grouped_host, "items_host": items_host}
                for f in fns.values():   # warm-up (scratch growth, module load, sort-algorithm choice)
                    f()
                    # the device-buffer calls only enqueue on `stream`, and a host-buffer call of the same context reuses their
                    # scratch without waiting for that stream: every call ends before the next starts
                    torch.cuda.synchronize()
                times = {k: [] for k in fns}
                for _ in range(args.rounds):
                    for k, f in fns.items():
                        ms, _ = timed(torch, f)
                        times[k].append(ms)
                    same = all(torch.equal(a, b) for a, b in zip(st_d["g"], st_d["i"])) and all(torch.equal(a, b) for a, b in zip(st_h["g"], st_h["i"]))
                    same = same and all(torch.equal(a.cpu(), b) for a, b in zip(st_d["g"], st_h["g"]))
                    assert same, (name, cname)
                r = {k: float(np.median(v)) for k, v in times.items()}
                r["all_rounds"] = times
                r["statuses_identical"] = True
                r["nonzero_statuses"] = int(sum(int((s != 0).sum()) for s in st_h["i"]))
                r["fallback_items_device"] = int(fb_d.item())
                r["fallback_items_host"] = int(fb_h.value)
                r["speedup_device"] = r["items_device"] / r["grouped_device"]
                r["speedup_host"] = r["items_host"] / r["grouped_host"]
                if cname == "16_failing":
                    bv.profile(True)
                    bv.profile_collect()
                    grouped_dev()
                    r["stages_grouped_device_profiled"] = bv.profile_collect()
                    items_dev()
                    r["stages_items_device_profiled"] = bv.profile_collect()
                    bv.profile(False)
                rcase[cname] = r
                print(name, cname, json.dumps({k: v for k, v in r.items() if not isinstance(v, (dict, list))}), flush=True)
                del pins, devs, st_d, st_h
                torch.cuda.empty_cache()
            ladder = ("0_failing", "1_failing", "16_failing", "256_failing", "10pct_invalid")
            rcase["crossover_device"] = next((c for c in ladder if rcase[c]["grouped_device"] > rcase[c]["items_device"]), "none up to 10 % invalid")
            rcase["crossover_host"] = next((c for c in ladder if rcase[c]["grouped_host"] > rcase[c]["items_host"]), "none up to 10 % invalid")
            res[name] = rcase
            with open(args.out + ".partial", "w") as f:
                json.dump(res, f, indent=1)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
