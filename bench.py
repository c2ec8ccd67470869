#!/usr/bin/env python3
"""bench.py -- Schnorr verifications per second on B200 (BASELINE.json metric), one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload single|double|vargen] [--log2n 20]
                    [--dump-outputs DIR]

A step is one pass of the verify path over one synthetic batch (default: BASELINE.json configs[1], 2^20 single
signatures with 10 % invalid items per GPU; weak scaling, every rank owns its own batch).
  value     whole-job verifications/s with the wire-format inputs already resident in HBM (device entry points,
            CUDA events on the launching stream, max over ranks)
  e2e       same metric through the host-buffer C ABI call a reference user would make (pinned host buffers,
            H2D + D2H inside the timed region)
  e2e_pageable  the same call from ordinary (pageable) numpy memory, what a Rust Vec<u8> is
  roofline  dominant kernel against the measured INT32-multiply peak (profiles/r01_microbench_int.json); this
            path is bound by the integer multiply pipe, not by HBM or tensor cores (DESIGN.md section 4).
            frac counts the CANONICAL algorithm's multiplies (SURVEY 8(d) contract); roofline.executed counts the
            IMAD.WIDE the kernels really execute (ncu, profiles/r*_executed_mac32.json) and is the pipe-efficiency figure
  strong_2p24   BASELINE.json configs[4]: a 2^24-item half single / half double batch through ONE context over all N
            GPUs and ONE jjs_verify_mixed host call (rank 0; under torchrun the other ranks wait on a CPU barrier)
  cpu_baseline  BASELINE.json configs[0]: 2^16 valid single signatures through the oracle's C port of the reference
            algorithm on all host threads
--impl reference times that CPU port on a bounded sample of the GPU arm's workload (same invalid mix; the reference is
Rust and cannot be built here; see DESIGN.md).
--dump-outputs DIR writes what the last timed step computed (see dump_outputs), so that two builds run with the same
arguments, and therefore the same seeded inputs, can be compared output for output.
"""
from __future__ import annotations

import argparse
import glob
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "schnorr_verifications_per_second"
UNIT = "verifications/s"
# canonical algorithmic work, SURVEY.md section 8(d) / Appendix C: MAC32 = one 32x32->64 multiply(-accumulate)
MAC32_M, MAC32_S = 136, 108
MAC32_PER_ITEM = {"single": 4399 * MAC32_M + 2964 * MAC32_S, "double": 7932 * MAC32_M + 5728 * MAC32_S, "vargen": 5808 * MAC32_M + 4248 * MAC32_S}
# per-launch units of the kernels (canonical counts): one equation u*B + c*PK (table + Straus + compare), one subgroup check
MAC32_EQUATION = (1358 + 68 + 2) * MAC32_M + (1008 + 4) * MAC32_S
MAC32_EQUATION_VARGEN = (1512 + 2 * 68 + 2) * MAC32_M + (1008 + 8) * MAC32_S
MAC32_SUBGROUP = (1134 + 68) * MAC32_M + (1008 + 4) * MAC32_S
MAC32_DECODE = 53 * MAC32_M + 272 * MAC32_S
MAC32_PERMUTATION = 865 * MAC32_M + 200 * MAC32_S
BYTES_IN = {"single": 128, "double": 192, "vargen": 160}


def int32_peak():
    """Measured IMAD.WIDE carry-chain issue rate on this pool's B200 (tools/microbench_int.cu), T MAC32/s."""
    path = os.path.join(ROOT, "profiles", "r01_microbench_int.json")
    try:
        data = json.load(open(path))
        for r in data["results"]:
            if r["kernel"].startswith("imad_wide_carry_chain (") :
                return float(r["mult_Tops_per_s"]), "measured: profiles/r01_microbench_int.json (mad.lo.cc/madc.hi.cc chains -> IMAD.WIDE.U32)"
    except Exception:
        pass
    return 32 * 148 * 1.965e9 / 1e12, "nominal: 32 IMAD.WIDE lanes/clk/SM x 148 SMs x 1.965 GHz"


class ClockSampler:
    """nvidia-smi streaming every 100 ms during the timed region (B200_PROFILING.md, clocks line)."""
    QUERY = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
        time.sleep(0.25)  # let the first samples land inside the timed region

    def stop(self):
        samples = []
        if self.proc is not None:
            self.proc.terminate()
            try:
                out, _ = self.proc.communicate(timeout=5)
            except Exception:
                self.proc.kill()
                out = ""
            samples = [[x.strip() for x in line.split(",")] for line in out.splitlines() if line.strip()]
        sm = sorted(int(s[0]) for s in samples if s and s[0].isdigit())
        mx = [int(s[1]) for s in samples if len(s) > 1 and s[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for s in samples if len(s) >= 6 for i in range(4) if s[2 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


def host_threads() -> int:
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def run_reference(args, rank, world):
    """CPU arm: the oracle's C port of the reference algorithm (kind 'port'), all host threads.  Each step verifies a bounded
    sample of the GPU arm's workload: oracle-generated valid items invalidated by the SAME routine, classes and fraction as the
    GPU arm's batches (jubjub_schnorr_b200.workload.invalidate: plain numpy, no kernel involved)."""
    if rank != 0:
        return
    if not args.log2n:
        args.log2n = 24 if args.workload == "mixed5" else 20
    import numpy as np
    from jubjub_schnorr_b200 import workload as wl
    from oracle import c_oracle as co
    co.build()
    threads = host_threads()
    sample = int(args.cpu_sample or 1 << 13)
    kinds = {"single": ["single"], "double": ["double"], "vargen": ["vargen"], "aggregate": ["aggregate"], "mixed4": ["vargen", "aggregate"],
             "mixed5": ["single", "double"]}[args.workload]
    per = sample // len(kinds)
    jobs = []
    for kind in kinds:
        frac = 0.05 if (kind == "aggregate" or args.workload == "mixed4") else 0.10
        if kind == "aggregate":
            signers = np.random.default_rng(1).choice(np.array([2, 3, 4], dtype=np.uint32), size=per)
            pks, off, sig, msg = co.gen_aggregate(0xB200, signers, threads=threads)
            k = max(1, int(round(frac * per)))
            sig[:k, 0] ^= 1
            expected = np.zeros(per, dtype=np.uint8)
            expected[:k] = 1
            jobs.append((lambda pks=pks, off=off, sig=sig, msg=msg: co.verify_aggregate(pks, off, sig, msg, threads=threads)[0], expected))
        else:
            variant = {"single": wl.SINGLE, "double": wl.DOUBLE, "vargen": wl.VARGEN}[kind]
            gen = {"single": co.gen_single, "double": co.gen_double, "vargen": co.gen_vargen}[kind]
            ver = {"single": co.verify_single, "double": co.verify_double, "vargen": co.verify_vargen}[kind]
            pk, sig, msg = gen(0xB200, per, threads=threads)
            pk, sig, msg, expected, _ = wl.invalidate(variant, pk, sig, msg, frac, seed=0xB200)
            jobs.append((lambda ver=ver, pk=pk, sig=sig, msg=msg: ver(pk, sig, msg, threads=threads)[0], expected))
    sample = per * len(kinds)
    for _ in range(args.warmup):
        for fn, _ in jobs:
            fn()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        results = [fn() for fn, _ in jobs]
    dt = time.perf_counter() - t0
    assert all(np.array_equal(st, exp) for st, (_, exp) in zip(results, jobs)), "CPU port disagrees with the constructed expectation"
    value = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "strong" if args.workload == "mixed5" else "weak", "vs_baseline": None,
        "dtype": "u64 (4x64-bit Montgomery limbs)", "data": "synthetic", "config": workload_config(args),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "per_thread": value / threads, "nproc": os.cpu_count(),
                         "sample": f"{sample} items per step drawn like the GPU arm's batch ({args.workload}: same generator classes and invalid fraction), "
                                   "oracle/jjs_oracle.c (reference algorithm restated in C; the Rust crate cannot be built here)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


PERMS = {"single": 2, "double": 3, "vargen": 2}
SLOTS = {"single": 2, "double": 4, "vargen": 3}
NEQ = {"single": 1, "double": 2, "vargen": 1}
MAC32_POINT = (53 + 1134 + 68) * MAC32_M + (272 + 1008 + 4) * MAC32_S      # decompress + subgroup check of one point
CONFIG_INDEX = {"single": 1, "double": 2, "vargen": 3, "aggregate": 3, "mixed4": 3, "mixed5": 4}


def aggregate_mac32(counts):
    """Canonical MAC32 of aggregate-key items (SURVEY Appendix C, aggregate(n)), split into the stages that do the work."""
    import numpy as np
    c = np.asarray(counts, dtype=np.int64)
    perms = c * ((2 + 2 * c + 3) // 4)
    decode = int((c * MAC32_DECODE).sum()) + len(c) * MAC32_POINT                      # n signer keys (decode only) + R
    agg = int((c * ((68 + 42 * 9) * MAC32_M + 4 * MAC32_S) + perms * MAC32_PERMUTATION).sum()) + len(c) * ((252 * 3 + 40) * MAC32_M + (252 * 4 + 255) * MAC32_S + MAC32_POINT - MAC32_DECODE)
    chall = len(c) * 2 * MAC32_PERMUTATION
    eq = len(c) * MAC32_EQUATION
    return {"decode": decode, "aggregate": agg, "challenge": chall, "equation": eq}


def plan_parts(args, n_gpus_total):
    """[(kind, items_per_gpu, invalid_fraction)] for one GPU."""
    n = 1 << args.log2n
    if args.workload in ("single", "double", "vargen", "aggregate"):
        return [(args.workload, n, 0.05 if args.workload == "aggregate" else 0.10)]
    if args.workload == "mixed4":   # BASELINE.json configs[3]: var-generator + aggregate-key halves, 5 % invalid
        return [("vargen", n // 2, 0.05), ("aggregate", n // 2, 0.05)]
    if args.workload == "mixed5":   # BASELINE.json configs[4]: 2^log2n items in total over all GPUs, half single half double
        from jubjub_schnorr_b200.sharding import shard_range
        lo, hi = shard_range(n // 2, 0, n_gpus_total)      # the largest contiguous slice of each half (slices differ by at most one item)
        per = max(1, hi - lo)
        return [("single", per, 0.10), ("double", per, 0.10)]
    raise SystemExit("unknown workload")


def workload_config(args):
    n = 1 << args.log2n
    desc = {
        "single": f"2^{args.log2n} single Schnorr signatures per GPU, 10% tampered/invalid",
        "double": f"2^{args.log2n} double Schnorr signatures (JJSCHDBL transcript, G and G') per GPU, 10% tampered/invalid",
        "vargen": f"2^{args.log2n} var-generator signatures (distinct generator per item) per GPU, 10% tampered/invalid",
        "aggregate": f"2^{args.log2n} SpeedyMuSig aggregate-key verifications (2-4 signers) per GPU, 5% invalid",
        "mixed4": f"2^{args.log2n - 1} var-generator + 2^{args.log2n - 1} aggregate-key (2-4 signers) verifications per GPU, 5% invalid",
        "mixed5": f"2^{args.log2n} items in total, half single half double, 10% invalid, split contiguously over {args.gpus} GPU(s)",
    }[args.workload]
    cfg = {"workload": f"{desc} (BASELINE.json configs[{CONFIG_INDEX[args.workload]}])", "items_per_gpu": n if args.workload != "mixed5" else n // args.gpus,
           "l2_policy": "inputs (>=128 MiB) plus >1 GiB of per-step scratch exceed the 126 MB L2; no explicit flush",
           "parallelism": f"{args.gpus} independent shard(s), no collective on the data path"}
    return cfg


class Part:
    """One homogeneous sub-batch resident on one device."""

    def __init__(self, bv, wl, kind, n, frac, seed, rank, dev_index, torch):
        self.kind, self.n, self.bv, self.dev_index, self.torch = kind, n, bv, dev_index, torch
        self.variant = {"single": wl.SINGLE, "double": wl.DOUBLE, "vargen": wl.VARGEN, "aggregate": None}[kind]
        if kind == "aggregate":
            self.pk, self.off, self.sig, self.msg, self.expected, cls = wl.make_aggregate_batch(bv, n, frac, seed=seed, rank=rank)
            self.counts = np.diff(self.off.astype(np.int64))
            names = wl.AGG_CLASSES
        else:
            self.pk, self.sig, self.msg, self.expected, cls = wl.make_batch(bv, self.variant, n, frac, seed=seed, rank=rank)
            self.off = None
            names = wl.CLASSES
        # Items whose equations the equation kernel evaluates: everything decodes and the keys are valid, i.e. status
        # Ok / InvalidSignature, or InvalidPoint caused by the signature point alone (the library drops the rest from the
        # kernel's work list).  The kernel's roofline counts these units only.
        sig_point_only = np.array([nm.startswith("R_") and st == 2 for nm, st in names], dtype=bool)
        cls = np.asarray(cls)
        self.n_equation_items = int(((self.expected <= 1) | ((cls >= 0) & sig_point_only[np.clip(cls, 0, len(names) - 1)])).sum())
        self.h2d = self.pk.nbytes + self.sig.nbytes + self.msg.nbytes + (self.off.nbytes if self.off is not None else 0)

    def to_device(self, dev):
        t = self.torch
        self.dev = dev
        self.stream = t.cuda.current_stream(dev)
        self.d = [t.from_numpy(x).to(dev) for x in ((self.pk, self.sig, self.msg) if self.off is None else (self.pk, self.sig, self.msg, self.off))]
        self.d_status = t.empty(self.n, dtype=t.uint8, device=dev)
        self.d_c = t.empty((self.n, 32), dtype=t.uint8, device=dev)

    def pin(self):
        t = self.torch
        self.h = [t.from_numpy(x).pin_memory() for x in (self.pk, self.sig, self.msg)]
        self.h_off = t.from_numpy(self.off.view(np.int32)).pin_memory() if self.off is not None else None
        self.h_status = t.empty(self.n, dtype=t.uint8).pin_memory()
        self.p_status = np.empty(self.n, dtype=np.uint8)     # pageable result buffer

    def host_part(self, pageable=False):
        """One jjs_part of the mixed host call: pinned torch tensors, or the pageable numpy arrays the batch was made in."""
        kind = 3 if self.off is not None else self.variant
        if pageable:
            return (kind, self.pk.ctypes.data, self.off.ctypes.data if self.off is not None else None, self.sig.ctypes.data, self.msg.ctypes.data, self.n,
                    self.p_status.ctypes.data, None, None, None)
        return (kind, self.h[0].data_ptr(), self.h_off.data_ptr() if self.h_off is not None else None, self.h[1].data_ptr(), self.h[2].data_ptr(), self.n,
                self.h_status.data_ptr(), None, None, None)

    def step_device(self):
        if self.off is None:
            self.bv.verify_device(self.variant, self.d[0].data_ptr(), self.d[1].data_ptr(), self.d[2].data_ptr(), self.n, self.d_status.data_ptr(),
                                  self.d_c.data_ptr(), stream=self.stream.cuda_stream, device_index=self.dev_index)
        else:
            self.bv.verify_aggregate_device(self.d[0].data_ptr(), self.d[3].data_ptr(), self.off, self.d[1].data_ptr(), self.d[2].data_ptr(), self.n,
                                            self.d_status.data_ptr(), self.d_c.data_ptr(), None, stream=self.stream.cuda_stream, device_index=self.dev_index)

    def canonical_mac32(self):
        """{stage: canonical MAC32 of this part for one step}"""
        if self.kind == "aggregate":
            d = aggregate_mac32(self.counts)
            d["equation"] = self.n_equation_items * MAC32_EQUATION
            return d
        chall = PERMS[self.kind] * MAC32_PERMUTATION
        eq = NEQ[self.kind] * (MAC32_EQUATION_VARGEN if self.kind == "vargen" else MAC32_EQUATION)
        # the rest of SURVEY's per-item figure is point decoding and the subgroup checks it counts (those of the key points)
        return {"decode": self.n * (MAC32_PER_ITEM[self.kind] - chall - eq), "challenge": self.n * chall, "equation": self.n_equation_items * eq,
                "aggregate": 0}

    def cpu_check(self, co, sample, threads):
        import numpy as np
        s = min(sample, self.n)
        if self.kind == "aggregate":
            st, _, _ = co.verify_aggregate(self.pk[: self.off[s]], self.off[: s + 1], self.sig[:s], self.msg[:s], threads=threads)
        else:
            over = {"single": co.verify_single, "double": co.verify_double, "vargen": co.verify_vargen}[self.kind]
            st, _ = over(self.pk[:s], self.sig[:s], self.msg[:s], threads=threads)
        assert np.array_equal(st, self.expected[:s]), "oracle and constructed expectation disagree on the sample"
        return s


DUMP_ITEMS = 1 << 19    # items dumped over the whole job, 68 bytes each: at most 34 MiB


def dump_outputs(out_dir, shards, rank, n_shards_total):
    """Writes, for every part of every shard of this process, what the device path returned in the last timed step:
    shard<g>_<kind>_status.npy (float32 status codes) and shard<g>_<kind>_challenge.npy (float64 [items, 8], the challenge
    scalar as eight little-endian 32-bit words, exact in float64).  A part larger than its share of DUMP_ITEMS is represented
    by a fixed sample of its items (sorted indices drawn with the part's size as the seed), the same in every run."""
    os.makedirs(out_dir, exist_ok=True)
    per_part = DUMP_ITEMS // (n_shards_total * len(shards[0]))
    for k, parts in enumerate(shards):
        g = rank * len(shards) + k
        for p in parts:
            idx = np.arange(p.n) if p.n <= per_part else np.sort(np.random.default_rng(p.n).choice(p.n, size=per_part, replace=False))
            status = p.d_status.cpu().numpy()[idx]
            c = p.d_c.cpu().numpy()[idx]
            np.save(os.path.join(out_dir, f"shard{g}_{p.kind}_status.npy"), status.astype(np.float32))
            np.save(os.path.join(out_dir, f"shard{g}_{p.kind}_challenge.npy"), np.ascontiguousarray(c).view("<u4").astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="single", choices=["single", "double", "vargen", "aggregate", "mixed4", "mixed5"])
    ap.add_argument("--log2n", type=int, default=0, help="log2 of the items per GPU (mixed5: of the whole job); default 20 (mixed5: 24)")
    ap.add_argument("--cpu-sample", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="skip the 2^24 strong-scaling sub-record")
    ap.add_argument("--strong-log2n", type=int, default=24)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    if not args.log2n:
        args.log2n = 24 if args.workload == "mixed5" else 20
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    from jubjub_schnorr_b200 import BatchVerifier
    from jubjub_schnorr_b200 import workload as wl

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version banner to stdout while the communicator is created; stdout must carry one JSON
        # line only, so fd 1 points at stderr until the first collective is through.
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    # under torchrun: one device per process; plain launch with --gpus N: one context over N devices
    devices = [local_rank] if world > 1 else list(range(args.gpus))
    n_gpus_total = world if world > 1 else len(devices)
    bv = BatchVerifier(devices)          # device entry points, one shard per device
    plan = plan_parts(args, n_gpus_total)
    shards = []                          # per device of this process: list of parts
    for k, dnum in enumerate(devices):
        dev = torch.device("cuda", dnum)
        parts = [Part(bv, wl, kind, n, frac, 0xB200 + 17 * j, rank * len(devices) + k, k, torch) for j, (kind, n, frac) in enumerate(plan)]
        for p in parts:
            p.to_device(dev)
        shards.append(parts)
    all_parts = [p for parts in shards for p in parts]
    items_per_device = sum(n for _, n, _ in plan)

    def barrier():
        if world > 1:
            dist.barrier()
        for d in devices:
            torch.cuda.synchronize(d)

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident measurement ("value") ------------------------------------------------------------
    def step_device():
        for p in all_parts:
            p.step_device()

    for _ in range(args.warmup):
        step_device()
    barrier()
    for p in all_parts:
        assert np.array_equal(p.d_status.cpu().numpy(), p.expected), f"GPU statuses differ from the constructed expectation ({p.kind})"
    sampler = ClockSampler(devices[0])
    sampler.start()
    launches0 = bv.launch_count
    events = []
    barrier()
    for parts in shards:
        with torch.cuda.device(parts[0].dev):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(parts[0].stream)
            events.append((e0, e1))
    for _ in range(args.steps):
        step_device()
    for parts, (e0, e1) in zip(shards, events):
        with torch.cuda.device(parts[0].dev):
            e1.record(parts[0].stream)
    barrier()
    ms_dev = max_over_ranks(max(e0.elapsed_time(e1) for e0, e1 in events))
    launches = bv.launch_count - launches0
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, shards, rank, n_gpus_total)
    # Stage breakdown from a second, untimed pass of the same K steps: with the per-stage timers on, the library keeps
    # every launch on one stream (the timed pass above overlaps neighbouring sub-chunks on two streams, which per-stage
    # CUDA events cannot attribute), so the stage times add up to slightly more than ms_per_step.
    bv.profile(True)
    for _ in range(args.steps):
        step_device()
    barrier()
    bv.profile(False)
    stages = bv.profile_collect()
    value = items_per_device * n_gpus_total * args.steps / (ms_dev * 1e-3)

    # ---- end to end through the host-buffer C ABI ("e2e") ---------------------------------------------------
    # ONE jjs_verify_mixed call per step carries every part; the library shards each part over the context's devices itself
    host_parts = shards[0] if len(devices) == 1 else [Part(bv, wl, kind, n * len(devices), frac, 0xE2E + 17 * j, rank, 0, torch) for j, (kind, n, frac) in enumerate(plan)]
    for p in host_parts:
        p.pin()

    def time_host(pageable):
        tuples = [p.host_part(pageable) for p in host_parts]
        for _ in range(max(1, args.warmup - 1)):
            bv.verify_mixed_ptr(tuples)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            bv.verify_mixed_ptr(tuples)
        barrier()
        dt = max_over_ranks(time.perf_counter() - t0)
        for p in host_parts:
            got = p.p_status if pageable else p.h_status.numpy()
            assert np.array_equal(got, p.expected), f"host-path statuses differ from the constructed expectation ({p.kind}, pageable={pageable})"
        return dt

    e2e_s = time_host(False)
    e2e_value = items_per_device * n_gpus_total * args.steps / e2e_s
    pageable_s = time_host(True)
    h2d = sum(p.h2d for p in host_parts)
    d2h = sum(p.n for p in host_parts)

    # ---- roofline of the dominant kernel ----------------------------------------------------------------------
    peak, peak_src = int32_peak()
    canon = {k: sum(p.canonical_mac32()[k] for p in shards[0]) for k in ("decode", "challenge", "aggregate", "equation")}
    stage_ms = {k: v[0] / max(1, args.steps) / len(devices) for k, v in stages.items()}
    dom = max(("decode", "challenge", "aggregate", "equation"), key=lambda k: stage_ms[k])
    achieved = canon[dom] / (stage_ms[dom] * 1e-3) / 1e12
    step_mac32 = sum(canon.values())
    step_achieved = step_mac32 * n_gpus_total / (ms_dev / args.steps * 1e-3) / 1e12 / n_gpus_total
    bytes_in = sum(p.h2d for p in shards[0])
    hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs") if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 6650.0
    units = {"decode": sum(p.n * SLOTS.get(p.kind, 1) for p in shards[0]), "challenge": sum(p.n_equation_items for p in shards[0]),
             "equation": sum(p.n_equation_items * NEQ.get(p.kind, 1) for p in shards[0]), "aggregate": sum(p.n for p in shards[0] if p.kind == "aggregate")}
    traffic = None
    try:  # DRAM bytes of the dominant kernel per step, from the committed ncu capture (bytes per unit x units in this step)
        traffic_file = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_traffic.json")))[-1]   # newest capture
        trk = json.load(open(traffic_file))["kernels"]
        vg_only = dom == "equation" and all(p.kind == "vargen" for p in shards[0])   # the var-generator equation kernel has its own capture
        tr = trk["k_equation_vargen"] if vg_only and "k_equation_vargen" in trk else trk["k_" + dom]
        traffic = tr["dram_bytes_per_unit"] * {"decode": units["decode"], "challenge": sum(p.n for p in shards[0]),
                                               "equation": sum(p.n * NEQ.get(p.kind, 1) for p in shards[0]), "aggregate": units["aggregate"]}[dom]
    except Exception:
        pass
    # executed multiplies: IMAD.WIDE / IMAD.HI thread instructions per unit of each kernel, counted by ncu on this build
    # (profiles/r*_executed_mac32.json, made by tools/ncu_executed.py from the source pages of the committed captures)
    executed = None
    try:
        ex_file = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_executed_mac32.json")))[-1]
        ex = json.load(open(ex_file))["per_unit"]
        per_stage = {"decode": 0.0, "challenge": 0.0, "equation": 0.0, "aggregate": 0.0}
        for p in shards[0]:
            if p.kind not in ex:
                raise KeyError(p.kind)
            if p.kind == "aggregate":
                # signer keys and signature points are decoded without a subgroup test: a key point of the single path minus
                # the difference the var-generator path shows for one more tested point (3 * vargen - 2 * single = a tested
                # point, so an untested one = 2 * single - that); the hash and the equation are the single path's
                tested = 3 * ex["vargen"]["k_decode"] - 2 * ex["single"]["k_decode"]
                untested = 2 * ex["single"]["k_decode"] - tested
                keys = int(p.counts.sum())
                per_stage["decode"] += untested * (keys + p.n)
                per_stage["challenge"] += ex["single"]["k_challenge"] * p.n_equation_items
                per_stage["equation"] += ex["single"]["k_equation"] * p.n_equation_items
                per_stage["aggregate"] += ex["aggregate"]["k_agg_coeffs"] * keys + ex["aggregate"]["k_aggregate"] * p.n
                continue
            per_stage["decode"] += ex[p.kind]["k_decode"] * p.n * SLOTS[p.kind]
            per_stage["challenge"] += ex[p.kind]["k_challenge"] * p.n_equation_items
            per_stage["equation"] += ex[p.kind]["k_equation"] * p.n_equation_items * NEQ[p.kind]
        if dom in per_stage:
            ex_dom = per_stage[dom] / (stage_ms[dom] * 1e-3) / 1e12
            ex_step = sum(per_stage.values()) / (ms_dev / args.steps * 1e-3) / 1e12
            executed = {"achieved": ex_dom, "frac": ex_dom / peak, "mac32_per_step_by_stage": per_stage,
                        "step": {"achieved": ex_step, "frac": ex_step / peak, "mac32_per_step_per_gpu": sum(per_stage.values())},
                        "source": os.path.relpath(ex_file, ROOT),
                        "note": "executed 32x32->64 multiplies (IMAD.WIDE + IMAD.HI thread instructions counted by ncu per unit of each kernel) x the units "
                                "of this step / measured time / peak: the integer-multiply pipe efficiency; rtest and finalize are left out (< 1 % of the step)"}
    except Exception:
        pass
    roofline = {"bound": "int32_mul", "kernel": {"decode": "k_decode", "challenge": "k_challenge", "aggregate": "k_aggregate", "equation": "k_equation"}[dom],
                "achieved": achieved, "peak": peak, "unit": "TMAC32/s", "frac": achieved / peak, "executed": executed, "traffic": traffic,
                "traffic_unit": "DRAM bytes per step (ncu dram__bytes_read.sum + dram__bytes_write.sum, the newest profiles/r*_ncu_traffic.json); secondary: the bound is the multiply pipe",
                "peak_source": peak_src,
                "ms_per_step": stage_ms[dom], "algorithmic_mac32_per_step": canon[dom],
                "note": "achieved = canonical MAC32 (SURVEY 8(d) / Appendix C operation counts at 136/108 MAC32 per field mul/sqr) of the kernel's units / its measured time "
                        "(equation kernel: only the equations it evaluates -- items that fail to decode or have an invalid key never reach it); "
                        "the implementation executes fewer multiplies than the canonical algorithm (Tate subgroup test, integer MDS, half-size scalars), so frac can exceed 1: "
                        "`executed` is the efficiency figure",
                "step": {"achieved": step_achieved, "frac": step_achieved / peak, "mac32_per_step_per_gpu": step_mac32},
                "stage_ms_per_step": stage_ms,
                "stage_timing": "per-stage CUDA events on the launching stream in a second pass of the same steps with the launches serialised "
                                "(the timed pass overlaps neighbouring sub-chunks on two streams); ms_per_step of the kernel above is from that pass",
                "hbm_secondary": {"algorithmic_GBps": (bytes_in + items_per_device * 33) / (ms_dev / args.steps * 1e-3) / 1e9, "measured_peak_GBps": hbm_peak}}

    # ---- strong scaling of the library's own sharding: BASELINE.json configs[4] -------------------------------------------------
    strong = None
    if not args.no_strong:
        gloo = dist.new_group(backend="gloo") if world > 1 else None     # the waiting ranks must not spin on their GPUs
        barrier()
        if rank == 0:
            strong = strong_scaling_record(args, torch, wl, BatchVerifier, n_gpus_total if world > 1 else len(devices))
        if gloo is not None:
            dist.barrier(group=gloo)

    # ---- CPU baseline beside it (rank 0, N = 1 only): BASELINE.json configs[0] -----------------------------------------------------
    cpu = None
    if rank == 0 and args.gpus == 1 and not args.no_cpu_baseline:
        from oracle import c_oracle as co
        co.build()
        threads = host_threads()
        shards[0][0].cpu_check(co, 512, threads)      # the oracle agrees with the GPU on the head of the timed batch
        n_cpu = int(args.cpu_sample or 1 << 16)
        pk, sig, msg = co.gen_single(0xB200, n_cpu, threads=threads)
        t0 = time.perf_counter()
        st, _ = co.verify_single(pk, sig, msg, threads=threads)
        dt = time.perf_counter() - t0
        assert not st.any()
        cpu = {"value": n_cpu / dt, "unit": UNIT, "cores": threads, "kind": "port", "per_thread": n_cpu / dt / threads, "nproc": os.cpu_count(),
               "sample": f"BASELINE.json configs[0]: {n_cpu} valid single signatures, PublicKey::verify restated in C (oracle/jjs_oracle.c), {threads} threads, one pass; "
                         "the first 512 items of the GPU batch went through the same port and agree with the GPU"}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "strong" if args.workload == "mixed5" else "weak", "vs_baseline": None,
                "dtype": "u32 (8x32-bit Montgomery limbs, IMAD.WIDE)", "data": "synthetic", "config": workload_config(args),
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": 1e3 * e2e_s / args.steps,
                        "host_memory": "pinned", "call": "one jjs_verify_mixed per step"},
                "e2e_pageable": {"value": items_per_device * n_gpus_total * args.steps / pageable_s, "unit": UNIT, "ms_per_step": 1e3 * pageable_s / args.steps,
                                 "host_memory": "pageable (numpy arrays, what a Rust Vec<u8> is)", "ratio_to_pinned": e2e_s / pageable_s},
                "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "strong_2p24": strong, "cpu_baseline": cpu, "impl": "b200"}
        print(json.dumps(line), flush=True)
    bv.close()
    if world > 1:
        dist.destroy_process_group()


def strong_scaling_record(args, torch, wl, BatchVerifier, n_devices):
    """BASELINE.json configs[4]: 2^24 items, half single half double, 10 % invalid, through ONE context over n_devices GPUs.
    e2e: one jjs_verify_mixed host call per step (pinned buffers; also pageable).  value: the same shards resident on the devices,
    enqueued through the device entry points, CUDA events per device, max over devices."""
    log2n = args.strong_log2n
    half = 1 << (log2n - 1)
    steps, warm = args.steps, 1
    with BatchVerifier(list(range(n_devices))) as sv:
        batches = [(wl.SINGLE,) + tuple(wl.make_batch(sv, wl.SINGLE, half, 0.10, seed=0x24A)[:4]), (wl.DOUBLE,) + tuple(wl.make_batch(sv, wl.DOUBLE, half, 0.10, seed=0x24B)[:4])]
        n = 2 * half
        pinned = [[torch.from_numpy(x).pin_memory() for x in b[1:4]] + [torch.empty(half, dtype=torch.uint8).pin_memory()] for b in batches]
        pstat = [np.empty(half, dtype=np.uint8) for _ in batches]
        t_pin = [(b[0], h[0].data_ptr(), None, h[1].data_ptr(), h[2].data_ptr(), half, h[3].data_ptr(), None, None, None) for b, h in zip(batches, pinned)]
        t_page = [(b[0], b[1].ctypes.data, None, b[2].ctypes.data, b[3].ctypes.data, half, st.ctypes.data, None, None, None) for b, st in zip(batches, pstat)]

        def sync_all():
            for k in range(n_devices):
                torch.cuda.synchronize(k)

        def timed(tuples):
            for _ in range(warm):
                sv.verify_mixed_ptr(tuples)
            sync_all()
            t0 = time.perf_counter()
            for _ in range(steps):
                sv.verify_mixed_ptr(tuples)
            return (time.perf_counter() - t0) / steps

        s_pin = timed(t_pin)
        for b, h in zip(batches, pinned):
            assert np.array_equal(h[3].numpy(), b[4]), "strong-scaling batch: statuses differ from the constructed expectation"
        s_page = timed(t_page)
        for b, st in zip(batches, pstat):
            assert np.array_equal(st, b[4]), "strong-scaling batch (pageable): statuses differ from the constructed expectation"
        # device-resident: contiguous shards of both kinds on every device
        per = ((half + n_devices - 1) // n_devices + 31) & ~31
        resident = []
        for k in range(n_devices):
            lo, hi = min(k * per, half), min(k * per + per, half)
            dev = torch.device("cuda", k)
            resident.append([(b[0], hi - lo, [torch.from_numpy(x[lo:hi]).to(dev) for x in b[1:4]], torch.empty(hi - lo, dtype=torch.uint8, device=dev), b[4][lo:hi])
                             for b in batches])

        def step_resident():
            for k, parts in enumerate(resident):
                stream = torch.cuda.current_stream(k).cuda_stream
                for variant, m, d, st, _ in parts:
                    if m:
                        sv.verify_device(variant, d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), m, st.data_ptr(), None, stream=stream, device_index=k)

        for _ in range(warm):
            step_resident()
        sync_all()
        events = []
        for k in range(n_devices):
            with torch.cuda.device(k):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(torch.cuda.current_stream(k))
                events.append((e0, e1))
        t0 = time.perf_counter()
        for _ in range(steps):
            step_resident()
        for k, (e0, e1) in enumerate(events):
            with torch.cuda.device(k):
                e1.record(torch.cuda.current_stream(k))
        sync_all()
        wall = (time.perf_counter() - t0) / steps
        ms_dev = max(e0.elapsed_time(e1) for e0, e1 in events) / steps
        for parts in resident:
            for _, m, _, st, exp in parts:
                assert np.array_equal(st.cpu().numpy(), exp), "strong-scaling batch (device-resident): statuses differ from the constructed expectation"
    return {"workload": f"2^{log2n} items, half single half double, 10% invalid (BASELINE.json configs[4]); one jjs_ctx over {n_devices} device(s), contiguous shards, no collective",
            "n_devices": n_devices, "items": n, "steps": steps, "warmup": warm,
            "value": n / (ms_dev * 1e-3), "ms_per_step": ms_dev, "value_wall_clock": n / wall,
            "e2e": {"value": n / s_pin, "ms_per_step": 1e3 * s_pin, "host_memory": "pinned", "call": "one jjs_verify_mixed",
                    "h2d_bytes_per_step": sum(sum(x.nbytes for x in b[1:4]) for b in batches), "d2h_bytes_per_step": n},
            "e2e_pageable": {"value": n / s_page, "ms_per_step": 1e3 * s_page, "ratio_to_pinned": s_pin / s_page},
            "unit": UNIT, "scaling": "strong"}


if __name__ == "__main__":
    main()
