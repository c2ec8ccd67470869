"""Pass plans and outputs of every verify entry point, for comparing two builds of the same ABI.

Runs a fixed matrix of calls on seeded inputs and writes one JSON record per call: the jjs_launch_count delta, the return code,
the profile_collect stage counts (profiling on), and a SHA-256 of every output (statuses, challenges, aggregate keys, bitmaps, the
whole-batch verdict, the grouped fallback count).  The matrix covers every host and device verify entry point at
n in {1, first_slice + 1, sub_chunk, sub_chunk + 1, chunk_items + 1, 3 sub_chunk + 5} of the context, on a jjs_init context and a
256 MiB jjs_init_limited context, with profiling off and on, and ends with an aggregate item with more signer keys than the limited
context's first key scratch.  Run it once per build (JJS_B200_LIB names the library) and compare the files:

    JJS_B200_LIB=old.so python tools/check_pass_plan.py --out a.json
    JJS_B200_LIB=new.so python tools/check_pass_plan.py --out b.json
    python tools/check_pass_plan.py --compare a.json b.json
"""
import argparse
import hashlib
import json
import os
import re
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SINGLE, DOUBLE, VARGEN, AGGREGATE = 0, 1, 2, 3
SEED = bytes(range(32))
LIMIT = 256 << 20


def sha(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def sizes_of(bv):
    chunk = bv.memory_info()["items_in_flight"]
    sub = chunk // 2
    first = min(1 << 17, sub)
    return chunk, [1, first + 1, sub, sub + 1, chunk + 1, 3 * sub + 5]


def make_pool(bv, n):
    from jubjub_schnorr_b200 import workload as wl
    pool = {}
    for v in (SINGLE, DOUBLE, VARGEN):
        pk, sig, msg, _, _ = wl.make_batch(bv, v, n, 0.1, seed=0xC4EC + v)
        pool[v] = (pk, sig, msg)
    pks, off, sig, msg, _, _ = wl.make_aggregate_batch(bv, n, 0.1, seed=0xC4EC)
    pool[AGGREGATE] = (pks, off, sig, msg)
    pool["typed"] = wl.make_typed_single_batch(bv, n, 0.1, seed=0xC4EC)[:3]
    kpks, idx, ksig, kmsg, _, _ = wl.make_keyed_batch(bv, SINGLE, 64, n, 0.1, seed=0xC4EC)   # 64 keys: the tables fit the limited context
    pool["keyed"] = (kpks, idx, ksig, kmsg)
    return pool


class Device:
    """the pool on the GPU, and fresh output buffers"""

    def __init__(self, pool):
        import torch
        self.t = torch
        self.d = {k: tuple(torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in v) for k, v in pool.items()}

    def ptr(self, key, i):
        return self.d[key][i].data_ptr()

    def zeros(self, *shape, dtype=None):
        return self.t.zeros(*shape, dtype=dtype or self.t.uint8, device="cuda")

    def stream(self):
        return self.t.cuda.current_stream().cuda_stream


def agg_host(pool, n):
    pks, off, sig, msg = pool[AGGREGATE]
    return pks[:off[n]], off[:n + 1], sig[:n], msg[:n]


def calls(bv, pool, dev, ks, n):
    """(name, fn) per entry point; fn returns the list of outputs to hash"""
    w = {v: tuple(a[:n] for a in pool[v]) for v in (SINGLE, DOUBLE, VARGEN)}
    apk, aoff, asig, amsg = agg_host(pool, n)
    t = dev.t
    out = []

    def host(name, fn):
        out.append((name, fn))
    host("single", lambda: list(bv.verify_single(*w[SINGLE], want_challenge=True)))
    host("double", lambda: list(bv.verify_double(*w[DOUBLE], want_challenge=True)))
    host("vargen", lambda: list(bv.verify_vargen(*w[VARGEN], want_challenge=True)))
    host("aggregate", lambda: list(bv.verify_aggregate(apk, aoff, asig, amsg, want_challenge=True, want_aggregate_key=True)))
    host("batch", lambda: [bv.verify_batch(*w[SINGLE])])
    host("batch_double", lambda: [bv.verify_batch_double(*w[DOUBLE])])
    host("batch_vargen", lambda: [bv.verify_batch_vargen(*w[VARGEN])])
    host("batch_aggregate", lambda: [bv.verify_batch_aggregate(apk, aoff, asig, amsg)])
    mixed_parts = [(SINGLE,) + w[SINGLE], (AGGREGATE, apk, asig, amsg, aoff)]
    host("mixed", lambda: [a for r in bv.verify_mixed(mixed_parts, want_challenge=True, want_bitmap=True) for a in r.values()])
    typed = tuple(a[:n] for a in pool["typed"])
    host("ext", lambda: list(bv.verify_ext(SINGLE, *typed, want_challenge=True)))
    host("challenge_only", lambda: [bv.challenge_only(DOUBLE, *w[DOUBLE])])
    kidx, ksig, kmsg = (a[:n] for a in pool["keyed"][1:])
    host("keyed", lambda: list(bv.verify_keyed(ks, kidx, ksig, kmsg, want_challenge=True, want_bitmap=True)))
    host("all_single", lambda: [np.int32(bv.verify_all(SINGLE, *w[SINGLE], seed=SEED))])
    host("all_double", lambda: [np.int32(bv.verify_all(DOUBLE, *w[DOUBLE], seed=SEED))])
    all_parts = [(VARGEN,) + w[VARGEN], (AGGREGATE, apk, asig, amsg, aoff)]
    host("all_mixed", lambda: [np.int32(bv.verify_all_mixed(all_parts, seed=SEED))])
    grp_parts = [(DOUBLE,) + w[DOUBLE], (AGGREGATE, apk, asig, amsg, aoff)]

    def grouped():
        res, fb = bv.verify_grouped(grp_parts, seed=SEED, want_challenge=True, want_bitmap=True)
        return [a for r in res for a in r.values()] + [np.uint64(fb)]
    host("grouped", grouped)

    def wire_device(v):
        def fn():
            st, c = dev.zeros(n), dev.zeros(n, 32)
            bv.verify_device(v, dev.ptr(v, 0), dev.ptr(v, 1), dev.ptr(v, 2), n, st.data_ptr(), c.data_ptr(), stream=dev.stream())
            return [st, c]
        return fn
    host("single_device", wire_device(SINGLE))
    host("double_device", wire_device(DOUBLE))
    host("vargen_device", wire_device(VARGEN))

    def aggregate_device():
        st, c, agg = dev.zeros(n), dev.zeros(n, 32), dev.zeros(n, 32)
        bv.verify_aggregate_device(dev.ptr(AGGREGATE, 0), dev.ptr(AGGREGATE, 1), aoff, dev.ptr(AGGREGATE, 2), dev.ptr(AGGREGATE, 3), n, st.data_ptr(),
                                   c.data_ptr(), agg.data_ptr(), stream=dev.stream())
        return [st, c, agg]
    host("aggregate_device", aggregate_device)

    def keyed_device():
        st, c = dev.zeros(n), dev.zeros(n, 32)
        bv.verify_keyed_device(ks, dev.ptr("keyed", 1), dev.ptr("keyed", 2), dev.ptr("keyed", 3), n, st.data_ptr(), c.data_ptr(), stream=dev.stream())
        return [st, c]
    host("keyed_device", keyed_device)

    def all_device(v):
        def fn():
            ok = dev.zeros(1, dtype=t.int32)
            bv.verify_all_device(v, dev.ptr(v, 0), dev.ptr(v, 1), dev.ptr(v, 2), n, ok.data_ptr(), seed=SEED, stream=dev.stream())
            return [ok]
        return fn
    host("all_single_device", all_device(SINGLE))
    host("all_double_device", all_device(DOUBLE))
    agg_dev = (dev.ptr(AGGREGATE, 0), dev.ptr(AGGREGATE, 2), dev.ptr(AGGREGATE, 3), n)

    def all_mixed_device():
        ok = dev.zeros(1, dtype=t.int32)
        parts = [(VARGEN, dev.ptr(VARGEN, 0), dev.ptr(VARGEN, 1), dev.ptr(VARGEN, 2), n), (AGGREGATE,) + agg_dev + (dev.ptr(AGGREGATE, 1), aoff)]
        bv.verify_all_mixed_device(parts, ok.data_ptr(), seed=SEED, stream=dev.stream())
        return [ok]
    host("all_mixed_device", all_mixed_device)

    def grouped_device():
        bufs = [(dev.zeros(n), dev.zeros(n, 32), None, dev.zeros((n + 31) // 32, dtype=t.int32)),
                (dev.zeros(n), dev.zeros(n, 32), dev.zeros(n, 32), dev.zeros((n + 31) // 32, dtype=t.int32))]
        ptr = lambda a: a.data_ptr() if a is not None else None  # noqa: E731
        fb = dev.zeros(1, dtype=t.int64)
        parts = [(DOUBLE, dev.ptr(DOUBLE, 0), dev.ptr(DOUBLE, 1), dev.ptr(DOUBLE, 2), n) + tuple(ptr(a) for a in bufs[0]),
                 (AGGREGATE,) + agg_dev + tuple(ptr(a) for a in bufs[1]) + (dev.ptr(AGGREGATE, 1), aoff)]
        bv.verify_grouped_device(parts, fb.data_ptr(), seed=SEED, stream=dev.stream())
        return [a for b in bufs for a in b if a is not None] + [fb]
    host("grouped_device", grouped_device)
    return out


def record(bv, fn, profiled):
    import torch
    from jubjub_schnorr_b200 import JjsError
    before = bv.launch_count
    try:
        outs = fn()
        torch.cuda.synchronize()
        r = {"rc": 0, "sha256": sha(*outs)}
    except JjsError as e:
        torch.cuda.synchronize()
        m = re.search(r"failed \((-?\d+)\)", str(e))
        r = {"rc": int(m.group(1)) if m else str(e)}
    r["launches"] = bv.launch_count - before
    if profiled:
        r["stages"] = {k: v[1] for k, v in bv.profile_collect().items()}
    return r


def run(out_path):
    import torch
    from jubjub_schnorr_b200 import BatchVerifier
    res = {"device": torch.cuda.get_device_name(0), "cases": {}}
    with BatchVerifier([0]) as bv0:
        chunk, sizes = sizes_of(bv0)
        pool = make_pool(bv0, max(sizes))
    dev = Device(pool)
    for ctx_name, limit in (("init", None), ("limited_256MiB", LIMIT)):
        with BatchVerifier([0], memory_limit=limit) as bv:
            chunk, sizes = sizes_of(bv)
            res[ctx_name] = {"items_in_flight": chunk, "sizes": sizes}
            ks = bv.keyset_create(SINGLE, pool["keyed"][0])
            for profiled in (False, True):
                bv.profile(profiled)
                for n in sizes:
                    for name, fn in calls(bv, pool, dev, ks, n):
                        key = f"{ctx_name}/{'profiled' if profiled else 'plain'}/{name}/n={n}"
                        res["cases"][key] = record(bv, fn, profiled)
                        print(key, res["cases"][key], flush=True)
                bv.profile(False)
            if limit:
                # one aggregate item with more signer keys than the first key scratch (half the capacity), then a short batch
                K = chunk // 2 + 1
                pks = np.ascontiguousarray(pool[AGGREGATE][0][:K])
                off = np.array([0, K], np.uint32)
                sig, msg = pool[AGGREGATE][2][:1], pool[AGGREGATE][3][:1]
                big = [(AGGREGATE, pks, sig, msg, off), (SINGLE,) + tuple(a[:5] for a in pool[SINGLE])]
                fns = {"mixed_big_item": lambda: [a for r in bv.verify_mixed(big, want_challenge=True) for a in r.values()],
                       "grouped_big_item": lambda: [a for r in bv.verify_grouped(big, seed=SEED, want_challenge=True)[0] for a in r.values()],
                       "all_mixed_big_item": lambda: [np.int32(bv.verify_all_mixed(big, seed=SEED))]}
                for name, fn in fns.items():
                    key = f"{ctx_name}/plain/{name}/K={K}"
                    res["cases"][key] = record(bv, fn, False)
                    print(key, res["cases"][key], flush=True)
            bv.keyset_destroy(ks)
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1, sort_keys=True)


def compare(a_path, b_path):
    a, b = json.load(open(a_path)), json.load(open(b_path))
    diffs = [k for k in sorted(set(a["cases"]) | set(b["cases"])) if a["cases"].get(k) != b["cases"].get(k)]
    for k in diffs:
        print("differs:", k, a["cases"].get(k), b["cases"].get(k))
    same_rest = {k: v for k, v in a.items() if k != "cases"} == {k: v for k, v in b.items() if k != "cases"}
    print(f"{len(a['cases'])} cases, {len(diffs)} differ; configuration {'equal' if same_rest else 'differs'}")
    return diffs


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("gpu_out", "check_pass_plan.json"))
    ap.add_argument("--compare", nargs=2, metavar=("A", "B"))
    args = ap.parse_args()
    if args.compare:
        compare(*args.compare)
    else:
        run(args.out)
