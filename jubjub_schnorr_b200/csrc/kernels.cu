// CUDA kernels (sm_100a) and the C ABI of libjjschnorr_b200.so.  See include/jjschnorr_b200.h for the
// contract and verify_core.cuh for the per-item stages.  One thread owns one point (decode, subgroup
// check), one item (challenge sponge, final status) or one verification equation (Straus-style
// u*B + c*PK); intermediates travel between the stages as SoA arrays of 32-byte field elements in HBM,
// so every warp access is a run of 128-bit vector loads.  There is deliberately no CPU path.
#include <cuda_runtime.h>
#include <cub/device/device_radix_sort.cuh>
#include <sys/random.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <new>
#include <thread>
#include <vector>

#include "../../include/jjschnorr_b200.h"
#include "keyset.cuh"
#include "multisig_core.cuh"
#include "rlc.cuh"
#include "sign_core.cuh"
#include "verify_core.cuh"
#include "safe_tag.h"

// The slot-based evaluation of the verification equation (csrc/fqs.cuh: field elements in shared memory, persistent kernel) is a
// compile-time alternative.  Measured on B200 (DESIGN.md section 8): it executes 6 % fewer multiply-pipe cycles and runs 4-7 %
// slower than the register-operand kernel, so it is off; tests/hostsim keeps its twin under test either way.
#ifndef JJS_EQ_V2
#define JJS_EQ_V2 0
#endif
#if JJS_EQ_V2
#include "fqs.cuh"
#else
#ifndef JJS_EQ_BLOCK
#define JJS_EQ_BLOCK 128
#endif
#endif

namespace tables {
#include "jjs_constants_tables.h"
}

using namespace jjs;

namespace {

#ifndef JJS_BLOCK
#define JJS_BLOCK 128
#endif
constexpr int BLOCK = JJS_BLOCK;
#ifndef JJS_EQ_MINBLOCKS
#define JJS_EQ_MINBLOCKS 4    // fixed-base equation kernel: 4 resident CTAs of 128 threads (128 registers, a few spills) beat 3 by 4 %
#endif
#ifndef JJS_EQ1_MINBLOCKS
#define JJS_EQ1_MINBLOCKS 4   // var-generator equation kernel
#endif
#ifndef JJS_AGG_MINBLOCKS
#define JJS_AGG_MINBLOCKS 4   // key-aggregation kernel (-1.9 % against 3)
#endif
#ifndef JJS_DEC_MINBLOCKS
#define JJS_DEC_MINBLOCKS 8   // decode and deferred-test kernels: 4 -> 12.62 ms per 2^21 points, 6 -> 12.49, 8 -> 12.41
#endif
#ifndef JJS_HASH_MINBLOCKS
#define JJS_HASH_MINBLOCKS 6  // hash kernels: 4 -> 12.78 ms per 2^20 challenges, 6 -> 12.66, 7 -> 12.92, 8 -> 13.06
#endif
#ifndef JJS_EQ_PERSISTENT
#define JJS_EQ_PERSISTENT 0   // measured (gpurun_out/ab2.log, DESIGN.md section 8): -22 % DRAM reads but +6 % time; off
#endif
constexpr size_t CHUNK_ITEMS = size_t(1) << 20;   // items per pipeline pass (jjs_init contexts)
constexpr size_t TAB_THREADS = size_t(1) << 20;   // threads served by the per-thread table scratch (four tables of 1152 B each)
constexpr size_t SUB_ITEMS = CHUNK_ITEMS / 2;      // items per scratch half
#ifndef JJS_SUB_CHUNK_LOG2
#define JJS_SUB_CHUNK_LOG2 19   // 2^18: 20.86 M/s device-resident on 2^20 singles, 2^19: 21.19 (fewer partially filled waves)
#endif
#ifndef JJS_FIRST_SLICE_LOG2
#define JJS_FIRST_SLICE_LOG2 17  // first slice of a host-buffer shard: short, so that compute starts while the rest is still being copied
#endif
constexpr size_t SUB_CHUNK = size_t(1) << JJS_SUB_CHUNK_LOG2;      // items per sub-chunk of an overlapped batch (<= SUB_ITEMS)
constexpr size_t AGG_KEYS_INITIAL = size_t(1) << 21;               // signer keys per scratch half of the aggregate path, first size
constexpr size_t TAGS_INITIAL = 1024;                              // SAFE tags of the multisig transcripts, first size

struct Fields {
    WireField f[4];
};

// thread t < slots * n decodes point field t / n of item t % n into index (slot_base + t / n) * n + t % n;
// bit s of subgroup_mask: run the subgroup test for slot s now (keys), else leave it to the equation stage (signature points)
__global__ void __launch_bounds__(BLOCK, JJS_DEC_MINBLOCKS) k_decode(Fields fields, int slots, int slot_base, size_t n, fq* pts_u, fq* pts_v,
                                                                      uint8_t* pflags, Tables T, uint32_t subgroup_mask) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (size_t)slots * n) return;
    int slot = (int)(t / n);
    size_t item = t - (size_t)slot * n;
    stage_decode(fields.f[slot], item, pts_u, pts_v, pflags, (size_t)(slot_base + slot) * n + item, T, (subgroup_mask >> slot) & 1u);
}

// typed inputs: thread t < slots * n normalises point t % slots of item t / slots (item-major, 160 bytes per point)
__global__ void __launch_bounds__(BLOCK, JJS_DEC_MINBLOCKS) k_decode_ext(const uint8_t* pts, int slots, size_t n, fq* pts_u, fq* pts_v, uint8_t* pflags,
                                                                          uint32_t subgroup_mask) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (size_t)slots * n) return;
    int slot = (int)(t / n);
    size_t item = t - (size_t)slot * n;
    stage_decode_ext(WireField{pts + 160 * (size_t)slot, (uint32_t)(160 * slots)}, item, pts_u, pts_v, pflags, (size_t)slot * n + item,
                     (subgroup_mask >> slot) & 1u);
}

// test-data utility: wire point -> JubJubExtended coordinates (u z, v z, z, u z, v) for a caller-chosen Montgomery z
__global__ void __launch_bounds__(BLOCK, JJS_DEC_MINBLOCKS) k_points_to_ext(const uint8_t* pts32, const uint8_t* z32, size_t n, uint8_t* out160, Tables T) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t w[8];
    fq u, v, z, c[5];
    wire_load(w, WireField{pts32, 32}, i);
    bool ok = point_from_wire(u, v, w, T);
    wire_load(z.l, WireField{z32, 32}, i);
    ok = ok && !ge_q(z.l);
    fq_mul(c[0], u, z);
    fq_mul(c[1], v, z);
    c[2] = z;
    c[3] = c[0];
    c[4] = v;
    uint4* o = reinterpret_cast<uint4*>(out160 + 160 * i);
#pragma unroll
    for (int k = 0; k < 5; k++) {
        o[2 * k] = ok ? make_uint4(c[k].l[0], c[k].l[1], c[k].l[2], c[k].l[3]) : make_uint4(0, 0, 0, 0);
        o[2 * k + 1] = ok ? make_uint4(c[k].l[4], c[k].l[5], c[k].l[6], c[k].l[7]) : make_uint4(0, 0, 0, 0);
    }
}

// ---- aggregate-key path: ordering of a chunk by signer count, entirely on the device -----------------------------------
// Items are bucketed by signer count (bucket 64 collects everything above 63) so that the lanes of a warp hash transcripts
// of one length and fold the same number of keys.  Three small kernels replace the host-side counting sort of round 1 (and
// the stream synchronisation it needed): histogram, exclusive scan over the 65 buckets, scatter.  The order inside a bucket
// depends on atomics; results are written by item index, so the outputs do not.
constexpr int AGG_BUCKETS = 65;
struct AggSort {
    uint32_t hist[AGG_BUCKETS], khist[AGG_BUCKETS];    // items / keys per bucket
    uint32_t ibase[AGG_BUCKETS], kbase[AGG_BUCKETS];   // first sorted item / key position of the bucket
    uint32_t cursor[AGG_BUCKETS], kcursor;             // scatter cursors (kcursor: keys of the open-ended bucket)
};
__global__ void __launch_bounds__(BLOCK) k_agg_hist(const uint32_t* offsets, size_t n, AggSort* c) {
    __shared__ uint32_t h[AGG_BUCKETS], kh[AGG_BUCKETS];
    for (int i = threadIdx.x; i < AGG_BUCKETS; i += blockDim.x) { h[i] = 0; kh[i] = 0; }
    __syncthreads();
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        uint32_t cnt = offsets[i + 1] - offsets[i], b = cnt < AGG_BUCKETS - 1 ? cnt : AGG_BUCKETS - 1;
        atomicAdd(&h[b], 1u);
        atomicAdd(&kh[b], cnt);
    }
    __syncthreads();
    for (int k = threadIdx.x; k < AGG_BUCKETS; k += blockDim.x) {
        if (h[k]) atomicAdd(&c->hist[k], h[k]);
        if (kh[k]) atomicAdd(&c->khist[k], kh[k]);
    }
}
__global__ void k_agg_scan(AggSort* c) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    uint32_t ib = 0, kb = 0;
    for (int b = 0; b < AGG_BUCKETS; b++) {
        c->ibase[b] = ib;
        c->kbase[b] = kb;
        ib += c->hist[b];
        kb += c->khist[b];
    }
}
// order[p]: item at sorted position p;  kmap[q] / kitem[q]: key (relative to the chunk's first key) and item at sorted key position q
__global__ void __launch_bounds__(BLOCK) k_agg_scatter(const uint32_t* offsets, uint32_t key_base, size_t n, AggSort* c, uint32_t* order, uint32_t* kmap,
                                                       uint32_t* kitem) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = i < n;
    uint32_t lo = 0, cnt = 0, b = 0xffffffffu;
    if (valid) {
        lo = offsets[i];
        cnt = offsets[i + 1] - lo;
        b = cnt < AGG_BUCKETS - 1 ? cnt : AGG_BUCKETS - 1;
    }
    // one atomic per distinct bucket of the warp
    const int lane = threadIdx.x & 31;
    uint32_t pos = 0;
    uint32_t remaining = __ballot_sync(0xffffffffu, valid);
    while (remaining) {
        int leader = __ffs(remaining) - 1;
        uint32_t bb = __shfl_sync(0xffffffffu, b, leader);
        uint32_t grp = __ballot_sync(0xffffffffu, valid && b == bb);
        uint32_t base = 0;
        if (lane == leader) base = atomicAdd(&c->cursor[bb], (uint32_t)__popc(grp));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (valid && b == bb) pos = base + __popc(grp & ((1u << lane) - 1u));
        remaining &= ~grp;
    }
    if (!valid) return;
    order[c->ibase[b] + pos] = (uint32_t)i;
    uint32_t kpos = b < AGG_BUCKETS - 1 ? c->kbase[b] + pos * cnt : c->kbase[b] + atomicAdd(&c->kcursor, cnt);
    for (uint32_t j = 0; j < cnt; j++) {
        kmap[kpos + j] = lo - key_base + j;
        kitem[kpos + j] = (uint32_t)i;
    }
}

// one thread hashes the delinearisation coefficient of ONE signer key (sorted key order: the threads of a warp hash transcripts of
// one length).  Per key rather than per item: an item with n signers costs n hashes of 2 + 2 n elements, and spread over n
// threads that work no longer depends on the signer count of the neighbouring items.
__global__ void __launch_bounds__(BLOCK, JJS_HASH_MINBLOCKS) k_agg_coeffs(const fq* keys_u, const fq* keys_v, const uint8_t* kflags,
                                                                          const uint32_t* offsets, const uint32_t* kmap, const uint32_t* kitem,
                                                                          uint32_t key_base, size_t n_keys, uint32_t* d_words, Tables T) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_keys) return;
    size_t item = kitem[t];
    stage_aggregate_coeff_key(keys_u, keys_v, kflags, offsets[item] - key_base, offsets[item + 1] - key_base, kmap[t], d_words, T.safe_tags);
}

// one thread folds the signer keys of one item into its aggregate key (slot 0 of the single-variant point arrays)
// `order` lists the items sorted by signer count, so the lanes of a warp loop over the same number of signers
__global__ void __launch_bounds__(BLOCK, JJS_AGG_MINBLOCKS) k_aggregate(const fq* keys_u, const fq* keys_v, const uint8_t* kflags, const uint32_t* offsets,
                                                     const uint32_t* order, uint32_t key_base, size_t n, fq* pts_u, fq* pts_v, uint8_t* pflags,
                                                     uint8_t* agg_out, fq* tab, size_t stride, uint32_t* d_words, Tables T) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    size_t item = order[t];
    uint32_t w[8];
    stage_aggregate(keys_u, keys_v, kflags, offsets[item] - key_base, offsets[item + 1] - key_base, pts_u, pts_v, pflags, item, w, tab + t, stride,
                    T.safe_tags, d_words);
    if (agg_out) {
        uint4* o = reinterpret_cast<uint4*>(agg_out + item * 32);
        o[0] = make_uint4(w[0], w[1], w[2], w[3]);
        o[1] = make_uint4(w[4], w[5], w[6], w[7]);
    }
}

// Work list of the hash and equation stages: the items that go on after decoding (verify_core.cuh, stage_item_ready).
// The others are settled by their flags, and leaving them out keeps every lane of the two heavy kernels busy on
// batches with many invalid items.  One warp ballot and one atomic per warp; also writes the scalar-range flag of every
// item, clears its equation results and zeroes the challenge words of the items that are left out.
__global__ void __launch_bounds__(BLOCK) k_work_list(int variant, const uint8_t* pflags, size_t n, WireField msg, WireField usc, bool require_valid_keys,
                                                     uint8_t* iflags, uint8_t* eqflags, uint32_t* cwords, uint32_t* list, uint32_t* count) {
    size_t item = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool ready = false;
    if (item < n) {
        bool ok = stage_scalars_ok(msg, usc, item);
        iflags[item] = ok ? IF_SCALARS_OK : 0;
        ready = stage_item_ready(variant, pflags, n, item, ok, require_valid_keys);
        eqflags[item] = 0;
        if (variant == VAR_DOUBLE) eqflags[n + item] = 0;
        if (!ready) {
            uint4* c = reinterpret_cast<uint4*>(cwords + item * 8);
            c[0] = make_uint4(0, 0, 0, 0);
            c[1] = make_uint4(0, 0, 0, 0);
        }
    }
    uint32_t mask = __ballot_sync(0xffffffffu, ready);
    if (mask == 0) return;
    int lane = threadIdx.x & 31, leader = __ffs(mask) - 1;
    uint32_t base = 0;
    if (lane == leader) base = atomicAdd(count, (uint32_t)__popc(mask));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (ready) list[base + __popc(mask & ((1u << lane) - 1u))] = (uint32_t)item;
}

// thread t < *count hashes the challenge of item list[t]
__global__ void __launch_bounds__(BLOCK, JJS_HASH_MINBLOCKS) k_challenge(int variant, const fq* pts_u, const fq* pts_v, size_t n, WireField msg,
                                                                         const uint32_t* list, const uint32_t* count, uint32_t* cwords) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= *count) return;
    stage_challenge_hash(variant, pts_u, pts_v, n, list[t], msg, cwords);
}

__global__ void __launch_bounds__(BLOCK) k_subgroup_check(WireField pts, size_t first, size_t count, int method, uint8_t* out, fq* tab,
                                                          size_t stride, Tables T) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    out[first + t] = subgroup_check(pts, first + t, method, tab + t, stride, T);
}

// thread T = first + t < neq * *count : equation T % neq of item list[T / neq].  Signature points whose subgroup
// membership the equation did not establish are appended to `rlist` (indices into the point arrays) for k_rtest.
// (instantiated per kind of equation: MODE 0 fixed base -- single, double -- and MODE 1 variable base -- var-gen; MODE 0 also per
// width W of the fixed-base tables)
template <int MODE, int W = FB_W>
__global__ void __launch_bounds__(BLOCK, MODE ? JJS_EQ1_MINBLOCKS : JJS_EQ_MINBLOCKS) k_equation(int variant, const fq* pts_u, const fq* pts_v, uint8_t* pflags, size_t n,
                                                    size_t first, size_t count, const uint32_t* list, const uint32_t* lcount, WireField usc,
                                                    const uint32_t* cwords, uint8_t* eqflags, fq* tab, size_t stride, Tables T,
                                                    uint32_t* rlist, uint32_t* rcount) {
    // Persistent form (JJS_EQ_PERSISTENT): the grid is one wave of resident CTAs and every thread walks the work list with the
    // grid's stride, so the two per-thread tables live in a scratch indexed by RESIDENT thread (stride = gridDim.x * blockDim.x,
    // ~130 MB in all, close to the L2's size) instead of by equation (600 MB per 2^18-item sub-chunk).
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int neq = variant == VAR_DOUBLE ? 2 : 1;
    const size_t total = (size_t)neq * *lcount, end = first + count < total ? first + count : total;
#if JJS_EQ_PERSISTENT
    const size_t step = (size_t)gridDim.x * blockDim.x;
#pragma unroll 1
    for (size_t g = first + t; g < end; g += step) {
#else
    {
        const size_t g = first + t;
        if (t >= count || g >= end) return;
#endif
        int eq = (int)(g % neq);
        size_t item = list[g / neq];
        bool need_r_test;
        bool ok = stage_equation_item<MODE, W>(variant, eq, pts_u, pts_v, pflags, n, item, (variant == VAR_DOUBLE && eq == 1) ? T.fb_gn : T.fb_g, usc, cwords,
                                            tab + t, tab + 36 * stride + t, stride, &need_r_test);
        if (need_r_test) {
            int pk_slot, r_slot, base_slot;
            equation_slots(variant, eq, pk_slot, r_slot, base_slot);
            rlist[atomicAdd(rcount, 1u)] = (uint32_t)((size_t)r_slot * n + item);
        }
        eqflags[(size_t)eq * n + item] = ok ? 1 : 0;
    }
}

// The same stage on the slot-based evaluation (fqs.cuh): field elements in shared memory, addressed by handle, so that no
// product needs its operands marshalled through registers.  Persistent: the grid is one wave of resident CTAs and every
// thread walks the work list with the grid's stride, which lets the two per-thread tables live in a scratch indexed by
// RESIDENT thread (gridDim.x * blockDim.x threads x 2 KiB, L2 sized) instead of by item.
#ifndef JJS_EQ2_MINBLOCKS
#define JJS_EQ2_MINBLOCKS 4
#endif
#if JJS_EQ_V2
__global__ void __launch_bounds__(JJS_EQ_BLOCK, JJS_EQ2_MINBLOCKS) k_equation2(int variant, const fq* pts_u, const fq* pts_v, uint8_t* pflags, size_t n,
                                                                                const uint32_t* list, const uint32_t* lcount, WireField usc,
                                                                                const uint32_t* cwords, uint8_t* eqflags, fq* tab, Tables T,
                                                                                uint32_t* rlist, uint32_t* rcount) {
    const Eq2Slots s = eq2_slots(threadIdx.x);
    const size_t nthreads = (size_t)gridDim.x * blockDim.x, tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int neq = variant == VAR_DOUBLE ? 2 : 1;
    const size_t total = (size_t)neq * *lcount;
#pragma unroll 1
    for (size_t g = tid; g < total; g += nthreads) {
        int eq = (int)(g % neq);
        size_t item = list[g / neq];
        bool need_r_test;
        bool ok = eq2_equation_item(s, variant, eq, pts_u, pts_v, pflags, n, item, (variant == VAR_DOUBLE && eq == 1) ? T.fb_gn : T.fb_g, usc, cwords,
                                    tab + tid, tab + EQ2_TAB_FQ * nthreads + tid, nthreads, &need_r_test);
        if (need_r_test) {
            int pk_slot, r_slot, base_slot;
            equation_slots(variant, eq, pk_slot, r_slot, base_slot);
            rlist[atomicAdd(rcount, 1u)] = (uint32_t)((size_t)r_slot * n + item);
        }
        eqflags[(size_t)eq * n + item] = ok ? 1 : 0;
    }
}

#endif  // JJS_EQ_V2

// deferred subgroup tests: thread t < *rcount tests point rlist[t]
__global__ void __launch_bounds__(BLOCK, JJS_DEC_MINBLOCKS) k_rtest(const fq* pts_u, const fq* pts_v, uint8_t* pflags, const uint32_t* rlist,
                                                                     const uint32_t* rcount) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= *rcount) return;
    stage_rtest(pts_u, pts_v, pflags, rlist[t]);
}

__global__ void __launch_bounds__(BLOCK) k_finalize(int variant, const uint8_t* pflags, const uint8_t* iflags, const uint8_t* eqflags,
                                                    const uint32_t* cwords, size_t n, uint8_t* status, uint8_t* c_out) {
    size_t item = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (item >= n) return;
    uint8_t fl = iflags[item];
    if (eqflags[item]) fl |= IF_EQ0_OK;
    if (variant == VAR_DOUBLE && eqflags[n + item]) fl |= IF_EQ1_OK;
    uint8_t st = stage_status(variant, pflags, fl, n, item);
    status[item] = st;
    if (c_out) {
        uint4 a = make_uint4(0, 0, 0, 0), b = a;
        if (st <= 1) {
            const uint4* p = reinterpret_cast<const uint4*>(cwords + item * 8);
            a = p[0];
            b = p[1];
        }
        uint4* o = reinterpret_cast<uint4*>(c_out + item * 32);
        o[0] = a;
        o[1] = b;
    }
}

// accept bitmap: bit (i % 32) of word i / 32 is set iff status[i] == 0; one warp ballot per word
__global__ void __launch_bounds__(BLOCK) k_bitmap(const uint8_t* status, size_t n, uint32_t* words) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool ok = i < n && status[i] == 0;
    uint32_t w = __ballot_sync(0xffffffffu, ok);
    if ((threadIdx.x & 31) == 0 && i < n) words[i >> 5] = w;
}

// ---- whole-batch verification (rlc.cuh): one random linear combination per call --------------------------------------------
__global__ void k_rlc_init(RlcAcc* acc) {
    if (blockIdx.x == 0 && threadIdx.x == 0) rlc_acc_init(*acc);
}
// Whether item `item` of a pass of m enters the combination: status 0 by the reference's precedence (every point decoded and
// valid, scalars in range) with the equation bits assumed
__device__ __forceinline__ bool rlc_item_valid(int variant, const uint8_t* pflags, const uint8_t* iflags, size_t m, size_t item) {
    return stage_status(variant, pflags, (uint8_t)(iflags[item] | IF_EQ0_OK | IF_EQ1_OK), m, item) == 0;
}
// thread = item: validity (rlc_item_valid), weights from the call-wide index base + item, sort entries of the item's group
// (item >> gshift; a whole-batch pass has one group) and the G scalars.  acc: the whole-batch accumulator, whose validity flag an
// invalid item clears (nullptr for a grouped pass, whose invalid items keep the status their flags give)
__global__ void __launch_bounds__(BLOCK) k_rlc_digits(int variant, const uint8_t* pflags, const uint8_t* iflags, const uint32_t* cwords, WireField usc, size_t m,
                                                      int gshift, RlcShape s, RlcSeed seed, uint64_t base, uint32_t* keys, uint32_t* vals, uint32_t* zu,
                                                      RlcAcc* acc) {
    const size_t item = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (item >= m) return;
    const bool valid = rlc_item_valid(variant, pflags, iflags, m, item);
    if (!valid && acc) acc->valid = 0;
    uint32_t u[8], c[8];
    wire_load(u, usc, item);
#pragma unroll
    for (int i = 0; i < 8; i++) c[i] = cwords[item * 8 + i];
    rlc_item_entries(keys + item * s.per_item, vals + item * s.per_item, zu + item * 8, zu + (m + item) * 8, variant, valid, c, u, seed, base + item, m, item,
                     s, (uint32_t)(item >> gshift));
}
__global__ void __launch_bounds__(BLOCK) k_rlc_bucket_init(ext* buckets, size_t nb) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nb) ext_identity(buckets[i]);
}
constexpr int RLC_SEG = 32;      // sorted entries per thread of a segment pass
constexpr int RLC_SLICE = 32;    // buckets per thread of the bucket reduction
__global__ void __launch_bounds__(BLOCK) k_rlc_segments0(const uint32_t* keys, const uint32_t* vals, const fq* pts_u, const fq* pts_v, size_t len, uint32_t sentinel,
                                                         ext* buckets, uint32_t* ckeys, ext* cpts, bool final_level) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    rlc_segment(keys, RlcAffineSrc{pts_u, pts_v, vals}, len, t, RLC_SEG, sentinel, buckets, ckeys, cpts, final_level);
}
__global__ void __launch_bounds__(BLOCK) k_rlc_segments(const uint32_t* keys, const ext* pts, size_t len, uint32_t sentinel, ext* buckets, uint32_t* ckeys,
                                                        ext* cpts, bool final_level) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    rlc_segment(keys, RlcExtSrc{pts}, len, t, RLC_SEG, sentinel, buckets, ckeys, cpts, final_level);
}
// thread = slice of RLC_SLICE buckets of one window (of every group's windows, nw = groups x nw_big)
__global__ void __launch_bounds__(BLOCK) k_rlc_slices(const ext* buckets, int nw, uint32_t per_window, ext* partial) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t slices = per_window / RLC_SLICE;
    if (t >= (size_t)nw * slices) return;
    const uint32_t w = (uint32_t)(t / slices), sl = (uint32_t)(t % slices);
    rlc_bucket_slice(partial[t], buckets + (size_t)w * per_window, sl * RLC_SLICE, (sl + 1) * RLC_SLICE);
}
// block = window, 32 threads: the window's slice sums
__global__ void __launch_bounds__(32) k_rlc_window_sums(const ext* partial, uint32_t slices, ext* W) {
    __shared__ ext part[32];
    ext acc;
    ext_identity(acc);
    for (uint32_t i = threadIdx.x; i < slices; i += 32) rlc_add(acc, partial[(size_t)blockIdx.x * slices + i]);
    part[threadIdx.x] = acc;
    __syncwarp();
    if (threadIdx.x == 0) {
        for (int k = 1; k < 32; k++) rlc_add(acc, part[k]);
        W[blockIdx.x] = acc;
    }
}
// one thread: Horner over the windows, added to the half's accumulator
__global__ void k_rlc_horner(const ext* W, int nw, int c, RlcAcc* acc) {
    if (blockIdx.x || threadIdx.x) return;
    ext P;
    rlc_horner(P, W, nw, c);
    rlc_add(acc->P, P);
}
// block = group of g items: the group's G (and G') scalar sums added into su[group], mod r (a whole-batch pass: one block, su =
// the accumulator's, g >= m).  Sums of up to 2^24 values below 2^252 fit in nine words, so the block adds exactly and reduces once.
constexpr int RLC_SUM_THREADS = 256;
__global__ void __launch_bounds__(RLC_SUM_THREADS) k_rlc_scalars(const uint32_t* zu, size_t m, size_t g, int neq, uint32_t (*su)[2][8]) {
    __shared__ uint32_t part[RLC_SUM_THREADS][9];
    const size_t lo = (size_t)blockIdx.x * g, hi = lo + g < m ? lo + g : m;
    for (int eq = 0; eq < neq; eq++) {
        uint32_t s[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
        // One block reads a whole pass of a whole-batch call, so the loads of four values are issued before their additions.
        const uint4* z = reinterpret_cast<const uint4*>(zu + (size_t)eq * m * 8);
        constexpr int AHEAD = 4;
        size_t i = lo + threadIdx.x;
        for (; i + (AHEAD - 1) * RLC_SUM_THREADS < hi; i += AHEAD * RLC_SUM_THREADS) {
            uint4 v[2 * AHEAD];
#pragma unroll
            for (int k = 0; k < AHEAD; k++) {
                v[2 * k] = z[2 * (i + k * RLC_SUM_THREADS)];
                v[2 * k + 1] = z[2 * (i + k * RLC_SUM_THREADS) + 1];
            }
#pragma unroll
            for (int k = 0; k < AHEAD; k++) {
                const uint32_t w[8] = {v[2 * k].x, v[2 * k].y, v[2 * k].z, v[2 * k].w, v[2 * k + 1].x, v[2 * k + 1].y, v[2 * k + 1].z, v[2 * k + 1].w};
                s[8] += add8c(s, s, w, 0u);
            }
        }
        for (; i < hi; i += RLC_SUM_THREADS) s[8] += add8c(s, s, zu + ((size_t)eq * m + i) * 8, 0u);
        for (int k = 0; k < 9; k++) part[threadIdx.x][k] = s[k];
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int t = 1; t < RLC_SUM_THREADS; t++) s[8] += part[t][8] + add8c(s, s, part[t], 0u);
            uint32_t wide[16] = {0}, red[8];
            for (int k = 0; k < 9; k++) wide[k] = s[k];
            fr_reduce_wide(red, wide, 9 * 32);
            fr_add(su[blockIdx.x][eq], su[blockIdx.x][eq], red);
        }
        __syncthreads();
    }
}
// thread = group: Horner over the group's windows, its G and G' terms added; verdict[group] = 1 iff the group's combination
// is the identity
template <int W>
__global__ void __launch_bounds__(BLOCK) k_rlc_verdicts(const ext* Wsum, int nw, int c, size_t groups, const uint32_t (*su)[2][8], Tables T,
                                                         uint8_t* verdict) {
    const size_t grp = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (grp >= groups) return;
    ext P;
    rlc_horner(P, Wsum + grp * (size_t)nw, nw, c);
    rlc_fixed_terms<W>(P, su[grp], true, T.fb_g, T.fb_gn);
    verdict[grp] = ext_is_identity(P) ? 1 : 0;
}
// thread = item of a grouped pass: an item that entered a group whose combination holds gets its equation bits; one that entered
// a failing group goes on the equation work list (the list and count of k_work_list, reset by the caller) and into *fallback.
// Items that did not enter keep cleared equation bits: their status comes from their flags.
__global__ void __launch_bounds__(BLOCK) k_rlc_gate(int variant, const uint8_t* pflags, const uint8_t* iflags, size_t m, int gshift, const uint8_t* verdict,
                                                    uint8_t* eqflags, uint32_t* list, uint32_t* count, unsigned long long* fallback) {
    const size_t item = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool redo = false;
    if (item < m && rlc_item_valid(variant, pflags, iflags, m, item)) {
        if (verdict[item >> gshift]) {
            eqflags[item] = 1;
            if (variant == VAR_DOUBLE) eqflags[m + item] = 1;
        } else {
            redo = true;
        }
    }
    const uint32_t mask = __ballot_sync(0xffffffffu, redo);
    if (mask == 0) return;
    const int lane = threadIdx.x & 31, leader = __ffs(mask) - 1;
    uint32_t at = 0;
    if (lane == leader) {
        at = atomicAdd(count, (uint32_t)__popc(mask));
        if (fallback) atomicAdd(fallback, (unsigned long long)__popc(mask));
    }
    at = __shfl_sync(0xffffffffu, at, leader);
    if (redo) list[at + __popc(mask & ((1u << lane) - 1u))] = (uint32_t)item;
}
struct RlcOut {
    ext P;
    uint32_t valid;
};
// one thread: the halves' accumulators summed, the G and G' terms added (a call may mix kinds, and a zero scalar sum adds the
// identity); writes the device's partial point (host entry point, summed over devices on the host) and / or the verdict
// (device entry point)
template <int W>
__global__ void k_rlc_finish(const RlcAcc* acc0, const RlcAcc* acc1, Tables T, RlcOut* out, int* all_valid) {
    if (blockIdx.x || threadIdx.x) return;
    ext P = acc0->P;
    uint32_t su[2][8], valid = acc0->valid;
    for (int i = 0; i < 8; i++) { su[0][i] = acc0->su[0][i]; su[1][i] = acc0->su[1][i]; }
    rlc_add(P, acc1->P);
    fr_add(su[0], su[0], acc1->su[0]);
    fr_add(su[1], su[1], acc1->su[1]);
    valid &= acc1->valid;
    rlc_fixed_terms<W>(P, su, true, T.fb_g, T.fb_gn);
    if (out) {
        out->P = P;
        out->valid = valid;
    }
    if (all_valid) *all_valid = (valid && ext_is_identity(P)) ? 1 : 0;
}

// Fixed-base tables of width W in two passes (curve.cuh, fb_combine_entries), LO = (W + 1) / 2, HI = W - LO.  Pass 1: the small
// tables of every window, affine points, small[w][0 .. 2^LO) = jl 2^(W w) B  and  small[w][2^LO .. 2^LO + 2^HI) = jh 2^(W w + LO) B.
template <int W>
__global__ void __launch_bounds__(BLOCK) k_fb_small(fq* small_u, fq* small_v, int which) {
    constexpr int LO = (W + 1) / 2, HI = W - LO, WINDOWS = (252 + W - 1) / W, SMALL = (1 << LO) + (1 << HI);
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= WINDOWS * SMALL) return;
    fq bu, bv, u, v;
    fq_load_const(bu, which ? JJS_C(GEN_NUMS_UV)[0] : JJS_C(GEN_UV)[0]);
    fq_load_const(bv, which ? JJS_C(GEN_NUMS_UV)[1] : JJS_C(GEN_UV)[1]);
    int w = t / SMALL, e = t % SMALL;
    if (e < (1 << LO)) fb_affine_multiple(u, v, bu, bv, w * W, e, LO);
    else fb_affine_multiple(u, v, bu, bv, w * W + LO, e - (1 << LO), HI);
    small_u[t] = u;
    small_v[t] = v;
}
// Pass 2: thread t combines entries [FB_BATCH t, FB_BATCH (t + 1)) of the table (FB_BATCH divides 2^LO, so they share jh).
template <int W>
__global__ void __launch_bounds__(BLOCK) k_fb_combine(niels* out, const fq* small_u, const fq* small_v) {
    constexpr int LO = (W + 1) / 2, HI = W - LO, WINDOWS = (252 + W - 1) / W, ENTRIES = 1 << W, SMALL = (1 << LO) + (1 << HI);
    static_assert((1 << LO) % FB_BATCH == 0, "a batch of table entries must share its high half");
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (size_t)WINDOWS * ENTRIES / FB_BATCH) return;
    size_t first = t * FB_BATCH;
    int w = (int)(first / ENTRIES), j = (int)(first % ENTRIES), jh = j >> LO, jl = j & ((1 << LO) - 1);
    const fq* su = small_u + (size_t)w * SMALL;
    const fq* sv = small_v + (size_t)w * SMALL;
    fb_combine_entries(out + first, su + jl, sv + jl, su[(1 << LO) + jh], sv[(1 << LO) + jh]);
}
// the definition, entry by entry (jjs_fb_table_check compares a sample of the built tables with it)
template <int W>
__global__ void __launch_bounds__(BLOCK) k_fb_check(const niels* table, int which, const uint32_t* entries, int n, uint32_t* mismatches) {
    constexpr int WINDOWS = (252 + W - 1) / W, ENTRIES = 1 << W;
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    fq u, v;
    fq_load_const(u, which ? JJS_C(GEN_NUMS_UV)[0] : JJS_C(GEN_UV)[0]);
    fq_load_const(v, which ? JJS_C(GEN_NUMS_UV)[1] : JJS_C(GEN_UV)[1]);
    niels e;
    uint32_t idx = entries[t] % (uint32_t)(WINDOWS * ENTRIES);
    fb_table_entry<W>(e, u, v, (int)(idx / ENTRIES), (int)(idx % ENTRIES));
    const niels& g = table[idx];
    if (!(fq_eq(e.ypx, g.ypx) && fq_eq(e.ymx, g.ymx) && fq_eq(e.t2d, g.t2d))) atomicAdd(mismatches, 1u);
}

// ---- registered key sets (keyset.cuh) --------------------------------------------------------------------------------
// Key points are numbered key-major (point p = key * nk + s, the order of the tables); the decoded points are slot-major
// (s * n_keys + key, as k_decode writes them).
// Table pass 1: thread p computes the window bases of key point p, bases[w * npts + p].  KW: the key-window width (keyset.cuh).
template <int KW>
__global__ void __launch_bounds__(BLOCK) k_keyset_bases(int variant, const fq* keys_u, const fq* keys_v, const uint8_t* kflags, size_t n_keys,
                                                        ext* bases) {
    const int nk = keyed_points(variant);
    const size_t npts = (size_t)nk * n_keys, p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= npts) return;
    const size_t k = (size_t)(p % nk) * n_keys + p / nk;
    fq u, v;
    keyed_table_base(u, v, keys_u[k], keys_v[k], kflags[k]);
    keyed_window_bases<KW>(bases + p, npts, u, v);
}
// Table pass 2: one thread per batch of KEYED_BATCH entries of one window of one key point.
JJS_HD constexpr int keyed_groups(int kw) { return keyed_entries(kw) / KEYED_BATCH; }
template <int KW>
__global__ void __launch_bounds__(BLOCK) k_keyset_combine(const ext* bases, size_t npts, niels* table) {
    constexpr int WINDOWS = keyed_windows(KW), ENTRIES = keyed_entries(KW), GROUPS = keyed_groups(KW);
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= npts * WINDOWS * GROUPS) return;
    const size_t p = t / (WINDOWS * GROUPS);
    const int r = (int)(t % (WINDOWS * GROUPS)), w = r / GROUPS, g = r % GROUPS;
    keyed_combine_entries<KW>(table + p * keyed_point_entries(KW) + (size_t)w * ENTRIES + (size_t)g * KEYED_BATCH, bases[(size_t)w * npts + p],
                              g * KEYED_BATCH + 1);
}
// the definition, entry by entry (jjs_keyset_table_check): flat index p * keyed_point_entries(KW) + w * keyed_entries(KW) + j - 1
template <int KW>
__global__ void __launch_bounds__(BLOCK) k_keyset_check(int variant, const fq* keys_u, const fq* keys_v, const uint8_t* kflags, size_t n_keys,
                                                        const niels* table, const uint32_t* entries, size_t n, uint32_t* mismatches) {
    constexpr int ENTRIES = keyed_entries(KW), POINT_ENTRIES = keyed_point_entries(KW);
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const int nk = keyed_points(variant);
    const size_t idx = (size_t)entries[t] % ((size_t)nk * n_keys * POINT_ENTRIES), p = idx / POINT_ENTRIES;
    const int e = (int)(idx % POINT_ENTRIES);
    const size_t k = (size_t)(p % nk) * n_keys + p / nk;
    fq u, v;
    keyed_table_base(u, v, keys_u[k], keys_v[k], kflags[k]);
    niels ref;
    keyed_table_entry<KW>(ref, u, v, e / ENTRIES, e % ENTRIES + 1);
    const niels& g = table[idx];
    if (!(fq_eq(ref.ypx, g.ypx) && fq_eq(ref.ymx, g.ymx) && fq_eq(ref.t2d, g.t2d))) atomicAdd(mismatches, 1u);
}
// key slots of the chunk's items from the key set, by index
__global__ void __launch_bounds__(BLOCK) k_keyed_gather(int variant, const fq* keys_u, const fq* keys_v, const uint8_t* kflags, size_t n_keys,
                                                        const uint32_t* key_index, size_t n, fq* pts_u, fq* pts_v, uint8_t* pflags) {
    const size_t item = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (item >= n) return;
    stage_keyed_gather(variant, keys_u, keys_v, kflags, n_keys, key_index[item], pts_u, pts_v, pflags, n, item);
}
// thread t < neq * *count: equation t % neq of item list[t / neq] under its registered key (stage_equation_keyed).  No per-thread
// table scratch: both products read precomputed tables.
#ifndef JJS_EQK_MINBLOCKS
#define JJS_EQK_MINBLOCKS 4
#endif
template <int W, int KW>
__global__ void __launch_bounds__(BLOCK, JJS_EQK_MINBLOCKS) k_equation_keyed(int variant, const fq* pts_u, const fq* pts_v, uint8_t* pflags, size_t n,
                                                                             const uint32_t* list, const uint32_t* lcount, WireField usc,
                                                                             const uint32_t* cwords, uint8_t* eqflags, const niels* ktab,
                                                                             const uint32_t* key_index, size_t n_keys, Tables T, uint32_t* rlist,
                                                                             uint32_t* rcount) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int neq = keyed_points(variant);
    if (t >= (size_t)neq * *lcount) return;
    const int eq = (int)(t % neq);
    const size_t item = list[t / neq];
    const uint32_t key = key_index[item];   // in range: items under an unknown index never reach the work list
    bool need_r_test = false;
    const bool ok = key < n_keys &&
                    stage_equation_keyed<W, KW>(variant, eq, pts_u, pts_v, pflags, n, item, eq == 1 ? T.fb_gn : T.fb_g,
                                                ktab + ((size_t)key * neq + eq) * keyed_point_entries(KW), usc, cwords, &need_r_test);
    if (need_r_test) {
        int pk_slot, r_slot, base_slot;
        equation_slots(variant, eq, pk_slot, r_slot, base_slot);
        rlist[atomicAdd(rcount, 1u)] = (uint32_t)((size_t)r_slot * n + item);
    }
    eqflags[(size_t)eq * n + item] = ok ? 1 : 0;
}

// one thread signs one item; inputs are 32-byte little-endian scalars, outputs the reference's wire bytes.
// The variant is a template parameter so that every array index below is static; W is the width of the fixed-base tables.
template <int VARIANT, int W = FB_W>
__global__ void __launch_bounds__(BLOCK) k_sign(const uint8_t* sk, const uint8_t* rnd, const uint8_t* gsc, const uint8_t* msg, size_t n,
                                                uint8_t* pk_out, uint8_t* sig_out, Tables T) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    constexpr int PKW = VARIANT == VAR_SINGLE ? 8 : 16, SGW = VARIANT == VAR_DOUBLE ? 24 : 16;
    uint32_t wsk[8], wrnd[8], wg[8], wm[8], pk[16], sig[24];
    wire_load(wsk, WireField{sk, 32}, i);
    wire_load(wrnd, WireField{rnd, 32}, i);
    wire_load(wm, WireField{msg, 32}, i);
    if (VARIANT == VAR_VARGEN) wire_load(wg, WireField{gsc, 32}, i);
    bool ok = sign_item<W>(VARIANT, wsk, wrnd, wg, wm, pk, sig, T);
    uint4* po = reinterpret_cast<uint4*>(pk_out + i * PKW * 4);
    uint4* so = reinterpret_cast<uint4*>(sig_out + i * SGW * 4);
#pragma unroll
    for (int k = 0; k < PKW / 4; k++) po[k] = ok ? make_uint4(pk[4 * k], pk[4 * k + 1], pk[4 * k + 2], pk[4 * k + 3]) : make_uint4(0, 0, 0, 0);
#pragma unroll
    for (int k = 0; k < SGW / 4; k++) so[k] = ok ? make_uint4(sig[4 * k], sig[4 * k + 1], sig[4 * k + 2], sig[4 * k + 3]) : make_uint4(0, 0, 0, 0);
}

// ---- multisig::combine ---------------------------------------------------------------------------------------------
struct MsigBuffers {
    fq *pu, *pv;           // [3K] decoded pk | R | S
    uint8_t* pf;           // [3K]
    uint32_t *d_words, *cd_words;  // [K][8]
    uint32_t* a_words;     // [n][8]
    fq *rsa_u, *rsa_v;     // [n]
    uint8_t* sflags;       // [n]
    uint8_t* share_ok;     // [K]
    const uint32_t *offsets, *owner, *order;
};

__global__ void __launch_bounds__(BLOCK) k_msig_session(MsigBuffers b, size_t K, size_t n, WireField msg, WireField zf, fq* tab, size_t stride, Tables T) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    size_t s = b.order[t];
    stage_msig_session(b.pu, b.pv, b.pf, K, b.offsets[s], b.offsets[s + 1], msg, zf, s, b.d_words, b.cd_words, b.a_words, b.rsa_u, b.rsa_v, b.sflags,
                       tab + t, stride, T.safe_tags);
}
template <int W = FB_W>
__global__ void __launch_bounds__(BLOCK, JJS_EQ_MINBLOCKS) k_msig_share(MsigBuffers b, size_t K, WireField zf, fq* tab, size_t stride, Tables T) {
    size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= K) return;
    size_t s = b.owner[j];
    bool ok = false;
    if (b.sflags[s] == (SF_DECODED | SF_NONEMPTY))
        ok = stage_msig_share<W>(b.pu, b.pv, K, j, zf, b.cd_words, b.a_words + 8 * s, T.fb_g, tab + j, tab + 36 * stride + j, stride);
    b.share_ok[j] = ok ? 1 : 0;
}
__global__ void __launch_bounds__(BLOCK) k_msig_finalize(MsigBuffers b, size_t n, WireField zf, uint8_t* status, uint32_t* bad, uint8_t* sig64) {
    size_t s = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    uint32_t sig[16], bi;
    uint8_t st = stage_msig_finalize(b.sflags, b.share_ok, b.offsets[s], b.offsets[s + 1], s, zf, b.rsa_u, b.rsa_v, &bi, sig);
    status[s] = st;
    bad[s] = bi;
    uint4* o = reinterpret_cast<uint4*>(sig64 + 64 * s);
#pragma unroll
    for (int k = 0; k < 4; k++) o[k] = make_uint4(sig[4 * k], sig[4 * k + 1], sig[4 * k + 2], sig[4 * k + 3]);
}

// Aggregate-key items for synthetic batches: signer keys pk_j = sk_j * G, the aggregate secret sum_j d_j sk_j with the
// reference's delinearisation coefficients, and an ordinary hedged signature under it (what a completed SpeedyMuSig
// session verifies as).  At most JJS_MAX_GEN_SIGNERS signers per item.
#define JJS_MAX_GEN_SIGNERS 8
template <int W = FB_W>
__global__ void __launch_bounds__(BLOCK) k_sign_aggregate(const uint8_t* sk, const uint32_t* offsets, const uint8_t* rnd, const uint8_t* msg, size_t n,
                                                          uint8_t* pks_out, uint8_t* sig_out, Tables T) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t lo = offsets[i], hi = offsets[i + 1];
    uint32_t cnt = hi - lo;
    fq ku[JJS_MAX_GEN_SIGNERS], kv[JJS_MAX_GEN_SIGNERS];
    uint32_t agg[8] = {0, 0, 0, 0, 0, 0, 0, 0}, ord[8], w[8];
    bool ok = cnt <= JJS_MAX_GEN_SIGNERS;
#pragma unroll
    for (int k = 0; k < 8; k++) ord[k] = JJS_C(R_ORDER)[k];
    if (ok) {
#pragma unroll 1
        for (uint32_t j = 0; j < cnt; j++) {
            wire_load(w, WireField{sk, 32}, lo + j);
            ok = ok && fr_wire_is_canonical(w);
            ext P;
            fixedbase_mul<W>(P, T.fb_g, w);
            ext_to_affine(ku[j], kv[j], P);
            uint32_t enc[8];
            point_to_wire(enc, ku[j], kv[j]);
            uint4* o = reinterpret_cast<uint4*>(pks_out + 32 * (size_t)(lo + j));
            o[0] = make_uint4(enc[0], enc[1], enc[2], enc[3]);
            o[1] = make_uint4(enc[4], enc[5], enc[6], enc[7]);
        }
#pragma unroll 1
        for (uint32_t j = 0; j < cnt; j++) {
            Sponge sp;
            sponge_start(sp, (int)(2 + 2 * cnt));
            sponge_absorb(sp, ku[j]);
            sponge_absorb(sp, kv[j]);
#pragma unroll 1
            for (uint32_t k = 0; k < cnt; k++) {
                sponge_absorb(sp, ku[k]);
                sponge_absorb(sp, kv[k]);
            }
            uint32_t dj[8], t[8], s[8];
            sponge_squeeze_truncated(dj, sp);
            wire_load(w, WireField{sk, 32}, lo + j);
            fr_mul(t, dj, w);
            add8(s, agg, t);  // < 2r < 2^256
            uint32_t borrow = sub8(t, s, ord);
#pragma unroll
            for (int k = 0; k < 8; k++) agg[k] = borrow ? s[k] : t[k];
        }
    }
    uint32_t wr[8], wm[8], pk[16], sig[24];
    wire_load(wr, WireField{rnd, 32}, i);
    wire_load(wm, WireField{msg, 32}, i);
    ok = ok && sign_item<W>(VAR_SINGLE, agg, wr, wr, wm, pk, sig, T);
    uint4* so = reinterpret_cast<uint4*>(sig_out + 64 * i);
#pragma unroll
    for (int k = 0; k < 4; k++) so[k] = ok ? make_uint4(sig[4 * k], sig[4 * k + 1], sig[4 * k + 2], sig[4 * k + 3]) : make_uint4(0, 0, 0, 0);
}

struct AggScratch {   // aggregate-key path, one per scratch half: decoded signer keys, their coefficients, the sorted orders
    fq *keys_u = nullptr, *keys_v = nullptr;
    uint8_t* kflags = nullptr;
    uint32_t *kcoef = nullptr, *kmap = nullptr, *kitem = nullptr, *order = nullptr;
    AggSort* sort = nullptr;
    size_t cap_keys = 0;
};

struct DeviceState {
    int device = -1;
    cudaStream_t stream = nullptr, copy_stream = nullptr;
    cudaEvent_t copied = nullptr;
    // two internal compute streams: consecutive sub-chunks of a batch alternate between them (each on its own half of
    // the scratch), so the last, partially filled wave of one kernel overlaps the first blocks of the next chunk's
    cudaStream_t sub[2] = {nullptr, nullptr};
    cudaEvent_t fork = nullptr, join[2] = {nullptr, nullptr};
    fq* root_tables = nullptr;
    uint8_t* dlog_hash = nullptr;
    niels* fb_g = nullptr;
    niels* fb_gn = nullptr;
    fq* safe_tags = nullptr;     // SAFE tags by number of absorbed elements (multisig transcripts of run-time length)
    size_t n_tags = 0;
    // pipeline scratch, sized for CHUNK_ITEMS items of the widest variant (4 points, 2 equations)
    fq *pts_u = nullptr, *pts_v = nullptr, *tab = nullptr;
    uint8_t *pflags = nullptr, *iflags = nullptr, *eqflags = nullptr;
    uint32_t* cwords = nullptr;
    uint32_t *rlist = nullptr, *rcount = nullptr;  // signature points awaiting the deferred subgroup test
    uint32_t* eqlist = nullptr;                    // items that go on to the hash and equation kernels (k_work_list)
    // persistent equation kernel: one wave of resident CTAs, two per-thread tables per resident thread, one such scratch
    // per compute stream (the two sub-chunk streams may run their equation kernels back to back or side by side)
    fq* eqtab = nullptr;
    size_t eqtab_half = 0;         // elements per stream's scratch
    int eq_grid = 0;
    AggScratch agg[2];
    // staging of the host-buffer entry points: one grow-only device buffer, carved up per call
    uint8_t* stage = nullptr;
    size_t stage_bytes = 0;
    // Device memory: `held` bytes allocated by the context on this device (key sets included); a memory-limited context
    // (jjs_init_limited) never lets it exceed `limit` (0: no limit, a jjs_init context).
    size_t limit = 0, held = 0;
    // The configuration (pick_config for limited contexts): width of the G / G' tables, items per pipeline pass, per scratch
    // half, per sub-chunk of an overlapped batch and in the first slice of a host-buffer shard, first size of the aggregate
    // key scratch and items per aggregate pass the order array serves.
    int fb_w = FB_W;
    size_t chunk_items = CHUNK_ITEMS, sub_items = SUB_ITEMS, sub_chunk = SUB_CHUNK, first_slice = size_t(1) << JJS_FIRST_SLICE_LOG2;
    size_t agg_keys_initial = AGG_KEYS_INITIAL, agg_items = CHUNK_ITEMS;
    Tables tables() const { return Tables{root_tables, dlog_hash, fb_g, fb_gn, safe_tags}; }
};

// Per-thread table scratch of a memory-limited context: TAB_ROWS field elements per item of capacity, the equation kernels'
// three 36-element tables (tabA, tabB = tabA + 36 stride, and the var-generator's third).
constexpr int TAB_ROWS = 3 * 36;
// Stride (threads served at once) in the table scratch of a region of `cap` items for a kernel with `rows` elements per thread.
// A jjs_init context's scratch holds the aggregation kernel's 4 x 68 rows for TAB_THREADS threads, and every kernel indexes it
// with that stride.  A limited context gives a region TAB_ROWS x cap elements: the largest power of two <= cap whose rows fit.
inline size_t tab_threads(const DeviceState& d, size_t cap, int rows) {
    if (!d.limit) return TAB_THREADS;
    size_t t = cap;
    while (t > 1 && t * rows > (size_t)TAB_ROWS * cap) t /= 2;
    return t;
}

// A slice of the pipeline scratch able to hold `cap` items of the widest variant; `tab` serves `cap` equation threads with stride
// `tstride`, or `acap` threads of the aggregation kernel with stride `astride` (tab_threads).
struct Region {
    fq *pts_u, *pts_v, *tab, *eqtab;
    uint8_t *pflags, *iflags, *eqflags;
    uint32_t *cwords, *rlist, *rcount, *eqlist;   // rcount[0]: deferred subgroup tests, rcount[2]: length of the work list
    size_t cap;
    int half;
    size_t tstride, astride, acap;
};
inline Region region_of(const DeviceState& d, size_t first_item, size_t cap, int half) {
    const size_t astride = tab_threads(d, cap, AGG_GROUP * R32_TAB_FQ);
    return Region{d.pts_u + 4 * first_item, d.pts_v + 4 * first_item, d.tab + (d.limit ? (size_t)TAB_ROWS * first_item : first_item),
                  d.eqtab + (size_t)(half & 1) * d.eqtab_half, d.pflags + 4 * first_item, d.iflags + first_item,
                  d.eqflags + 2 * first_item, d.cwords + 8 * first_item, d.rlist + 2 * first_item, d.rcount + 4 * (half & 1), d.eqlist + 2 * first_item, cap,
                  half & 1, tab_threads(d, cap, TAB_ROWS), astride, astride < cap ? astride : cap};
}
inline Region region_whole(const DeviceState& d) { return region_of(d, 0, d.chunk_items, 0); }
inline Region region_half(const DeviceState& d, size_t j) { return region_of(d, (j & 1) * d.sub_items, d.sub_items, (int)(j & 1)); }

// A registered key set (jjs_keyset_create / _limited), copied to every device of the context: the decoded key points slot-major
// as k_decode writes them (point s of key k at s * n_keys + k), their flags, and the window tables of width key_bits key-major
// (keyset.cuh; the table of point s of key k starts at entry (k * nk + s) * keyed_point_entries(key_bits)).  key_bits 0: no
// tables, the points only; items then run the per-item equation of run_chunk.
struct KeySetDev {
    fq *u = nullptr, *v = nullptr;
    uint8_t* flags = nullptr;
    niels* table = nullptr;
};
struct KeySet {
    int variant = VAR_SINGLE;
    int key_bits = KEYED_W;
    size_t n_keys = 0;
    std::vector<KeySetDev> dev;
};

}  // namespace

struct StageRecord {
    int stage;
    int device;
    cudaEvent_t e0, e1;
};

struct jjs_ctx {
    std::vector<DeviceState> dev;
    bool ready = false;              // jjs_init succeeded on every device; nothing else may touch the devices
    std::mutex mu;                   // guards err and records (the host entry points run one worker thread per device)
    char err[512];
    std::atomic<uint64_t> launches{0};
    bool profile = false;
    std::vector<StageRecord> records;
    std::vector<fq> tags;            // host copy of the SAFE tag table
    std::vector<KeySet*> keysets;    // registered key sets by handle (nullptr once destroyed; handles are not reused)
};

namespace {

int fail(jjs_ctx* ctx, int code, const char* fmt, ...) {
    if (ctx) {
        std::lock_guard<std::mutex> lock(ctx->mu);
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(ctx->err, sizeof(ctx->err), fmt, ap);
        va_end(ap);
    }
    return code;
}

#define JJS_CUDA(ctx, call)                                                                                   \
    do {                                                                                                      \
        cudaError_t e_ = (call);                                                                              \
        if (e_ != cudaSuccess) return fail(ctx, e_ == cudaErrorMemoryAllocation ? JJS_ERR_NOMEM : JJS_ERR_CUDA, \
                                           "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

// Every entry point starts here: a context whose jjs_init failed exists only so that the caller can read the reason.
#define JJS_ENTER(ctx)                                                                                         \
    do {                                                                                                      \
        if (!(ctx)) return JJS_ERR_ARGUMENT;                                                                  \
        if (!(ctx)->ready || (ctx)->dev.empty()) return JJS_ERR_CUDA; /* err keeps the message of jjs_init */ \
        { std::lock_guard<std::mutex> lock_((ctx)->mu); (ctx)->err[0] = 0; }                                  \
    } while (0)

// Optional per-stage timing: CUDA events recorded on the launching stream around each stage's launches.
struct StageTimer {
    jjs_ctx* ctx;
    StageRecord rec;
    bool on;
    StageTimer(jjs_ctx* c, int device, int stage, cudaStream_t s) : ctx(c), on(c->profile) {
        if (!on) return;
        rec.stage = stage;
        rec.device = device;
        cudaEventCreate(&rec.e0);
        cudaEventCreate(&rec.e1);
        cudaEventRecord(rec.e0, s);
    }
    void stop(cudaStream_t s) {
        if (!on) return;
        cudaEventRecord(rec.e1, s);
        std::lock_guard<std::mutex> lock(ctx->mu);
        ctx->records.push_back(rec);
    }
};

inline unsigned blocks_for(size_t threads) { return (unsigned)((threads + BLOCK - 1) / BLOCK); }
inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Allocator of one device of a context: `held` counts every allocation, and a memory-limited context refuses one that would
// cross its limit.  A dry run only adds the sizes up: the policy of jjs_init_limited (footprint) runs the allocation code of a
// configuration that way, so what it plans and what a context holds cannot drift apart.
struct DevAlloc {
    jjs_ctx* ctx;
    DeviceState* d;   // nullptr: dry run
    size_t total = 0;
    template <typename T>
    int operator()(T** p, size_t bytes) {
        total += bytes;
        if (!d) return JJS_SUCCESS;
        *p = nullptr;
        if (d->limit && d->held + bytes > d->limit)
            return fail(ctx, JJS_ERR_NOMEM, "device %d: %zu more bytes would exceed the context's memory limit of %zu bytes (%zu held)", d->device, bytes,
                        d->limit, d->held);
        cudaError_t e = cudaMalloc((void**)p, bytes);
        if (e != cudaSuccess) {
            *p = nullptr;
            cudaGetLastError();
            return fail(ctx, e == cudaErrorMemoryAllocation ? JJS_ERR_NOMEM : JJS_ERR_CUDA, "cudaMalloc of %zu bytes on device %d failed: %s", bytes,
                        d->device, cudaGetErrorString(e));
        }
        d->held += bytes;
        return JJS_SUCCESS;
    }
};
inline DevAlloc dev_alloc(jjs_ctx* ctx, DeviceState& d) { return DevAlloc{ctx, &d}; }
template <typename T>
void dev_free(DeviceState& d, T*& p, size_t bytes) {
    if (!p) return;
    cudaFree(p);
    p = nullptr;
    d.held -= bytes;
}
// a growth of `more` bytes that frees `less` first: refused up front on a limited context, which then keeps what it has
int check_growth(jjs_ctx* ctx, const DeviceState& d, size_t less, size_t more, const char* what) {
    if (d.limit && d.held - less + more > d.limit)
        return fail(ctx, JJS_ERR_NOMEM, "device %d: growing the %s to %zu bytes would exceed the context's memory limit of %zu bytes (%zu held)", d.device,
                    what, more, d.limit, d.held);
    return JJS_SUCCESS;
}

inline size_t fb_table_bytes(int w) { return sizeof(niels) * (size_t)fb_windows(w) << w; }

// constant tables and the fixed-base tables of width d.fb_w
int alloc_tables(DevAlloc& A, DeviceState& d) {
    int rc = A(&d.root_tables, sizeof(tables::ROOT_TABLES));
    if (!rc) rc = A(&d.dlog_hash, sizeof(tables::DLOG_HASH));
    if (!rc) rc = A(&d.fb_g, fb_table_bytes(d.fb_w));
    if (!rc) rc = A(&d.fb_gn, fb_table_bytes(d.fb_w));
    return rc;
}

// pipeline scratch for `cap` items of the widest variant (4 points, 2 equations) and `tab_fq` elements of per-thread tables
int alloc_pipeline(DevAlloc& A, DeviceState& d, size_t cap, size_t tab_fq) {
    int rc = A(&d.pts_u, sizeof(fq) * 4 * cap);
    if (!rc) rc = A(&d.pts_v, sizeof(fq) * 4 * cap);
    if (!rc) rc = A(&d.pflags, 4 * cap);
    if (!rc) rc = A(&d.iflags, cap);
    if (!rc) rc = A(&d.eqflags, 2 * cap);
    if (!rc) rc = A(&d.cwords, 32 * cap);
    if (!rc) rc = A(&d.rlist, sizeof(uint32_t) * 2 * cap);
    if (!rc) rc = A(&d.rcount, 8 * sizeof(uint32_t));
    if (!rc) rc = A(&d.eqlist, sizeof(uint32_t) * 2 * cap);
    if (!rc) rc = A(&d.tab, sizeof(fq) * tab_fq);
    return rc;
}

// one half of the aggregate path's scratch: `keys` signer keys; the order and sort state are allocated once
inline size_t agg_key_bytes(size_t keys) { return keys * (2 * sizeof(fq) + 1 + 32 + 2 * sizeof(uint32_t)); }
int alloc_agg_half(DevAlloc& A, const DeviceState& d, AggScratch& a, size_t keys) {
    int rc = A(&a.keys_u, sizeof(fq) * keys);
    if (!rc) rc = A(&a.keys_v, sizeof(fq) * keys);
    if (!rc) rc = A(&a.kflags, keys);
    if (!rc) rc = A(&a.kcoef, 32 * keys);
    if (!rc) rc = A(&a.kmap, sizeof(uint32_t) * keys);
    if (!rc) rc = A(&a.kitem, sizeof(uint32_t) * keys);
    if (!rc && !a.order) rc = A(&a.order, sizeof(uint32_t) * d.agg_items);
    if (!rc && !a.sort) rc = A(&a.sort, sizeof(AggSort));
    if (!rc) a.cap_keys = keys;
    return rc;
}
void free_agg_keys(DeviceState& d, AggScratch& a) {
    const size_t k = a.cap_keys;
    dev_free(d, a.keys_u, sizeof(fq) * k); dev_free(d, a.keys_v, sizeof(fq) * k); dev_free(d, a.kflags, k); dev_free(d, a.kcoef, 32 * k);
    dev_free(d, a.kmap, sizeof(uint32_t) * k); dev_free(d, a.kitem, sizeof(uint32_t) * k);
    a.cap_keys = 0;
}

// ---- memory-limited contexts (jjs_init_limited) -------------------------------------------------------------------------------
// A configuration is the width W of the G / G' tables and the capacity C, the items per pipeline pass.  From C follow the
// scratch halves (C / 2 items), the sub-chunks of an overlapped batch (C / 2), the first host slice (at most 2^17), the table
// scratch (TAB_ROWS x C elements: the equation kernels' three tables; aggregate and multisig passes are cut to the items whose
// 4 x 68-element tables fit, tab_threads), the aggregate passes (C / 8 items per half) and their key scratch (4 keys per item),
// and the staging of the host-buffer entry points (LIMITED_STAGE_PER_ITEM bytes per item of capacity: a window of C double
// items with challenges, or a signing chunk of C items).  No persistent-equation scratch (eqtab).
constexpr size_t LIMITED_MIN_ITEMS = size_t(1) << 12, LIMITED_STAGE_PER_ITEM = 320;
void configure_limited(DeviceState& d, int w, size_t cap) {
    d.fb_w = w;
    d.chunk_items = cap;
    d.sub_items = cap / 2;
    d.sub_chunk = cap / 2;
    d.first_slice = d.sub_chunk < d.first_slice ? d.sub_chunk : d.first_slice;
    d.agg_items = tab_threads(d, d.sub_items, AGG_GROUP * R32_TAB_FQ);
    d.agg_keys_initial = 4 * d.agg_items;
}
// what a limited context allocates on a device at init besides alloc_tables and the first SAFE tag table (ensure_tags)
int alloc_limited_scratch(DevAlloc& A, DeviceState& d) {
    int rc = alloc_pipeline(A, d, d.chunk_items, (size_t)TAB_ROWS * d.chunk_items);
    for (int h = 0; h < 2 && !rc; h++) rc = alloc_agg_half(A, d, d.agg[h], d.agg_keys_initial);
    if (!rc) rc = A(&d.stage, LIMITED_STAGE_PER_ITEM * d.chunk_items);
    if (!rc) d.stage_bytes = LIMITED_STAGE_PER_ITEM * d.chunk_items;
    return rc;
}
// bytes a limited context of width w and capacity cap holds on a device after init: a dry run of its allocations
size_t footprint(int w, size_t cap) {
    DeviceState d;
    d.limit = 1;   // tab_threads of a limited context
    configure_limited(d, w, cap);
    DevAlloc A{nullptr, nullptr};
    alloc_tables(A, d);
    alloc_limited_scratch(A, d);
    return A.total + sizeof(fq) * TAGS_INITIAL;
}
// The policy: the largest capacity in [2^12, 2^20] whose scratch fits in `limit` beside the 12-bit tables, then the device's
// default width instead if its tables fit as well.  The fastest configuration inside the limit: the capacity decides whether one
// pass fills the GPU, the width costs about 2 % (DESIGN.md section 11).  False if not even the smallest one fits.
bool pick_config(size_t limit, int* w, size_t* cap) {
    for (size_t c = CHUNK_ITEMS; c >= LIMITED_MIN_ITEMS; c /= 2) {
        if (footprint(FB_W_SMALL, c) > limit) continue;
        *cap = c;
        *w = footprint(FB_W, c) <= limit ? FB_W : FB_W_SMALL;
        return true;
    }
    return false;
}

int ensure_scratch(jjs_ctx* ctx, DeviceState& d) {
    if (d.pts_u) return JJS_SUCCESS;
    JJS_CUDA(ctx, cudaSetDevice(d.device));
    DevAlloc A = dev_alloc(ctx, d);
    int rc = alloc_pipeline(A, d, CHUNK_ITEMS, (size_t)AGG_GROUP * R32_TAB_FQ * TAB_THREADS);   // the key-aggregation kernel's four tables per thread
    if (rc) return rc;
    {
        cudaDeviceProp prop;
        JJS_CUDA(ctx, cudaGetDeviceProperties(&prop, d.device));
        int per_sm = 0;
#if JJS_EQ_V2
        const size_t smem = sizeof(uint4) * 2 * EQ2_SLOTS * JJS_EQ_BLOCK;
        JJS_CUDA(ctx, cudaFuncSetAttribute(k_equation2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        JJS_CUDA(ctx, cudaFuncSetAttribute(k_equation2, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        JJS_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_equation2, JJS_EQ_BLOCK, smem));
        const size_t per_thread = 2 * EQ2_TAB_FQ, block = JJS_EQ_BLOCK;
#else
        JJS_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_equation<1>, BLOCK, 0));
        const size_t per_thread = 3 * 36, block = BLOCK;   // the var-gen equation builds three tables
#endif
        if (per_sm < 1) return fail(ctx, JJS_ERR_CUDA, "the equation kernel does not fit on an SM of device %d", d.device);
        d.eq_grid = per_sm * prop.multiProcessorCount;
        d.eqtab_half = per_thread * (size_t)d.eq_grid * block;
        rc = A(&d.eqtab, sizeof(fq) * 2 * d.eqtab_half);
        if (rc) return rc;
    }
    return JJS_SUCCESS;
}

// grow-only staging buffer of the host-buffer entry points; growing waits for the device (nothing of this context is in
// flight at that point: the host entry points are synchronous)
int ensure_stage(jjs_ctx* ctx, DeviceState& d, size_t bytes) {
    if (bytes <= d.stage_bytes) return JJS_SUCCESS;
    int rc = check_growth(ctx, d, d.stage_bytes, bytes, "staging buffer");
    if (rc) return rc;
    JJS_CUDA(ctx, cudaSetDevice(d.device));
    JJS_CUDA(ctx, cudaDeviceSynchronize());
    dev_free(d, d.stage, d.stage_bytes);
    d.stage_bytes = 0;
    DevAlloc A = dev_alloc(ctx, d);
    rc = A(&d.stage, bytes);
    if (rc) return rc;
    d.stage_bytes = bytes;
    return JJS_SUCCESS;
}

// SAFE tags up to `n_absorb` absorbed elements on device d (multisig transcripts).  The table is sized at jjs_init for
// 1 024 elements (511 signers per aggregate key, 255 participants per session); a larger transcript grows it, which
// waits for the device once.
int ensure_tags(jjs_ctx* ctx, DeviceState& d, size_t n_absorb) {
    if (n_absorb < d.n_tags) return JJS_SUCCESS;
    size_t want = d.n_tags ? d.n_tags : TAGS_INITIAL;
    while (want <= n_absorb) want *= 2;
    int rc = check_growth(ctx, d, sizeof(fq) * d.n_tags, sizeof(fq) * want, "SAFE tag table");
    if (rc) return rc;
    {
        std::lock_guard<std::mutex> lock(ctx->mu);
        while (ctx->tags.size() < want) {
            fq t;
            safe_tag_mont(t.l, (uint32_t)ctx->tags.size());
            ctx->tags.push_back(t);
        }
    }
    JJS_CUDA(ctx, cudaSetDevice(d.device));
    JJS_CUDA(ctx, cudaDeviceSynchronize());
    dev_free(d, d.safe_tags, sizeof(fq) * d.n_tags);
    d.n_tags = 0;
    DevAlloc A = dev_alloc(ctx, d);
    rc = A(&d.safe_tags, sizeof(fq) * want);
    if (rc) return rc;
    JJS_CUDA(ctx, cudaMemcpy(d.safe_tags, ctx->tags.data(), sizeof(fq) * want, cudaMemcpyHostToDevice));
    d.n_tags = want;
    return JJS_SUCCESS;
}

// key scratch of the aggregate path, both halves; growing waits for the device
int ensure_agg_scratch(jjs_ctx* ctx, DeviceState& d, size_t keys) {
    if (keys <= d.agg[0].cap_keys) return JJS_SUCCESS;
    size_t want = d.agg[0].cap_keys ? d.agg[0].cap_keys : d.agg_keys_initial;
    while (want < keys) want *= 2;
    int rc = check_growth(ctx, d, 2 * agg_key_bytes(d.agg[0].cap_keys), 2 * agg_key_bytes(want), "aggregate key scratch");
    if (rc) return rc;
    JJS_CUDA(ctx, cudaSetDevice(d.device));
    JJS_CUDA(ctx, cudaDeviceSynchronize());
    for (int h = 0; h < 2; h++) free_agg_keys(d, d.agg[h]);
    DevAlloc A = dev_alloc(ctx, d);
    for (int h = 0; h < 2; h++) {
        rc = alloc_agg_half(A, d, d.agg[h], want);
        if (rc) {
            for (int k = 0; k <= h; k++) free_agg_keys(d, d.agg[k]);
            return rc;
        }
    }
    return JJS_SUCCESS;
}

void variant_fields(int variant, const uint8_t* pk, const uint8_t* sig, const uint8_t* msg, Fields& pts, WireField& fmsg, WireField& fu) {
    fmsg = WireField{msg, 32};
    if (variant == VAR_SINGLE) {
        pts.f[0] = WireField{pk, 32};
        pts.f[1] = WireField{sig + 32, 64};
        pts.f[2] = pts.f[3] = WireField{nullptr, 0};
        fu = WireField{sig, 64};
    } else if (variant == VAR_DOUBLE) {
        pts.f[0] = WireField{pk, 64};
        pts.f[1] = WireField{pk + 32, 64};
        pts.f[2] = WireField{sig + 32, 96};
        pts.f[3] = WireField{sig + 64, 96};
        fu = WireField{sig, 96};
    } else {
        pts.f[0] = WireField{pk, 64};
        pts.f[1] = WireField{pk + 32, 64};
        pts.f[2] = WireField{sig + 32, 64};
        pts.f[3] = WireField{nullptr, 0};
        fu = WireField{sig, 64};
    }
}
inline size_t pk_size(int variant) { return variant == VAR_SINGLE ? 32 : 64; }
inline size_t sig_size(int variant) { return variant == VAR_DOUBLE ? 96 : 64; }

// keys (and the var-gen generator) get their subgroup test in k_decode; signature points get it from the equation
inline uint32_t key_slot_mask(int variant) { return variant == VAR_SINGLE ? 1u : 3u; }

// Hash stage for a chunk of m <= R.cap items: the work list, then the sponge of the items on it.
int enqueue_challenges(jjs_ctx* ctx, DeviceState& d, const Region& R, int variant, size_t m, const WireField& fmsg, const WireField& fu,
                       cudaStream_t stream, bool require_valid_keys) {
    StageTimer t1(ctx, d.device, 1, stream);
    JJS_CUDA(ctx, cudaMemsetAsync(R.rcount + 2, 0, sizeof(uint32_t), stream));
    k_work_list<<<blocks_for(m), BLOCK, 0, stream>>>(variant, R.pflags, m, fmsg, fu, require_valid_keys, R.iflags, R.eqflags, R.cwords, R.eqlist,
                                                    R.rcount + 2);
    k_challenge<<<blocks_for(m), BLOCK, 0, stream>>>(variant, R.pts_u, R.pts_v, m, fmsg, R.eqlist, R.rcount + 2, R.cwords);
    t1.stop(stream);
    ctx->launches += 2;
    return JJS_SUCCESS;
}

// Equation stage for a chunk of m <= R.cap items (after enqueue_challenges, whose work list it shares): the
// equations, then the deferred subgroup tests they asked for.
int enqueue_equations(jjs_ctx* ctx, DeviceState& d, const Region& R, int variant, size_t m, const WireField& fu, cudaStream_t stream) {
    const int neq = variant == VAR_DOUBLE ? 2 : 1;
    Tables T = d.tables();
    StageTimer t3(ctx, d.device, 3, stream);
    JJS_CUDA(ctx, cudaMemsetAsync(R.rcount, 0, sizeof(uint32_t), stream));
#if JJS_EQ_V2
    {
        const size_t smem = sizeof(uint4) * 2 * EQ2_SLOTS * JJS_EQ_BLOCK;
        const size_t want = (neq * m + JJS_EQ_BLOCK - 1) / JJS_EQ_BLOCK;
        const unsigned grid = (unsigned)(want < (size_t)d.eq_grid ? want : (size_t)d.eq_grid);
        k_equation2<<<grid, JJS_EQ_BLOCK, smem, stream>>>(variant, R.pts_u, R.pts_v, R.pflags, m, R.eqlist, R.rcount + 2, fu, R.cwords, R.eqflags,
                                                         R.eqtab, T, R.rlist, R.rcount);
        ctx->launches++;
    }
#elif JJS_EQ_PERSISTENT
    {
        const size_t want = blocks_for(neq * m);
        const unsigned grid = (unsigned)(want < (size_t)d.eq_grid ? want : (size_t)d.eq_grid);
        (variant == VAR_VARGEN ? k_equation<1> : k_equation<0>)<<<grid, BLOCK, 0, stream>>>(variant, R.pts_u, R.pts_v, R.pflags, m, 0, neq * m, R.eqlist, R.rcount + 2, fu,
                                                                                            R.cwords, R.eqflags, R.eqtab, (size_t)d.eq_grid * BLOCK, T, R.rlist, R.rcount);
        ctx->launches++;
    }
#else
    const auto keq = variant == VAR_VARGEN ? k_equation<1> : (d.fb_w == FB_W_SMALL ? k_equation<0, FB_W_SMALL> : k_equation<0>);
    for (size_t first = 0; first < neq * m; first += R.cap) {
        size_t cnt = neq * m - first < R.cap ? neq * m - first : R.cap;
        keq<<<blocks_for(cnt), BLOCK, 0, stream>>>(variant, R.pts_u, R.pts_v, R.pflags, m, first, cnt, R.eqlist, R.rcount + 2, fu, R.cwords, R.eqflags, R.tab,
                                                   R.tstride, T, R.rlist, R.rcount);
        ctx->launches++;
    }
#endif
    t3.stop(stream);
    StageTimer t5(ctx, d.device, 5, stream);
    k_rtest<<<blocks_for(neq * m), BLOCK, 0, stream>>>(R.pts_u, R.pts_v, R.pflags, R.rlist, R.rcount);
    ctx->launches++;
    t5.stop(stream);
    return JJS_SUCCESS;
}

// The tail of a chunk of m items: enqueue_equations, then the statuses (and challenges, c_out may be null).
int finish_chunk(jjs_ctx* ctx, DeviceState& d, const Region& R, int variant, size_t m, const WireField& fu, uint8_t* status, uint8_t* c_out,
                 cudaStream_t stream) {
    int rc = enqueue_equations(ctx, d, R, variant, m, fu, stream);
    if (rc) return rc;
    StageTimer t4(ctx, d.device, 4, stream);
    k_finalize<<<blocks_for(m), BLOCK, 0, stream>>>(variant, R.pflags, R.iflags, R.eqflags, R.cwords, m, status, c_out);
    t4.stop(stream);
    ctx->launches++;
    return JJS_SUCCESS;
}

// The whole pipeline for one chunk of m <= R.cap items (device pointers) on `stream`.
int run_chunk(jjs_ctx* ctx, DeviceState& d, const Region& R, int variant, const uint8_t* pk, const uint8_t* sig, const uint8_t* msg, size_t m,
              uint8_t* status, uint8_t* c_out, cudaStream_t stream, bool challenge_only) {
    const int slots = variant_slots(variant);
    Tables T = d.tables();
    Fields pts;
    WireField fmsg, fu;
    variant_fields(variant, pk, sig, msg, pts, fmsg, fu);
    StageTimer t0(ctx, d.device, 0, stream);
    k_decode<<<blocks_for(slots * m), BLOCK, 0, stream>>>(pts, slots, 0, m, R.pts_u, R.pts_v, R.pflags, T, key_slot_mask(variant));
    t0.stop(stream);
    ctx->launches++;
    int rc = enqueue_challenges(ctx, d, R, variant, m, fmsg, fu, stream, !challenge_only);
    if (rc) return rc;
    if (challenge_only) {
        JJS_CUDA(ctx, cudaMemcpyAsync(c_out, R.cwords, 32 * m, cudaMemcpyDeviceToDevice, stream));
        return JJS_SUCCESS;
    }
    return finish_chunk(ctx, d, R, variant, m, fu, status, c_out, stream);
}

// Typed inputs: the same pipeline behind k_decode_ext (points as JubJubExtended coordinates, 160 bytes each, item-major).
int run_chunk_ext(jjs_ctx* ctx, DeviceState& d, const Region& R, int variant, const uint8_t* pts, const uint8_t* u32, const uint8_t* msg, size_t m,
                  uint8_t* status, uint8_t* c_out, cudaStream_t stream) {
    const int slots = variant_slots(variant);
    WireField fmsg{msg, 32}, fu{u32, 32};
    StageTimer t0(ctx, d.device, 0, stream);
    k_decode_ext<<<blocks_for(slots * m), BLOCK, 0, stream>>>(pts, slots, m, R.pts_u, R.pts_v, R.pflags, key_slot_mask(variant));
    t0.stop(stream);
    ctx->launches++;
    int rc = enqueue_challenges(ctx, d, R, variant, m, fmsg, fu, stream, true);
    return rc ? rc : finish_chunk(ctx, d, R, variant, m, fu, status, c_out, stream);
}

// The front of an aggregate-key chunk of m items with K <= cap_keys signer keys, on `stream`: signer keys and R decoded, the
// ordering by signer count, the coefficients, the aggregate keys into slot 0 (the aggregation kernel's tables at `tab`,
// serving `stride` >= m threads), then the work list and challenges.  R's subgroup test runs at decode when `r_test`, else it
// is left to the equation.  d_keys: the chunk's first key; d_offsets: the chunk's m + 1 offsets (absolute, first = key_lo).
int enqueue_aggregate_front(jjs_ctx* ctx, DeviceState& d, const Region& R, const uint8_t* d_keys, const uint32_t* d_offsets, uint32_t key_lo, size_t K,
                            const uint8_t* d_sig, const uint8_t* d_msg, size_t m, uint8_t* d_agg, fq* tab, size_t stride, bool r_test,
                            cudaStream_t stream) {
    AggScratch& A = d.agg[R.half];
    Tables T = d.tables();
    Fields fk, fr;
    fk.f[0] = WireField{d_keys, 32};
    fr.f[0] = WireField{d_sig + 32, 64};
    fk.f[1] = fk.f[2] = fk.f[3] = fr.f[1] = fr.f[2] = fr.f[3] = WireField{nullptr, 0};
    WireField fmsg{d_msg, 32}, fu{d_sig, 64};
    StageTimer t0(ctx, d.device, 0, stream);
    if (K) k_decode<<<blocks_for(K), BLOCK, 0, stream>>>(fk, 1, 0, K, A.keys_u, A.keys_v, A.kflags, T, 0u);
    k_decode<<<blocks_for(m), BLOCK, 0, stream>>>(fr, 1, 1, m, R.pts_u, R.pts_v, R.pflags, T, r_test ? 1u : 0u);
    t0.stop(stream);
    StageTimer t2(ctx, d.device, 2, stream);
    JJS_CUDA(ctx, cudaMemsetAsync(A.sort, 0, sizeof(AggSort), stream));
    k_agg_hist<<<blocks_for(m), BLOCK, 0, stream>>>(d_offsets, m, A.sort);
    k_agg_scan<<<1, 32, 0, stream>>>(A.sort);
    k_agg_scatter<<<blocks_for(m), BLOCK, 0, stream>>>(d_offsets, key_lo, m, A.sort, A.order, A.kmap, A.kitem);
    if (K) k_agg_coeffs<<<blocks_for(K), BLOCK, 0, stream>>>(A.keys_u, A.keys_v, A.kflags, d_offsets, A.kmap, A.kitem, key_lo, K, A.kcoef, T);
    k_aggregate<<<blocks_for(m), BLOCK, 0, stream>>>(A.keys_u, A.keys_v, A.kflags, d_offsets, A.order, key_lo, m, R.pts_u, R.pts_v, R.pflags, d_agg, tab,
                                                    stride, A.kcoef, T);
    t2.stop(stream);
    ctx->launches += 7;
    return enqueue_challenges(ctx, d, R, VAR_SINGLE, m, fmsg, fu, stream, true);
}

// aggregate_pk(..).verify(..) for one chunk of m <= R.acap items with K <= cap_keys signer keys; everything on `stream`,
// nothing on the host.  Arguments as enqueue_aggregate_front.
int run_chunk_aggregate(jjs_ctx* ctx, DeviceState& d, const Region& R, const uint8_t* d_keys, const uint32_t* d_offsets, uint32_t key_lo, size_t K,
                        const uint8_t* d_sig, const uint8_t* d_msg, size_t m, uint8_t* d_status, uint8_t* d_c, uint8_t* d_agg, cudaStream_t stream) {
    WireField fu{d_sig, 64};
    int rc = enqueue_aggregate_front(ctx, d, R, d_keys, d_offsets, key_lo, K, d_sig, d_msg, m, d_agg, R.tab, R.astride, false, stream);
    return rc ? rc : finish_chunk(ctx, d, R, VAR_SINGLE, m, fu, d_status, d_c, stream);
}

// The pipeline for one chunk of m <= R.cap items under a registered key set (device pointers, key_index: the chunk's first
// index).  The key slots are gathered from the key set instead of decoded; only the signature points go through k_decode,
// with their subgroup test deferred.  Hash, deferred tests and status are the kernels of run_chunk; so is the equation under a
// points-only set, which has no tables.
int run_chunk_keyed(jjs_ctx* ctx, DeviceState& d, const Region& R, const KeySet& ks, const KeySetDev& kd, const uint32_t* key_index, const uint8_t* sig,
                    const uint8_t* msg, size_t m, uint8_t* status, uint8_t* c_out, cudaStream_t stream) {
    const int variant = ks.variant, nk = keyed_points(variant);
    const uint32_t sgs = (uint32_t)sig_size(variant);
    Tables T = d.tables();
    Fields fr;
    fr.f[0] = WireField{sig + 32, sgs};
    fr.f[1] = variant == VAR_DOUBLE ? WireField{sig + 64, sgs} : WireField{nullptr, 0};
    fr.f[2] = fr.f[3] = WireField{nullptr, 0};
    WireField fmsg{msg, 32}, fu{sig, sgs};
    StageTimer t0(ctx, d.device, 0, stream);
    k_keyed_gather<<<blocks_for(m), BLOCK, 0, stream>>>(variant, kd.u, kd.v, kd.flags, ks.n_keys, key_index, m, R.pts_u, R.pts_v, R.pflags);
    k_decode<<<blocks_for(nk * m), BLOCK, 0, stream>>>(fr, nk, nk, m, R.pts_u, R.pts_v, R.pflags, T, 0u);
    t0.stop(stream);
    ctx->launches += 2;
    int rc = enqueue_challenges(ctx, d, R, variant, m, fmsg, fu, stream, true);
    if (rc) return rc;
    if (ks.key_bits == 0) return finish_chunk(ctx, d, R, variant, m, fu, status, c_out, stream);   // points only
    StageTimer t3(ctx, d.device, 3, stream);
    JJS_CUDA(ctx, cudaMemsetAsync(R.rcount, 0, sizeof(uint32_t), stream));
    const auto keq = with_key_width(ks.key_bits, [&](auto kw) {
        return d.fb_w == FB_W_SMALL ? k_equation_keyed<FB_W_SMALL, kw.value> : k_equation_keyed<FB_W, kw.value>;
    });
    keq<<<blocks_for(nk * m), BLOCK, 0, stream>>>(variant, R.pts_u, R.pts_v, R.pflags, m, R.eqlist, R.rcount + 2, fu, R.cwords, R.eqflags, kd.table,
                                                  key_index, ks.n_keys, T, R.rlist, R.rcount);
    t3.stop(stream);
    StageTimer t5(ctx, d.device, 5, stream);
    k_rtest<<<blocks_for(nk * m), BLOCK, 0, stream>>>(R.pts_u, R.pts_v, R.pflags, R.rlist, R.rcount);
    t5.stop(stream);
    StageTimer t4(ctx, d.device, 4, stream);
    k_finalize<<<blocks_for(m), BLOCK, 0, stream>>>(variant, R.pflags, R.iflags, R.eqflags, R.cwords, m, status, c_out);
    t4.stop(stream);
    ctx->launches += 3;
    return JJS_SUCCESS;
}

// ---- whole-batch verification: one pass of the combination ----------------------------------------------------------------
// No per-item equation runs on this path, so its scratch is the region's equation-table scratch: TAB_ROWS field elements
// (3 456 bytes) per item of capacity, contiguous from rlc_base.  On a limited context that is R.tab itself; a jjs_init
// context's table scratch is laid out by row for the equation kernels (column = thread), so each half takes a contiguous
// half of the whole allocation instead (4 352 bytes per item of a half).  The half's accumulator takes the last RLC_ACC_BYTES
// of those 3 456 per item: the pass buffers (rlc_plan) and the aggregation tables of an aggregate pass (rlc_agg_items) stay
// below it, so no pass of the call overwrites what earlier passes on the half accumulated, and the two halves stay disjoint.
constexpr size_t RLC_ROW_BYTES = sizeof(fq) * TAB_ROWS, RLC_ACC_BYTES = 256;
static_assert(sizeof(RlcAcc) <= RLC_ACC_BYTES, "the accumulator must fit its slot");
inline uint8_t* rlc_base(const DeviceState& d, const Region& R) {
    if (d.limit) return reinterpret_cast<uint8_t*>(R.tab);
    return reinterpret_cast<uint8_t*>(d.tab) + (size_t)R.half * (sizeof(fq) * AGG_GROUP * R32_TAB_FQ * TAB_THREADS / 2);
}
inline size_t rlc_pass_bytes(const Region& R) { return RLC_ROW_BYTES * R.cap - RLC_ACC_BYTES; }
inline RlcAcc* rlc_acc(const DeviceState& d, const Region& R) { return reinterpret_cast<RlcAcc*>(rlc_base(d, R) + rlc_pass_bytes(R)); }
// Items of an aggregate pass: as many as the aggregation kernel's per-thread tables (stride = this count) fit below the
// accumulator, and the order array serves.
constexpr size_t AGG_TAB_BYTES = sizeof(fq) * AGG_GROUP * R32_TAB_FQ;
inline size_t rlc_agg_items(const DeviceState& d, const Region& R) {
    size_t t = rlc_pass_bytes(R) / AGG_TAB_BYTES;
    if (t > R.cap) t = R.cap;
    return t < d.agg_items ? t : d.agg_items;
}

// Where the buffers of a pass of m items in G groups with window width c go, in bytes from rlc_base; `total` is what it needs.
// A grouped pass (jjs_verify_grouped) also keeps each group's scalar sums and verdict; a whole-batch pass (G = 1) keeps its sums
// in the half's accumulator and has neither.
struct RlcPlan {
    RlcShape s;
    size_t entries, n1, n2, cub_bytes;
    size_t o_zu, o_keys[2], o_vals[2], o_cub, o_buckets, o_ck[2], o_cp[2], o_partial, o_W, o_su, o_verdict, total;
};
inline int rlc_plan(RlcPlan& p, int variant, size_t m, int c, size_t groups, bool grouped) {
    p.s = rlc_shape(variant, c, groups);
    p.entries = m * (size_t)p.s.per_item;
    p.n1 = 2 * rlc_segments(p.entries, RLC_SEG);
    p.n2 = 2 * rlc_segments(p.n1, RLC_SEG);
    cub::DoubleBuffer<uint32_t> kb(nullptr, nullptr), vb(nullptr, nullptr);
    p.cub_bytes = 0;
    if (cub::DeviceRadixSort::SortPairs(nullptr, p.cub_bytes, kb, vb, (int)p.entries, 0, p.s.end_bit) != cudaSuccess) return JJS_ERR_CUDA;
    const size_t neq = variant == VAR_DOUBLE ? 2 : 1, nb = p.s.sentinel, slices = nb / RLC_SLICE;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o += align_up(bytes, 256); return at; };
    p.o_zu = take(32 * neq * m);
    for (int k = 0; k < 2; k++) { p.o_keys[k] = take(4 * p.entries); p.o_vals[k] = take(4 * p.entries); }
    p.o_cub = take(p.cub_bytes);
    p.o_buckets = take(sizeof(ext) * nb);
    p.o_ck[0] = take(4 * p.n1); p.o_cp[0] = take(sizeof(ext) * p.n1);
    p.o_ck[1] = take(4 * p.n2); p.o_cp[1] = take(sizeof(ext) * p.n2);
    p.o_partial = take(sizeof(ext) * slices);
    p.o_W = take(sizeof(ext) * groups * p.s.nw_big);
    p.o_su = grouped ? take(sizeof(uint32_t) * 16 * groups) : 0;
    p.o_verdict = grouped ? take(groups) : 0;
    p.total = o;
    return JJS_SUCCESS;
}
// The window width of a pass: the cheapest c whose buffers fit the region's scratch, by a count of point additions (one per
// sort entry, about 2.3 mixed-addition equivalents per bucket of every group for the running sums).  It follows from the point
// and group counts alone.
inline int rlc_choose(jjs_ctx* ctx, RlcPlan& best, int variant, size_t m, size_t groups, bool grouped, size_t budget) {
    double best_cost = 0;
    bool found = false;
    for (int c = RLC_C_MIN; c <= RLC_C_MAX; c++) {
        RlcPlan p;
        if (rlc_plan(p, variant, m, c, groups, grouped)) return fail(ctx, JJS_ERR_CUDA, "radix sort: temporary storage query failed");
        if (p.total > budget) continue;
        const double cost = (double)p.entries + 2.3 * (double)p.s.sentinel;
        if (!found || cost < best_cost) { best = p; best_cost = cost; found = true; }
    }
    if (!found) return fail(ctx, JJS_ERR_NOMEM, "whole-batch verification: %zu items do not fit the pass scratch of %zu bytes", m, budget);
    return JJS_SUCCESS;
}

// log2 of the items per group of a grouped pass (jjs_verify_grouped; DESIGN.md section 14 has the sweep that chose it).  0: one
// group per pass.  A build-time define for A/B measurements only; the header promises groups of at most 2^16 items.
#ifndef JJS_GROUP_LOG2
#define JJS_GROUP_LOG2 12
#endif
static_assert(JJS_GROUP_LOG2 >= 0 && JJS_GROUP_LOG2 <= 16, "groups hold at most 2^16 items");
constexpr int RLC_ONE_GROUP = 31;   // the group shift of a pass that is one group (passes hold fewer than 2^31 items)

// The per-item outputs of a grouped pass (device pointers at the pass's first item; c and agg may be null) and the call's
// count of items verified one by one (may be null).
struct GroupedOut {
    uint8_t *status, *c, *agg;
    unsigned long long* fallback;
};

// One pass of m <= R.cap items of kind `kind` (JJS_KIND_*, device pointers), with every point subgroup-tested before it enters:
// single, double and var-generator items decode every slot with its test, then work list and challenges; aggregate items
// (m <= rlc_agg_items; pk = the pass's first signer key, offsets, key_lo and K as run_chunk_aggregate) run the front of the
// aggregate path with R's test on, its aggregation tables in the pass scratch.  `base`: position of the pass's first item in
// the whole call.
// Whole-batch (out == nullptr): the combination of the pass is added into the half's accumulator.  Grouped: every group of
// 2^JJS_GROUP_LOG2 consecutive items gets its own combination and verdict, the items of failing groups run the per-item equations
// (their tables in the half's own pass scratch), and the pass's statuses are written to `out`.
int run_chunk_rlc(jjs_ctx* ctx, DeviceState& d, const Region& R, int kind, const uint8_t* pk, const uint32_t* offsets, uint32_t key_lo, size_t K,
                  const uint8_t* sig, const uint8_t* msg, size_t m, uint64_t base, const RlcSeed& seed, cudaStream_t stream,
                  const GroupedOut* out = nullptr) {
    const bool agg = kind == JJS_KIND_AGGREGATE;
    const int variant = agg ? VAR_SINGLE : kind, neq = variant == VAR_DOUBLE ? 2 : 1;
    const int gshift = out && JJS_GROUP_LOG2 ? JJS_GROUP_LOG2 : RLC_ONE_GROUP;
    const size_t g = size_t(1) << gshift, groups = (m + g - 1) >> gshift;
    RlcPlan p;
    int rc = rlc_choose(ctx, p, variant, m, groups, out != nullptr, rlc_pass_bytes(R));
    if (rc) return rc;
    uint8_t* B = rlc_base(d, R);
    WireField fu;
    if (agg) {
        fu = WireField{sig, 64};
        rc = enqueue_aggregate_front(ctx, d, R, pk, offsets, key_lo, K, sig, msg, m, out ? out->agg : nullptr, reinterpret_cast<fq*>(B), rlc_agg_items(d, R),
                                     true, stream);
    } else {
        const int slots = variant_slots(variant);
        Fields pts;
        WireField fmsg;
        variant_fields(variant, pk, sig, msg, pts, fmsg, fu);
        StageTimer t0(ctx, d.device, 0, stream);
        k_decode<<<blocks_for(slots * m), BLOCK, 0, stream>>>(pts, slots, 0, m, R.pts_u, R.pts_v, R.pflags, d.tables(), (1u << slots) - 1u);
        t0.stop(stream);
        ctx->launches++;
        rc = enqueue_challenges(ctx, d, R, variant, m, fmsg, fu, stream, true);
    }
    if (rc) return rc;
    RlcAcc* acc = out ? nullptr : rlc_acc(d, R);
    uint32_t* zu = reinterpret_cast<uint32_t*>(B + p.o_zu);
    StageTimer t3(ctx, d.device, 3, stream);
    k_rlc_digits<<<blocks_for(m), BLOCK, 0, stream>>>(variant, R.pflags, R.iflags, R.cwords, fu, m, gshift, p.s, seed, base,
                                                       reinterpret_cast<uint32_t*>(B + p.o_keys[0]), reinterpret_cast<uint32_t*>(B + p.o_vals[0]), zu, acc);
    cub::DoubleBuffer<uint32_t> kb(reinterpret_cast<uint32_t*>(B + p.o_keys[0]), reinterpret_cast<uint32_t*>(B + p.o_keys[1]));
    cub::DoubleBuffer<uint32_t> vb(reinterpret_cast<uint32_t*>(B + p.o_vals[0]), reinterpret_cast<uint32_t*>(B + p.o_vals[1]));
    size_t cub_bytes = p.cub_bytes;
    JJS_CUDA(ctx, cub::DeviceRadixSort::SortPairs(B + p.o_cub, cub_bytes, kb, vb, (int)p.entries, 0, p.s.end_bit, stream));
    ext* buckets = reinterpret_cast<ext*>(B + p.o_buckets);
    k_rlc_bucket_init<<<blocks_for(p.s.sentinel), BLOCK, 0, stream>>>(buckets, p.s.sentinel);
    // level 0 on the sorted pairs, then the merge levels on the carries until one segment is left
    size_t len = p.entries;
    size_t segs = rlc_segments(len, RLC_SEG);
    k_rlc_segments0<<<blocks_for(segs), BLOCK, 0, stream>>>(kb.Current(), vb.Current(), R.pts_u, R.pts_v, len, p.s.sentinel, buckets,
                                                            reinterpret_cast<uint32_t*>(B + p.o_ck[0]), reinterpret_cast<ext*>(B + p.o_cp[0]), segs == 1);
    ctx->launches += 4;
    for (int lv = 0; segs > 1; lv ^= 1) {
        len = 2 * segs;
        segs = rlc_segments(len, RLC_SEG);
        k_rlc_segments<<<blocks_for(segs), BLOCK, 0, stream>>>(reinterpret_cast<const uint32_t*>(B + p.o_ck[lv]), reinterpret_cast<const ext*>(B + p.o_cp[lv]), len,
                                                               p.s.sentinel, buckets, reinterpret_cast<uint32_t*>(B + p.o_ck[lv ^ 1]),
                                                               reinterpret_cast<ext*>(B + p.o_cp[lv ^ 1]), segs == 1);
        ctx->launches++;
    }
    const uint32_t slices = p.s.buckets_per_window / RLC_SLICE;
    const int nwin = (int)(groups * p.s.nw_big);   // every group's windows
    ext* partial = reinterpret_cast<ext*>(B + p.o_partial);
    ext* W = reinterpret_cast<ext*>(B + p.o_W);
    k_rlc_slices<<<blocks_for((size_t)nwin * slices), BLOCK, 0, stream>>>(buckets, nwin, p.s.buckets_per_window, partial);
    k_rlc_window_sums<<<nwin, 32, 0, stream>>>(partial, slices, W);
    ctx->launches += 2;
    if (!out) {
        k_rlc_horner<<<1, 1, 0, stream>>>(W, p.s.nw_big, p.s.c, acc);
        k_rlc_scalars<<<1, RLC_SUM_THREADS, 0, stream>>>(zu, m, g, neq, &acc->su);
        t3.stop(stream);
        ctx->launches += 2;
        return JJS_SUCCESS;
    }
    // grouped: the verdicts are consumed into the equation bits and the work list before any equation runs, so the fallback
    // equations may take the whole pass scratch for their tables.  Not R.tab with R.tstride: on a jjs_init context those rows
    // span both halves' pass scratch, and the other half's pass may be running.
    auto* su = reinterpret_cast<uint32_t(*)[2][8]>(B + p.o_su);
    uint8_t* verdict = B + p.o_verdict;
    JJS_CUDA(ctx, cudaMemsetAsync(su, 0, sizeof(uint32_t) * 16 * groups, stream));
    k_rlc_scalars<<<(unsigned)groups, RLC_SUM_THREADS, 0, stream>>>(zu, m, g, neq, su);
    (d.fb_w == FB_W_SMALL ? k_rlc_verdicts<FB_W_SMALL> : k_rlc_verdicts<FB_W>)<<<blocks_for(groups), BLOCK, 0, stream>>>(W, p.s.nw_big, p.s.c, groups, su,
                                                                                                                      d.tables(), verdict);
    JJS_CUDA(ctx, cudaMemsetAsync(R.rcount + 2, 0, sizeof(uint32_t), stream));
    k_rlc_gate<<<blocks_for(m), BLOCK, 0, stream>>>(variant, R.pflags, R.iflags, m, gshift, verdict, R.eqflags, R.eqlist, R.rcount + 2, out->fallback);
    t3.stop(stream);
    ctx->launches += 3;
    Region F = R;
    F.tab = reinterpret_cast<fq*>(B);
    F.tstride = R.cap;
    return finish_chunk(ctx, d, F, variant, m, fu, out->status, out->c, stream);
}

// Sub-chunks of an overlapped batch alternate between the two internal streams and scratch halves: kernels of neighbouring
// sub-chunks overlap, which hides the partially filled last wave of every launch (per-thread work is uniform, so a launch
// ends with SMs idling for up to one block duration).  With per-stage profiling on, everything stays on `stream` so that
// the stage timers do not overlap.
struct Overlap {
    jjs_ctx* ctx;
    DeviceState& d;
    cudaStream_t stream;
    bool on;
    size_t i = 0;
    Overlap(jjs_ctx* c, DeviceState& dev, cudaStream_t s, bool enable) : ctx(c), d(dev), stream(s), on(enable && !c->profile) {}
    int begin() {
        if (!on) return JJS_SUCCESS;
        JJS_CUDA(ctx, cudaEventRecord(d.fork, stream));
        for (int k = 0; k < 2; k++) JJS_CUDA(ctx, cudaStreamWaitEvent(d.sub[k], d.fork, 0));
        return JJS_SUCCESS;
    }
    cudaStream_t next_stream() const { return on ? d.sub[i & 1] : stream; }
    void advance() { i++; }
    int end() {
        if (!on) return JJS_SUCCESS;
        for (int k = 0; k < 2; k++) {
            JJS_CUDA(ctx, cudaEventRecord(d.join[k], d.sub[k]));
            JJS_CUDA(ctx, cudaStreamWaitEvent(stream, d.join[k], 0));
        }
        return JJS_SUCCESS;
    }
};

// Chunks of an aggregate-key batch: at most `max_items` items and `max_keys` signer keys each (an item with more keys than
// that forms a chunk of its own, for which the caller grows the key scratch first).
inline size_t agg_chunk_end(const uint32_t* offsets, size_t first, size_t n, size_t max_items, size_t max_keys) {
    size_t end = first;
    while (end < n && end - first < max_items && (size_t)(offsets[end + 1] - offsets[first]) <= max_keys) end++;
    return end == first ? first + 1 : end;
}
inline size_t agg_max_item_keys(const uint32_t* offsets, size_t n) {
    size_t mx = 0;
    for (size_t i = 0; i < n; i++) {
        size_t c = offsets[i + 1] - offsets[i];
        if (c > mx) mx = c;
    }
    return mx;
}

// ---- parts and passes -----------------------------------------------------------------------------------------------------
// A call verifies one or more PARTS (each a homogeneous batch: one of the three wire variants, aggregate-key items, typed items,
// items under a registered key set, or the whole-batch or grouped items of one kind).  A host-buffer call cuts every part into
// shards, one per device of the context (small parts go whole to the least loaded device), and every device is driven by its
// own host thread: copies in on the copy stream, pipeline slices alternating between the two compute streams, results copied
// out at the end, one synchronisation.  A single host thread would serialise the devices whenever the caller's memory is
// pageable (cudaMemcpyAsync from pageable memory returns only after staging).  A device-buffer call runs its parts on one device
// and the caller's stream (run_device_parts).  Both cut a part into passes with pass_end and run every pass through run_pass.
enum PartMode : int { PART_WIRE = 0, PART_AGGREGATE = 1, PART_TYPED = 2, PART_KEYED = 3, PART_ALL = 4, PART_GROUPED = 5 };
// whole-batch verification: the devices' partial points and validity flags, summed on the host as the devices finish;
// grouped verification: the items the devices verified one by one
struct RlcSink {
    std::mutex mu;
    ext P;
    bool valid = true;
    uint64_t fallback = 0;
    RlcSink() { ext_identity(P); }
    void add(const RlcOut& o) {
        std::lock_guard<std::mutex> lock(mu);
        rlc_add(P, o.P);
        valid = valid && o.valid;
    }
    void add_fallback(uint64_t items) {
        std::lock_guard<std::mutex> lock(mu);
        fallback += items;
    }
};
// One part of a call; its buffers are the host's (host-buffer calls) or the device's (device-buffer calls).
struct Part {
    int mode = PART_WIRE;
    int variant = VAR_SINGLE;                  // wire, typed and keyed parts: VAR_*; the others: the part's JJS_KIND_*
    const uint8_t *pk = nullptr, *sig = nullptr, *msg = nullptr;   // typed: pk = points_ext160, sig = u32;  keyed: pk = the uint32
                                                                   // key indices;  aggregate: pk = the signer keys
    const uint32_t* offsets = nullptr;         // aggregate only: the n + 1 offsets beside the other buffers,
    const uint32_t* h_offsets = nullptr;       // and their host copy, which plans the passes (the same array in a host-buffer call)
    size_t n = 0;
    uint8_t *status = nullptr, *c_out = nullptr, *agg_out = nullptr;
    uint32_t* bitmap = nullptr;
    bool challenge_only = false;
    const KeySet* keys = nullptr;              // keyed only
    const RlcSeed* seed = nullptr;             // whole-batch and grouped only: the weights' seed, where the devices' results go (one
    RlcSink* sink = nullptr;                   // sink per host-buffer call) and the position of the part's first item in the call
    uint64_t base = 0;
};
inline bool part_rlc(const Part& p) { return p.mode == PART_ALL || p.mode == PART_GROUPED; }
inline bool part_aggregate(const Part& p) { return p.mode == PART_AGGREGATE || (part_rlc(p) && p.variant == JJS_KIND_AGGREGATE); }
// Bytes per item of a part's pk and sig buffers; pk of an aggregate part: per signer key.
struct Strides {
    size_t pk, sig;
};
inline Strides part_strides(const Part& p) {
    if (part_aggregate(p)) return {32, 64};
    if (p.mode == PART_TYPED) return {160 * (size_t)variant_slots(p.variant), 32};
    if (p.mode == PART_KEYED) return {sizeof(uint32_t), sig_size(p.variant)};
    return {pk_size(p.variant), sig_size(p.variant)};
}
struct Shard {
    size_t lo, hi;
};

inline double part_weight(const Part& p) {   // relative cost of one item (executed multiplies, single = 1)
    if (part_aggregate(p)) {
        double avg = p.n ? (double)(p.h_offsets[p.n] - p.h_offsets[0]) / (double)p.n : 0.0;
        return 1.0 + 0.75 * avg;
    }
    return p.variant == VAR_DOUBLE ? 1.9 : (p.variant == VAR_VARGEN ? 1.4 : 1.0);
}

// shards[part][device].  Large parts are split evenly (every device then carries the same share of every kind, so the
// devices finish together whatever the mix); parts too small to be worth splitting go whole to the least loaded device.
constexpr size_t MIN_SPLIT_ITEMS = 8192;
void plan_shards(const std::vector<Part>& parts, size_t g, std::vector<std::vector<Shard>>& shards) {
    shards.assign(parts.size(), std::vector<Shard>(g, Shard{0, 0}));
    std::vector<double> load(g, 0.0);
    for (size_t p = 0; p < parts.size(); p++) {
        const size_t n = parts[p].n;
        if (n >= g * MIN_SPLIT_ITEMS) {
            const size_t per = ((n + g - 1) / g + 31) & ~size_t(31);   // shards start on a bitmap word
            for (size_t k = 0; k < g; k++) {
                size_t lo = k * per < n ? k * per : n, hi = lo + per < n ? lo + per : n;
                shards[p][k] = Shard{lo, hi};
                load[k] += part_weight(parts[p]) * (double)(hi - lo);
            }
        }
    }
    for (size_t p = 0; p < parts.size(); p++) {
        const size_t n = parts[p].n;
        if (n == 0 || n >= g * MIN_SPLIT_ITEMS) continue;
        size_t best = 0;
        for (size_t k = 1; k < g; k++)
            if (load[k] < load[best]) best = k;
        shards[p][best] = Shard{0, n};
        load[best] += part_weight(parts[p]) * (double)n;
    }
}

// Checks part P of a host-buffer call, or of a device-buffer call (on_device), which also needs the host copy of an aggregate
// part's offsets and a status buffer (a host-buffer call may take a bitmap instead).  `part` >= 0: the message names the part.
int validate_part(jjs_ctx* ctx, const Part& P, bool on_device, long part = -1) {
    const bool agg = part_aggregate(P), offsets = P.offsets && (P.h_offsets || !on_device);
    const char* why = [&]() -> const char* {
        if (P.mode != PART_AGGREGATE && (P.variant < 0 || P.variant > (part_rlc(P) ? JJS_KIND_AGGREGATE : VAR_VARGEN)))
            return part_rlc(P) ? "bad kind" : "bad variant";
        if (part_rlc(P) && agg && !offsets)   // whole-batch and grouped parts are checked for these even when empty
            return on_device ? "an aggregate part needs its offsets on the device and on the host" : "an aggregate part needs its offsets";
        if (P.mode == PART_GROUPED && !P.status && !P.bitmap) return "a part needs a status or a bitmap output";
        if (P.n == 0) return nullptr;
        if (P.challenge_only) return !P.pk || !P.sig || !P.msg || !P.c_out ? "null buffer" : nullptr;
        if (!P.sig || !P.msg) return "null buffer";
        if (P.mode != PART_ALL && !P.status && (on_device || !P.bitmap)) return on_device ? "null buffer (a device call needs a status buffer)" : "null buffer";
        if (!agg) return P.pk ? nullptr : "null buffer";
        if (!offsets) return "null buffer";
        for (size_t i = 0; i < P.n; i++)
            if (P.h_offsets[i + 1] < P.h_offsets[i]) return "offsets must be non-decreasing";
        return P.h_offsets[P.n] > P.h_offsets[0] && !P.pk ? "null key buffer" : nullptr;
    }();
    if (!why) return JJS_SUCCESS;
    return part < 0 ? fail(ctx, JJS_ERR_ARGUMENT, "%s", why) : fail(ctx, JJS_ERR_ARGUMENT, "part %ld: %s", part, why);
}

// End of the pass of part P that starts at item `off` of n and takes at most `want` items.  An aggregate pass also holds no more
// items than the aggregation tables of region R serve (in the pass scratch for whole-batch and grouped parts) and no more signer
// keys than the key scratch (agg_chunk_end on h_offsets, the host offsets of the n items).
inline size_t pass_end(const DeviceState& d, const Region& R, const Part& P, const uint32_t* h_offsets, size_t off, size_t n, size_t want) {
    if (!part_aggregate(P)) return off + (n - off < want ? n - off : want);
    const size_t most = part_rlc(P) ? rlc_agg_items(d, R) : R.acap;
    return agg_chunk_end(h_offsets, off, n, want < most ? want : most, d.agg[0].cap_keys);
}

// Scratch on device d for items [ranges[p].lo, ranges[p].hi) of every part p: the pipeline scratch, then the SAFE tags and the
// aggregate key scratch for the most signer keys of one item.  Growing either waits for the device.
int prepare_parts(jjs_ctx* ctx, DeviceState& d, const std::vector<Part>& parts, const std::vector<Shard>& ranges) {
    int rc = ensure_scratch(ctx, d);
    bool agg = false;
    size_t most = 0;
    for (size_t p = 0; p < parts.size(); p++) {
        if (!part_aggregate(parts[p]) || ranges[p].hi == ranges[p].lo) continue;
        agg = true;
        const size_t mc = agg_max_item_keys(parts[p].h_offsets + ranges[p].lo, ranges[p].hi - ranges[p].lo);
        if (mc > most) most = mc;
    }
    if (!rc && agg) rc = ensure_tags(ctx, d, 2 + 2 * most);
    if (!rc && agg) rc = ensure_agg_scratch(ctx, d, most > d.agg_keys_initial ? most : d.agg_keys_initial);
    return rc;
}

// Device buffers of a part from its item `first` on: the caller's (device-buffer calls, first = 0) or the staging of device_job.
// pk of an aggregate part is at signer key `key0`; status, c and agg may be null.
struct PartPtrs {
    const uint8_t *pk, *sig, *msg;
    const uint32_t* offsets;
    uint8_t *status, *c, *agg;
    size_t first;
    uint32_t key0;
};

// One pass of items [off, off + cnt) after b.first of part P, on device k in region R on `stream`: the run_chunk* of the part's
// mode.  fallback: a grouped call's count of the items verified one by one.
int run_pass(jjs_ctx* ctx, size_t k, const Region& R, const Part& P, const PartPtrs& b, size_t off, size_t cnt, cudaStream_t stream,
             unsigned long long* fallback) {
    DeviceState& d = ctx->dev[k];
    const Strides s = part_strides(P);
    const uint8_t *sig = b.sig + s.sig * off, *msg = b.msg + 32 * off;
    uint8_t* status = b.status ? b.status + off : nullptr;
    uint8_t* c = b.c ? b.c + 32 * off : nullptr;
    uint8_t* agg = b.agg ? b.agg + 32 * off : nullptr;
    const GroupedOut go{status, c, agg, fallback};
    const GroupedOut* out = P.mode == PART_GROUPED ? &go : nullptr;
    const uint64_t base = P.base + b.first + off;
    if (part_aggregate(P)) {
        const uint32_t key_lo = P.h_offsets[b.first + off];
        const size_t K = P.h_offsets[b.first + off + cnt] - key_lo;
        const uint8_t* keys = b.pk + s.pk * (size_t)(key_lo - b.key0);
        if (P.mode == PART_AGGREGATE) return run_chunk_aggregate(ctx, d, R, keys, b.offsets + off, key_lo, K, sig, msg, cnt, status, c, agg, stream);
        return run_chunk_rlc(ctx, d, R, JJS_KIND_AGGREGATE, keys, b.offsets + off, key_lo, K, sig, msg, cnt, base, *P.seed, stream, out);
    }
    const uint8_t* pk = b.pk + s.pk * off;
    switch (P.mode) {
    case PART_WIRE: return run_chunk(ctx, d, R, P.variant, pk, sig, msg, cnt, status, c, stream, P.challenge_only);
    case PART_TYPED: return run_chunk_ext(ctx, d, R, P.variant, pk, sig, msg, cnt, status, c, stream);
    case PART_KEYED:
        return run_chunk_keyed(ctx, d, R, *P.keys, P.keys->dev[k], reinterpret_cast<const uint32_t*>(pk), sig, msg, cnt, status, c, stream);
    default: return run_chunk_rlc(ctx, d, R, P.variant, pk, nullptr, 0, 0, sig, msg, cnt, base, *P.seed, stream, out);
    }
}

// Enqueue `parts` (device pointers, checked) on device k: the work is ordered after what `stream` holds now and `stream` waits
// for it.  Per-item wire and keyed parts that do not overlap run passes of chunk_items in the whole region (twice a half's
// capacity, so a double pass launches its equations once instead of twice); every other pass takes up to sub_chunk items in the
// next scratch half.  Whole-batch parts (all_valid set) add into the halves' accumulators and the verdict is written to
// *all_valid, also when there are no items.  Grouped parts write their items' outputs, and *fallback (may be null) counts the
// items verified one by one.  Enqueue-only unless a scratch has to grow (prepare_parts).
int run_device_parts(jjs_ctx* ctx, size_t k, const std::vector<Part>& parts, cudaStream_t stream, int* all_valid, unsigned long long* fallback) {
    DeviceState& d = ctx->dev[k];
    JJS_CUDA(ctx, cudaSetDevice(d.device));
    size_t n = 0;
    std::vector<Shard> ranges;
    for (const Part& P : parts) {
        ranges.push_back(Shard{0, P.n});
        n += P.n;
    }
    int rc = prepare_parts(ctx, d, parts, ranges);
    if (rc) return rc;
    if (fallback) JJS_CUDA(ctx, cudaMemsetAsync(fallback, 0, sizeof(unsigned long long), stream));
    Overlap ov(ctx, d, stream, n > d.sub_chunk);
    rc = ov.begin();
    if (rc) return rc;
    for (int h = 0; h < 2 && all_valid; h++) {
        k_rlc_init<<<1, 1, 0, ov.on ? d.sub[h] : stream>>>(rlc_acc(d, region_half(d, h)));
        ctx->launches++;
    }
    for (const Part& P : parts) {
        const bool whole = !ov.on && (P.mode == PART_WIRE || P.mode == PART_KEYED);
        const PartPtrs b{P.pk, P.sig, P.msg, P.offsets, P.status, P.c_out, P.agg_out, 0, 0};
        for (size_t off = 0; off < P.n; ov.advance()) {
            const Region R = whole ? region_whole(d) : region_half(d, ov.i);
            const size_t end = pass_end(d, R, P, P.h_offsets, off, P.n, whole ? d.chunk_items : d.sub_chunk);
            rc = run_pass(ctx, k, R, P, b, off, end - off, ov.next_stream(), fallback);
            if (rc) return rc;
            off = end;
        }
    }
    rc = ov.end();
    if (rc) return rc;
    for (const Part& P : parts) {
        if (!P.bitmap || !P.n) continue;
        k_bitmap<<<blocks_for(P.n), BLOCK, 0, stream>>>(P.status, P.n, P.bitmap);
        ctx->launches++;
    }
    if (all_valid) {
        (d.fb_w == FB_W_SMALL ? k_rlc_finish<FB_W_SMALL> : k_rlc_finish<FB_W>)<<<1, 1, 0, stream>>>(
            rlc_acc(d, region_half(d, 0)), rlc_acc(d, region_half(d, 1)), d.tables(), nullptr, all_valid);
        ctx->launches++;
    }
    JJS_CUDA(ctx, cudaGetLastError());
    return JJS_SUCCESS;
}

// ---- host-buffer calls ------------------------------------------------------------------------------------------------------
struct StagedPart {   // device staging of one part's shard
    uint8_t *pk = nullptr, *sig = nullptr, *msg = nullptr, *status = nullptr, *c = nullptr, *agg = nullptr;
    uint32_t *offsets = nullptr, *bitmap = nullptr;
};

// bytes of the pk buffer of items [lo, hi) of part P (aggregate parts: of their signer keys)
inline size_t part_pk_bytes(const Part& P, size_t lo, size_t hi) {
    return part_strides(P).pk * (part_aggregate(P) ? (size_t)(P.h_offsets[hi] - P.h_offsets[lo]) : hi - lo);
}

// Everything device k does for one call.  Runs on its own host thread when the context has several devices.
int device_job(jjs_ctx* ctx, size_t k, const std::vector<Part>& parts, const std::vector<std::vector<Shard>>& shards) {
    DeviceState& d = ctx->dev[k];
    std::vector<Shard> mine(parts.size());
    bool any = false;
    for (size_t p = 0; p < parts.size(); p++) {
        mine[p] = shards[p][k];
        any = any || mine[p].hi > mine[p].lo;
    }
    if (!any) return JJS_SUCCESS;
    JJS_CUDA(ctx, cudaSetDevice(d.device));
    int rc = prepare_parts(ctx, d, parts, mine);
    if (rc) return rc;
    // staging layout
    std::vector<StagedPart> st(parts.size());
    std::vector<size_t> o_pk(parts.size()), o_sig(parts.size()), o_msg(parts.size()), o_st(parts.size()), o_c(parts.size()), o_agg(parts.size()),
        o_off(parts.size()), o_bm(parts.size());
    size_t total = 0;
    for (size_t p = 0; p < parts.size(); p++) {
        const Part& P = parts[p];
        const size_t lo = mine[p].lo, hi = mine[p].hi, m = hi - lo;
        if (!m) continue;
        o_pk[p] = total; total += align_up(part_pk_bytes(P, lo, hi), 256);
        o_sig[p] = total; total += align_up(part_strides(P).sig * m, 256);
        o_msg[p] = total; total += align_up(32 * m, 256);
        o_st[p] = total; total += align_up(m, 256);
        o_c[p] = total; total += align_up(32 * m, 256);
        o_bm[p] = total; total += align_up(4 * ((m + 31) / 32), 256);
        if (part_aggregate(P)) {
            o_agg[p] = total; total += align_up(32 * m, 256);
            o_off[p] = total; total += align_up(4 * (m + 1), 256);
        }
    }
    int p_grp = -1;                     // the first grouped part with items here, if any: its sink gets the device's fallback count,
    for (size_t p = 0; p < parts.size() && p_grp < 0; p++)   // which is staged after the parts
        if (parts[p].mode == PART_GROUPED && mine[p].hi > mine[p].lo) p_grp = (int)p;
    const size_t o_fb = total;
    if (p_grp >= 0) total += 256;
    rc = ensure_stage(ctx, d, total);
    if (rc) return rc;
    unsigned long long* d_fb = p_grp >= 0 ? reinterpret_cast<unsigned long long*>(d.stage + o_fb) : nullptr;
    if (d_fb) JJS_CUDA(ctx, cudaMemsetAsync(d_fb, 0, sizeof(unsigned long long), d.copy_stream));   // before every slice's copies
    const bool serial = ctx->profile;   // stage timers must not overlap
    int p_all = -1;                     // the first whole-batch part with items here, if any: all of them add into the accumulators of
    for (size_t p = 0; p < parts.size() && p_all < 0; p++)   // both halves, which start out empty
        if (parts[p].mode == PART_ALL && mine[p].hi > mine[p].lo) p_all = (int)p;
    if (p_all >= 0)
        for (int h = 0; h < 2; h++) {
            k_rlc_init<<<1, 1, 0, serial ? d.stream : d.sub[h]>>>(rlc_acc(d, region_half(d, h)));
            ctx->launches++;
        }
    size_t j = 0;                       // slice counter of this device: slices alternate between the compute streams / scratch halves
    for (size_t p = 0; p < parts.size(); p++) {
        const Part& P = parts[p];
        const size_t lo = mine[p].lo, hi = mine[p].hi, m = hi - lo;
        if (!m) continue;
        StagedPart& S = st[p];
        S.pk = d.stage + o_pk[p]; S.sig = d.stage + o_sig[p]; S.msg = d.stage + o_msg[p]; S.status = d.stage + o_st[p]; S.c = d.stage + o_c[p];
        S.bitmap = reinterpret_cast<uint32_t*>(d.stage + o_bm[p]);
        const uint32_t* ho = part_aggregate(P) ? P.h_offsets + lo : nullptr;   // host offsets of this shard
        if (ho) {
            S.agg = d.stage + o_agg[p];
            S.offsets = reinterpret_cast<uint32_t*>(d.stage + o_off[p]);
            JJS_CUDA(ctx, cudaMemcpyAsync(S.offsets, ho, 4 * (m + 1), cudaMemcpyHostToDevice, d.copy_stream));
        }
        const Strides s = part_strides(P);
        const bool want_c = P.c_out != nullptr || P.challenge_only;
        const PartPtrs b{S.pk, S.sig, S.msg, S.offsets, S.status, want_c ? S.c : nullptr, P.agg_out ? S.agg : nullptr, lo, ho ? ho[0] : 0u};
        // Pipeline slices: slice j + 1 is copied in on the copy stream while slice j is being verified (the kernels of one
        // slice run far longer than its copy); the first slice of a device is short so that compute starts early.
        for (size_t off = 0; off < m; j++) {
            cudaStream_t cs = serial ? d.stream : d.sub[j & 1];
            const Region R = region_half(d, j);
            const size_t end = pass_end(d, R, P, ho, off, m, j == 0 ? d.first_slice : d.sub_chunk), cnt = end - off;
            if (ho) {
                const size_t K = ho[end] - ho[off];
                if (K) JJS_CUDA(ctx, cudaMemcpyAsync(S.pk + s.pk * (ho[off] - ho[0]), P.pk + s.pk * ho[off], s.pk * K, cudaMemcpyHostToDevice, d.copy_stream));
            } else {
                JJS_CUDA(ctx, cudaMemcpyAsync(S.pk + off * s.pk, P.pk + (lo + off) * s.pk, cnt * s.pk, cudaMemcpyHostToDevice, d.copy_stream));
            }
            JJS_CUDA(ctx, cudaMemcpyAsync(S.sig + off * s.sig, P.sig + (lo + off) * s.sig, cnt * s.sig, cudaMemcpyHostToDevice, d.copy_stream));
            JJS_CUDA(ctx, cudaMemcpyAsync(S.msg + off * 32, P.msg + (lo + off) * 32, cnt * 32, cudaMemcpyHostToDevice, d.copy_stream));
            JJS_CUDA(ctx, cudaEventRecord(d.copied, d.copy_stream));
            JJS_CUDA(ctx, cudaStreamWaitEvent(cs, d.copied, 0));
            rc = run_pass(ctx, k, R, P, b, off, cnt, cs, d_fb);
            if (rc) return rc;
            off = end;
        }
    }
    if (!serial)
        for (int q = 0; q < 2; q++) {
            JJS_CUDA(ctx, cudaEventRecord(d.join[q], d.sub[q]));
            JJS_CUDA(ctx, cudaStreamWaitEvent(d.stream, d.join[q], 0));
        }
    for (size_t p = 0; p < parts.size(); p++) {
        const Part& P = parts[p];
        const size_t lo = mine[p].lo, hi = mine[p].hi, m = hi - lo;
        if (!m) continue;
        const StagedPart& S = st[p];
        if (!P.challenge_only && P.status) JJS_CUDA(ctx, cudaMemcpyAsync(P.status + lo, S.status, m, cudaMemcpyDeviceToHost, d.stream));
        if (P.c_out) JJS_CUDA(ctx, cudaMemcpyAsync(P.c_out + lo * 32, S.c, m * 32, cudaMemcpyDeviceToHost, d.stream));
        if (P.agg_out) JJS_CUDA(ctx, cudaMemcpyAsync(P.agg_out + lo * 32, S.agg, m * 32, cudaMemcpyDeviceToHost, d.stream));
        if (P.bitmap) {
            k_bitmap<<<blocks_for(m), BLOCK, 0, d.stream>>>(S.status, m, S.bitmap);
            ctx->launches++;
            JJS_CUDA(ctx, cudaMemcpyAsync(P.bitmap + lo / 32, S.bitmap, 4 * ((m + 31) / 32), cudaMemcpyDeviceToHost, d.stream));
        }
    }
    RlcOut out;
    if (p_all >= 0) {   // the device's partial point: both halves' accumulators and the G terms, staged in the part's challenge slot
        RlcOut* d_out = reinterpret_cast<RlcOut*>(st[p_all].c);
        (d.fb_w == FB_W_SMALL ? k_rlc_finish<FB_W_SMALL> : k_rlc_finish<FB_W>)<<<1, 1, 0, d.stream>>>(
            rlc_acc(d, region_half(d, 0)), rlc_acc(d, region_half(d, 1)), d.tables(), d_out, nullptr);
        ctx->launches++;
        JJS_CUDA(ctx, cudaMemcpyAsync(&out, d_out, sizeof(RlcOut), cudaMemcpyDeviceToHost, d.stream));
    }
    unsigned long long fb = 0;
    if (d_fb) JJS_CUDA(ctx, cudaMemcpyAsync(&fb, d_fb, sizeof(fb), cudaMemcpyDeviceToHost, d.stream));
    JJS_CUDA(ctx, cudaGetLastError());
    JJS_CUDA(ctx, cudaStreamSynchronize(d.stream));
    if (p_all >= 0) parts[p_all].sink->add(out);
    if (p_grp >= 0) parts[p_grp].sink->add_fallback(fb);
    return JJS_SUCCESS;
}

// Device staging that device_job lays out for items [lo, hi) of part P.
inline size_t part_stage_bytes(const Part& P, size_t lo, size_t hi) {
    const size_t m = hi - lo;
    size_t b = align_up(part_pk_bytes(P, lo, hi), 256) + align_up(part_strides(P).sig * m, 256) + 2 * align_up(32 * m, 256) + align_up(m, 256) +
               align_up(4 * ((m + 31) / 32), 256);
    if (part_aggregate(P)) b += align_up(32 * m, 256) + align_up(4 * (m + 1), 256);
    return b;
}
// The largest window [lo, end) of part P whose staging fits `budget` bytes, ending on a bitmap word (or at hi); at least one word.
size_t window_end(const Part& P, size_t lo, size_t hi, size_t budget) {
    size_t good = 1, bad = (hi - lo + 31) / 32 + 1;   // in bitmap words
    while (bad - good > 1) {
        const size_t mid = (good + bad) / 2, end = lo + 32 * mid < hi ? lo + 32 * mid : hi;
        if (part_stage_bytes(P, lo, end) <= budget) good = mid;
        else bad = mid;
    }
    return lo + 32 * good < hi ? lo + 32 * good : hi;
}
// A memory-limited context cannot stage a whole shard: it runs device_job window by window, each window as large as the staging
// buffer it reserved at init allows (or grows within its limit for a window of one bitmap word), so batches of any size stream
// through it.  Each window is verified and copied back before the next is staged.
int device_job_windows(jjs_ctx* ctx, size_t k, const std::vector<Part>& parts, const std::vector<std::vector<Shard>>& shards) {
    DeviceState& d = ctx->dev[k];
    std::vector<std::vector<Shard>> win(parts.size(), std::vector<Shard>(ctx->dev.size(), Shard{0, 0}));
    bool grouped = false;   // device_job stages a grouped call's fallback count after the parts
    for (const Part& P : parts) grouped = grouped || P.mode == PART_GROUPED;
    const size_t budget = d.stage_bytes - (grouped ? 256 : 0);
    for (size_t p = 0; p < parts.size(); p++) {
        const size_t hi = shards[p][k].hi;
        for (size_t off = shards[p][k].lo; off < hi;) {
            const size_t end = window_end(parts[p], off, hi, budget);
            win[p][k] = Shard{off, end};
            int rc = device_job(ctx, k, parts, win);
            if (rc) return rc;
            off = end;
        }
        win[p][k] = Shard{0, 0};
    }
    return JJS_SUCCESS;
}

// device_job, and on failure a drain of the device: nothing may still be reading or writing the caller's buffers when the
// call returns
int device_job_drained(jjs_ctx* ctx, size_t k, const std::vector<Part>& parts, const std::vector<std::vector<Shard>>& shards) {
    int rc = ctx->dev[k].limit ? device_job_windows(ctx, k, parts, shards) : device_job(ctx, k, parts, shards);
    if (rc) {
        cudaSetDevice(ctx->dev[k].device);
        cudaDeviceSynchronize();
    }
    return rc;
}

// A host-buffer call of checked parts.
int run_parts(jjs_ctx* ctx, const std::vector<Part>& parts) {
    bool any = false;
    for (const Part& P : parts) any = any || P.n > 0;
    if (!any) return JJS_SUCCESS;
    const size_t g = ctx->dev.size();
    std::vector<std::vector<Shard>> shards;
    plan_shards(parts, g, shards);
    std::vector<int> rcs(g, JJS_SUCCESS);
    if (g == 1) {
        rcs[0] = device_job_drained(ctx, 0, parts, shards);
    } else {
        std::vector<std::thread> workers;
        workers.reserve(g);
        for (size_t k = 0; k < g; k++) workers.emplace_back([&, k] { rcs[k] = device_job_drained(ctx, k, parts, shards); });
        for (auto& w : workers) w.join();
    }
    for (size_t k = 0; k < g; k++)
        if (rcs[k]) return rcs[k];
    return JJS_SUCCESS;
}
// A host-buffer call of one part.
int run_part(jjs_ctx* ctx, const Part& P) {
    JJS_ENTER(ctx);
    int rc = validate_part(ctx, P, false);
    return rc ? rc : run_parts(ctx, {P});
}

Part wire_part(int variant, const uint8_t* pk, const uint8_t* sig, const uint8_t* msg, size_t n, uint8_t* status, uint8_t* c_out, uint32_t* bitmap) {
    return Part{PART_WIRE, variant, pk, sig, msg, nullptr, nullptr, n, status, c_out, nullptr, bitmap};
}
Part aggregate_part(const uint8_t* pks, const uint32_t* offsets, const uint32_t* h_offsets, const uint8_t* sig, const uint8_t* msg, size_t n,
                    uint8_t* status, uint8_t* c_out, uint8_t* agg_out, uint32_t* bitmap) {
    return Part{PART_AGGREGATE, JJS_KIND_AGGREGATE, pks, sig, msg, offsets, h_offsets, n, status, c_out, agg_out, bitmap};
}

// The checked parts of a jjs_part array: per-item parts (mode PART_WIRE: wire or aggregate parts by kind), or the whole-batch
// (PART_ALL: no per-item outputs) or grouped (PART_GROUPED) parts of one call, whose items are weighted by their position in the
// call.  The parts of a device-buffer call (on_device) take the host copies of the aggregate parts' offsets from h_offsets.
int parts_from_jjs(jjs_ctx* ctx, const jjs_part* parts, size_t n_parts, int mode, bool on_device, const uint32_t* const* h_offsets,
                   const RlcSeed* seed, RlcSink* sink, std::vector<Part>& out) {
    out.reserve(n_parts);
    uint64_t base = 0;
    for (size_t i = 0; i < n_parts; i++) {
        const jjs_part& p = parts[i];
        if (p.kind < JJS_KIND_SINGLE || p.kind > JJS_KIND_AGGREGATE) return fail(ctx, JJS_ERR_ARGUMENT, "part %zu: bad kind", i);
        if (mode == PART_ALL && (p.status || p.c32 || p.aggpk32 || p.accept_bitmap))
            return fail(ctx, JJS_ERR_ARGUMENT, "part %zu: whole-batch verification has no per-item outputs", i);
        const bool agg = p.kind == JJS_KIND_AGGREGATE;
        const uint32_t* ho = !agg ? nullptr : !on_device ? p.offsets : h_offsets ? h_offsets[i] : nullptr;
        Part P{mode == PART_WIRE && agg ? (int)PART_AGGREGATE : mode, p.kind, p.pk, p.sig, p.msg32, agg ? p.offsets : nullptr, ho, p.n, p.status,
               p.c32, agg ? p.aggpk32 : nullptr, p.accept_bitmap};
        P.seed = seed;
        P.sink = sink;
        P.base = base;
        base += p.n;
        int rc = validate_part(ctx, P, on_device, (long)i);
        if (rc) return rc;
        out.push_back(P);
    }
    return JJS_SUCCESS;
}

// multisig::combine for n ragged sessions (host buffers, device 0); a chunk holds as many sessions as the table scratch serves
// threads of k_msig_session and as many participants as it serves threads of k_msig_share (2^20 each on a jjs_init context)
int run_msig(jjs_ctx* ctx, const uint8_t* pks, const uint8_t* Rs, const uint8_t* Ss, const uint8_t* zs, const uint32_t* offsets, const uint8_t* msg,
             size_t n, uint8_t* share_ok, uint8_t* status, uint32_t* bad, uint8_t* sig) {
    JJS_ENTER(ctx);
    if (n == 0) return JJS_SUCCESS;
    if (!offsets || !msg || !status) return fail(ctx, JJS_ERR_ARGUMENT, "null buffer");
    if (offsets[0] != 0) return fail(ctx, JJS_ERR_ARGUMENT, "offsets[0] must be 0");
    for (size_t i = 0; i < n; i++)
        if (offsets[i + 1] < offsets[i]) return fail(ctx, JJS_ERR_ARGUMENT, "offsets must be non-decreasing");
    if (offsets[n] && (!pks || !Rs || !Ss || !zs)) return fail(ctx, JJS_ERR_ARGUMENT, "null buffer");
    DeviceState& d = ctx->dev[0];
    int rc = ensure_scratch(ctx, d);
    if (!rc) rc = ensure_tags(ctx, d, 3 + 4 * agg_max_item_keys(offsets, n));
    if (rc) return rc;
    JJS_CUDA(ctx, cudaSetDevice(d.device));
    Tables T = d.tables();
    const size_t sess_stride = tab_threads(d, d.chunk_items, AGG_GROUP * R32_TAB_FQ), share_stride = tab_threads(d, d.chunk_items, 2 * 36);
    const size_t max_sessions = sess_stride < d.chunk_items ? sess_stride : d.chunk_items;
    std::vector<uint32_t> rel, owner, order;
    for (size_t s0 = 0; s0 < n;) {
        size_t s1 = s0;
        while (s1 < n && s1 - s0 < max_sessions && offsets[s1 + 1] - offsets[s0] <= share_stride) s1++;
        if (s1 == s0) return fail(ctx, JJS_ERR_ARGUMENT, "a session has more than %zu participants", share_stride);
        const size_t m = s1 - s0, K = offsets[s1] - offsets[s0], k0 = offsets[s0];
        rel.resize(m + 1);
        owner.resize(K ? K : 1);
        order.resize(m);
        size_t hist[34] = {0};
        for (size_t i = 0; i <= m; i++) rel[i] = offsets[s0 + i] - (uint32_t)k0;
        for (size_t i = 0; i < m; i++) {
            uint32_t c = rel[i + 1] - rel[i];
            for (uint32_t j = rel[i]; j < rel[i + 1]; j++) owner[j] = (uint32_t)i;
            hist[(c > 32 ? 32 : c) + 1]++;
        }
        for (int b = 0; b < 33; b++) hist[b + 1] += hist[b];
        for (size_t i = 0; i < m; i++) {
            uint32_t c = rel[i + 1] - rel[i];
            order[hist[c > 32 ? 32 : c]++] = (uint32_t)i;
        }
        // one device buffer: wire inputs | decoded points | scalars | results | index arrays
        size_t o = 0;
        auto take = [&](size_t bytes) { size_t at = o; o += (bytes + 255) / 256 * 256; return at; };
        size_t o_pk = take(32 * K), o_R = take(32 * K), o_S = take(32 * K), o_z = take(32 * K), o_msg = take(32 * m), o_pu = take(sizeof(fq) * 3 * K),
               o_pv = take(sizeof(fq) * 3 * K), o_pf = take(3 * K), o_d = take(32 * K), o_cd = take(32 * K), o_a = take(32 * m), o_ru = take(sizeof(fq) * m),
               o_rv = take(sizeof(fq) * m), o_sf = take(m), o_ok = take(K), o_off = take(4 * (m + 1)), o_own = take(4 * K), o_ord = take(4 * m),
               o_st = take(m), o_bad = take(4 * m), o_sig = take(64 * m);
        rc = ensure_stage(ctx, d, o);
        if (rc) return rc;
        uint8_t* B = d.stage;
        cudaStream_t st = d.stream;
        cudaError_t ce = cudaSuccess;
        auto up = [&](size_t at, const void* src, size_t bytes) { if (ce == cudaSuccess && bytes) ce = cudaMemcpyAsync(B + at, src, bytes, cudaMemcpyHostToDevice, st); };
        up(o_pk, pks + 32 * k0, 32 * K); up(o_R, Rs + 32 * k0, 32 * K); up(o_S, Ss + 32 * k0, 32 * K); up(o_z, zs + 32 * k0, 32 * K);
        up(o_own, owner.data(), 4 * K); up(o_msg, msg + 32 * s0, 32 * m); up(o_off, rel.data(), 4 * (m + 1)); up(o_ord, order.data(), 4 * m);
        MsigBuffers b;
        b.pu = reinterpret_cast<fq*>(B + o_pu); b.pv = reinterpret_cast<fq*>(B + o_pv); b.pf = B + o_pf;
        b.d_words = reinterpret_cast<uint32_t*>(B + o_d); b.cd_words = reinterpret_cast<uint32_t*>(B + o_cd); b.a_words = reinterpret_cast<uint32_t*>(B + o_a);
        b.rsa_u = reinterpret_cast<fq*>(B + o_ru); b.rsa_v = reinterpret_cast<fq*>(B + o_rv); b.sflags = B + o_sf; b.share_ok = B + o_ok;
        b.offsets = reinterpret_cast<uint32_t*>(B + o_off); b.owner = reinterpret_cast<uint32_t*>(B + o_own); b.order = reinterpret_cast<uint32_t*>(B + o_ord);
        Fields f;
        f.f[0] = WireField{B + o_pk, 32}; f.f[1] = WireField{B + o_R, 32}; f.f[2] = WireField{B + o_S, 32}; f.f[3] = WireField{nullptr, 0};
        WireField fmsg{B + o_msg, 32}, fz{B + o_z, 32};
        if (K) k_decode<<<blocks_for(3 * K), BLOCK, 0, st>>>(f, 3, 0, K, b.pu, b.pv, b.pf, T, 0u);
        k_msig_session<<<blocks_for(m), BLOCK, 0, st>>>(b, K, m, fmsg, fz, d.tab, sess_stride, T);
        if (K) (d.fb_w == FB_W_SMALL ? k_msig_share<FB_W_SMALL> : k_msig_share<>)<<<blocks_for(K), BLOCK, 0, st>>>(b, K, fz, d.tab, share_stride, T);
        k_msig_finalize<<<blocks_for(m), BLOCK, 0, st>>>(b, m, fz, B + o_st, reinterpret_cast<uint32_t*>(B + o_bad), B + o_sig);
        ctx->launches += 4;
        auto down = [&](void* dst, size_t at, size_t bytes) { if (ce == cudaSuccess && bytes) ce = cudaMemcpyAsync(dst, B + at, bytes, cudaMemcpyDeviceToHost, st); };
        down(status + s0, o_st, m);
        if (bad) down(bad + s0, o_bad, 4 * m);
        if (sig) down(sig + 64 * s0, o_sig, 64 * m);
        if (share_ok) down(share_ok + k0, o_ok, K);
        cudaError_t e = cudaStreamSynchronize(st);   // also the drain of the error path: the host vectors above are reused by the next chunk
        if (ce != cudaSuccess) e = ce;
        if (e != cudaSuccess) return fail(ctx, JJS_ERR_CUDA, "multisig combine failed: %s", cudaGetErrorString(e));
        s0 = s1;
    }
    return JJS_SUCCESS;
}

int run_sign(jjs_ctx* ctx, int variant, const uint8_t* sk, const uint8_t* rnd, const uint8_t* gsc, const uint8_t* msg, size_t n, uint8_t* pk_out,
             uint8_t* sig_out) {
    JJS_ENTER(ctx);
    if (variant < 0 || variant > 2) return fail(ctx, JJS_ERR_ARGUMENT, "bad variant");
    if (n == 0) return JJS_SUCCESS;
    if (!sk || !rnd || !msg || !pk_out || !sig_out || (variant == VAR_VARGEN && !gsc)) return fail(ctx, JJS_ERR_ARGUMENT, "null buffer");
    DeviceState& d = ctx->dev[0];
    JJS_CUDA(ctx, cudaSetDevice(d.device));
    const size_t pks = pk_size(variant), sgs = sig_size(variant);
    const size_t chunk = n < d.chunk_items ? n : d.chunk_items;
    int rc = ensure_stage(ctx, d, chunk * (4 * 32 + pks + sgs));
    if (rc) return rc;
    uint8_t* buf = d.stage;
    uint8_t *d_sk = buf, *d_rnd = buf + 32 * chunk, *d_g = buf + 64 * chunk, *d_msg = buf + 96 * chunk, *d_pk = buf + 128 * chunk,
            *d_sig = d_pk + pks * chunk;
    for (size_t off = 0; off < n; off += chunk) {
        size_t m = n - off < chunk ? n - off : chunk;
        cudaError_t ce = cudaMemcpyAsync(d_sk, sk + 32 * off, 32 * m, cudaMemcpyHostToDevice, d.stream);
        if (ce == cudaSuccess) ce = cudaMemcpyAsync(d_rnd, rnd + 32 * off, 32 * m, cudaMemcpyHostToDevice, d.stream);
        if (ce == cudaSuccess && variant == VAR_VARGEN) ce = cudaMemcpyAsync(d_g, gsc + 32 * off, 32 * m, cudaMemcpyHostToDevice, d.stream);
        if (ce == cudaSuccess) ce = cudaMemcpyAsync(d_msg, msg + 32 * off, 32 * m, cudaMemcpyHostToDevice, d.stream);
        if (ce == cudaSuccess) {
            const bool small = d.fb_w == FB_W_SMALL;
            const auto ks = variant == VAR_SINGLE ? (small ? k_sign<VAR_SINGLE, FB_W_SMALL> : k_sign<VAR_SINGLE>)
                            : variant == VAR_DOUBLE ? (small ? k_sign<VAR_DOUBLE, FB_W_SMALL> : k_sign<VAR_DOUBLE>)
                                                    : (small ? k_sign<VAR_VARGEN, FB_W_SMALL> : k_sign<VAR_VARGEN>);
            ks<<<blocks_for(m), BLOCK, 0, d.stream>>>(d_sk, d_rnd, d_g, d_msg, m, d_pk, d_sig, d.tables());
            ctx->launches++;
            ce = cudaMemcpyAsync(pk_out + pks * off, d_pk, pks * m, cudaMemcpyDeviceToHost, d.stream);
        }
        if (ce == cudaSuccess) ce = cudaMemcpyAsync(sig_out + sgs * off, d_sig, sgs * m, cudaMemcpyDeviceToHost, d.stream);
        cudaError_t e = cudaStreamSynchronize(d.stream);
        if (ce != cudaSuccess) e = ce;
        if (e != cudaSuccess) return fail(ctx, JJS_ERR_CUDA, "sign batch failed: %s", cudaGetErrorString(e));
    }
    return JJS_SUCCESS;
}

// G / G' tables of width W in two passes (k_fb_small, k_fb_combine)
template <int W>
int build_fb_tables(jjs_ctx* ctx, DeviceState& d) {
    constexpr int LO = (W + 1) / 2, HI = W - LO, WINDOWS = (252 + W - 1) / W, SMALL = (1 << LO) + (1 << HI);
    const size_t small_bytes = sizeof(fq) * WINDOWS * SMALL;
    fq *small_u = nullptr, *small_v = nullptr;
    DevAlloc A = dev_alloc(ctx, d);
    int rc = A(&small_u, small_bytes);
    if (!rc) rc = A(&small_v, small_bytes);
    if (!rc) {
        for (int which = 0; which < 2; which++) {
            k_fb_small<W><<<blocks_for(WINDOWS * SMALL), BLOCK, 0, d.stream>>>(small_u, small_v, which);
            k_fb_combine<W><<<blocks_for((size_t)WINDOWS * ((size_t)1 << W) / FB_BATCH), BLOCK, 0, d.stream>>>(which ? d.fb_gn : d.fb_g, small_u, small_v);
        }
        ctx->launches += 4;
    }
    cudaError_t e1 = cudaGetLastError(), e2 = cudaStreamSynchronize(d.stream);
    dev_free(d, small_u, small_bytes);
    dev_free(d, small_v, small_bytes);
    if (rc) return rc;
    JJS_CUDA(ctx, e1);
    JJS_CUDA(ctx, e2);
    return JJS_SUCCESS;
}

// Constant tables, fixed-base tables and SAFE tags of one device; a memory-limited context (d.limit set, configure_limited
// applied) also allocates all its scratch here.
int init_device(jjs_ctx* ctx, DeviceState& d) {
    JJS_CUDA(ctx, cudaSetDevice(d.device));
    cudaDeviceProp prop;
    JJS_CUDA(ctx, cudaGetDeviceProperties(&prop, d.device));
    if (prop.major != 10) return fail(ctx, JJS_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", d.device, prop.major, prop.minor);
    JJS_CUDA(ctx, cudaStreamCreateWithFlags(&d.stream, cudaStreamNonBlocking));
    JJS_CUDA(ctx, cudaStreamCreateWithFlags(&d.copy_stream, cudaStreamNonBlocking));
    JJS_CUDA(ctx, cudaEventCreateWithFlags(&d.copied, cudaEventDisableTiming));
    JJS_CUDA(ctx, cudaEventCreateWithFlags(&d.fork, cudaEventDisableTiming));
    for (int k = 0; k < 2; k++) {
        JJS_CUDA(ctx, cudaStreamCreateWithFlags(&d.sub[k], cudaStreamNonBlocking));
        JJS_CUDA(ctx, cudaEventCreateWithFlags(&d.join[k], cudaEventDisableTiming));
    }
    DevAlloc A = dev_alloc(ctx, d);
    int rc = alloc_tables(A, d);
    if (rc) return rc;
    JJS_CUDA(ctx, cudaMemcpy(d.root_tables, tables::ROOT_TABLES, sizeof(tables::ROOT_TABLES), cudaMemcpyHostToDevice));
    JJS_CUDA(ctx, cudaMemcpy(d.dlog_hash, tables::DLOG_HASH, sizeof(tables::DLOG_HASH), cudaMemcpyHostToDevice));
    rc = d.fb_w == FB_W_SMALL ? build_fb_tables<FB_W_SMALL>(ctx, d) : build_fb_tables<FB_W>(ctx, d);
    if (!rc) rc = ensure_tags(ctx, d, TAGS_INITIAL - 1);
    if (!rc && d.limit) rc = alloc_limited_scratch(A, d);
    return rc;
}

void free_device(DeviceState& d) {
    if (d.device < 0) return;
    cudaSetDevice(d.device);
    cudaDeviceSynchronize();
    cudaFree(d.root_tables); cudaFree(d.dlog_hash); cudaFree(d.fb_g); cudaFree(d.fb_gn); cudaFree(d.safe_tags);
    cudaFree(d.pts_u); cudaFree(d.pts_v); cudaFree(d.tab); cudaFree(d.eqtab); cudaFree(d.pflags); cudaFree(d.iflags); cudaFree(d.eqflags); cudaFree(d.cwords);
    cudaFree(d.rlist); cudaFree(d.rcount); cudaFree(d.eqlist); cudaFree(d.stage);
    for (int h = 0; h < 2; h++) {
        AggScratch& a = d.agg[h];
        cudaFree(a.keys_u); cudaFree(a.keys_v); cudaFree(a.kflags); cudaFree(a.kcoef); cudaFree(a.kmap); cudaFree(a.kitem); cudaFree(a.order); cudaFree(a.sort);
    }
    if (d.stream) cudaStreamDestroy(d.stream);
    if (d.copy_stream) cudaStreamDestroy(d.copy_stream);
    if (d.copied) cudaEventDestroy(d.copied);
    if (d.fork) cudaEventDestroy(d.fork);
    for (int k = 0; k < 2; k++) {
        if (d.sub[k]) cudaStreamDestroy(d.sub[k]);
        if (d.join[k]) cudaEventDestroy(d.join[k]);
    }
}

// a per-item device-buffer call of one part on the caller's stream
int device_entry(jjs_ctx* ctx, int device_index, const Part& P, void* stream) {
    JJS_ENTER(ctx);
    if (device_index < 0 || (size_t)device_index >= ctx->dev.size()) return fail(ctx, JJS_ERR_ARGUMENT, "device_index out of range");
    int rc = validate_part(ctx, P, true);
    if (rc || P.n == 0) return rc;
    return run_device_parts(ctx, (size_t)device_index, {P}, (cudaStream_t)stream, nullptr, nullptr);
}

// small synchronous utilities on device 0: copy in, one kernel, copy out
template <typename Launch>
int run_small(jjs_ctx* ctx, const char* what, size_t in_bytes, size_t out_bytes, const void* const* srcs, const size_t* src_bytes, int n_src, void* dst,
              Launch launch) {
    DeviceState& d = ctx->dev[0];
    JJS_CUDA(ctx, cudaSetDevice(d.device));
    int rc = ensure_stage(ctx, d, align_up(in_bytes, 256) + out_bytes);
    if (rc) return rc;
    cudaError_t ce = cudaSuccess;
    size_t at = 0;
    for (int i = 0; i < n_src && ce == cudaSuccess; i++) {
        if (src_bytes[i]) ce = cudaMemcpyAsync(d.stage + at, srcs[i], src_bytes[i], cudaMemcpyHostToDevice, d.stream);
        at += src_bytes[i];
    }
    uint8_t* d_out = d.stage + align_up(in_bytes, 256);
    if (ce == cudaSuccess) {
        launch(d, d.stage, d_out);
        ce = cudaGetLastError();
    }
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(dst, d_out, out_bytes, cudaMemcpyDeviceToHost, d.stream);
    cudaError_t e = cudaStreamSynchronize(d.stream);
    if (ce != cudaSuccess) e = ce;
    if (e != cudaSuccess) return fail(ctx, JJS_ERR_CUDA, "%s failed: %s", what, cudaGetErrorString(e));
    return JJS_SUCCESS;
}

// ---- registered key sets ----------------------------------------------------------------------------------------
// Device memory of a key set of npts key points: decoded points and flags, and the tables of width kw (none for kw = 0).
inline size_t keyset_point_bytes(size_t npts) { return npts * (2 * sizeof(fq) + 1); }
inline size_t keyset_table_bytes(size_t npts, int kw) { return kw ? sizeof(niels) * npts * keyed_point_entries(kw) : 0; }

struct DeviceTemp {   // scratch of one key-set build, freed on every path out
    DeviceState& d;
    size_t bytes;
    uint8_t* p = nullptr;
    ~DeviceTemp() { dev_free(d, p, bytes); }
};

// Everything a key set of npts key points at width kw allocates on a device, in order: what it keeps (points, flags, tables),
// then the build's scratch (the wire keys and, with tables, the window bases of every key point).
int alloc_keyset(DevAlloc& A, KeySetDev& kd, size_t npts, int kw, uint8_t** wire, uint8_t** bases) {
    int rc = A(&kd.u, sizeof(fq) * npts);
    if (!rc) rc = A(&kd.v, sizeof(fq) * npts);
    if (!rc) rc = A(&kd.flags, npts);
    if (!rc && kw) rc = A(&kd.table, keyset_table_bytes(npts, kw));
    if (!rc) rc = A(wire, 32 * npts);
    if (!rc && kw) rc = A(bases, sizeof(ext) * npts * keyed_windows(kw));
    return rc;
}
// The most a key set of npts key points at width kw holds on a device, while its tables are built: a dry run of alloc_keyset.
size_t keyset_peak(size_t npts, int kw) {
    DevAlloc A{nullptr, nullptr};
    KeySetDev kd;
    uint8_t *wire = nullptr, *bases = nullptr;
    alloc_keyset(A, kd, npts, kw, &wire, &bases);
    return A.total;
}

// Key set `ks` on device d: copy the wire keys in, decode them with the subgroup test, build the tables (keyset.cuh) unless the
// set holds points only.  key_status (optional) receives 0 / 2 / 3 per key.
int keyset_build(jjs_ctx* ctx, DeviceState& d, const KeySet& ks, KeySetDev& kd, const uint8_t* pk, uint8_t* key_status) {
    JJS_CUDA(ctx, cudaSetDevice(d.device));
    const int nk = keyed_points(ks.variant), kw = ks.key_bits;
    const size_t npts = (size_t)nk * ks.n_keys;
    DeviceTemp wire{d, 32 * npts}, bases{d, kw ? sizeof(ext) * npts * keyed_windows(kw) : 0};
    // a limited context refuses a key set that would cross its limit before allocating any of it
    const size_t need = keyset_peak(npts, kw);
    if (d.limit && d.held + need > d.limit)
        return fail(ctx, JJS_ERR_NOMEM, "key set: %zu bytes on device %d would exceed the context's memory limit of %zu bytes (%zu held)", need, d.device,
                    d.limit, d.held);
    DevAlloc A = dev_alloc(ctx, d);
    int rc = alloc_keyset(A, kd, npts, kw, &wire.p, &bases.p);
    if (rc) return rc;
    cudaStream_t st = d.stream;
    // undecodable keys leave their coordinates unwritten; zero them so that gathering them copies defined values
    JJS_CUDA(ctx, cudaMemsetAsync(kd.u, 0, sizeof(fq) * npts, st));
    JJS_CUDA(ctx, cudaMemsetAsync(kd.v, 0, sizeof(fq) * npts, st));
    JJS_CUDA(ctx, cudaMemcpyAsync(wire.p, pk, 32 * npts, cudaMemcpyHostToDevice, st));
    const uint8_t* w = wire.p;
    Fields f;
    f.f[0] = WireField{w, (uint32_t)(32 * nk)};
    f.f[1] = nk == 2 ? WireField{w + 32, 64} : WireField{nullptr, 0};
    f.f[2] = f.f[3] = WireField{nullptr, 0};
    k_decode<<<blocks_for(npts), BLOCK, 0, st>>>(f, nk, 0, ks.n_keys, kd.u, kd.v, kd.flags, d.tables(), 3u);
    ctx->launches++;
    if (kw) {
        with_key_width(kw, [&](auto kwc) {
            constexpr int KW = kwc.value;
            k_keyset_bases<KW><<<blocks_for(npts), BLOCK, 0, st>>>(ks.variant, kd.u, kd.v, kd.flags, ks.n_keys, reinterpret_cast<ext*>(bases.p));
            k_keyset_combine<KW><<<blocks_for(npts * keyed_windows(KW) * keyed_groups(KW)), BLOCK, 0, st>>>(reinterpret_cast<const ext*>(bases.p), npts,
                                                                                                            kd.table);
        });
        ctx->launches += 2;
    }
    JJS_CUDA(ctx, cudaGetLastError());
    std::vector<uint8_t> flags;
    if (key_status) {
        flags.resize(npts);
        JJS_CUDA(ctx, cudaMemcpyAsync(flags.data(), kd.flags, npts, cudaMemcpyDeviceToHost, st));
    }
    JJS_CUDA(ctx, cudaStreamSynchronize(st));
    for (size_t k = 0; key_status && k < ks.n_keys; k++) key_status[k] = keyed_key_status(ks.variant, flags.data(), ks.n_keys, k);
    return JJS_SUCCESS;
}

// The layout of jjs_keyset_create_limited for npts key points per device: the widest key-window width KEYED_MAX_W ..
// KEYED_MIN_W whose peak (keyset_peak) is at most `budget` and, on a limited context, at most what the limit leaves on every
// device; else points only (0) if that fits; else -1.  One width serves the whole set on every device.
int pick_key_bits(const jjs_ctx* ctx, size_t npts, size_t budget) {
    size_t room = budget;
    for (const DeviceState& d : ctx->dev)
        if (d.limit) room = std::min(room, d.limit > d.held ? d.limit - d.held : size_t(0));
    for (int kw = KEYED_MAX_W; kw >= KEYED_MIN_W; kw--)
        if (keyset_peak(npts, kw) <= room) return kw;
    return keyset_peak(npts, 0) <= room ? 0 : -1;
}

void keyset_free(jjs_ctx* ctx, KeySet* ks) {
    const size_t npts = (size_t)keyed_points(ks->variant) * ks->n_keys;
    for (size_t k = 0; k < ks->dev.size(); k++) {
        KeySetDev& kd = ks->dev[k];
        if (!kd.u && !kd.v && !kd.flags && !kd.table) continue;
        DeviceState& d = ctx->dev[k];
        cudaSetDevice(d.device);
        cudaDeviceSynchronize();   // work enqueued by the device entry point may still read the tables
        dev_free(d, kd.u, sizeof(fq) * npts); dev_free(d, kd.v, sizeof(fq) * npts); dev_free(d, kd.flags, npts);
        dev_free(d, kd.table, keyset_table_bytes(npts, ks->key_bits));
    }
    delete ks;
}

// Register a key set of kind `kind` at key-window width key_bits (0: points only) on every device: jjs_keyset_create and
// jjs_keyset_create_limited after their argument checks.
int keyset_register(jjs_ctx* ctx, int kind, int key_bits, const uint8_t* pk, size_t n_keys, uint8_t* key_status_or_null, int* keyset_out) {
    KeySet* ks = new (std::nothrow) KeySet();
    if (!ks) return fail(ctx, JJS_ERR_NOMEM, "key set: out of host memory");
    ks->variant = kind;
    ks->key_bits = key_bits;
    ks->n_keys = n_keys;
    ks->dev.resize(ctx->dev.size());
    for (size_t k = 0; k < ctx->dev.size(); k++) {
        int rc = keyset_build(ctx, ctx->dev[k], *ks, ks->dev[k], pk, k == 0 ? key_status_or_null : nullptr);
        if (rc) {
            keyset_free(ctx, ks);
            return rc;
        }
    }
    std::lock_guard<std::mutex> lock(ctx->mu);
    ctx->keysets.push_back(ks);
    *keyset_out = (int)(ctx->keysets.size() - 1);
    return JJS_SUCCESS;
}
// the arguments both create calls refuse
int keyset_check_args(jjs_ctx* ctx, int kind, const uint8_t* pk, size_t n_keys, int* keyset_out) {
    if (kind != JJS_KIND_SINGLE && kind != JJS_KIND_DOUBLE) return fail(ctx, JJS_ERR_ARGUMENT, "key sets hold single or double keys (kind %d)", kind);
    if (n_keys == 0 || n_keys > 0xffffffffu) return fail(ctx, JJS_ERR_ARGUMENT, "n_keys must be in [1, 2^32)");
    if (!pk || !keyset_out) return fail(ctx, JJS_ERR_ARGUMENT, "null buffer");
    return JJS_SUCCESS;
}

// The weights' seed: the caller's 32 bytes, or 32 fresh bytes from the operating system
int rlc_seed(jjs_ctx* ctx, const uint8_t* seed32_or_null, RlcSeed& seed) {
    uint8_t b[32];
    if (seed32_or_null) {
        memcpy(b, seed32_or_null, 32);
    } else {
        for (size_t got = 0; got < 32;) {
            ssize_t r = getrandom(b + got, 32 - got, 0);
            if (r < 0) {
                if (errno == EINTR) continue;
                return fail(ctx, JJS_ERR_ARGUMENT, "getrandom failed: %s", strerror(errno));
            }
            got += (size_t)r;
        }
    }
    for (int i = 0; i < 8; i++) seed.w[i] = (uint32_t)b[4 * i] | (uint32_t)b[4 * i + 1] << 8 | (uint32_t)b[4 * i + 2] << 16 | (uint32_t)b[4 * i + 3] << 24;
    return JJS_SUCCESS;
}
// kinds of the whole-batch entry points; on a context whose jjs_init failed the refusal keeps the reason of the failure
int rlc_check_kind(jjs_ctx* ctx, int kind) {
    if (kind == JJS_KIND_SINGLE || kind == JJS_KIND_DOUBLE) return JJS_SUCCESS;
    if (ctx && ctx->ready) return fail(ctx, JJS_ERR_ARGUMENT, "whole-batch verification takes single or double items (kind %d)", kind);
    return JJS_ERR_ARGUMENT;
}

KeySet* keyset_lookup(jjs_ctx* ctx, int handle) {
    std::lock_guard<std::mutex> lock(ctx->mu);
    return handle >= 0 && (size_t)handle < ctx->keysets.size() ? ctx->keysets[handle] : nullptr;
}

}  // namespace

extern "C" {

#define JJS_API __attribute__((visibility("default")))

}  // extern "C"

namespace {
// jjs_init and jjs_init_limited; limit 0: no limit
int init_context(const int* devices, int n_devices, size_t limit, jjs_ctx** out) {
    if (!out || n_devices < 1 || n_devices > 64) return JJS_ERR_ARGUMENT;
    *out = nullptr;
    jjs_ctx* ctx = new (std::nothrow) jjs_ctx();
    if (!ctx) return JJS_ERR_NOMEM;
    ctx->err[0] = 0;
    *out = ctx;   // on failure the context is returned unusable, only so that the caller can read the reason: no CPU fallback
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count < 1)
        return fail(ctx, JJS_ERR_CUDA, "no CUDA device available: %s", e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    int w = FB_W;
    size_t cap = CHUNK_ITEMS;
    if (limit) {
#if JJS_EQ_V2 || JJS_EQ_PERSISTENT
        return fail(ctx, JJS_ERR_ARGUMENT, "memory-limited contexts are not available in a build with the persistent equation kernel");
#endif
        if (!pick_config(limit, &w, &cap))
            return fail(ctx, JJS_ERR_NOMEM, "a device memory limit of %zu bytes is below the smallest configuration, %zu bytes (%d-bit tables, %zu items per pass)",
                        limit, footprint(FB_W_SMALL, LIMITED_MIN_ITEMS), FB_W_SMALL, LIMITED_MIN_ITEMS);
    }
    ctx->dev.resize(n_devices);
    for (int i = 0; i < n_devices; i++) {
        int ord = devices ? devices[i] : i;
        if (ord < 0 || ord >= count) return fail(ctx, JJS_ERR_ARGUMENT, "device ordinal %d not present (%d devices)", ord, count);
        for (int k = 0; k < i; k++)
            if (ctx->dev[k].device == ord) return fail(ctx, JJS_ERR_ARGUMENT, "device ordinal %d listed twice", ord);
        DeviceState& d = ctx->dev[i];
        d.device = ord;
        if (limit) {
            d.limit = limit;
            configure_limited(d, w, cap);
        }
        int rc = init_device(ctx, d);
        if (rc) {
            if (limit) {   // nothing is left allocated
                for (auto& dv : ctx->dev) free_device(dv);
                ctx->dev.clear();
            }
            return rc;
        }
    }
    ctx->ready = true;
    return JJS_SUCCESS;
}
}  // namespace

extern "C" {

JJS_API int jjs_init(const int* devices, int n_devices, jjs_ctx** out) { return init_context(devices, n_devices, 0, out); }

JJS_API int jjs_init_limited(const int* devices, int n_devices, size_t device_memory_limit, jjs_ctx** out) {
    if (device_memory_limit == 0) {
        if (out) *out = nullptr;
        return JJS_ERR_ARGUMENT;
    }
    return init_context(devices, n_devices, device_memory_limit, out);
}

JJS_API int jjs_memory_info(const jjs_ctx* ctx, int device_index, uint64_t* bytes_held, int* fb_window_bits, uint64_t* items_in_flight) {
    if (!ctx) return JJS_ERR_ARGUMENT;
    if (!ctx->ready || ctx->dev.empty()) return JJS_ERR_CUDA;
    if (device_index < 0 || (size_t)device_index >= ctx->dev.size()) return fail(const_cast<jjs_ctx*>(ctx), JJS_ERR_ARGUMENT, "device_index out of range");
    const DeviceState& d = ctx->dev[device_index];
    if (bytes_held) *bytes_held = d.held;
    if (fb_window_bits) *fb_window_bits = d.fb_w;
    if (items_in_flight) *items_in_flight = d.chunk_items;
    return JJS_SUCCESS;
}

JJS_API void jjs_destroy(jjs_ctx* ctx) {
    if (!ctx) return;
    for (KeySet* ks : ctx->keysets)
        if (ks) keyset_free(ctx, ks);
    for (auto& d : ctx->dev) free_device(d);
    delete ctx;
}

JJS_API const char* jjs_last_error(const jjs_ctx* ctx) { return ctx ? ctx->err : "null context"; }
JJS_API int jjs_device_count(const jjs_ctx* ctx) { return ctx && ctx->ready ? (int)ctx->dev.size() : 0; }
JJS_API uint64_t jjs_launch_count(const jjs_ctx* ctx) { return ctx ? ctx->launches.load() : 0; }

JJS_API int jjs_verify_single(jjs_ctx* ctx, const uint8_t* pk32, const uint8_t* sig64, const uint8_t* msg32, size_t n, uint8_t* status,
                              uint8_t* c32_or_null) {
    return run_part(ctx, wire_part(VAR_SINGLE, pk32, sig64, msg32, n, status, c32_or_null, nullptr));
}
JJS_API int jjs_verify_double(jjs_ctx* ctx, const uint8_t* pk64, const uint8_t* sig96, const uint8_t* msg32, size_t n, uint8_t* status,
                              uint8_t* c32_or_null) {
    return run_part(ctx, wire_part(VAR_DOUBLE, pk64, sig96, msg32, n, status, c32_or_null, nullptr));
}
JJS_API int jjs_verify_vargen(jjs_ctx* ctx, const uint8_t* pk64, const uint8_t* sig64, const uint8_t* msg32, size_t n, uint8_t* status,
                              uint8_t* c32_or_null) {
    return run_part(ctx, wire_part(VAR_VARGEN, pk64, sig64, msg32, n, status, c32_or_null, nullptr));
}
JJS_API int jjs_verify_aggregate(jjs_ctx* ctx, const uint8_t* pks32, const uint32_t* offsets, const uint8_t* sig64, const uint8_t* msg32, size_t n,
                                 uint8_t* status, uint8_t* c32_or_null, uint8_t* aggpk32_or_null) {
    if (ctx && ctx->ready && n && !status) return fail(ctx, JJS_ERR_ARGUMENT, "null buffer");
    return run_part(ctx, aggregate_part(pks32, offsets, offsets, sig64, msg32, n, status, c32_or_null, aggpk32_or_null, nullptr));
}
JJS_API int jjs_verify_batch(jjs_ctx* ctx, const uint8_t* pk32, const uint8_t* sig64, const uint8_t* msg32, size_t n, uint32_t* accept_bitmap) {
    if (ctx && ctx->ready && n && !accept_bitmap) return fail(ctx, JJS_ERR_ARGUMENT, "null buffer");
    return run_part(ctx, wire_part(VAR_SINGLE, pk32, sig64, msg32, n, nullptr, nullptr, accept_bitmap));
}
JJS_API int jjs_verify_batch_double(jjs_ctx* ctx, const uint8_t* pk64, const uint8_t* sig96, const uint8_t* msg32, size_t n, uint32_t* accept_bitmap) {
    if (ctx && ctx->ready && n && !accept_bitmap) return fail(ctx, JJS_ERR_ARGUMENT, "null buffer");
    return run_part(ctx, wire_part(VAR_DOUBLE, pk64, sig96, msg32, n, nullptr, nullptr, accept_bitmap));
}
JJS_API int jjs_verify_batch_vargen(jjs_ctx* ctx, const uint8_t* pk64, const uint8_t* sig64, const uint8_t* msg32, size_t n, uint32_t* accept_bitmap) {
    if (ctx && ctx->ready && n && !accept_bitmap) return fail(ctx, JJS_ERR_ARGUMENT, "null buffer");
    return run_part(ctx, wire_part(VAR_VARGEN, pk64, sig64, msg32, n, nullptr, nullptr, accept_bitmap));
}
JJS_API int jjs_verify_batch_aggregate(jjs_ctx* ctx, const uint8_t* pks32, const uint32_t* offsets, const uint8_t* sig64, const uint8_t* msg32, size_t n,
                                       uint32_t* accept_bitmap) {
    if (ctx && ctx->ready && n && !accept_bitmap) return fail(ctx, JJS_ERR_ARGUMENT, "null buffer");
    return run_part(ctx, aggregate_part(pks32, offsets, offsets, sig64, msg32, n, nullptr, nullptr, nullptr, accept_bitmap));
}
JJS_API int jjs_verify_mixed(jjs_ctx* ctx, const jjs_part* parts, size_t n_parts) {
    JJS_ENTER(ctx);
    if (n_parts && !parts) return fail(ctx, JJS_ERR_ARGUMENT, "null buffer");
    std::vector<Part> hp;
    int rc = parts_from_jjs(ctx, parts, n_parts, PART_WIRE, false, nullptr, nullptr, nullptr, hp);
    return rc ? rc : run_parts(ctx, hp);
}
JJS_API int jjs_status_bitmap_device(jjs_ctx* ctx, int device_index, const uint8_t* d_status, size_t n, uint32_t* d_accept_bitmap, void* cuda_stream) {
    JJS_ENTER(ctx);
    if (device_index < 0 || (size_t)device_index >= ctx->dev.size()) return fail(ctx, JJS_ERR_ARGUMENT, "device_index out of range");
    if (n == 0) return JJS_SUCCESS;
    if (!d_status || !d_accept_bitmap) return fail(ctx, JJS_ERR_ARGUMENT, "null buffer");
    JJS_CUDA(ctx, cudaSetDevice(ctx->dev[device_index].device));
    k_bitmap<<<blocks_for(n), BLOCK, 0, (cudaStream_t)cuda_stream>>>(d_status, n, d_accept_bitmap);
    ctx->launches++;
    JJS_CUDA(ctx, cudaGetLastError());
    return JJS_SUCCESS;
}
JJS_API int jjs_verify_single_device(jjs_ctx* ctx, int device_index, const uint8_t* d_pk32, const uint8_t* d_sig64, const uint8_t* d_msg32,
                                     size_t n, uint8_t* d_status, uint8_t* d_c32_or_null, void* cuda_stream) {
    return device_entry(ctx, device_index, wire_part(VAR_SINGLE, d_pk32, d_sig64, d_msg32, n, d_status, d_c32_or_null, nullptr), cuda_stream);
}
JJS_API int jjs_verify_double_device(jjs_ctx* ctx, int device_index, const uint8_t* d_pk64, const uint8_t* d_sig96, const uint8_t* d_msg32,
                                     size_t n, uint8_t* d_status, uint8_t* d_c32_or_null, void* cuda_stream) {
    return device_entry(ctx, device_index, wire_part(VAR_DOUBLE, d_pk64, d_sig96, d_msg32, n, d_status, d_c32_or_null, nullptr), cuda_stream);
}
JJS_API int jjs_verify_vargen_device(jjs_ctx* ctx, int device_index, const uint8_t* d_pk64, const uint8_t* d_sig64, const uint8_t* d_msg32,
                                     size_t n, uint8_t* d_status, uint8_t* d_c32_or_null, void* cuda_stream) {
    return device_entry(ctx, device_index, wire_part(VAR_VARGEN, d_pk64, d_sig64, d_msg32, n, d_status, d_c32_or_null, nullptr), cuda_stream);
}
JJS_API int jjs_verify_aggregate_device(jjs_ctx* ctx, int device_index, const uint8_t* d_pks32, const uint32_t* d_offsets, const uint32_t* h_offsets,
                                        const uint8_t* d_sig64, const uint8_t* d_msg32, size_t n, uint8_t* d_status, uint8_t* d_c32_or_null,
                                        uint8_t* d_aggpk32_or_null, void* cuda_stream) {
    return device_entry(ctx, device_index,
                        aggregate_part(d_pks32, d_offsets, h_offsets, d_sig64, d_msg32, n, d_status, d_c32_or_null, d_aggpk32_or_null, nullptr), cuda_stream);
}
JJS_API int jjs_verify_ext(jjs_ctx* ctx, int variant, const uint8_t* points_ext160, const uint8_t* u32, const uint8_t* msg32, size_t n,
                           uint8_t* status, uint8_t* c32_or_null) {
    if (ctx && ctx->ready && n && !status) return fail(ctx, JJS_ERR_ARGUMENT, "null buffer");
    return run_part(ctx, Part{PART_TYPED, variant, points_ext160, u32, msg32, nullptr, nullptr, n, status, c32_or_null});
}
JJS_API int jjs_challenge_only(jjs_ctx* ctx, int variant, const uint8_t* pk, const uint8_t* sig, const uint8_t* msg32, size_t n, uint8_t* c32) {
    Part P = wire_part(variant, pk, sig, msg32, n, nullptr, c32, nullptr);
    P.challenge_only = true;
    return run_part(ctx, P);
}
JJS_API int jjs_subgroup_check(jjs_ctx* ctx, const uint8_t* points32, size_t n, int method, uint8_t* out) {
    JJS_ENTER(ctx);
    if (method < 0 || method > 1) return fail(ctx, JJS_ERR_ARGUMENT, "bad method");
    if (n == 0) return JJS_SUCCESS;
    if (!points32 || !out) return fail(ctx, JJS_ERR_ARGUMENT, "null buffer");
    int rc = ensure_scratch(ctx, ctx->dev[0]);
    if (rc) return rc;
    const void* srcs[1] = {points32};
    const size_t bytes[1] = {32 * n};
    return run_small(ctx, "subgroup check", 32 * n, n, srcs, bytes, 1, out, [&](DeviceState& d, uint8_t* in, uint8_t* o) {
        const size_t stride = tab_threads(d, d.chunk_items, 36);
        for (size_t first = 0; first < n; first += stride) {
            size_t cnt = n - first < stride ? n - first : stride;
            k_subgroup_check<<<blocks_for(cnt), BLOCK, 0, d.stream>>>(WireField{in, 32}, first, cnt, method, o, d.tab, stride, d.tables());
            ctx->launches++;
        }
    });
}
JJS_API int jjs_fb_table_check(jjs_ctx* ctx, int which, const uint32_t* entries, size_t n, uint32_t* mismatches) {
    JJS_ENTER(ctx);
    if (which < 0 || which > 1) return fail(ctx, JJS_ERR_ARGUMENT, "bad table");
    if (!mismatches) return fail(ctx, JJS_ERR_ARGUMENT, "null buffer");
    *mismatches = 0;
    if (n == 0) return JJS_SUCCESS;
    if (!entries) return fail(ctx, JJS_ERR_ARGUMENT, "null buffer");
    const void* srcs[1] = {entries};
    const size_t bytes[1] = {4 * n};
    uint32_t count = 0;
    int rc = run_small(ctx, "fixed-base table check", 4 * n, 4, srcs, bytes, 1, &count, [&](DeviceState& d, uint8_t* in, uint8_t* o) {
        cudaMemsetAsync(o, 0, 4, d.stream);
        (d.fb_w == FB_W_SMALL ? k_fb_check<FB_W_SMALL> : k_fb_check<FB_W>)<<<blocks_for(n), BLOCK, 0, d.stream>>>(which ? d.fb_gn : d.fb_g, which, reinterpret_cast<const uint32_t*>(in), (int)n,
                                                         reinterpret_cast<uint32_t*>(o));
        ctx->launches++;
    });
    *mismatches = count;
    return rc;
}
JJS_API int jjs_sign_aggregate_batch(jjs_ctx* ctx, const uint8_t* sk32, const uint32_t* offsets, const uint8_t* rnd32, const uint8_t* msg32, size_t n,
                                     uint8_t* pks32_out, uint8_t* sig64_out) {
    JJS_ENTER(ctx);
    if (n == 0) return JJS_SUCCESS;
    if (!sk32 || !offsets || !rnd32 || !msg32 || !pks32_out || !sig64_out) return fail(ctx, JJS_ERR_ARGUMENT, "null buffer");
    if (offsets[0] != 0) return fail(ctx, JJS_ERR_ARGUMENT, "offsets[0] must be 0");
    for (size_t i = 0; i < n; i++)
        if (offsets[i + 1] < offsets[i]) return fail(ctx, JJS_ERR_ARGUMENT, "offsets must be non-decreasing");
    const size_t K = offsets[n];
    const size_t off_bytes = align_up(4 * (n + 1), 32);
    const void* srcs[4] = {sk32, offsets, rnd32, msg32};
    const size_t bytes[4] = {32 * K, off_bytes, 32 * n, 32 * n};   // the offsets slot is padded; only 4 (n + 1) bytes are meaningful
    // the padded tail of the offsets copy must stay inside the caller's array: copy exactly, pad on the device side
    const size_t exact[4] = {32 * K, 4 * (n + 1), 32 * n, 32 * n};
    DeviceState& d = ctx->dev[0];
    JJS_CUDA(ctx, cudaSetDevice(d.device));
    const size_t in_bytes = bytes[0] + bytes[1] + bytes[2] + bytes[3];
    int rc = ensure_stage(ctx, d, align_up(in_bytes, 256) + 32 * K + 64 * n);
    if (rc) return rc;
    cudaError_t ce = cudaSuccess;
    size_t at = 0;
    for (int i = 0; i < 4 && ce == cudaSuccess; i++) {
        if (exact[i]) ce = cudaMemcpyAsync(d.stage + at, srcs[i], exact[i], cudaMemcpyHostToDevice, d.stream);
        at += bytes[i];
    }
    uint8_t *b = d.stage, *o_pks = d.stage + align_up(in_bytes, 256), *o_sig = o_pks + 32 * K;
    if (ce == cudaSuccess) {
        (d.fb_w == FB_W_SMALL ? k_sign_aggregate<FB_W_SMALL> : k_sign_aggregate<>)<<<blocks_for(n), BLOCK, 0, d.stream>>>(b, reinterpret_cast<uint32_t*>(b + bytes[0]), b + bytes[0] + bytes[1],
                                                              b + bytes[0] + bytes[1] + bytes[2], n, o_pks, o_sig, d.tables());
        ctx->launches++;
        ce = cudaGetLastError();
    }
    if (ce == cudaSuccess && K) ce = cudaMemcpyAsync(pks32_out, o_pks, 32 * K, cudaMemcpyDeviceToHost, d.stream);
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(sig64_out, o_sig, 64 * n, cudaMemcpyDeviceToHost, d.stream);
    cudaError_t e = cudaStreamSynchronize(d.stream);
    if (ce != cudaSuccess) e = ce;
    if (e != cudaSuccess) return fail(ctx, JJS_ERR_CUDA, "sign aggregate batch failed: %s", cudaGetErrorString(e));
    return JJS_SUCCESS;
}
JJS_API int jjs_points_to_ext(jjs_ctx* ctx, const uint8_t* points32, const uint8_t* z_mont32, size_t n, uint8_t* out160) {
    JJS_ENTER(ctx);
    if (n == 0) return JJS_SUCCESS;
    if (!points32 || !z_mont32 || !out160) return fail(ctx, JJS_ERR_ARGUMENT, "null buffer");
    const void* srcs[2] = {points32, z_mont32};
    const size_t bytes[2] = {32 * n, 32 * n};
    return run_small(ctx, "points_to_ext", 64 * n, 160 * n, srcs, bytes, 2, out160, [&](DeviceState& d, uint8_t* in, uint8_t* o) {
        k_points_to_ext<<<blocks_for(n), BLOCK, 0, d.stream>>>(in, in + 32 * n, n, o, d.tables());
        ctx->launches++;
    });
}
JJS_API int jjs_multisig_combine(jjs_ctx* ctx, const uint8_t* pks32, const uint8_t* R32, const uint8_t* S32, const uint8_t* z32, const uint32_t* offsets,
                                 const uint8_t* msg32, size_t n, uint8_t* share_ok_or_null, uint8_t* status, uint32_t* bad_index_or_null,
                                 uint8_t* sig64_or_null) {
    return run_msig(ctx, pks32, R32, S32, z32, offsets, msg32, n, share_ok_or_null, status, bad_index_or_null, sig64_or_null);
}
JJS_API void jjs_profile_enable(jjs_ctx* ctx, int on) {
    if (ctx) ctx->profile = on != 0;
}
JJS_API int jjs_profile_collect(jjs_ctx* ctx, double* stage_ms, uint64_t* stage_count) {
    if (!ctx || !stage_ms || !stage_count) return JJS_ERR_ARGUMENT;
    for (int i = 0; i < JJS_N_STAGES; i++) { stage_ms[i] = 0; stage_count[i] = 0; }
    std::vector<StageRecord> records;
    {
        std::lock_guard<std::mutex> lock(ctx->mu);
        records.swap(ctx->records);
    }
    int rc = JJS_SUCCESS;
    for (auto& r : records) {
        cudaSetDevice(r.device);
        float ms = 0;
        cudaError_t e = cudaEventSynchronize(r.e1);
        if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, r.e0, r.e1);
        cudaEventDestroy(r.e0);
        cudaEventDestroy(r.e1);
        if (e != cudaSuccess) {
            if (rc == JJS_SUCCESS) rc = fail(ctx, JJS_ERR_CUDA, "profile collect: %s", cudaGetErrorString(e));
            continue;
        }
        stage_ms[r.stage] += ms;
        stage_count[r.stage]++;
    }
    return rc;
}
JJS_API int jjs_keyset_create(jjs_ctx* ctx, int kind, const uint8_t* pk, size_t n_keys, uint8_t* key_status_or_null, int* keyset_out) {
    JJS_ENTER(ctx);
    int rc = keyset_check_args(ctx, kind, pk, n_keys, keyset_out);
    return rc ? rc : keyset_register(ctx, kind, KEYED_W, pk, n_keys, key_status_or_null, keyset_out);
}
JJS_API int jjs_keyset_create_limited(jjs_ctx* ctx, int kind, const uint8_t* pk, size_t n_keys, size_t bytes_per_device, uint8_t* key_status_or_null,
                                      int* keyset_out) {
    JJS_ENTER(ctx);
    int rc = keyset_check_args(ctx, kind, pk, n_keys, keyset_out);
    if (rc) return rc;
    if (bytes_per_device == 0) return fail(ctx, JJS_ERR_ARGUMENT, "bytes_per_device must be positive");
    const size_t npts = (size_t)keyed_points(kind) * n_keys;
    const int key_bits = pick_key_bits(ctx, npts, bytes_per_device);
    if (key_bits < 0)
        return fail(ctx, JJS_ERR_NOMEM, "key set: even its decoded points (the smallest layout) need %zu bytes per device while they are built, beyond the "
                    "budget of %zu bytes or what the context's memory limit leaves", keyset_peak(npts, 0), bytes_per_device);
    return keyset_register(ctx, kind, key_bits, pk, n_keys, key_status_or_null, keyset_out);
}
JJS_API int jjs_keyset_info(const jjs_ctx* ctx, int keyset, int* key_window_bits, uint64_t* bytes_per_device) {
    if (!ctx) return JJS_ERR_ARGUMENT;
    if (!ctx->ready || ctx->dev.empty()) return JJS_ERR_CUDA;
    jjs_ctx* c = const_cast<jjs_ctx*>(ctx);   // the handle table's lock and the error message
    const KeySet* ks = keyset_lookup(c, keyset);
    if (!ks) return fail(c, JJS_ERR_ARGUMENT, "unknown key set %d", keyset);
    const size_t npts = (size_t)keyed_points(ks->variant) * ks->n_keys;
    if (key_window_bits) *key_window_bits = ks->key_bits;
    if (bytes_per_device) *bytes_per_device = keyset_point_bytes(npts) + keyset_table_bytes(npts, ks->key_bits);
    return JJS_SUCCESS;
}
JJS_API int jjs_keyset_destroy(jjs_ctx* ctx, int keyset) {
    JJS_ENTER(ctx);
    KeySet* ks = nullptr;
    {
        std::lock_guard<std::mutex> lock(ctx->mu);
        if (keyset >= 0 && (size_t)keyset < ctx->keysets.size()) std::swap(ks, ctx->keysets[keyset]);
    }
    if (!ks) return fail(ctx, JJS_ERR_ARGUMENT, "unknown key set %d", keyset);
    keyset_free(ctx, ks);
    return JJS_SUCCESS;
}
JJS_API int jjs_verify_keyed(jjs_ctx* ctx, int keyset, const uint32_t* key_index, const uint8_t* sig, const uint8_t* msg32, size_t n,
                             uint8_t* status_or_null, uint8_t* c32_or_null, uint32_t* accept_bitmap_or_null) {
    JJS_ENTER(ctx);
    const KeySet* ks = keyset_lookup(ctx, keyset);
    if (!ks) return fail(ctx, JJS_ERR_ARGUMENT, "unknown key set %d", keyset);
    return run_part(ctx, Part{PART_KEYED, ks->variant, reinterpret_cast<const uint8_t*>(key_index), sig, msg32, nullptr, nullptr, n, status_or_null,
                              c32_or_null, nullptr, accept_bitmap_or_null, false, ks});
}
JJS_API int jjs_verify_keyed_device(jjs_ctx* ctx, int device_index, int keyset, const uint32_t* d_key_index, const uint8_t* d_sig,
                                    const uint8_t* d_msg32, size_t n, uint8_t* d_status, uint8_t* d_c32_or_null, void* cuda_stream) {
    JJS_ENTER(ctx);
    const KeySet* ks = keyset_lookup(ctx, keyset);
    if (!ks) return fail(ctx, JJS_ERR_ARGUMENT, "unknown key set %d", keyset);
    return device_entry(ctx, device_index, Part{PART_KEYED, ks->variant, reinterpret_cast<const uint8_t*>(d_key_index), d_sig, d_msg32, nullptr, nullptr, n,
                                                d_status, d_c32_or_null, nullptr, nullptr, false, ks},
                        cuda_stream);
}
JJS_API int jjs_keyset_table_check(jjs_ctx* ctx, int keyset, const uint32_t* entries, size_t n, uint32_t* mismatches) {
    JJS_ENTER(ctx);
    const KeySet* ks = keyset_lookup(ctx, keyset);
    if (!ks) return fail(ctx, JJS_ERR_ARGUMENT, "unknown key set %d", keyset);
    if (ks->key_bits == 0) return fail(ctx, JJS_ERR_ARGUMENT, "key set %d holds points only: no table", keyset);
    if (!mismatches) return fail(ctx, JJS_ERR_ARGUMENT, "null buffer");
    *mismatches = 0;
    if (n == 0) return JJS_SUCCESS;
    if (!entries) return fail(ctx, JJS_ERR_ARGUMENT, "null buffer");
    const void* srcs[1] = {entries};
    const size_t bytes[1] = {4 * n};
    const KeySetDev& kd = ks->dev[0];
    uint32_t count = 0;
    int rc = run_small(ctx, "key-set table check", 4 * n, 4, srcs, bytes, 1, &count, [&](DeviceState& d, uint8_t* in, uint8_t* o) {
        cudaMemsetAsync(o, 0, 4, d.stream);
        with_key_width(ks->key_bits, [&](auto kw) {
            k_keyset_check<kw.value><<<blocks_for(n), BLOCK, 0, d.stream>>>(ks->variant, kd.u, kd.v, kd.flags, ks->n_keys, kd.table,
                                                                          reinterpret_cast<const uint32_t*>(in), n, reinterpret_cast<uint32_t*>(o));
        });
        ctx->launches++;
    });
    *mismatches = count;
    return rc;
}
JJS_API int jjs_verify_all(jjs_ctx* ctx, int kind, const uint8_t* pk, const uint8_t* sig, const uint8_t* msg32, size_t n, const uint8_t* seed32_or_null,
                           int* all_valid) {
    int rc = rlc_check_kind(ctx, kind);
    if (rc) return rc;
    JJS_ENTER(ctx);
    if (!all_valid) return fail(ctx, JJS_ERR_ARGUMENT, "null buffer");
    *all_valid = 0;
    RlcSeed seed;
    rc = rlc_seed(ctx, seed32_or_null, seed);
    if (rc) return rc;
    RlcSink sink;
    Part P{PART_ALL, kind, pk, sig, msg32, nullptr, nullptr, n};
    P.seed = &seed;
    P.sink = &sink;
    rc = run_part(ctx, P);
    if (rc) return rc;
    *all_valid = sink.valid && ext_is_identity(sink.P) ? 1 : 0;
    return JJS_SUCCESS;
}
JJS_API int jjs_verify_all_device(jjs_ctx* ctx, int device_index, int kind, const uint8_t* d_pk, const uint8_t* d_sig, const uint8_t* d_msg32, size_t n,
                                  const uint8_t* seed32_or_null, int* d_all_valid, void* cuda_stream) {
    int rc = rlc_check_kind(ctx, kind);
    if (rc) return rc;
    JJS_ENTER(ctx);
    if (device_index < 0 || (size_t)device_index >= ctx->dev.size()) return fail(ctx, JJS_ERR_ARGUMENT, "device_index out of range");
    if (!d_all_valid) return fail(ctx, JJS_ERR_ARGUMENT, "null buffer");
    RlcSeed seed;
    Part P{PART_ALL, kind, d_pk, d_sig, d_msg32, nullptr, nullptr, n};
    P.seed = &seed;
    rc = validate_part(ctx, P, true);
    if (!rc) rc = rlc_seed(ctx, seed32_or_null, seed);
    if (rc) return rc;
    return run_device_parts(ctx, (size_t)device_index, {P}, (cudaStream_t)cuda_stream, d_all_valid, nullptr);
}
JJS_API int jjs_verify_all_mixed(jjs_ctx* ctx, const jjs_part* parts, size_t n_parts, const uint8_t* seed32_or_null, int* all_valid) {
    JJS_ENTER(ctx);
    if (!all_valid || (n_parts && !parts)) return fail(ctx, JJS_ERR_ARGUMENT, "null buffer");
    *all_valid = 0;
    RlcSeed seed;
    RlcSink sink;
    std::vector<Part> hp;
    int rc = parts_from_jjs(ctx, parts, n_parts, PART_ALL, false, nullptr, &seed, &sink, hp);
    if (!rc) rc = rlc_seed(ctx, seed32_or_null, seed);
    if (!rc) rc = run_parts(ctx, hp);
    if (rc) return rc;
    *all_valid = sink.valid && ext_is_identity(sink.P) ? 1 : 0;
    return JJS_SUCCESS;
}
JJS_API int jjs_verify_all_mixed_device(jjs_ctx* ctx, int device_index, const jjs_part* parts, size_t n_parts, const uint32_t* const* h_offsets_or_null,
                                        const uint8_t* seed32_or_null, int* d_all_valid, void* cuda_stream) {
    JJS_ENTER(ctx);
    if (device_index < 0 || (size_t)device_index >= ctx->dev.size()) return fail(ctx, JJS_ERR_ARGUMENT, "device_index out of range");
    if (!d_all_valid || (n_parts && !parts)) return fail(ctx, JJS_ERR_ARGUMENT, "null buffer");
    RlcSeed seed;
    std::vector<Part> dp;
    int rc = parts_from_jjs(ctx, parts, n_parts, PART_ALL, true, h_offsets_or_null, &seed, nullptr, dp);
    if (!rc) rc = rlc_seed(ctx, seed32_or_null, seed);
    if (rc) return rc;
    return run_device_parts(ctx, (size_t)device_index, dp, (cudaStream_t)cuda_stream, d_all_valid, nullptr);
}
JJS_API int jjs_verify_grouped(jjs_ctx* ctx, const jjs_part* parts, size_t n_parts, const uint8_t* seed32_or_null, uint64_t* fallback_items_or_null) {
    JJS_ENTER(ctx);
    if (n_parts && !parts) return fail(ctx, JJS_ERR_ARGUMENT, "null buffer");
    if (fallback_items_or_null) *fallback_items_or_null = 0;
    RlcSeed seed;
    RlcSink sink;
    std::vector<Part> hp;
    int rc = parts_from_jjs(ctx, parts, n_parts, PART_GROUPED, false, nullptr, &seed, &sink, hp);
    if (!rc) rc = rlc_seed(ctx, seed32_or_null, seed);
    if (!rc) rc = run_parts(ctx, hp);
    if (rc) return rc;
    if (fallback_items_or_null) *fallback_items_or_null = sink.fallback;
    return JJS_SUCCESS;
}
JJS_API int jjs_verify_grouped_device(jjs_ctx* ctx, int device_index, const jjs_part* parts, size_t n_parts, const uint32_t* const* h_offsets_or_null,
                                      const uint8_t* seed32_or_null, uint64_t* d_fallback_items_or_null, void* cuda_stream) {
    JJS_ENTER(ctx);
    if (device_index < 0 || (size_t)device_index >= ctx->dev.size()) return fail(ctx, JJS_ERR_ARGUMENT, "device_index out of range");
    if (n_parts && !parts) return fail(ctx, JJS_ERR_ARGUMENT, "null buffer");
    RlcSeed seed;
    std::vector<Part> dp;
    int rc = parts_from_jjs(ctx, parts, n_parts, PART_GROUPED, true, h_offsets_or_null, &seed, nullptr, dp);
    if (!rc) rc = rlc_seed(ctx, seed32_or_null, seed);
    if (rc) return rc;
    return run_device_parts(ctx, (size_t)device_index, dp, (cudaStream_t)cuda_stream, nullptr,
                            reinterpret_cast<unsigned long long*>(d_fallback_items_or_null));
}
JJS_API int jjs_sign_batch(jjs_ctx* ctx, int variant, const uint8_t* sk32, const uint8_t* rnd32, const uint8_t* gen_scalar32_or_null,
                           const uint8_t* msg32, size_t n, uint8_t* pk_out, uint8_t* sig_out) {
    return run_sign(ctx, variant, sk32, rnd32, gen_scalar32_or_null, msg32, n, pk_out, sig_out);
}

}  // extern "C"
