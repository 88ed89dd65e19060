// primitives_harness.cu — test code, not product: C entry points that run one primitive of radix_sort.cuh or scan.cuh the way
// the pipeline drives it (rs_init_device, rs_plan, rs_sort_pairs / rs_sort_packed, scan_apply / scan_flags / scan_segmax /
// compact_unordered on one stream, device lambdas as functors).  tests/test_primitives_gpu.py compiles it with the product's
// nvcc flags into a temporary directory and compares every result with a plain NumPy reference.
//
// Host-array entry points copy their inputs in, run the primitive once and copy every output back.  The big_* entry points
// generate inputs on the device at the top of each primitive's size contract (n = 2^30 - 1 sorted pairs, n = 2^31 - 1 scanned
// elements, too large for a host reference) and check the result with a plain kernel that shares no logic with the
// primitive; they return the number of mismatches and the first bad index.
//
// Return codes: 0 done; 1 CUDA error (message in msg); 2 not enough free device memory for the case (message in msg);
// 3 bad argument.  Every allocation is freed before returning.
#include "common.cuh"
#include "scan.cuh"
#include "radix_sort.cuh"

#include <string.h>
#include <string>
#include <vector>

using namespace swg;

namespace {

enum { PH_OK = 0, PH_CUDA = 1, PH_NOMEM = 2, PH_ARG = 3 };

struct NoMem {
    size_t need, free_bytes;
};

// one stream and the allocations of one call; the destructor frees them on every way out
struct Run {
    cudaStream_t st = nullptr;
    int sm_count = 0;
    LaunchCounter lc;
    std::vector<void *> allocs;
    Run() {
        SWG_CUDA(cudaSetDevice(0));
        SWG_CUDA(cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, 0));
        rs_init_device();
        SWG_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    }
    ~Run() {
        if (st) cudaStreamSynchronize(st);
        for (void *p : allocs) cudaFree(p);
        if (st) cudaStreamDestroy(st);
    }
    template <class T> T *alloc(size_t n) {
        void *p = nullptr;
        SWG_CUDA(cudaMalloc(&p, sizeof(T) * (n ? n : 1)));
        allocs.push_back(p);
        return reinterpret_cast<T *>(p);
    }
    template <class T> void h2d(T *d, const T *h, size_t n) {
        if (n) SWG_CUDA(cudaMemcpyAsync(d, h, sizeof(T) * n, cudaMemcpyHostToDevice, st));
    }
    template <class T> void d2h(T *h, const T *d, size_t n) {
        if (n) SWG_CUDA(cudaMemcpyAsync(h, d, sizeof(T) * n, cudaMemcpyDeviceToHost, st));
    }
    void sync() {
        SWG_CUDA(cudaGetLastError());
        SWG_CUDA(cudaStreamSynchronize(st));
    }
};

// the large cases need tens of GB: refuse before allocating when the device does not have them free (with 1 GiB to spare)
static void need_free(size_t bytes) {
    SWG_CUDA(cudaSetDevice(0));
    size_t fr = 0, tot = 0;
    SWG_CUDA(cudaMemGetInfo(&fr, &tot));
    if (fr < bytes + ((size_t)1 << 30)) throw NoMem{bytes, fr};
}

template <class F> static int guarded(char *msg, int cap, F body) {
    if (msg && cap > 0) msg[0] = 0;
    try {
        return body();
    } catch (const CudaError &e) {
        if (msg && cap > 0) snprintf(msg, cap, "%s (%s:%d)", cudaGetErrorString(e.code), e.file, e.line);
        return PH_CUDA;
    } catch (const NoMem &e) {
        if (msg && cap > 0)
            snprintf(msg, cap, "needs %.1f GB of device memory, %.1f GB free", e.need / 1e9, e.free_bytes / 1e9);
        return PH_NOMEM;
    }
}

// ---- host-array entry points -------------------------------------------------------------------------------------------------
static int sort_pairs_body(u32 n, int bits, const u64 *keys, const u32 *vals, u64 *keys_out, u32 *vals_out) {
    if (bits < 1 || bits > 64) return PH_ARG;
    Run r;
    u64 *k = r.alloc<u64>(n), *k2 = r.alloc<u64>(n);
    u32 *v = r.alloc<u32>(n), *v2 = r.alloc<u32>(n);
    r.h2d(k, keys, n);
    r.h2d(v, vals, n);
    const RadixSortPlan p = rs_plan(n, 0, bits);
    void *tmp = r.alloc<char>(p.temp_bytes);
    rs_sort_pairs(p, k, k2, v, v2, tmp, r.st, r.sm_count, r.lc);
    r.d2h(keys_out, k, n);
    r.d2h(vals_out, v, n);
    r.sync();
    return PH_OK;
}

// info: c0, passes, pack_pass, timed_passes of the returned PackedSort
static int sort_packed_body(u32 n, int key_bits, int ib, int gap_cb, const u64 *keys, const u32 *vals, u64 *words_out, int *info) {
    if (key_bits < 1 || key_bits > 64 || ib < 1 || ib > 32) return PH_ARG;
    Run r;
    u64 *k = r.alloc<u64>(n), *k2 = r.alloc<u64>(n);
    u32 *v = r.alloc<u32>(n), *v2 = r.alloc<u32>(n);
    r.h2d(k, keys, n);
    r.h2d(v, vals, n);
    const RadixSortPlan p = rs_plan(n, 0, key_bits);
    void *tmp = r.alloc<char>(p.temp_bytes);
    const PackedSort ps = rs_sort_packed(n, key_bits, ib, k, k2, v, v2, tmp, p, r.st, r.sm_count, r.lc, nullptr, nullptr, gap_cb);
    if (n) r.d2h(words_out, ps.packed, n);
    r.sync();
    info[0] = ps.c0;
    info[1] = ps.passes;
    info[2] = ps.pack_pass;
    info[3] = ps.timed_passes;
    return PH_OK;
}

// excl[i], seen[i]: the exclusive prefix and the value out(i, ...) received; calls[i]: how often out(i, ...) ran
static int scan_apply_body(u32 n, const u32 *vals, u32 *excl, u32 *seen, u32 *calls, u32 *total) {
    Run r;
    u32 *in = r.alloc<u32>(n), *ex = r.alloc<u32>(n), *sv = r.alloc<u32>(n), *cl = r.alloc<u32>(n), *tot = r.alloc<u32>(1);
    u32 *tmp = r.alloc<u32>(scan_temp_u32(n));
    r.h2d(in, vals, n);
    SWG_CUDA(cudaMemsetAsync(cl, 0, sizeof(u32) * (n ? n : 1), r.st));
    SWG_CUDA(cudaMemsetAsync(tot, 0xFF, sizeof(u32), r.st));
    const u32 *cin = in;
    scan_apply([=] __device__(u32 i) -> u32 { return cin[i]; },
               [=] __device__(u32 i, u32 e, u32 v) {
                   ex[i] = e;
                   sv[i] = v;
                   atomicAdd(&cl[i], 1u);
               },
               n, tmp, tot, r.st, r.lc);
    r.d2h(excl, ex, n);
    r.d2h(seen, sv, n);
    r.d2h(calls, cl, n);
    r.d2h(total, tot, 1);
    r.sync();
    return PH_OK;
}

static int scan_flags_body(u32 n, const u8 *flags, u32 *excl, u32 *seen, u32 *calls, u32 *total) {
    Run r;
    u8 *f = r.alloc<u8>(n);
    u32 *ex = r.alloc<u32>(n), *sv = r.alloc<u32>(n), *cl = r.alloc<u32>(n), *tot = r.alloc<u32>(1);
    u32 *tmp = r.alloc<u32>(scan_temp_u32(n));
    r.h2d(f, flags, n);
    SWG_CUDA(cudaMemsetAsync(cl, 0, sizeof(u32) * (n ? n : 1), r.st));
    SWG_CUDA(cudaMemsetAsync(tot, 0xFF, sizeof(u32), r.st));
    const u8 *cf = f;
    scan_flags([=] __device__(u32 i) -> bool { return cf[i] != 0; },
               [=] __device__(u32 i, u32 e, u32 v) {
                   ex[i] = e;
                   sv[i] = v;
                   atomicAdd(&cl[i], 1u);
               },
               n, tmp, tot, r.st, r.lc);
    r.d2h(excl, ex, n);
    r.d2h(seen, sv, n);
    r.d2h(calls, cl, n);
    r.d2h(total, tot, 1);
    r.sync();
    return PH_OK;
}

static int scan_segmax_body(u32 n, const u8 *head, const u32 *val, u32 *out, u32 *calls) {
    Run r;
    u8 *h = r.alloc<u8>(n);
    u32 *v = r.alloc<u32>(n), *o = r.alloc<u32>(n), *cl = r.alloc<u32>(n);
    u32 *tmp = r.alloc<u32>(scan_temp_u32(n));
    r.h2d(h, head, n);
    r.h2d(v, val, n);
    SWG_CUDA(cudaMemsetAsync(cl, 0, sizeof(u32) * (n ? n : 1), r.st));
    const u8 *ch = h;
    const u32 *cv = v;
    scan_segmax([=] __device__(u32 i) -> bool { return ch[i] != 0; }, [=] __device__(u32 i) -> u32 { return cv[i]; },
                [=] __device__(u32 i, u32 m) {
                    o[i] = m;
                    atomicAdd(&cl[i], 1u);
                },
                n, tmp, r.st, r.lc);
    r.d2h(out, o, n);
    r.d2h(calls, cl, n);
    r.sync();
    return PH_OK;
}

// slot[i]: the slot out(i, slot) received, NONE32 where out(i, ...) never ran
static int compact_unordered_body(u32 n, const u8 *pred, u32 *slot, u32 *calls, u32 *count) {
    Run r;
    u8 *f = r.alloc<u8>(n);
    u32 *s = r.alloc<u32>(n), *cl = r.alloc<u32>(n), *cnt = r.alloc<u32>(1);
    r.h2d(f, pred, n);
    SWG_CUDA(cudaMemsetAsync(s, 0xFF, sizeof(u32) * (n ? n : 1), r.st));
    SWG_CUDA(cudaMemsetAsync(cl, 0, sizeof(u32) * (n ? n : 1), r.st));
    SWG_CUDA(cudaMemsetAsync(cnt, 0xFF, sizeof(u32), r.st));
    const u8 *cf = f;
    compact_unordered([=] __device__(u32 i) -> bool { return cf[i] != 0; },
                      [=] __device__(u32 i, u32 sl) {
                          s[i] = sl;
                          atomicAdd(&cl[i], 1u);
                      },
                      n, cnt, r.st, r.lc);
    r.d2h(slot, s, n);
    r.d2h(calls, cl, n);
    r.d2h(count, cnt, 1);
    r.sync();
    return PH_OK;
}

// ---- device-generated cases at the top of the size contracts ---------------------------------------------------------------
__device__ __forceinline__ void note_bad(u64 i, unsigned long long *bad, unsigned long long *first) {
    atomicAdd(bad, 1ull);
    atomicMin(first, (unsigned long long)i);
}

// sort: key(i) = i mod m, payload i.  Sorted position of i: r*q + min(r, n mod m) + i div m  (r = i mod m, q = n div m)
__global__ void k_big_sort_gen(u64 *keys, u32 *vals, u32 n, u32 m) {
    for (u64 i = blockIdx.x * (u64)blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        keys[i] = i % m;
        vals[i] = (u32)i;
    }
}
__device__ __forceinline__ u64 big_sort_pos(u64 i, u64 n, u64 m) {
    const u64 r = i % m, q = n / m;
    return r * q + (r < n % m ? r : n % m) + i / m;
}
// pairs: (keys[p], vals[p]); packed (ib > 0): word[p] = (key << ib) | payload
__global__ void k_big_sort_check(const u64 *keys, const u32 *vals, int ib, u32 n, u32 m, unsigned long long *bad,
                                 unsigned long long *first) {
    for (u64 p = blockIdx.x * (u64)blockDim.x + threadIdx.x; p < n; p += (u64)gridDim.x * blockDim.x) {
        const u64 w = keys[p];
        const u64 i = ib ? (w & (((u64)1 << ib) - 1)) : (u64)vals[p];
        const u64 key = ib ? (w >> ib) : w;
        if (i >= n || key != i % m || big_sort_pos(i, n, m) != p) note_bad(p, bad, first);
    }
}

static int big_sort_body(u32 m, int packed, unsigned long long *mismatches, unsigned long long *first_bad) {
    if (m == 0) return PH_ARG;
    const u32 n = RS_VAL_MASK;      // 2^30 - 1: the largest n whose digit counts fit the 30-bit tile status words
    const int bits = 32;            // 4 passes: the digits above i mod m are constant, so one digit's count reaches n
    const int ib = 30;              // packed: c0 == 0 (32 + 30 <= 64), pass 0 packs
    const RadixSortPlan p = rs_plan(n, 0, bits);
    need_free(sizeof(u64) * 2 * (size_t)n + sizeof(u32) * 2 * (size_t)n + p.temp_bytes);
    Run r;
    u64 *k = r.alloc<u64>(n), *k2 = r.alloc<u64>(n);
    u32 *v = r.alloc<u32>(n), *v2 = r.alloc<u32>(n);
    void *tmp = r.alloc<char>(p.temp_bytes);
    unsigned long long *d = r.alloc<unsigned long long>(2), h[2] = {0, ~0ull};
    r.h2d(d, h, 2);
    const u32 grid = (u32)r.sm_count * 8;
    k_big_sort_gen<<<grid, 256, 0, r.st>>>(k, v, n, m);
    if (packed) {
        const PackedSort ps = rs_sort_packed(n, bits, ib, k, k2, v, v2, tmp, p, r.st, r.sm_count, r.lc);
        if (ps.c0 != 0) return PH_ARG;
        k_big_sort_check<<<grid, 256, 0, r.st>>>(ps.packed, nullptr, ib, n, m, d, d + 1);
    } else {
        rs_sort_pairs(p, k, k2, v, v2, tmp, r.st, r.sm_count, r.lc);
        k_big_sort_check<<<grid, 256, 0, r.st>>>(k, v, 0, n, m, d, d + 1);
    }
    r.d2h(h, d, 2);
    r.sync();
    *mismatches = h[0];
    *first_bad = h[1];
    return PH_OK;
}

// scans at n = 2^31 - 1.  Cases:
//   0  scan_apply, v(i) = 2046 if i mod 1024 == 1023 else 0   excl(i) = 2046 (i div 1024); total 4 290 770 946, near 2^32
//   1  scan_apply, v(i) = i mod 3                              excl(i) = 3 (i div 3) + (1 if i mod 3 == 2)
//   2  scan_flags, every flag set                              excl(i) = i
//   3  scan_flags, flag(i) = (i mod 3 == 0)                    excl(i) = ceil(i / 3)
//   4  scan_segmax over hashed heads and values (see seg_head / seg_val), checked by one thread per segment
//   5  compact_unordered, pred(i) = (i mod 3 == 0)             every selected i one slot in [0, count), every slot hit once
__device__ __forceinline__ u32 mix32(u64 x) {
    x ^= x >> 33;
    x *= 0xff51afd7ed558ccdull;
    x ^= x >> 33;
    x *= 0xc4ceb9fe1a85ec53ull;
    x ^= x >> 33;
    return (u32)x;
}
__device__ __forceinline__ u32 big_apply_val(int which, u64 i) { return which == 0 ? (i % 1024 == 1023 ? 2046u : 0u) : (u32)(i % 3); }
__device__ __forceinline__ u64 big_apply_excl(int which, u64 i) {
    if (which == 0) return 2046 * (i / 1024);
    const u64 r = i % 3;
    return 3 * (i / 3) + (r == 2 ? 1 : 0);
}
__device__ __forceinline__ bool big_flag(int which, u64 i) { return which == 2 || i % 3 == 0; }
__device__ __forceinline__ u64 big_flag_excl(int which, u64 i) { return which == 2 ? i : (i + 2) / 3; }

// segments: the input is cut into regions of 2^16 elements (32 tiles of 2048); each region draws how its heads fall —
// at every element, sparse, one in ~4096 (segments over several tiles), on every tile edge, one element off the tile edges,
// or none (a segment crosses the region and its 32-tile look-back rounds) — and how its values fall: hashed over the whole
// u32 range with 0 and 0xFFFFFFFF frequent, descending (the carry into each tile decides the maximum), or heavy-tailed.
__device__ __forceinline__ bool seg_head(u64 i) {
    const u32 rm = mix32((i >> 16) * 2 + 1) % 6, h = mix32(i * 3 + 7);
    switch (rm) {
    case 0: return true;
    case 1: return (h & 7) == 0;
    case 2: return (h & 4095) == 0;
    case 3: return i % SC_TILE == 0;
    case 4: return i % SC_TILE == 1 || i % SC_TILE == SC_TILE - 1;
    default: return false;
    }
}
__device__ __forceinline__ u32 seg_val(u64 i) {
    const u32 vm = mix32((i >> 16) * 2) % 3, h = mix32(i * 5 + 11);
    if (vm == 0) return (h % 97 == 0) ? 0xFFFFFFFFu : (h % 89 == 0) ? 0u : h;
    if (vm == 1) return 0xFFFFFFFFu - (u32)i;
    return h >> (h & 31);
}

__global__ void k_big_scan_gen(int which, u32 n, u32 *val, u8 *flag) {
    for (u64 i = blockIdx.x * (u64)blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        if (which <= 1) val[i] = big_apply_val(which, i);
        else if (which <= 3) flag[i] = big_flag(which, i);
        else if (which == 4) { flag[i] = seg_head(i); val[i] = seg_val(i); }
        else flag[i] = i % 3 == 0;
    }
}
__global__ void k_big_scan_check(int which, u32 n, const u32 *out, u32 total, unsigned long long *bad, unsigned long long *first) {
    for (u64 i = blockIdx.x * (u64)blockDim.x + threadIdx.x; i <= n; i += (u64)gridDim.x * blockDim.x) {
        const u64 want = which <= 1 ? big_apply_excl(which, i) : big_flag_excl(which, i);
        if (i == n) { if (want != total) note_bad(i, bad, first); }  // index n stands for the total
        else if (want != out[i]) note_bad(i, bad, first);
    }
}
// the plain reference of the segmented max: one thread per segment start walks its segment in order
__global__ void k_big_segmax_check(u32 n, const u8 *head, const u32 *val, const u32 *out, unsigned long long *bad,
                                   unsigned long long *first) {
    for (u64 s = blockIdx.x * (u64)blockDim.x + threadIdx.x; s < n; s += (u64)gridDim.x * blockDim.x) {
        if (s != 0 && !head[s]) continue;
        u32 m = val[s];
        for (u64 j = s; j < n && (j == s || !head[j]); j++) {
            m = max(m, val[j]);
            if (out[j] != m) { note_bad(j, bad, first); break; }
        }
    }
}
__global__ void k_big_compact_check(u32 n, const u8 *pred, const u32 *slot, u32 count, u32 *hits, unsigned long long *bad,
                                    unsigned long long *first) {
    for (u64 i = blockIdx.x * (u64)blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const u32 s = slot[i];
        if (!pred[i]) { if (s != NONE32) note_bad(i, bad, first); }
        else if (s >= count) note_bad(i, bad, first);
        else atomicAdd(&hits[s], 1u);
    }
}
__global__ void k_hits_check(u32 count, const u32 *hits, unsigned long long *bad, unsigned long long *first) {
    for (u64 s = blockIdx.x * (u64)blockDim.x + threadIdx.x; s < count; s += (u64)gridDim.x * blockDim.x)
        if (hits[s] != 1) note_bad(s, bad, first);
}

static int big_scan_body(int which, unsigned long long *mismatches, unsigned long long *first_bad, u32 *total) {
    if (which < 0 || which > 5) return PH_ARG;
    const u32 n = 0x7FFFFFFFu; // 2^31 - 1: the context's record limit
    const bool has_val = which <= 1 || which == 4, has_flag = which >= 2;
    need_free(sizeof(u32) * (size_t)n * (has_val ? 2 : 1) + (has_flag ? (size_t)n : 0) + (which == 5 ? sizeof(u32) * ((size_t)n / 3 + 1) : 0) +
              sizeof(u32) * scan_temp_u32(n));
    Run r;
    u32 *val = has_val ? r.alloc<u32>(n) : nullptr, *out = r.alloc<u32>(n), *tot = r.alloc<u32>(1);
    u8 *flag = has_flag ? r.alloc<u8>(n) : nullptr;
    u32 *tmp = r.alloc<u32>(scan_temp_u32(n));
    unsigned long long *d = r.alloc<unsigned long long>(2), h[2] = {0, ~0ull};
    r.h2d(d, h, 2);
    SWG_CUDA(cudaMemsetAsync(out, 0xFF, sizeof(u32) * (size_t)n, r.st)); // an element out() never reached keeps 0xFFFFFFFF
    SWG_CUDA(cudaMemsetAsync(tot, 0xFF, sizeof(u32), r.st));
    const u32 grid = (u32)r.sm_count * 8;
    k_big_scan_gen<<<grid, 256, 0, r.st>>>(which, n, val, flag);
    const u32 *cv = val;
    const u8 *cf = flag;
    if (which <= 1) {
        scan_apply([=] __device__(u32 i) -> u32 { return cv[i]; }, [=] __device__(u32 i, u32 e, u32) { out[i] = e; }, n, tmp, tot, r.st, r.lc);
    } else if (which <= 3) {
        scan_flags([=] __device__(u32 i) -> bool { return cf[i] != 0; }, [=] __device__(u32 i, u32 e, u32) { out[i] = e; }, n, tmp, tot,
                   r.st, r.lc);
    } else if (which == 4) {
        scan_segmax([=] __device__(u32 i) -> bool { return cf[i] != 0; }, [=] __device__(u32 i) -> u32 { return cv[i]; },
                    [=] __device__(u32 i, u32 m) { out[i] = m; }, n, tmp, r.st, r.lc);
    } else {
        compact_unordered([=] __device__(u32 i) -> bool { return cf[i] != 0; }, [=] __device__(u32 i, u32 s) { out[i] = s; }, n, tot, r.st,
                          r.lc);
    }
    u32 total_h = 0;
    r.d2h(&total_h, tot, 1);
    r.sync();
    if (which <= 3) {
        k_big_scan_check<<<grid, 256, 0, r.st>>>(which, n, out, total_h, d, d + 1);
    } else if (which == 4) {
        k_big_segmax_check<<<grid, 256, 0, r.st>>>(n, flag, val, out, d, d + 1);
    } else {
        const u32 want = (n + 2) / 3;
        if (total_h != want) { // index n stands for the count
            *mismatches = 1;
            *first_bad = n;
            *total = total_h;
            return PH_OK;
        }
        u32 *hits = r.alloc<u32>(want);
        SWG_CUDA(cudaMemsetAsync(hits, 0, sizeof(u32) * (size_t)want, r.st));
        k_big_compact_check<<<grid, 256, 0, r.st>>>(n, flag, out, total_h, hits, d, d + 1);
        k_hits_check<<<grid, 256, 0, r.st>>>(total_h, hits, d, d + 1);
    }
    r.d2h(h, d, 2);
    r.sync();
    *mismatches = h[0];
    *first_bad = h[1];
    *total = total_h;
    return PH_OK;
}

} // namespace

extern "C" {

int ph_sort_pairs(u32 n, int bits, const u64 *keys, const u32 *vals, u64 *keys_out, u32 *vals_out, char *msg, int cap) {
    return guarded(msg, cap, [&] { return sort_pairs_body(n, bits, keys, vals, keys_out, vals_out); });
}
int ph_sort_packed(u32 n, int key_bits, int ib, int gap_cb, const u64 *keys, const u32 *vals, u64 *words_out, int *info, char *msg,
                   int cap) {
    return guarded(msg, cap, [&] { return sort_packed_body(n, key_bits, ib, gap_cb, keys, vals, words_out, info); });
}
int ph_scan_apply(u32 n, const u32 *vals, u32 *excl, u32 *seen, u32 *calls, u32 *total, char *msg, int cap) {
    return guarded(msg, cap, [&] { return scan_apply_body(n, vals, excl, seen, calls, total); });
}
int ph_scan_flags(u32 n, const u8 *flags, u32 *excl, u32 *seen, u32 *calls, u32 *total, char *msg, int cap) {
    return guarded(msg, cap, [&] { return scan_flags_body(n, flags, excl, seen, calls, total); });
}
int ph_scan_segmax(u32 n, const u8 *head, const u32 *val, u32 *out, u32 *calls, char *msg, int cap) {
    return guarded(msg, cap, [&] { return scan_segmax_body(n, head, val, out, calls); });
}
int ph_compact_unordered(u32 n, const u8 *pred, u32 *slot, u32 *calls, u32 *count, char *msg, int cap) {
    return guarded(msg, cap, [&] { return compact_unordered_body(n, pred, slot, calls, count); });
}
int ph_big_sort(u32 m, int packed, unsigned long long *mismatches, unsigned long long *first_bad, char *msg, int cap) {
    return guarded(msg, cap, [&] { return big_sort_body(m, packed, mismatches, first_bad); });
}
int ph_big_scan(int which, unsigned long long *mismatches, unsigned long long *first_bad, u32 *total, char *msg, int cap) {
    return guarded(msg, cap, [&] { return big_scan_body(which, mismatches, first_bad, total); });
}

} // extern "C"
