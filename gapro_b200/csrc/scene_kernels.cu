// Scene-level kernels of the gapro_b200 hot path (sm_100a): superpoint densification, floor
// slab, fused containment + occupancy, feature pooling, index-list compaction, per-superpoint
// resolution and the broadcast to points.  HBM-bound integer / compare work: no tensor cores.
#include <cub/cub.cuh>

#include <vector>

#include "common.cuh"

#define FULL_MASK 0xffffffffu

// =============================================================================================
// U — densification (gen_ps_utils.py:312)
// =============================================================================================
__global__ void k_id_minmax(const int64_t* __restrict__ spp_raw, const int64_t* __restrict__ pt_off, int n_scenes,
                            int64_t n, long long* __restrict__ mn, long long* __restrict__ mx) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool valid = i < n;
    int sc = 0;
    long long v = 0;
    if (valid) {
        sc = gapro_find_segment<int64_t>(pt_off, n_scenes, i);
        v = spp_raw[i];
    }
    // warp-uniform scene: reduce first, one atomic pair per warp
    int sc0 = __shfl_sync(FULL_MASK, sc, 0);
    bool uniform = __all_sync(FULL_MASK, valid && sc == sc0);
    if (uniform) {
        long long lo = v, hi = v;
        for (int o = 16; o; o >>= 1) {
            long long a = __shfl_xor_sync(FULL_MASK, lo, o), b = __shfl_xor_sync(FULL_MASK, hi, o);
            lo = a < lo ? a : lo;
            hi = b > hi ? b : hi;
        }
        if ((threadIdx.x & 31) == 0) {
            atomicMin(mn + sc, lo);
            atomicMax(mx + sc, hi);
        }
    } else if (valid) {
        atomicMin(mn + sc, v);
        atomicMax(mx + sc, v);
    }
}

__global__ void k_fill_minmax(long long* mn, long long* mx, int n_scenes) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_scenes) {
        mn[i] = INT64_MAX;
        mx[i] = INT64_MIN;
    }
}

__global__ void k_build_keys(const int64_t* __restrict__ spp_raw, const int64_t* __restrict__ pt_off, int n_scenes,
                             int64_t n, const long long* __restrict__ mn, int id_bits, uint64_t* __restrict__ keys,
                             uint32_t* __restrict__ vals) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int sc = gapro_find_segment<int64_t>(pt_off, n_scenes, i);
    uint64_t rel = (uint64_t)(spp_raw[i] - mn[sc]);
    keys[i] = ((uint64_t)sc << id_bits) | rel;
    vals[i] = (uint32_t)i;
}

__global__ void k_heads(const uint64_t* __restrict__ keys, int64_t n, int32_t* __restrict__ head) {
    int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    head[k] = (k == 0 || keys[k] != keys[k - 1]) ? 1 : 0;
}

__global__ void k_densify_finish(const uint64_t* __restrict__ keys, const int32_t* __restrict__ perm,
                                 const int32_t* __restrict__ head, const int32_t* __restrict__ gsum,
                                 const int64_t* __restrict__ pt_off, int n_scenes, int64_t n, int id_bits,
                                 int32_t* __restrict__ spp_gid, int32_t* __restrict__ seg_off,
                                 int32_t* __restrict__ spp_off_dev) {
    int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    int g = gsum[k] - 1;
    spp_gid[perm[k]] = g;
    if (head[k]) seg_off[g] = (int32_t)k;
    int sc = (int)(keys[k] >> id_bits);
    if (k == pt_off[sc]) spp_off_dev[sc] = g;   // first sorted position of scene sc
    if (k == n - 1) {
        seg_off[g + 1] = (int32_t)n;
        spp_off_dev[n_scenes] = g + 1;
    }
}

struct DensifyWs {
    size_t keys_in, keys_out, vals_in, head, gsum, cub_tmp, cub_bytes, minmax, pt_off, spp_off, total;
};

static DensifyWs densify_layout(int64_t n, int32_t n_scenes) {
    DensifyWs w;
    size_t o = 0;
    auto take = [&](size_t bytes) {
        size_t r = o;
        o += gapro_align_up(bytes, 256);
        return r;
    };
    w.keys_in = take(n * 8);
    w.keys_out = take(n * 8);
    w.vals_in = take(n * 4);
    w.head = take(n * 4);
    w.gsum = take(n * 4);
    size_t sort_bytes = 0, scan_bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (uint64_t*)nullptr, (uint64_t*)nullptr, (uint32_t*)nullptr,
                                    (uint32_t*)nullptr, (int)n, 0, 64);
    cub::DeviceScan::InclusiveSum(nullptr, scan_bytes, (int32_t*)nullptr, (int32_t*)nullptr, (int)n);
    w.cub_bytes = sort_bytes > scan_bytes ? sort_bytes : scan_bytes;
    w.cub_tmp = take(w.cub_bytes);
    w.minmax = take((size_t)n_scenes * 16);
    w.pt_off = take((size_t)(n_scenes + 1) * 8);
    w.spp_off = take((size_t)(n_scenes + 1) * 4);
    w.total = o;
    return w;
}

extern "C" size_t gapro_densify_workspace_bytes(int64_t n_points, int32_t n_scenes) {
    if (n_points <= 0 || n_scenes <= 0) return 0;
    return densify_layout(n_points, n_scenes).total;
}

static int bit_length_u64(uint64_t v) {
    int b = 0;
    while (v) {
        ++b;
        v >>= 1;
    }
    return b;
}

extern "C" int gapro_densify_spp(const int64_t* spp_raw, const int64_t* pt_off, int32_t n_scenes, int32_t* spp_gid,
                                 int32_t* perm, int32_t* seg_off, int32_t* spp_off, void* ws, size_t ws_bytes,
                                 void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GAPRO_REQUIRE(spp_raw && pt_off && spp_gid && perm && seg_off && spp_off && ws, "gapro_densify_spp: null pointer");
    GAPRO_REQUIRE(n_scenes > 0, "gapro_densify_spp: n_scenes must be positive");
    int64_t n = pt_off[n_scenes];
    GAPRO_REQUIRE(pt_off[0] == 0 && n > 0 && n < (int64_t)INT32_MAX, "gapro_densify_spp: bad point offsets (n=%lld)",
                  (long long)n);
    for (int s = 0; s < n_scenes; ++s)
        GAPRO_REQUIRE(pt_off[s + 1] > pt_off[s], "gapro_densify_spp: scene %d has no points", s);
    DensifyWs w = densify_layout(n, n_scenes);
    if (ws_bytes < w.total) {
        gapro_set_error("gapro_densify_spp: workspace %zu < %zu bytes", ws_bytes, w.total);
        return GAPRO_ERR_WORKSPACE;
    }
    char* base = (char*)ws;
    uint64_t* keys_in = (uint64_t*)(base + w.keys_in);
    uint64_t* keys_out = (uint64_t*)(base + w.keys_out);
    uint32_t* vals_in = (uint32_t*)(base + w.vals_in);
    int32_t* head = (int32_t*)(base + w.head);
    int32_t* gsum = (int32_t*)(base + w.gsum);
    long long* mn = (long long*)(base + w.minmax);
    long long* mx = mn + n_scenes;
    int64_t* pt_off_dev = (int64_t*)(base + w.pt_off);
    int32_t* spp_off_dev = (int32_t*)(base + w.spp_off);

    GAPRO_CUDA_TRY(cudaMemcpyAsync(pt_off_dev, pt_off, (size_t)(n_scenes + 1) * 8, cudaMemcpyHostToDevice, stream));
    const int T = 256;
    const unsigned G = (unsigned)((n + T - 1) / T);
    k_fill_minmax<<<(n_scenes + T - 1) / T, T, 0, stream>>>(mn, mx, n_scenes);
    k_id_minmax<<<G, T, 0, stream>>>(spp_raw, pt_off_dev, n_scenes, n, mn, mx);
    GAPRO_KERNEL_CHECK();
    std::vector<long long> h_mm((size_t)2 * n_scenes);
    GAPRO_CUDA_TRY(cudaMemcpyAsync(h_mm.data(), mn, (size_t)n_scenes * 16, cudaMemcpyDeviceToHost, stream));
    GAPRO_CUDA_TRY(cudaStreamSynchronize(stream));
    int id_bits = 1;
    for (int s = 0; s < n_scenes; ++s) {
        uint64_t range = (uint64_t)(h_mm[n_scenes + s] - h_mm[s]);
        int b = bit_length_u64(range);
        if (b > id_bits) id_bits = b;
    }
    int sc_bits = bit_length_u64((uint64_t)(n_scenes - 1));
    GAPRO_REQUIRE(id_bits <= 40 && id_bits + sc_bits <= 64,
                  "gapro_densify_spp: superpoint id range needs %d bits (max 40)", id_bits);

    k_build_keys<<<G, T, 0, stream>>>(spp_raw, pt_off_dev, n_scenes, n, mn, id_bits, keys_in, vals_in);
    GAPRO_KERNEL_CHECK();
    size_t tmp_bytes = w.cub_bytes;
    GAPRO_CUDA_TRY(cub::DeviceRadixSort::SortPairs(base + w.cub_tmp, tmp_bytes, keys_in, keys_out, vals_in,
                                                   (uint32_t*)perm, (int)n, 0, id_bits + sc_bits, stream));
    k_heads<<<G, T, 0, stream>>>(keys_out, n, head);
    GAPRO_KERNEL_CHECK();
    tmp_bytes = w.cub_bytes;
    GAPRO_CUDA_TRY(cub::DeviceScan::InclusiveSum(base + w.cub_tmp, tmp_bytes, head, gsum, (int)n, stream));
    k_densify_finish<<<G, T, 0, stream>>>(keys_out, perm, head, gsum, pt_off_dev, n_scenes, n, id_bits, spp_gid,
                                          seg_off, spp_off_dev);
    GAPRO_KERNEL_CHECK();
    GAPRO_CUDA_TRY(cudaMemcpyAsync(spp_off, spp_off_dev, (size_t)(n_scenes + 1) * 4, cudaMemcpyDeviceToHost, stream));
    GAPRO_CUDA_TRY(cudaStreamSynchronize(stream));
    return GAPRO_OK;
}

// =============================================================================================
// F — floor slab (gen_ps_utils.py:317-326)
// =============================================================================================
__device__ __forceinline__ unsigned long long dbl_to_ordered(double d) {
    unsigned long long b = (unsigned long long)__double_as_longlong(d);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double ordered_to_dbl(unsigned long long u) {
    unsigned long long b = (u >> 63) ? (u & 0x7fffffffffffffffull) : ~u;
    return __longlong_as_double((long long)b);
}

__global__ void k_extent_init(unsigned long long* scratch, int n_scenes) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_scenes * 6) scratch[i] = (i % 6) < 3 ? ~0ull : 0ull;
}

// one block handles a chunk of 4096 consecutive points; scene looked up per point
__global__ void k_extent(const double* __restrict__ xyz, const int64_t* __restrict__ pt_off, int n_scenes, int64_t n,
                         unsigned long long* __restrict__ scratch) {
    const int PER = 16;
    int64_t base = ((int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31)) * PER;   // warp's first point
    int lane = threadIdx.x & 31;
    int cur = -1;
    unsigned long long lo[3], hi[3];
    for (int it = 0; it < PER; ++it) {
        int64_t i = base + (int64_t)it * 32 + lane;
        bool valid = i < n;
        int sc = valid ? gapro_find_segment<int64_t>(pt_off, n_scenes, i) : -2;
        if (sc != cur) {
            if (cur >= 0)
                for (int d = 0; d < 3; ++d) {
                    atomicMin(scratch + cur * 6 + d, lo[d]);
                    atomicMax(scratch + cur * 6 + 3 + d, hi[d]);
                }
            cur = sc;
            for (int d = 0; d < 3; ++d) {
                lo[d] = ~0ull;
                hi[d] = 0ull;
            }
        }
        if (valid)
            for (int d = 0; d < 3; ++d) {
                unsigned long long u = dbl_to_ordered(xyz[3 * i + d]);
                lo[d] = u < lo[d] ? u : lo[d];
                hi[d] = u > hi[d] ? u : hi[d];
            }
    }
    // warp-level combine when the whole warp ended in the same scene
    int c0 = __shfl_sync(FULL_MASK, cur, 0);
    if (__all_sync(FULL_MASK, cur == c0) && c0 >= 0) {
        for (int d = 0; d < 3; ++d)
            for (int o = 16; o; o >>= 1) {
                unsigned long long a = __shfl_xor_sync(FULL_MASK, lo[d], o), b = __shfl_xor_sync(FULL_MASK, hi[d], o);
                lo[d] = a < lo[d] ? a : lo[d];
                hi[d] = b > hi[d] ? b : hi[d];
            }
        if (lane == 0)
            for (int d = 0; d < 3; ++d) {
                atomicMin(scratch + c0 * 6 + d, lo[d]);
                atomicMax(scratch + c0 * 6 + 3 + d, hi[d]);
            }
    } else if (cur >= 0) {
        for (int d = 0; d < 3; ++d) {
            atomicMin(scratch + cur * 6 + d, lo[d]);
            atomicMax(scratch + cur * 6 + 3 + d, hi[d]);
        }
    }
}

__global__ void k_floor_write(const unsigned long long* __restrict__ scratch, const int32_t* __restrict__ box_off,
                              int n_scenes, double ground_h, double* __restrict__ boxes, double* __restrict__ vol) {
    int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_scenes) return;
    double lo[3], hi[3];
    for (int d = 0; d < 3; ++d) {
        lo[d] = ordered_to_dbl(scratch[s * 6 + d]);
        hi[d] = ordered_to_dbl(scratch[s * 6 + 3 + d]);
    }
    int b = box_off[s + 1] - 1;
    double fb[6] = {lo[0], lo[1], lo[2], hi[0], hi[1], __dadd_rn(lo[2], ground_h)};
    double v = 1.0;
    for (int d = 0; d < 3; ++d) {
        boxes[6 * b + d] = fb[d];
        boxes[6 * b + 3 + d] = fb[3 + d];
        double e = __dsub_rn(fb[3 + d], fb[d]);
        e = e < 0.001 ? 0.001 : e;
        v = __dmul_rn(v, e);
    }
    vol[b] = v;
}

extern "C" int gapro_floor_boxes(const double* xyz, const int64_t* pt_off_dev, const int32_t* box_off_dev,
                                 int32_t n_scenes, int64_t n_points, double ground_h, double* boxes,
                                 double* boxes_vol, uint64_t* scratch, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GAPRO_REQUIRE(xyz && pt_off_dev && box_off_dev && boxes && boxes_vol && scratch, "gapro_floor_boxes: null pointer");
    GAPRO_REQUIRE(n_scenes > 0 && n_points > 0, "gapro_floor_boxes: empty batch");
    k_extent_init<<<(n_scenes * 6 + 255) / 256, 256, 0, stream>>>((unsigned long long*)scratch, n_scenes);
    const int T = 256, PER = 16;
    unsigned G = (unsigned)((n_points + (int64_t)T * PER - 1) / ((int64_t)T * PER));
    k_extent<<<G, T, 0, stream>>>(xyz, pt_off_dev, n_scenes, n_points, (unsigned long long*)scratch);
    k_floor_write<<<(n_scenes + 127) / 128, 128, 0, stream>>>((const unsigned long long*)scratch, box_off_dev, n_scenes,
                                                               ground_h, boxes, boxes_vol);
    GAPRO_KERNEL_CHECK();
    return GAPRO_OK;
}

// =============================================================================================
// A + A' — containment + occupancy (gen_ps_utils.py:349-351, 359-363), one warp per superpoint
// =============================================================================================
// One warp per superpoint.  Pass 1 gathers the superpoint's points and reduces their extent; pass 2
// lets lane b classify box 32w+b against that extent: "contains" (every point inside: count = size)
// and "disjoint" (count = 0) are decided without touching the points again — exact, because the
// containment test is a conjunction of per-axis interval tests — and only boxes that cut through the
// superpoint are counted point by point with a warp ballot.
// Warp-wide min / max of doubles with two integer REDUX operations each: doubles are mapped to
// order-preserving uint64 keys, the high words are reduced first, then the low words among the
// lanes that hold the winning high word.  Exact (no floating-point arithmetic involved).
__device__ __forceinline__ unsigned long long dbl_key(double d) {
    unsigned long long b = (unsigned long long)__double_as_longlong(d);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double key_dbl(unsigned long long u) {
    unsigned long long b = (u >> 63) ? (u & 0x7fffffffffffffffull) : ~u;
    return __longlong_as_double((long long)b);
}
__device__ __forceinline__ double warp_min(double v) {
    const unsigned long long u = dbl_key(v);
    const unsigned hi = (unsigned)(u >> 32), lo = (unsigned)u;
    const unsigned mhi = __reduce_min_sync(FULL_MASK, hi);
    const unsigned mlo = __reduce_min_sync(FULL_MASK, hi == mhi ? lo : 0xffffffffu);
    return key_dbl(((unsigned long long)mhi << 32) | mlo);
}
__device__ __forceinline__ double warp_max(double v) {
    const unsigned long long u = dbl_key(v);
    const unsigned hi = (unsigned)(u >> 32), lo = (unsigned)u;
    const unsigned mhi = __reduce_max_sync(FULL_MASK, hi);
    const unsigned mlo = __reduce_max_sync(FULL_MASK, hi == mhi ? lo : 0u);
    return key_dbl(((unsigned long long)mhi << 32) | mlo);
}

// scene of global superpoint g: one coalesced load of the offsets + a ballot instead of a chain of
// dependent binary-search loads
__device__ __forceinline__ int warp_find_scene(const int32_t* __restrict__ spp_off, int n_scenes, int g, int lane) {
    int sc = -1;
    for (int base = 0; base <= n_scenes; base += 32) {
        const int i = base + lane;
        const bool le = (i <= n_scenes) && (spp_off[i] <= g);
        sc += __popc(__ballot_sync(FULL_MASK, le));
    }
    return sc;
}

template <int WORDS>
__global__ void __launch_bounds__(256)
k_occupancy(const double* __restrict__ xyz, const int32_t* __restrict__ perm, const int32_t* __restrict__ seg_off,
            const int32_t* __restrict__ spp_off, const int32_t* __restrict__ box_off, const double* __restrict__ boxes,
            int n_scenes, int s_total, double margin, float thresh, uint32_t* __restrict__ occ_bits,
            int32_t* __restrict__ n_bbs, int32_t* __restrict__ cnt_in, int32_t* __restrict__ excl_cnt,
            int32_t* __restrict__ inter_cnt) {
    const int lane = threadIdx.x & 31;
    const int g = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (g >= s_total) return;
    const int start = seg_off[g], end = seg_off[g + 1];
    const int cnt = end - start;
    const int sc = warp_find_scene(spp_off, n_scenes, g, lane);
    const int b0 = box_off[sc];
    const int nb = box_off[sc + 1] - b0;

    // pass 1: extent of the superpoint; the first 32 points stay in registers
    double px = 0, py = 0, pz = 0;
    const bool pvalid = start + lane < end;
    if (pvalid) {
        const int64_t p = perm[start + lane];
        px = xyz[3 * p];
        py = xyz[3 * p + 1];
        pz = xyz[3 * p + 2];
    }
    const double INF = __longlong_as_double(0x7ff0000000000000LL);
    double lx = pvalid ? px : INF, ly = pvalid ? py : INF, lz = pvalid ? pz : INF;
    double hx = pvalid ? px : -INF, hy = pvalid ? py : -INF, hz = pvalid ? pz : -INF;
    for (int k = start + 32 + lane; k < end; k += 32) {
        const int64_t p = perm[k];
        const double x = xyz[3 * p], y = xyz[3 * p + 1], z = xyz[3 * p + 2];
        lx = fmin(lx, x); ly = fmin(ly, y); lz = fmin(lz, z);
        hx = fmax(hx, x); hy = fmax(hy, y); hz = fmax(hz, z);
    }
    lx = warp_min(lx); ly = warp_min(ly); lz = warp_min(lz);
    hx = warp_max(hx); hy = warp_max(hy); hz = warp_max(hz);

    const float fcnt = (float)cnt;
    uint32_t bits[WORDS];
    int total = 0;
#pragma unroll
    for (int w = 0; w < WORDS; ++w) {
        const int b = 32 * w + lane;
        int count = 0;
        bool partial = false;
        if (b < nb) {
            const double* bx = boxes + 6 * (size_t)(b0 + b);
            // margins in float64 on the float64 boxes (gen_ps_utils.py:350)
            const double l0 = __dsub_rn(bx[0], margin), l1 = __dsub_rn(bx[1], margin), l2 = __dsub_rn(bx[2], margin);
            const double h0 = __dadd_rn(bx[3], margin), h1 = __dadd_rn(bx[4], margin), h2 = __dadd_rn(bx[5], margin);
            const bool contains = lx >= l0 && ly >= l1 && lz >= l2 && hx <= h0 && hy <= h1 && hz <= h2;
            const bool disjoint = hx < l0 || hy < l1 || hz < l2 || lx > h0 || ly > h1 || lz > h2;
            count = contains ? cnt : 0;
            partial = !contains && !disjoint;
        }
        uint32_t pmask = __ballot_sync(FULL_MASK, partial);
        while (pmask) {
            const int bb = __ffs(pmask) - 1;
            pmask &= pmask - 1;
            const double* bx = boxes + 6 * (size_t)(b0 + 32 * w + bb);      // warp-uniform address
            const double l0 = __dsub_rn(bx[0], margin), l1 = __dsub_rn(bx[1], margin), l2 = __dsub_rn(bx[2], margin);
            const double h0 = __dadd_rn(bx[3], margin), h1 = __dadd_rn(bx[4], margin), h2 = __dadd_rn(bx[5], margin);
            bool in = pvalid && px >= l0 && py >= l1 && pz >= l2 && px <= h0 && py <= h1 && pz <= h2;
            int c = __popc(__ballot_sync(FULL_MASK, in));
            for (int base = start + 32; base < end; base += 32) {
                const int k = base + lane;
                in = false;
                if (k < end) {
                    const int64_t p = perm[k];
                    const double x = xyz[3 * p], y = xyz[3 * p + 1], z = xyz[3 * p + 2];
                    in = x >= l0 && y >= l1 && z >= l2 && x <= h0 && y <= h1 && z <= h2;
                }
                c += __popc(__ballot_sync(FULL_MASK, in));
            }
            if (lane == bb) count = c;
        }
        const bool occ = (b < nb) && (__fdiv_rn((float)count, fcnt) >= thresh);
        bits[w] = __ballot_sync(FULL_MASK, occ);
        total += __popc(bits[w]);
        if (cnt_in) cnt_in[((size_t)g * WORDS + w) * 32 + lane] = count;
        if (lane == 0) occ_bits[(size_t)g * WORDS + w] = bits[w];
    }
    if (lane == 0) {
        n_bbs[g] = total;
        if (total == 1) {
#pragma unroll
            for (int w = 0; w < WORDS; ++w)
                if (bits[w]) atomicAdd(excl_cnt + b0 + 32 * w + __ffs(bits[w]) - 1, 1);
        } else if (total >= 2) {
            const int stride = 32 * WORDS;
            int32_t* ic = inter_cnt + (size_t)sc * stride * stride;
#pragma unroll
            for (int w1 = 0; w1 < WORDS; ++w1) {
                uint32_t m1 = bits[w1];
                while (m1) {
                    int i1 = 32 * w1 + __ffs(m1) - 1;
                    m1 &= m1 - 1;
#pragma unroll
                    for (int w2 = 0; w2 < WORDS; ++w2) {
                        if (w2 < w1) continue;
                        uint32_t m2 = bits[w2];
                        while (m2) {
                            int i2 = 32 * w2 + __ffs(m2) - 1;
                            m2 &= m2 - 1;
                            if (i2 > i1) atomicAdd(ic + (size_t)i1 * stride + i2, 1);
                        }
                    }
                }
            }
        }
    }
}

extern "C" int gapro_occupancy(const double* xyz, const int32_t* perm, const int32_t* seg_off,
                               const int32_t* spp_off_dev, const int32_t* box_off_dev, const double* boxes,
                               int32_t n_scenes, int32_t s_total, int32_t n_boxes, int32_t words, double margin,
                               float thresh, uint32_t* occ_bits, int32_t* n_bbs, int32_t* cnt_in, int32_t* excl_cnt,
                               int32_t* inter_cnt, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GAPRO_REQUIRE(xyz && perm && seg_off && spp_off_dev && box_off_dev && boxes && occ_bits && n_bbs && excl_cnt &&
                      inter_cnt,
                  "gapro_occupancy: null pointer");
    GAPRO_REQUIRE(n_scenes > 0 && s_total > 0 && n_boxes > 0, "gapro_occupancy: empty batch");
    GAPRO_REQUIRE(words == 1 || words == 2 || words == 4 || words == 8,
                  "gapro_occupancy: words must be 1, 2, 4 or 8 (got %d; at most 256 boxes per scene)", words);
    GAPRO_CUDA_TRY(cudaMemsetAsync(excl_cnt, 0, (size_t)n_boxes * 4, stream));
    GAPRO_CUDA_TRY(cudaMemsetAsync(inter_cnt, 0, (size_t)n_scenes * 32 * words * 32 * words * 4, stream));
    const int T = 256, WPB = T / 32;
    unsigned G = (unsigned)((s_total + WPB - 1) / WPB);
#define LAUNCH_OCC(W)                                                                                              \
    k_occupancy<W><<<G, T, 0, stream>>>(xyz, perm, seg_off, spp_off_dev, box_off_dev, boxes, n_scenes, s_total,    \
                                        margin, thresh, occ_bits, n_bbs, cnt_in, excl_cnt, inter_cnt)
    switch (words) {
        case 1: LAUNCH_OCC(1); break;
        case 2: LAUNCH_OCC(2); break;
        case 4: LAUNCH_OCC(4); break;
        default: LAUNCH_OCC(8); break;
    }
#undef LAUNCH_OCC
    GAPRO_KERNEL_CHECK();
    return GAPRO_OK;
}

// =============================================================================================
// Source point of the "dist" rule.  gen_pseudo_label computes, for the points that lie in several
// boxes, point_inds = nonzero(bb_occupancy[num_BBs_per_point > 1])[0] (gen_ps_utils.py:516) - row
// numbers of the COMPACTED sub-matrix - and then reads coords_float[point_inds] (:526): the k-th
// multi-box point of a scene is measured from the coordinates of point k of that scene.  To return what
// the reference returns, dist_src[p] = scene base + (number of multi-box points before p in the scene)
// for multi-box points, p otherwise: per-point flag, exclusive scan, subtract the scan at the scene base.
// =============================================================================================
__device__ __forceinline__ int find_scene_pt(const int64_t* __restrict__ pt_off, int n_scenes, int64_t p) {
    int lo = 0, hi = n_scenes;            // pt_off[lo] <= p < pt_off[hi]
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (pt_off[mid] <= p) lo = mid; else hi = mid;
    }
    return lo;
}

__global__ void __launch_bounds__(256)
k_multibox_flag(const double* __restrict__ xyz, const int64_t* __restrict__ pt_off, const int32_t* __restrict__ box_off,
                const float* __restrict__ boxes, int n_scenes, int64_t n, int32_t* __restrict__ flag) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const int sc = find_scene_pt(pt_off, n_scenes, p);
    const double x = xyz[3 * p], y = xyz[3 * p + 1], z = xyz[3 * p + 2];
    const float MARGIN = 0.005f;
    int n_in = 0;
    for (int b = box_off[sc]; b < box_off[sc + 1]; ++b) {
        const float* bx = boxes + 6 * (size_t)b;
        n_in += x >= (double)__fsub_rn(bx[0], MARGIN) && y >= (double)__fsub_rn(bx[1], MARGIN) &&
                z >= (double)__fsub_rn(bx[2], MARGIN) && x <= (double)__fadd_rn(bx[3], MARGIN) &&
                y <= (double)__fadd_rn(bx[4], MARGIN) && z <= (double)__fadd_rn(bx[5], MARGIN);
    }
    flag[p] = n_in > 1;
}

__global__ void __launch_bounds__(256)
k_multibox_src(const int32_t* __restrict__ flag, const int32_t* __restrict__ scan, const int64_t* __restrict__ pt_off,
               int n_scenes, int64_t n, int32_t* __restrict__ dist_src) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const int64_t base = pt_off[find_scene_pt(pt_off, n_scenes, p)];
    dist_src[p] = flag[p] ? (int32_t)(base + (scan[p] - scan[base])) : (int32_t)p;
}

struct MultiboxWs {
    size_t flag, scan, cub_tmp, cub_bytes, total;
};
static MultiboxWs multibox_layout(int64_t n) {
    MultiboxWs w;
    w.flag = 0;
    w.scan = gapro_align_up((size_t)n * 4, 256);
    w.cub_tmp = w.scan + gapro_align_up((size_t)n * 4, 256);
    w.cub_bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, w.cub_bytes, (int32_t*)nullptr, (int32_t*)nullptr, (int)n);
    w.total = w.cub_tmp + gapro_align_up(w.cub_bytes, 256);
    return w;
}

extern "C" size_t gapro_multibox_workspace_bytes(int64_t n_points) {
    if (n_points <= 0) return 0;
    return multibox_layout(n_points).total;
}

extern "C" int gapro_multibox_sources(const double* xyz, const int64_t* pt_off_dev, const int32_t* box_off_dev,
                                      const float* boxes, int32_t n_scenes, int64_t n_points, int32_t* dist_src,
                                      void* ws, size_t ws_bytes, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GAPRO_REQUIRE(xyz && pt_off_dev && box_off_dev && boxes && dist_src && ws, "gapro_multibox_sources: null pointer");
    GAPRO_REQUIRE(n_scenes > 0 && n_points > 0 && n_points < (int64_t)INT32_MAX, "gapro_multibox_sources: empty batch");
    const MultiboxWs w = multibox_layout(n_points);
    if (ws_bytes < w.total) {
        gapro_set_error("gapro_multibox_sources: workspace %zu < %zu bytes", ws_bytes, w.total);
        return GAPRO_ERR_WORKSPACE;
    }
    char* base = (char*)ws;
    int32_t* flag = (int32_t*)(base + w.flag);
    int32_t* scan = (int32_t*)(base + w.scan);
    const int T = 256;
    const unsigned G = (unsigned)((n_points + T - 1) / T);
    k_multibox_flag<<<G, T, 0, stream>>>(xyz, pt_off_dev, box_off_dev, boxes, n_scenes, n_points, flag);
    GAPRO_KERNEL_CHECK();
    size_t tmp = w.cub_bytes;
    GAPRO_CUDA_TRY(cub::DeviceScan::ExclusiveSum(base + w.cub_tmp, tmp, flag, scan, (int)n_points, stream));
    k_multibox_src<<<G, T, 0, stream>>>(flag, scan, pt_off_dev, n_scenes, n_points, dist_src);
    GAPRO_KERNEL_CHECK();
    return GAPRO_OK;
}

// =============================================================================================
// Heuristic labelers (SURVEY section 8f): gen_pseudo_label_box2mask (gen_ps_utils.py:242-290) and
// gen_pseudo_label (:485-569) + spp_align_label (:99-129).  Per-POINT containment in the instance
// boxes (margins evaluated in float32, the dtype of instance_box there), per-point rule for points
// in several boxes (smallest volume / nearest centre / none), then a majority vote per superpoint
// over the labels {background, box 0, box 1, ...} (first maximum wins), optionally restricted to
// boxes that hold >= occ_thresh of the superpoint.  One warp per superpoint, same extent
// pre-classification as k_occupancy.
// =============================================================================================
template <int WORDS>
__global__ void __launch_bounds__(256)
k_heuristic(const double* __restrict__ xyz, const int32_t* __restrict__ perm, const int32_t* __restrict__ seg_off,
            const int32_t* __restrict__ spp_off, const int32_t* __restrict__ box_off, const float* __restrict__ boxes,
            const float* __restrict__ vol, const int32_t* __restrict__ dist_src, int n_scenes, int s_total, int rule,
            int spp_align, float occ_thresh, int32_t* __restrict__ inst_spp, int32_t* __restrict__ inst_pt) {
    const int lane = threadIdx.x & 31;
    const int g = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (g >= s_total) return;
    const int start = seg_off[g], end = seg_off[g + 1];
    const int cnt = end - start;
    const int sc = warp_find_scene(spp_off, n_scenes, g, lane);
    const int b0 = box_off[sc];
    const int nb = box_off[sc + 1] - b0;
    const float MARGIN = 0.005f;
    // extent of the superpoint
    const double INF = __longlong_as_double(0x7ff0000000000000LL);
    double lx = INF, ly = INF, lz = INF, hx = -INF, hy = -INF, hz = -INF;
    for (int k = start + lane; k < end; k += 32) {
        const int64_t p = perm[k];
        const double x = xyz[3 * p], y = xyz[3 * p + 1], z = xyz[3 * p + 2];
        lx = fmin(lx, x); ly = fmin(ly, y); lz = fmin(lz, z);
        hx = fmax(hx, x); hy = fmax(hy, y); hz = fmax(hz, z);
    }
    lx = warp_min(lx); ly = warp_min(ly); lz = warp_min(lz);
    hx = warp_max(hx); hy = warp_max(hy); hz = warp_max(hz);
    // classify the boxes: lane b of word w looks at box 32w+b
    uint32_t all_in[WORDS], cuts[WORDS];
#pragma unroll
    for (int w = 0; w < WORDS; ++w) {
        const int b = 32 * w + lane;
        bool contains = false, partial = false;
        if (b < nb) {
            const float* bx = boxes + 6 * (size_t)(b0 + b);
            const double l0 = (double)__fsub_rn(bx[0], MARGIN), l1 = (double)__fsub_rn(bx[1], MARGIN),
                         l2 = (double)__fsub_rn(bx[2], MARGIN);
            const double h0 = (double)__fadd_rn(bx[3], MARGIN), h1 = (double)__fadd_rn(bx[4], MARGIN),
                         h2 = (double)__fadd_rn(bx[5], MARGIN);
            contains = lx >= l0 && ly >= l1 && lz >= l2 && hx <= h0 && hy <= h1 && hz <= h2;
            const bool disjoint = hx < l0 || hy < l1 || hz < l2 || lx > h0 || ly > h1 || lz > h2;
            partial = !contains && !disjoint;
        }
        all_in[w] = __ballot_sync(FULL_MASK, contains);
        cuts[w] = __ballot_sync(FULL_MASK, partial);
    }
    int votes[WORDS], inside[WORDS];      // lane b of word w: votes / points inside for box 32w+b
#pragma unroll
    for (int w = 0; w < WORDS; ++w) votes[w] = inside[w] = 0;
    int votes_bg = 0;
    for (int base = start; base < end; base += 32) {
        const int k = base + lane;
        const bool valid = k < end;
        int64_t p = 0;
        double x = 0, y = 0, z = 0;
        if (valid) {
            p = perm[k];
            x = xyz[3 * p];
            y = xyz[3 * p + 1];
            z = xyz[3 * p + 2];
        }
        // per-point containment mask
        uint32_t mask[WORDS];
        int n_in = 0;
#pragma unroll
        for (int w = 0; w < WORDS; ++w) {
            uint32_t m = valid ? all_in[w] : 0u;
            uint32_t c = cuts[w];
            while (c) {
                const int bb = __ffs(c) - 1;
                c &= c - 1;
                const float* bx = boxes + 6 * (size_t)(b0 + 32 * w + bb);
                const bool in = valid && x >= (double)__fsub_rn(bx[0], MARGIN) && y >= (double)__fsub_rn(bx[1], MARGIN) &&
                                z >= (double)__fsub_rn(bx[2], MARGIN) && x <= (double)__fadd_rn(bx[3], MARGIN) &&
                                y <= (double)__fadd_rn(bx[4], MARGIN) && z <= (double)__fadd_rn(bx[5], MARGIN);
                m |= (uint32_t)in << bb;
            }
            mask[w] = m;
            n_in += __popc(m);
        }
        // label: 0 background, b+1 box b, (rule "none": several boxes -> background for the vote, -2 per point)
        int label = 0;
        if (n_in == 1) {
#pragma unroll
            for (int w = 0; w < WORDS; ++w)
                if (mask[w]) label = 32 * w + __ffs(mask[w]);
        } else if (n_in > 1 && rule != 2) {
            double best = 0.0;
            int arg = -1;
            double qx = x, qy = y, qz = z;
            if (rule == 1) {
                // gen_ps_utils.py:526 measures the k-th multi-box point of the scene from the coordinates of
                // point k (it indexes coords_float with row numbers of the compacted sub-matrix): dist_src
                const int64_t q = dist_src[p];
                qx = xyz[3 * q];
                qy = xyz[3 * q + 1];
                qz = xyz[3 * q + 2];
            }
#pragma unroll
            for (int w = 0; w < WORDS; ++w) {
                uint32_t m = mask[w];
                while (m) {
                    const int b = 32 * w + __ffs(m) - 1;
                    m &= m - 1;
                    double key;
                    if (rule == 0) {
                        key = (double)vol[b0 + b];
                    } else {
                        const float* bx = boxes + 6 * (size_t)(b0 + b);
                        const double cx = (double)__fdiv_rn(__fadd_rn(bx[0], bx[3]), 2.0f);
                        const double cy = (double)__fdiv_rn(__fadd_rn(bx[1], bx[4]), 2.0f);
                        const double cz = (double)__fdiv_rn(__fadd_rn(bx[2], bx[5]), 2.0f);
                        const double dx = __dsub_rn(qx, cx), dy = __dsub_rn(qy, cy), dz = __dsub_rn(qz, cz);
                        key = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
                    }
                    if (arg < 0 || key < best) {
                        best = key;
                        arg = b;
                    }
                }
            }
            label = arg + 1;
        }
        if (!spp_align && valid) inst_pt[p] = (n_in > 1 && rule == 2) ? -2 : label - 1;
        // votes of this chunk
        votes_bg += __popc(__ballot_sync(FULL_MASK, valid && label == 0));
#pragma unroll
        for (int w = 0; w < WORDS; ++w) {
            uint32_t cand = all_in[w] | cuts[w];
            while (cand) {
                const int bb = __ffs(cand) - 1;
                cand &= cand - 1;
                const int v = __popc(__ballot_sync(FULL_MASK, valid && label == 32 * w + bb + 1));
                const int c = __popc(__ballot_sync(FULL_MASK, (mask[w] >> bb) & 1u));
                if (lane == bb) {
                    votes[w] += v;
                    inside[w] += c;
                }
            }
        }
    }
    if (!spp_align) return;
    // majority vote (first maximum wins: background first, then boxes in increasing index)
    uint32_t best_key = ((uint32_t)votes_bg << 10) | 1023u;            // key = votes * 1024 + (1023 - label)
    const float fcnt = (float)cnt;
#pragma unroll
    for (int w = 0; w < WORDS; ++w) {
        int v = votes[w];
        if (occ_thresh >= 0.0f && !(__fdiv_rn((float)inside[w], fcnt) >= occ_thresh)) v = 0;
        const int label = 32 * w + lane + 1;
        const uint32_t key = (32 * w + lane < nb) ? (((uint32_t)v << 10) | (uint32_t)(1023 - label)) : 0u;
        const uint32_t m = __reduce_max_sync(FULL_MASK, key);
        best_key = m > best_key ? m : best_key;
    }
    if (lane == 0) inst_spp[g] = (int)(1023u - (best_key & 1023u)) - 1;      // label - 1: -1 = background
}

extern "C" int gapro_heuristic_labels(const double* xyz, const int32_t* perm, const int32_t* seg_off,
                                      const int32_t* spp_off_dev, const int32_t* box_off_dev, const float* boxes,
                                      const float* boxes_vol, const int32_t* dist_src, int32_t n_scenes,
                                      int32_t s_total, int32_t words, int32_t rule, int32_t spp_align, float occ_thresh,
                                      int32_t* inst_spp, int32_t* inst_pt, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GAPRO_REQUIRE(xyz && perm && seg_off && spp_off_dev && box_off_dev && boxes && boxes_vol, "gapro_heuristic_labels: null pointer");
    GAPRO_REQUIRE(spp_align ? inst_spp != nullptr : inst_pt != nullptr, "gapro_heuristic_labels: missing output array");
    GAPRO_REQUIRE(rule >= 0 && rule <= 2, "gapro_heuristic_labels: rule must be 0 (volume), 1 (dist) or 2 (none)");
    GAPRO_REQUIRE(rule != 1 || dist_src != nullptr,
                  "gapro_heuristic_labels: rule 1 (dist) needs dist_src from gapro_multibox_sources");
    GAPRO_REQUIRE(n_scenes > 0 && s_total > 0, "gapro_heuristic_labels: empty batch");
    GAPRO_REQUIRE(words == 1 || words == 2 || words == 4 || words == 8,
                  "gapro_heuristic_labels: words must be 1, 2, 4 or 8 (at most 256 boxes per scene)");
    const int T = 256, WPB = T / 32;
    unsigned G = (unsigned)((s_total + WPB - 1) / WPB);
#define LAUNCH_H(W)                                                                                                 \
    k_heuristic<W><<<G, T, 0, stream>>>(xyz, perm, seg_off, spp_off_dev, box_off_dev, boxes, boxes_vol, dist_src,   \
                                        n_scenes, s_total, rule, spp_align, occ_thresh, inst_spp, inst_pt)
    switch (words) {
        case 1: LAUNCH_H(1); break;
        case 2: LAUNCH_H(2); break;
        case 4: LAUNCH_H(4); break;
        default: LAUNCH_H(8); break;
    }
#undef LAUNCH_H
    GAPRO_KERNEL_CHECK();
    return GAPRO_OK;
}

// =============================================================================================
// Heuristic labels -> final labels (gen_ps_utils.py:283-288 / :559-564).  Scene-local box index b >= 0:
// sem = cls[box_off[scene] + b], inst = b; -1 (background): sem = instance_classes, inst = -100; -2 (undecided
// under rule "none", per point only): sem = inst = -100.  Superpoint-aligned results become the 16-byte records
// (sem, inst, 1.0f, 0) of k_broadcast; per-point results are written directly.  One thread per element.
// =============================================================================================
__device__ __forceinline__ int2 heuristic_final(int b, int sc, const int32_t* __restrict__ box_off,
                                                const int64_t* __restrict__ cls, int instance_classes) {
    if (b >= 0) return make_int2((int32_t)cls[box_off[sc] + b], b);
    return make_int2(b == -1 ? instance_classes : -100, -100);
}

__global__ void __launch_bounds__(256)
k_heuristic_final_spp(const int32_t* __restrict__ inst_spp, const int32_t* __restrict__ spp_off,
                      const int32_t* __restrict__ box_off, const int64_t* __restrict__ cls, int instance_classes,
                      int n_scenes, int s_total, int4* __restrict__ packed_spp) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= s_total) return;
    const int b = inst_spp[g];
    const int2 r = heuristic_final(b, b >= 0 ? gapro_find_segment(spp_off, n_scenes, g) : 0, box_off, cls,
                                   instance_classes);
    packed_spp[g] = make_int4(r.x, r.y, __float_as_int(1.0f), 0);
}

__global__ void __launch_bounds__(256)
k_heuristic_final_pt(const int32_t* __restrict__ inst_pt, const int64_t* __restrict__ pt_off,
                     const int32_t* __restrict__ box_off, const int64_t* __restrict__ cls, int instance_classes,
                     int n_scenes, int64_t n, int32_t* __restrict__ sem, int32_t* __restrict__ inst) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const int b = inst_pt[p];
    const int2 r = heuristic_final(b, b >= 0 ? find_scene_pt(pt_off, n_scenes, p) : 0, box_off, cls, instance_classes);
    sem[p] = r.x;
    inst[p] = r.y;
}

extern "C" int gapro_heuristic_finalize(const int32_t* inst_spp, const int32_t* inst_pt, const int32_t* spp_off_dev,
                                        const int64_t* pt_off_dev, const int32_t* box_off_dev,
                                        const int64_t* boxes_cls, int32_t instance_classes, int32_t n_scenes,
                                        int32_t s_total, int64_t n_points, int32_t spp_align, void* packed_spp,
                                        int32_t* sem, int32_t* inst, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GAPRO_REQUIRE(box_off_dev && boxes_cls, "gapro_heuristic_finalize: null pointer");
    GAPRO_REQUIRE(n_scenes > 0, "gapro_heuristic_finalize: n_scenes must be positive");
    const int T = 256;
    if (spp_align) {
        GAPRO_REQUIRE(inst_spp && spp_off_dev, "gapro_heuristic_finalize: null pointer");
        GAPRO_REQUIRE(packed_spp, "gapro_heuristic_finalize: missing output array (packed_spp)");
        GAPRO_REQUIRE(s_total > 0, "gapro_heuristic_finalize: empty batch");
        GAPRO_REQUIRE((uintptr_t)packed_spp % 16 == 0, "gapro_heuristic_finalize: packed_spp must be 16-byte aligned");
        k_heuristic_final_spp<<<(unsigned)((s_total + T - 1) / T), T, 0, stream>>>(
            inst_spp, spp_off_dev, box_off_dev, boxes_cls, instance_classes, n_scenes, s_total, (int4*)packed_spp);
    } else {
        GAPRO_REQUIRE(inst_pt && pt_off_dev, "gapro_heuristic_finalize: null pointer");
        GAPRO_REQUIRE(sem && inst, "gapro_heuristic_finalize: missing output array (sem, inst)");
        GAPRO_REQUIRE(n_points > 0, "gapro_heuristic_finalize: empty batch");
        k_heuristic_final_pt<<<(unsigned)((n_points + T - 1) / T), T, 0, stream>>>(
            inst_pt, pt_off_dev, box_off_dev, boxes_cls, instance_classes, n_scenes, n_points, sem, inst);
    }
    GAPRO_KERNEL_CHECK();
    return GAPRO_OK;
}

// =============================================================================================
// B — feature pooling (gen_ps_utils.py:357): float32 sum in point-index order, / float32 count
// =============================================================================================
// One warp per superpoint.  For every chunk of 32 points the warp loads the point indices with one
// coalesced read, issues all D*32 feature gathers at once (independent loads, one memory latency),
// stages them in shared memory, and lanes d < D then replay the float32 adds strictly in point
// order — the index-ordered float32 sum of torch_scatter's CPU kernel, bit for bit.
constexpr int POOL_WARPS = 8;

template <int DT>     // DT > 0: feature dimension known at compile time (cheap index arithmetic); 0: runtime D
__global__ void __launch_bounds__(32 * POOL_WARPS)
k_pool_feats(const float* __restrict__ feats, const int32_t* __restrict__ perm, const int32_t* __restrict__ seg_off,
             int s_total, int D_, float* __restrict__ out) {
    const int D = DT > 0 ? DT : D_;
    extern __shared__ float pool_smem[];               // [POOL_WARPS][32 * D]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = blockIdx.x * POOL_WARPS + warp;
    if (g >= s_total) return;
    float* stage = pool_smem + (size_t)warp * 32 * D;
    const int start = seg_off[g], end = seg_off[g + 1];
    float acc[2] = {0.0f, 0.0f};                       // lane handles dims lane and lane + 32 (D <= 64)
    for (int base = start; base < end; base += 32) {
        const int n = min(32, end - base);
        const int myp = (lane < n) ? perm[base + lane] : 0;
        const int total = n * D;
        for (int e0 = 0; e0 < total; e0 += 32) {           // warp-uniform trip count (full-mask shuffles)
            const int e = e0 + lane;
            const int ec = min(e, total - 1);
            const int pt = ec / D, d = ec - pt * D;
            const int p = __shfl_sync(FULL_MASK, myp, pt);
            if (e < total) stage[e] = feats[(int64_t)p * D + d];
        }
        __syncwarp();
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int d = lane + 32 * h;
            if (d < D) {
                float a = acc[h];
                for (int pt = 0; pt < n; ++pt) a = __fadd_rn(a, stage[pt * D + d]);
                acc[h] = a;
            }
        }
        __syncwarp();
    }
    const float fcnt = (float)(end - start);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int d = lane + 32 * h;
        if (d < D) out[(int64_t)g * D + d] = __fdiv_rn(acc[h], fcnt);
    }
}

extern "C" int gapro_pool_feats(const float* feats, const int32_t* perm, const int32_t* seg_off, int32_t s_total,
                                int32_t D, float* out, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GAPRO_REQUIRE(feats && perm && seg_off && out, "gapro_pool_feats: null pointer");
    GAPRO_REQUIRE(s_total > 0 && D > 0, "gapro_pool_feats: empty input");
    GAPRO_REQUIRE(D <= 64, "gapro_pool_feats: feature dimension %d > 64", D);
    const size_t smem = (size_t)POOL_WARPS * 32 * D * sizeof(float);
    static bool attr = false;
    if (!attr) {
        GAPRO_CUDA_TRY(cudaFuncSetAttribute(k_pool_feats<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
        attr = true;
    }
    const unsigned grid = (unsigned)((s_total + POOL_WARPS - 1) / POOL_WARPS);
    if (D == 6)
        k_pool_feats<6><<<grid, 32 * POOL_WARPS, smem, stream>>>(feats, perm, seg_off, s_total, D, out);
    else if (D == 32)
        k_pool_feats<32><<<grid, 32 * POOL_WARPS, smem, stream>>>(feats, perm, seg_off, s_total, D, out);
    else
        k_pool_feats<0><<<grid, 32 * POOL_WARPS, smem, stream>>>(feats, perm, seg_off, s_total, D, out);
    GAPRO_KERNEL_CHECK();
    return GAPRO_OK;
}

// =============================================================================================
// Index lists by warp-ballot compaction (torch.nonzero at gen_ps_utils.py:405, 428-429)
// =============================================================================================
__global__ void __launch_bounds__(256)
k_compact_lists(const uint32_t* __restrict__ occ_bits, const int32_t* __restrict__ n_bbs,
                const int32_t* __restrict__ spp_off, int words, const int32_t* __restrict__ list_scene,
                const int32_t* __restrict__ list_b1, const int32_t* __restrict__ list_b2,
                const int32_t* __restrict__ list_off, int32_t* __restrict__ out_idx) {
    __shared__ int warp_cnt[8];
    __shared__ int running;
    const int l = blockIdx.x;
    const int sc = list_scene[l], b1 = list_b1[l], b2 = list_b2[l];
    const int g0 = spp_off[sc], g1 = spp_off[sc + 1];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int32_t* out = out_idx + list_off[l];
    if (threadIdx.x == 0) running = 0;
    __syncthreads();
    for (int base = g0; base < g1; base += 256) {
        const int g = base + threadIdx.x;
        bool keep = false;
        if (g < g1) {
            const uint32_t* row = occ_bits + (size_t)g * words;
            bool in1 = (row[b1 >> 5] >> (b1 & 31)) & 1u;
            keep = b2 < 0 ? (in1 && n_bbs[g] == 1) : (in1 && ((row[b2 >> 5] >> (b2 & 31)) & 1u));
        }
        const uint32_t bal = __ballot_sync(FULL_MASK, keep);
        if (lane == 0) warp_cnt[wid] = __popc(bal);
        __syncthreads();
        int before = running;
        for (int w = 0; w < wid; ++w) before += warp_cnt[w];
        if (keep) out[before + __popc(bal & ((1u << lane) - 1u))] = g;
        __syncthreads();
        if (threadIdx.x == 0) {
            int tot = 0;
            for (int w = 0; w < 8; ++w) tot += warp_cnt[w];
            running += tot;
        }
        __syncthreads();
    }
}

extern "C" int gapro_compact_lists(const uint32_t* occ_bits, const int32_t* n_bbs, const int32_t* spp_off_dev,
                                   int32_t words, const int32_t* list_scene, const int32_t* list_b1,
                                   const int32_t* list_b2, const int32_t* list_off, int32_t n_lists, int32_t* out_idx,
                                   void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (n_lists == 0) return GAPRO_OK;
    GAPRO_REQUIRE(occ_bits && n_bbs && spp_off_dev && list_scene && list_b1 && list_b2 && list_off && out_idx,
                  "gapro_compact_lists: null pointer");
    GAPRO_REQUIRE(n_lists > 0 && words > 0, "gapro_compact_lists: bad sizes");
    k_compact_lists<<<n_lists, 256, 0, stream>>>(occ_bits, n_bbs, spp_off_dev, words, list_scene, list_b1, list_b2,
                                                 list_off, out_idx);
    GAPRO_KERNEL_CHECK();
    return GAPRO_OK;
}

// =============================================================================================
// S0 + M + D + per-superpoint labels (gen_ps_utils.py:365-383, 412-446, 450-476): one CTA / scene
// =============================================================================================
__global__ void __launch_bounds__(512)
k_resolve_spp(const uint32_t* __restrict__ occ_bits, const int32_t* __restrict__ n_bbs, int words,
              const int32_t* __restrict__ spp_off, const int32_t* __restrict__ box_off,
              const double* __restrict__ boxes_vol, const int64_t* __restrict__ boxes_cls,
              const int32_t* __restrict__ n_fg, int instance_classes, const int32_t* __restrict__ ev_off,
              const int32_t* __restrict__ ev_kind, const int32_t* __restrict__ ev_b1, const int32_t* __restrict__ ev_b2,
              const int32_t* __restrict__ ev_list_off, const int32_t* __restrict__ ev_list_len,
              const int32_t* __restrict__ ev_gp_off, const int32_t* __restrict__ lists_idx,
              const float* __restrict__ gp_conf, const uint8_t* __restrict__ gp_label, const float* __restrict__ gp_mu,
              const float* __restrict__ gp_var, int32_t* __restrict__ sem_spp, int32_t* __restrict__ inst_spp,
              float* __restrict__ prob_spp, float* __restrict__ mu_spp, float* __restrict__ var_spp,
              int4* __restrict__ packed_spp) {
    const int sc = blockIdx.x;
    const int g0 = spp_off[sc], g1 = spp_off[sc + 1];
    const int b0 = box_off[sc];
    // S0: trivial assignment (:365-383).  inst == -100 doubles as "undetermined".
    for (int g = g0 + threadIdx.x; g < g1; g += blockDim.x) {
        const int nb = n_bbs[g];
        int inst = -100;
        float prob = 0.0f;
        if (nb == 1) {
            for (int w = 0; w < words; ++w) {
                uint32_t b = occ_bits[(size_t)g * words + w];
                if (b) inst = 32 * w + __ffs(b) - 1;
            }
            prob = 1.0f;
        } else if (nb == 0) {
            inst = -1;
            prob = 1.0f;
        }
        inst_spp[g] = inst;
        prob_spp[g] = prob;
        mu_spp[g] = -100.0f;
        var_spp[g] = -100.0f;
    }
    __syncthreads();
    // M: events in loop order (:411-446)
    for (int e = ev_off[sc]; e < ev_off[sc + 1]; ++e) {
        const int kind = ev_kind[e], b1 = ev_b1[e], b2 = ev_b2[e];
        const int32_t* list = lists_idx + ev_list_off[e];
        const int len = ev_list_len[e];
        const int gp = ev_gp_off[e];
        for (int r = threadIdx.x; r < len; r += blockDim.x) {
            const int g = list[r];
            if (kind == GAPRO_EV_GP) {
                const float conf = gp_conf[gp + r];
                if (prob_spp[g] < conf) {                      // strict, float32 (:438)
                    inst_spp[g] = gp_label[gp + r] ? b2 : b1;   // :440-441
                    prob_spp[g] = conf;
                    mu_spp[g] = gp_mu[gp + r];
                    var_spp[g] = gp_var[gp + r];
                }
            } else {
                inst_spp[g] = (kind == GAPRO_EV_NEST_B1) ? b1 : b2;
                prob_spp[g] = 1.0f;
            }
        }
        __syncthreads();
    }
    // D: smallest-volume fallback (:450-464) and per-superpoint labels (:467-476)
    const int nfg = n_fg[sc];
    for (int g = g0 + threadIdx.x; g < g1; g += blockDim.x) {
        int inst = inst_spp[g];
        if (n_bbs[g] > 1 && inst == -100) {
            double best = 0.0;
            int arg = -1;
            for (int w = 0; w < words; ++w) {
                uint32_t m = occ_bits[(size_t)g * words + w];
                while (m) {
                    int b = 32 * w + __ffs(m) - 1;
                    m &= m - 1;
                    double v = boxes_vol[b0 + b];
                    if (arg < 0 || v < best) {
                        best = v;
                        arg = b;
                    }
                }
            }
            inst = arg;
            prob_spp[g] = 1.0f;
        }
        int sem = -100, inst_out = -100;
        if (inst >= 0) {
            sem = (int)boxes_cls[b0 + inst];
            inst_out = inst;
        } else if (inst == -1) {
            sem = instance_classes;
        }
        if (inst_out >= nfg) inst_out = -100;
        sem_spp[g] = sem;
        inst_spp[g] = inst_out;
        if (packed_spp) packed_spp[g] = make_int4(sem, inst_out, __float_as_int(prob_spp[g]), 0);
    }
}

extern "C" int gapro_resolve_spp(const uint32_t* occ_bits, const int32_t* n_bbs, int32_t words,
                                 const int32_t* spp_off_dev, const int32_t* box_off_dev, const double* boxes_vol,
                                 const int64_t* boxes_cls, const int32_t* n_fg, int32_t instance_classes,
                                 int32_t n_scenes, const int32_t* ev_off, const int32_t* ev_kind, const int32_t* ev_b1,
                                 const int32_t* ev_b2, const int32_t* ev_list_off, const int32_t* ev_list_len,
                                 const int32_t* ev_gp_off, const int32_t* lists_idx, const float* gp_conf,
                                 const uint8_t* gp_label, const float* gp_mu, const float* gp_var, int32_t* sem_spp,
                                 int32_t* inst_spp, float* prob_spp, float* mu_spp, float* var_spp, void* packed_spp,
                                 void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GAPRO_REQUIRE(occ_bits && n_bbs && spp_off_dev && box_off_dev && boxes_vol && boxes_cls && n_fg && ev_off &&
                      sem_spp && inst_spp && prob_spp && mu_spp && var_spp,
                  "gapro_resolve_spp: null pointer");
    GAPRO_REQUIRE(n_scenes > 0 && words > 0, "gapro_resolve_spp: bad sizes");
    k_resolve_spp<<<n_scenes, 512, 0, stream>>>(occ_bits, n_bbs, words, spp_off_dev, box_off_dev, boxes_vol, boxes_cls,
                                                n_fg, instance_classes, ev_off, ev_kind, ev_b1, ev_b2, ev_list_off,
                                                ev_list_len, ev_gp_off, lists_idx, gp_conf, gp_label, gp_mu, gp_var,
                                                sem_spp, inst_spp, prob_spp, mu_spp, var_spp, (int4*)packed_spp);
    GAPRO_KERNEL_CHECK();
    return GAPRO_OK;
}

// =============================================================================================
// E — broadcast to points (gen_ps_utils.py:478-480)
// =============================================================================================
__global__ void __launch_bounds__(256)
k_broadcast(const int32_t* __restrict__ spp_gid, int64_t n, const int4* __restrict__ packed_spp,
            int32_t* __restrict__ sem, int32_t* __restrict__ inst, float* __restrict__ prob) {
    // 4 points per thread: one 128-bit load of ids, four 128-bit gathers of (sem, inst, prob) records
    // from the L2-resident per-superpoint table, three 128-bit stores; scalar tail
    int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t n4 = n >> 2;
    if (q < n4) {
        const int4 g = __ldcs(reinterpret_cast<const int4*>(spp_gid) + q);
        const int4 a = __ldg(packed_spp + g.x), b = __ldg(packed_spp + g.y), c = __ldg(packed_spp + g.z),
                   d = __ldg(packed_spp + g.w);
        __stcs(reinterpret_cast<int4*>(sem) + q, make_int4(a.x, b.x, c.x, d.x));
        __stcs(reinterpret_cast<int4*>(inst) + q, make_int4(a.y, b.y, c.y, d.y));
        __stcs(reinterpret_cast<int4*>(prob) + q, make_int4(a.z, b.z, c.z, d.z));
    } else if (q == n4) {
        for (int64_t k = n4 << 2; k < n; ++k) {
            const int4 a = packed_spp[spp_gid[k]];
            sem[k] = a.x;
            inst[k] = a.y;
            prob[k] = __int_as_float(a.z);
        }
    }
}

extern "C" int gapro_broadcast_labels(const int32_t* spp_gid, int64_t n_points, const void* packed_spp, int32_t* sem,
                                      int32_t* inst, float* prob, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GAPRO_REQUIRE(spp_gid && packed_spp && sem && inst && prob, "gapro_broadcast_labels: null pointer");
    GAPRO_REQUIRE(n_points > 0, "gapro_broadcast_labels: empty input");
    GAPRO_REQUIRE(((uintptr_t)spp_gid % 16 == 0) && ((uintptr_t)sem % 16 == 0) && ((uintptr_t)inst % 16 == 0) &&
                      ((uintptr_t)prob % 16 == 0) && ((uintptr_t)packed_spp % 16 == 0),
                  "gapro_broadcast_labels: arrays must be 16-byte aligned");
    int64_t threads = (n_points >> 2) + 1;
    k_broadcast<<<(unsigned)((threads + 255) / 256), 256, 0, stream>>>(spp_gid, n_points, (const int4*)packed_spp, sem,
                                                                       inst, (float*)prob);
    GAPRO_KERNEL_CHECK();
    return GAPRO_OK;
}

// =============================================================================================
// Random-gather microbenchmark: the roofline of the gather-bound stages.  k_occupancy and k_pool_feats read
// every point once, but through `perm` (points grouped by superpoint), i.e. as 24-byte records at random
// addresses.  This kernel does nothing else: coalesced index read, one independent 24-byte gather per
// record (4 records per thread in flight), a sum that is never stored.  Timed by the caller (bench.py).
// =============================================================================================
__global__ void __launch_bounds__(256)
k_gather_peak(const int32_t* __restrict__ idx, const double* __restrict__ table, int64_t n, double* __restrict__ sink) {
    const int64_t base = (int64_t)blockIdx.x * 1024 + threadIdx.x;
    int64_t p[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int64_t k = base + 256 * i;
        p[i] = k < n ? (int64_t)idx[k] : -1;
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 4; ++i)
        if (p[i] >= 0) s += table[3 * p[i]] + table[3 * p[i] + 1] + table[3 * p[i] + 2];
    if (s == 1.2345e300) sink[0] = s;      // keeps the loads alive
}

extern "C" int gapro_gather_peak(const int32_t* idx, const double* table, int64_t n_records, double* sink,
                                 void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GAPRO_REQUIRE(idx && table && sink && n_records > 0, "gapro_gather_peak: bad arguments");
    k_gather_peak<<<(unsigned)((n_records + 1023) / 1024), 256, 0, stream>>>(idx, table, n_records, sink);
    GAPRO_KERNEL_CHECK();
    return GAPRO_OK;
}
