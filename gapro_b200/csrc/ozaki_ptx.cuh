// tcgen05 / mbarrier / bulk-copy PTX wrappers, the digit-plane constants, the digit-plane slicing of one block and
// the tile main loop shared by the stand-alone product (ozaki.cu) and the batched GP phases (gp_ozaki.cuh).
// sm_100a only.
#pragma once
#include <stdint.h>

#include "common.cuh"

namespace oz {

constexpr int OZ_MAXS = 8;      // 8 accumulators of 64 columns = the 512 TMEM columns of an SM
constexpr int OZ_BM = 128, OZ_BN = 64, OZ_BK = 64;
constexpr int OZ_BLK = 64 * 64;                 // bytes of one (64 vectors x 64 k) block of a digit plane
constexpr int OZ_THREADS = 192;

__host__ __device__ constexpr int oz_stage_bytes(int S) { return S * (2 * OZ_BLK + OZ_BLK); }
__host__ __device__ constexpr int oz_stages(int S) { return S <= 6 ? 3 : 2; }      // 227 KB of shared memory per CTA
__host__ __device__ constexpr int oz_smem_bytes(int S) { return oz_stages(S) * oz_stage_bytes(S) + 1024 + 256; }

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(bar), "r"(parity)
            : "memory");
    } while (!ok);
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_i8(uint32_t tmem_c, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}"
        ::"r"(tmem_c), "l"(da), "l"(db), "r"(idesc), "r"(accumulate), "r"(0u)
        : "memory");
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, int32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major operand tile, 64-byte swizzle: rows of 64 bytes, 8-row atoms of 512 bytes (SBO), version 1 (sm_100)
__device__ __forceinline__ uint64_t umma_desc_sw64(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | (1ull << 16) | ((uint64_t)(512 >> 4) << 32) | (1ull << 46) | (4ull << 61);
}
// kind::i8: D = S32 (c_format 2), A and B signed 8 bit (format 1), both K-major, N >> 3 at bit 17, M >> 4 at bit 24
constexpr uint32_t OZ_IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(OZ_BN >> 3) << 17) | ((uint32_t)(OZ_BM >> 4) << 24);


// one (vector, 16-k chunk) of a staged 64 x 64 block -> 16 bytes of each of the S digit planes, written at the
// 64-byte-swizzled position of the K-major shared-memory layout.  y: the 16 values already scaled to |y| < 64.
template <int S>
__device__ __forceinline__ void emit_digits(double (&y)[16], uint8_t* dst, size_t plane) {
#pragma unroll
    for (int s = 0; s < S; ++s) {
        uint32_t w[4];
#pragma unroll
        for (int p = 0; p < 4; ++p) {
            uint32_t word = 0;
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const int j = 4 * p + b;
                const double q = rint(y[j]);               // |q| <= 64
                y[j] = (y[j] - q) * 128.0;                 // exact: the next 7 bits, |.| <= 64
                word |= ((uint32_t)(int)q & 0xffu) << (8 * b);
            }
            w[p] = word;
        }
        *reinterpret_cast<uint4*>(dst + s * plane) = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

// Block (kb, rb) - vectors 64 rb.., k 64 kb.. - of the S digit planes of an operand: the 64 x 64 block of
// x(v, k) ks(k), zero where !valid(v, k), is staged in shared memory, then every thread writes one (vector, 16-k chunk)
// of each plane.  X is [vectors, k] row-major (trans = 0) or [k, vectors] (trans = 1); ks (optional) scales along k.
// The digits are those of x inv(v) post, |.| < 64: inv(v) is 2^-e times 64 or 1, post the other factor (each caller
// keeps its own order of the two exact power-of-two scalings).  planes: [S][kb_total][rb_total] blocks of 4 KB.
template <int S, class Valid, class Inv>
__device__ __forceinline__ void oz_slice_block(const double* X, int ld, bool trans, const double* ks, int kb, int rb,
                                               const Valid& valid, const Inv& inv, double post, uint8_t* planes,
                                               int kb_total, int rb_total) {
    constexpr int LD = 68;                         // + k/16 skew: conflict-free 16-double reads per (vector, chunk)
    __shared__ double blk[64 * LD + 8];
    const int v0 = rb * 64, k0 = kb * 64;
    for (int e = threadIdx.x; e < 64 * 64; e += 256) {
        const int a = e >> 6, b = e & 63;          // b runs along the contiguous direction of X
        const int v = trans ? b : a, k = trans ? a : b;
        double x = 0.0;
        if (valid(v0 + v, k0 + k)) {
            x = trans ? X[(size_t)(k0 + k) * ld + v0 + v] : X[(size_t)(v0 + v) * ld + k0 + k];
            if (ks) x *= ks[k0 + k];
        }
        blk[v * LD + k + (k >> 4)] = x;
    }
    __syncthreads();
    const int t = threadIdx.x;
    const int atom = t >> 5, r = (t & 31) >> 2, c = t & 3;
    const int v = 8 * atom + r;
    const double iv = inv(v0 + v);
    double y[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) y[j] = blk[v * LD + 16 * c + j + c] * iv * post;      // |y| < 64
    uint8_t* dst = planes + ((size_t)kb * rb_total + rb) * OZ_BLK + atom * 512 + r * 64 + ((c ^ ((r >> 1) & 3)) * 16);
    emit_digits<S>(y, dst, (size_t)kb_total * rb_total * OZ_BLK);
}

// One 128 x 64 output tile of A B^T from S digit planes per operand, warp-specialised:
//   warp 0    producer: per 64-deep k-block ONE mbarrier transaction of S x (8 KB + 4 KB) `cp.async.bulk` copies
//             (the digit planes are stored in global memory block by block ALREADY in the 64-byte-swizzled K-major
//             shared-memory layout the UMMA descriptors describe, so a plain bulk copy lands them ready to use);
//   warp 1    one elected thread issues tcgen05.mma.cta_group::1.kind::i8 (M = 128, N = 64, K = 32) for all pairs
//             s + t < S of the k-block into S TMEM accumulators (S x 64 columns), tcgen05.commit releases the stage;
//   warps 2-5 epilogue: tcgen05.ld the S accumulators of their 32 TMEM lanes, float64 recombination, then
//             epi(row, c, acc) for tile row `row` and columns 16c .. 16c+15:
//             acc[j] = sum_g 2^-(12+7g) acc_g[row][16c + j], not yet scaled (zeros when nkb == 0).
// oz_stages(S) stages of S x 12 KB in oz_smem_bytes(S) of dynamic shared memory; 512 TMEM columns, one CTA per SM.
// a (b): plane 0 of the operand at the tile's first k-block and its two (one) 64-vector blocks; a_kstride: bytes from
// one k-block to the next, a_plane: bytes from one plane to the next.
template <int S, class Epi>
__device__ __forceinline__ void oz_tile(uint8_t* smem_raw, const uint8_t* a, size_t a_kstride, size_t a_plane,
                                        const uint8_t* b, size_t b_kstride, size_t b_plane, int nkb, const Epi& epi) {
    constexpr int STAGE = oz_stage_bytes(S);
    constexpr int NST = oz_stages(S);
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + NST * STAGE);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * NST + 1);
    const uint32_t full0 = smem_u32(bars), empty0 = smem_u32(bars + NST), tfull = smem_u32(bars + 2 * NST);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int s = 0; s < NST; ++s) {
            mbar_init(full0 + 8 * s, 1);
            mbar_init(empty0 + 8 * s, 1);
        }
        mbar_init(tfull, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            for (int i = 0; i < nkb; ++i) {
                const int st = i % NST;
                mbar_wait(empty0 + 8 * st, ((i / NST) & 1) ^ 1);
                mbar_expect_tx(full0 + 8 * st, (uint32_t)STAGE);
                const uint32_t dst = smem_u32(smem + st * STAGE);
                const uint8_t* ga = a + (size_t)i * a_kstride;
                const uint8_t* gb = b + (size_t)i * b_kstride;
#pragma unroll
                for (int s = 0; s < S; ++s) {
                    bulk_g2s(dst + s * 2 * OZ_BLK, ga + s * a_plane, 2 * OZ_BLK, full0 + 8 * st);
                    bulk_g2s(dst + S * 2 * OZ_BLK + s * OZ_BLK, gb + s * b_plane, OZ_BLK, full0 + 8 * st);
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        if (lane == 0) {
            for (int i = 0; i < nkb; ++i) {
                const int st = i % NST;
                mbar_wait(full0 + 8 * st, (i / NST) & 1);
                tc_fence_after();
                const uint32_t sa = smem_u32(smem + st * STAGE), sb = sa + S * 2 * OZ_BLK;
#pragma unroll
                for (int kk = 0; kk < OZ_BK / 32; ++kk) {
#pragma unroll
                    for (int s = 0; s < S; ++s) {
                        const uint64_t da = umma_desc_sw64(sa + s * 2 * OZ_BLK + kk * 32);
#pragma unroll
                        for (int t = 0; t + s < S; ++t) {
                            const uint64_t db = umma_desc_sw64(sb + t * OZ_BLK + kk * 32);
                            tc_mma_i8(tmem + (uint32_t)((s + t) * OZ_BN), da, db, OZ_IDESC, (i | kk | s) != 0);
                        }
                    }
                }
                tc_commit(empty0 + 8 * st);      // frees the stage when these MMAs have read it
            }
            tc_commit(tfull);                    // accumulators complete
        }
        __syncwarp();
    } else {
        // epilogue warps 2..5: TMEM lane quarter = warp % 4
        const int q = warp & 3;
        const int row = 32 * q + lane;
        if (nkb > 0) {
            mbar_wait(tfull, 0);
            tc_fence_after();
        }
#pragma unroll 1
        for (int c = 0; c < OZ_BN / 16; ++c) {
            double acc[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) acc[j] = 0.0;
            if (nkb > 0) {
                // the S accumulators in two batches (register budget), smallest weights first
#pragma unroll
                for (int h = (S - 1) / 4; h >= 0; --h) {
                    int32_t v[4][16];
#pragma unroll
                    for (int g = 0; g < 4; ++g)
                        if (4 * h + g < S)
                            tc_ld16(tmem + ((uint32_t)(32 * q) << 16) + (uint32_t)((4 * h + g) * OZ_BN + 16 * c), v[g]);
                    tc_wait_ld();
#pragma unroll
                    for (int g = 3; g >= 0; --g) {
                        if (4 * h + g < S) {
                            const double w = __longlong_as_double((long long)(1023 - (12 + 7 * (4 * h + g))) << 52);   // 2^-(12+7g)
#pragma unroll
                            for (int j = 0; j < 16; ++j) acc[j] = fma((double)v[g][j], w, acc[j]);
                        }
                    }
                }
            }
            epi(row, c, acc);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        __syncwarp();
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
    }
}

}  // namespace oz
