// Float64 tile products on the 5th-generation tensor cores (tcgen05, sm_100a) by integer slicing ("Ozaki scheme").
//
// tcgen05.mma has no f64 kind and the FP64 DMMA path tops out at ~37 TFLOP/s on B200, so a float64 product
// C = A B^T is computed from EXACT int8 products instead:
//
//   every row of A (and of B) is scaled by a power of two so that |x| < 1 and cut into S signed digits,
//       x = 2^e (q_0 2^-6 + q_1 2^-13 + ... + q_{S-1} 2^-(6+7(S-1))) + O(2^-(7S)),   |q_s| <= 64  (int8),
//   the digit planes are multiplied pairwise on the tensor cores (kind::i8, int32 accumulators in TMEM - exact:
//   |q q'| <= 2^12, K <= 2^13, at most S pairs per accumulator), pairs with s + t >= S are dropped (they are below
//   the truncation of the operands), and the S accumulators are recombined in float64 in the epilogue:
//       C_ij = 2^(e_i + e'_j) * sum_g 2^-(12 + 7g) * acc_g[i][j],   acc_g = sum_{s+t=g} sum_k q_s[i][k] q'_t[j][k].
//   Error: <= (S+1) 2^-(7S) of the row-max x row-max x K bound (1.6e-12 at S = 6), i.e. normwise like a float64
//   GEMM with a ~1e4 larger unit roundoff; S(S+1)/2 = 21 int8 products per float64 product at S = 6.
//
// Kernel k_oz_gemm: one CTA per 128 x 64 output tile, the warp-specialised main loop oz_tile (ozaki_ptx.cuh) with an
// epilogue that scales and stores.  oz_stages(S) stages of S x 12 KB: three of 72 KB (216 KB of shared memory) at
// S = 6, two of 96 KB (192 KB) at S = 8; 512 TMEM columns allocated, one CTA per SM.
#include <vector>

#include "common.cuh"
#include "ozaki_ptx.cuh"

namespace {

using namespace oz;

struct OzGemm {
    const uint8_t* a;       // digit planes of the A operand: [S][kb][rb64][4 KB]
    const uint8_t* b;
    int a_rb, b_rb;         // 64-vector blocks per plane row (a_rb even)
    int kb_total;           // 64-deep k-blocks per plane
    const double* sa;       // 2^e per A vector, 2^e' per B vector
    const double* sb;
    double* C;
    int ldc, M, N;          // valid output extent
    int tiles_n;            // 64-wide tiles per row of tiles
};

template <int S>
__global__ void __launch_bounds__(OZ_THREADS, 1) k_oz_gemm(OzGemm P) {
    extern __shared__ __align__(1024) uint8_t oz_smem[];
    const int ti = blockIdx.x / P.tiles_n, tj = blockIdx.x % P.tiles_n;
    const auto epi = [&](int row, int c, const double(&acc)[16]) {
        const int gr = ti * OZ_BM + row, gc0 = tj * OZ_BN + 16 * c;
        if (gr >= P.M) return;
        const double sa = P.sa[gr];
        double* out = P.C + (size_t)gr * P.ldc + gc0;
#pragma unroll
        for (int j = 0; j < 16; ++j)
            if (gc0 + j < P.N) out[j] = acc[j] * sa * P.sb[gc0 + j];
    };
    const size_t a_kstride = (size_t)P.a_rb * OZ_BLK, b_kstride = (size_t)P.b_rb * OZ_BLK;
    oz_tile<S>(oz_smem, P.a + (size_t)2 * ti * OZ_BLK, a_kstride, P.kb_total * a_kstride, P.b + (size_t)tj * OZ_BLK,
               b_kstride, P.kb_total * b_kstride, P.kb_total, epi);
}

// ---------------------------------------------------------------------------------------------
// digit planes
// ---------------------------------------------------------------------------------------------
// scale[v] = 2^e with max_k |x(v,k) ks(k)| * 2^-e in [1/2, 1)  (1 for an all-zero vector)
// trans = 0: vector v = row v of X (k along the row); trans = 1: vector v = column v of X (k down the column)
__global__ void __launch_bounds__(256)
k_oz_vecscale(const double* __restrict__ X, int ld, int nvec, int K, int trans, const double* __restrict__ ks,
              double* __restrict__ scale) {
    __shared__ double red[4][64];
    double m = 0.0;
    if (!trans) {
        const int v = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
        if (v < nvec)
            for (int k = lane; k < K; k += 32) m = fmax(m, fabs(X[(size_t)v * ld + k] * (ks ? ks[k] : 1.0)));
        for (int o = 16; o; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (lane == 0 && v < nvec) scale[v] = m > 0.0 ? ldexp(1.0, ilogb(m) + 1) : 1.0;
    } else {
        const int c = threadIdx.x & 63, rg = threadIdx.x >> 6, v = blockIdx.x * 64 + c;
        if (v < nvec)
            for (int k = rg; k < K; k += 4) m = fmax(m, fabs(X[(size_t)k * ld + v] * (ks ? ks[k] : 1.0)));
        red[rg][c] = m;
        __syncthreads();
        if (rg == 0 && v < nvec) {
            m = fmax(fmax(red[0][c], red[1][c]), fmax(red[2][c], red[3][c]));
            scale[v] = m > 0.0 ? ldexp(1.0, ilogb(m) + 1) : 1.0;
        }
    }
}

// grid (k-blocks, 64-vector blocks): one 4 KB block of each of the S planes per CTA
template <int S>
__global__ void __launch_bounds__(256)
k_oz_slice(const double* __restrict__ X, int ld, int nvec, int K, int trans, const double* __restrict__ ks,
           const double* __restrict__ scale, uint8_t* __restrict__ planes, int rb_total, int kb_total) {
    oz_slice_block<S>(
        X, ld, trans, ks, blockIdx.x, blockIdx.y, [&](int v, int k) { return v < nvec && k < K; },
        [&](int v) { return v < nvec ? 1.0 / scale[v] : 0.0; }, 64.0,      // exact: a power of two
        planes, kb_total, rb_total);
}

struct OzWs {
    size_t a_planes, b_planes, sa, sb, total;
    int a_rb, b_rb, kb;
};
OzWs oz_layout(int M, int N, int K, int S) {
    OzWs w;
    w.a_rb = (M + OZ_BM - 1) / OZ_BM * 2;
    w.b_rb = (N + OZ_BN - 1) / OZ_BN;
    w.kb = (K + OZ_BK - 1) / OZ_BK;
    size_t o = 0;
    w.a_planes = o;
    o += gapro_align_up((size_t)S * w.kb * w.a_rb * OZ_BLK, 1024);
    w.b_planes = o;
    o += gapro_align_up((size_t)S * w.kb * w.b_rb * OZ_BLK, 1024);
    w.sa = o;
    o += gapro_align_up((size_t)w.a_rb * 64 * 8, 256);
    w.sb = o;
    o += gapro_align_up((size_t)w.b_rb * 64 * 8, 256);
    w.total = o;
    return w;
}

template <int S>
int oz_run(const double* A, int lda, int transA, const double* ks, const double* B, int ldb, int transB, int M, int N,
           int K, double* C, int ldc, void* ws, const OzWs& L, int reps, float* ms_slice, float* ms_gemm,
           cudaStream_t stream) {
    uint8_t* ap = (uint8_t*)ws + L.a_planes;
    uint8_t* bp = (uint8_t*)ws + L.b_planes;
    double* sa = (double*)((char*)ws + L.sa);
    double* sb = (double*)((char*)ws + L.sb);
    static bool attr_done[64] = {};      // (one flag per template instantiation and device)
    int dev = 0;
    GAPRO_CUDA_TRY(cudaGetDevice(&dev));
    if (!attr_done[dev & 63]) {
        GAPRO_CUDA_TRY(cudaFuncSetAttribute(k_oz_gemm<S>, cudaFuncAttributeMaxDynamicSharedMemorySize, oz_smem_bytes(S)));
        attr_done[dev & 63] = true;
    }
    cudaEvent_t e0, e1, e2;
    GAPRO_CUDA_TRY(cudaEventCreate(&e0));
    GAPRO_CUDA_TRY(cudaEventCreate(&e1));
    GAPRO_CUDA_TRY(cudaEventCreate(&e2));
    OzGemm P{ap, bp, L.a_rb, L.b_rb, L.kb, sa, sb, C, ldc, M, N, L.b_rb};
    const int tiles = (L.a_rb / 2) * L.b_rb;
    for (int rep = 0; rep < reps; ++rep) {
        GAPRO_CUDA_TRY(cudaEventRecord(e0, stream));
        k_oz_vecscale<<<transA ? (M + 63) / 64 : (M + 7) / 8, 256, 0, stream>>>(A, lda, M, K, transA, ks, sa);
        k_oz_vecscale<<<transB ? (N + 63) / 64 : (N + 7) / 8, 256, 0, stream>>>(B, ldb, N, K, transB, nullptr, sb);
        k_oz_slice<S><<<dim3(L.kb, L.a_rb), 256, 0, stream>>>(A, lda, M, K, transA, ks, sa, ap, L.a_rb, L.kb);
        k_oz_slice<S><<<dim3(L.kb, L.b_rb), 256, 0, stream>>>(B, ldb, N, K, transB, nullptr, sb, bp, L.b_rb, L.kb);
        GAPRO_CUDA_TRY(cudaEventRecord(e1, stream));
        k_oz_gemm<S><<<tiles, OZ_THREADS, oz_smem_bytes(S), stream>>>(P);
        GAPRO_CUDA_TRY(cudaEventRecord(e2, stream));
    }
    GAPRO_KERNEL_CHECK();
    GAPRO_CUDA_TRY(cudaEventSynchronize(e2));
    if (ms_slice) GAPRO_CUDA_TRY(cudaEventElapsedTime(ms_slice, e0, e1));
    if (ms_gemm) GAPRO_CUDA_TRY(cudaEventElapsedTime(ms_gemm, e1, e2));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaEventDestroy(e2);
    return GAPRO_OK;
}

}  // namespace

extern "C" size_t gapro_ozaki_workspace_bytes(int32_t M, int32_t N, int32_t K, int32_t S) {
    if (M <= 0 || N <= 0 || K <= 0 || S < 2 || S > OZ_MAXS) return 0;
    return oz_layout(M, N, K, S).total;
}

// C[M, N] = op(A) op(B)^T in float64 through int8 digit planes on tcgen05.  trans = 0: the operand is stored
// [vectors, K] row-major; trans = 1: [K, vectors] row-major.  kscale (optional, K doubles) multiplies the A operand
// along k.  The last of `reps` runs is timed: ms_slice (scaling + digit planes), ms_gemm (the tcgen05 kernel).
extern "C" int gapro_ozaki_gemm(const double* A, int32_t lda, int32_t transA, const double* kscale, const double* B,
                                int32_t ldb, int32_t transB, int32_t M, int32_t N, int32_t K, int32_t S, double* C,
                                int32_t ldc, void* ws, size_t ws_bytes, int32_t reps, float* ms_slice, float* ms_gemm,
                                void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GAPRO_REQUIRE(A && B && C && ws, "gapro_ozaki_gemm: null pointer");
    GAPRO_REQUIRE(M > 0 && N > 0 && K > 0 && K <= 8192 && S >= 2 && S <= OZ_MAXS && reps >= 1,
                  "gapro_ozaki_gemm: bad sizes (K <= 8192 keeps the int32 accumulators exact; 2 <= S <= %d)", OZ_MAXS);
    const OzWs L = oz_layout(M, N, K, S);
    if (ws_bytes < L.total) {
        gapro_set_error("gapro_ozaki_gemm: workspace %zu < %zu bytes", ws_bytes, L.total);
        return GAPRO_ERR_WORKSPACE;
    }
    GAPRO_REQUIRE(((uintptr_t)ws & 1023) == 0, "gapro_ozaki_gemm: workspace must be 1024-byte aligned");
    switch (S) {
        case 2: return oz_run<2>(A, lda, transA, kscale, B, ldb, transB, M, N, K, C, ldc, ws, L, reps, ms_slice, ms_gemm, stream);
        case 3: return oz_run<3>(A, lda, transA, kscale, B, ldb, transB, M, N, K, C, ldc, ws, L, reps, ms_slice, ms_gemm, stream);
        case 4: return oz_run<4>(A, lda, transA, kscale, B, ldb, transB, M, N, K, C, ldc, ws, L, reps, ms_slice, ms_gemm, stream);
        case 5: return oz_run<5>(A, lda, transA, kscale, B, ldb, transB, M, N, K, C, ldc, ws, L, reps, ms_slice, ms_gemm, stream);
        case 6: return oz_run<6>(A, lda, transA, kscale, B, ldb, transB, M, N, K, C, ldc, ws, L, reps, ms_slice, ms_gemm, stream);
        case 7: return oz_run<7>(A, lda, transA, kscale, B, ldb, transB, M, N, K, C, ldc, ws, L, reps, ms_slice, ms_gemm, stream);
        default: return oz_run<8>(A, lda, transA, kscale, B, ldb, transB, M, N, K, C, ldc, ws, L, reps, ms_slice, ms_gemm, stream);
    }
}
