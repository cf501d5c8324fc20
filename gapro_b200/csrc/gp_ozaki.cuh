// The O(M^3) tile products of the GP step on tcgen05 for LARGE regions (included by gp_fit.cu inside its
// anonymous namespace; needs Region, Layout, GpParams, adam_update, Phase).
//
// A float64 product is evaluated from exact int8 digit-plane products (see ozaki.cu for the arithmetic and the
// error bound).  Per training step of a large region: 14 operand slicings (k_oz_vecmax_b + k_oz_slice_b: every
// operand matrix in the orientation its product contracts over, scaled per row / column by a power of two) and
// 8 launches of k_oz_gemm_b<PH> with the same fused epilogues as k_gemm<PH> (Adam on T, G_A assembly, the
// symmetrisations).  The products contract over the same triangular k-ranges as the DMMA path, in 64-deep blocks.
// Small regions keep the DMMA path; prediction keeps it for every region (1 of 51 passes).
#pragma once
#include "ozaki_ptx.cuh"

enum OzMat { OM_LINV = 0, OM_KZX, OM_T, OM_A, OM_BM, OM_GA };
enum OzBuf { OB_LR = 0, OB_LC, OB_X1, OB_X2, OB_X3, OB_COUNT };

// Digits per operand: 8, a 2^-55 truncation per operand (ozaki.cu).  6 and 7 digits (2^-41, 2^-48) miss the 1e-6
// parity bar on the golden regions (DESIGN.md section 4.1).
constexpr int OZ_S = 8;

__host__ __device__ inline int oz_rb(int Mp) { return (Mp + 127) / 128 * 2; }                // 64-vector blocks per plane row
__host__ __device__ inline size_t oz_plane_bytes(int Mp) { return (size_t)(Mp / 64) * oz_rb(Mp) * oz::OZ_BLK; }
__host__ __device__ inline size_t oz_buf_bytes(int Mp) { return (size_t)OZ_S * oz_plane_bytes(Mp); }
__host__ __device__ inline long long oz_region_doubles(int Mp) {
    return (long long)OB_COUNT * ((long long)(oz_buf_bytes(Mp) / 8) + (long long)oz_rb(Mp) * 64);
}
__device__ __forceinline__ uint8_t* oz_buf(double* ws, const Region& R, int b) {
    return reinterpret_cast<uint8_t*>(ws + R.oz_base) + (size_t)b * oz_buf_bytes(R.Mp);
}
__device__ __forceinline__ double* oz_scale(double* ws, const Region& R, int b) {
    return ws + R.oz_base + (long long)OB_COUNT * (long long)(oz_buf_bytes(R.Mp) / 8) + (long long)b * oz_rb(R.Mp) * 64;
}
__device__ __forceinline__ const double* oz_src(const Layout& lay, const double* base, const Region& R, int mat, int& ld) {
    switch (mat) {
        case OM_LINV: ld = R.Mp; return base + lay.Linv;
        case OM_KZX: ld = R.Wp; return base + lay.Kzx;
        case OM_T: ld = R.Mp; return base + lay.T;
        case OM_A: ld = R.Wp; return base + lay.A;
        case OM_BM: ld = R.Wp; return base + lay.Bm;
        default: ld = R.Mp; return base + lay.GA;
    }
}
// flags of a slicing
constexpr int OZF_TRANS = 1;   // vector v = column v of the matrix (k runs down the column); else row v
constexpr int OZF_GV = 2;      // multiply along k by g_v (the dT product A diag(g_v) B^T)
constexpr int OZF_YTRI = 4;    // source holds Y only in the tiles k_oz_gemm_b<PH_Y> wrote: (k, j) with 64*(j/64) <= 128*(k/128)+127

__device__ __forceinline__ bool oz_valid(int v, int k, int M, int flags) {
    if (v >= M || k >= M) return false;
    if (flags & OZF_YTRI) return ((v >> 6) << 6) <= ((k >> 7) << 7) + 127;
    return true;
}

// The scale buffer of an operand holds max_k |x(v, k)| per vector as a float64 bit pattern (positive doubles order like
// unsigned integers): zeroed by k_oz_zero_b, raised by k_oz_vecmax_b with atomicMax - grid (64-vector block, k-chunk),
// so that ONE large region still fills the GPU - and turned into the power-of-two scale 2^e, max 2^-e in [1/2, 1),
// where it is used (oz_pow2).
constexpr int OZ_KCH = 512;      // k-range of one k_oz_vecmax_b CTA

__device__ __forceinline__ double oz_pow2(double m) { return (m > 0.0 && m < 1e300) ? ldexp(1.0, ilogb(m) + 1) : 1.0; }

__global__ void __launch_bounds__(64)
k_oz_zero_b(const Region* __restrict__ regs, const int2* __restrict__ vblocks, double* __restrict__ ws, int buf) {
    const int2 vb = vblocks[blockIdx.x];
    const Region R = regs[vb.x];
    oz_scale(ws, R, buf)[vb.y * 64 + threadIdx.x] = 0.0;
}

__global__ void __launch_bounds__(256)
k_oz_vecmax_b(const Region* __restrict__ regs, const int2* __restrict__ vblocks, GpParams prm, double* __restrict__ ws,
              int mat, int flags, int buf) {
    __shared__ double red[4][64];
    const int2 vb = vblocks[blockIdx.x];
    const Region R = regs[vb.x];
    const int M = R.M;
    const int k_lo = blockIdx.y * OZ_KCH, k_hi = min(M, k_lo + OZ_KCH);
    if (k_lo >= M) return;
    const Layout lay = make_layout(R.Mp, R.Np, R.Wp, prm.D);
    const double* base = ws + R.base;
    int ld;
    const double* X = oz_src(lay, base, R, mat, ld);
    const double* ks = (flags & OZF_GV) ? base + lay.gv : nullptr;
    unsigned long long* mx = reinterpret_cast<unsigned long long*>(oz_scale(ws, R, buf));
    if (!(flags & OZF_TRANS)) {
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        for (int r = 0; r < 8; ++r) {
            const int v = vb.y * 64 + warp * 8 + r;
            if (v >= M) break;
            double m = 0.0;
            for (int k = k_lo + lane; k < k_hi; k += 32) m = fmax(m, fabs(X[(size_t)v * ld + k] * (ks ? ks[k] : 1.0)));
            for (int o = 16; o; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
            if (lane == 0 && m > 0.0) atomicMax(mx + v, (unsigned long long)__double_as_longlong(m));
        }
    } else {
        const int c = threadIdx.x & 63, rg = threadIdx.x >> 6, v = vb.y * 64 + c;
        double m = 0.0;
        if (v < M)
            for (int k = k_lo + rg; k < k_hi; k += 4)
                if (oz_valid(v, k, M, flags)) m = fmax(m, fabs(X[(size_t)k * ld + v] * (ks ? ks[k] : 1.0)));
        red[rg][c] = m;
        __syncthreads();
        if (rg == 0 && v < M) {
            m = fmax(fmax(red[0][c], red[1][c]), fmax(red[2][c], red[3][c]));
            if (m > 0.0) atomicMax(mx + v, (unsigned long long)__double_as_longlong(m));
        }
    }
}

// one 4 KB block (64 vectors x 64 k) of each of the OZ_S digit planes per CTA; table entry (region, kb, rb)
__global__ void __launch_bounds__(256)
k_oz_slice_b(const Region* __restrict__ regs, const int4* __restrict__ blocks, GpParams prm, double* __restrict__ ws,
             int mat, int flags, int buf) {
    const int4 e4 = blocks[blockIdx.x];
    const Region R = regs[e4.x];
    const Layout lay = make_layout(R.Mp, R.Np, R.Wp, prm.D);
    const double* base = ws + R.base;
    int ld;
    const double* X = oz_src(lay, base, R, mat, ld);
    const double* ks = (flags & OZF_GV) ? base + lay.gv : nullptr;
    const double* scale = oz_scale(ws, R, buf);
    const int M = R.M;
    oz::oz_slice_block<OZ_S>(
        X, ld, flags & OZF_TRANS, ks, e4.y, e4.z, [&](int v, int k) { return oz_valid(v, k, M, flags); },
        [&](int v) { return v < M ? 64.0 / oz_pow2(scale[v]) : 0.0; }, 1.0,      // exact: a power of two
        oz_buf(ws, R, buf), R.Mp / 64, oz_rb(R.Mp));      // oz_plane_bytes(R.Mp) per plane
}

// C tile (128 x 64) of phase PH for one large region; table entry (region, ti, tj)
template <int PH>
__global__ void __launch_bounds__(oz::OZ_THREADS, 1)
k_oz_gemm_b(const Region* __restrict__ regs, const int4* __restrict__ tiles, GpParams prm, double* __restrict__ ws,
            int abuf, int bbuf) {
    using namespace oz;
    extern __shared__ __align__(1024) uint8_t oz_smem_b[];
    const int4 t4 = tiles[blockIdx.x];
    const Region R = regs[t4.x];
    const int ti = t4.y, tj = t4.z;
    const int kbt = (R.M + 63) >> 6;                 // k-blocks that hold data
    // contraction range in 64-deep blocks (the triangular structure of the operands, as in k_gemm)
    int k0 = 0, k1 = kbt;
    if (PH == PH_A || PH == PH_GA) k1 = min(kbt, 2 * ti + 2);             // A operand lower triangular: k <= i
    if (PH == PH_B || PH == PH_GC || PH == PH_GK) k0 = min(kbt, 2 * ti);  // A operand = transposed lower: k >= i
    if (PH == PH_Y) k0 = min(kbt, tj);                                    // B operand = L^-1 columns: k >= j
    // the phase epilogue of one 16-column chunk of tile row `row`
    const auto epi = [&](int row, int c, double(&acc)[16]) {
        const int Mp = R.Mp, Wp = R.Wp, M = R.M;
        const int gr = ti * OZ_BM + row, gc0 = tj * OZ_BN + 16 * c;
        if (gr >= Mp || gc0 >= Mp) return;                  // outside the allocated matrix (128-row tiles overhang)
        const Layout lay = make_layout(R.Mp, R.Np, R.Wp, prm.D);
        double* base = ws + R.base;
        const double sa = gr < M ? oz_pow2(oz_scale(ws, R, abuf)[gr]) : 0.0;
        const double* sbv = oz_scale(ws, R, bbuf);
#pragma unroll
        for (int j = 0; j < 16; ++j) acc[j] = (gc0 + j < M) ? acc[j] * sa * oz_pow2(sbv[gc0 + j]) : 0.0;
        if (PH == PH_A || PH == PH_B) {
            double* out = base + (PH == PH_A ? lay.A : lay.Bm) + (size_t)gr * Wp + gc0;
#pragma unroll
            for (int j = 0; j < 16; j += 2) *reinterpret_cast<double2*>(out + j) = make_double2(acc[j], acc[j + 1]);
        } else if (PH == PH_GA) {        // G_A = m g_mu^T + 2 (T B - A) diag(g_v)
            const double2* Am = reinterpret_cast<const double2*>(base + lay.A + (size_t)gr * Wp + gc0);
            const double mi = base[lay.m + gr];
            const double2* gmu = reinterpret_cast<const double2*>(base + lay.gmu + gc0);
            const double2* gv = reinterpret_cast<const double2*>(base + lay.gv + gc0);
            double2* out = reinterpret_cast<double2*>(base + lay.GA + (size_t)gr * Mp + gc0);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const double2 a = Am[j], u = gmu[j], w = gv[j];
                out[j] = make_double2(mi * u.x + 2.0 * w.x * (acc[2 * j] - a.x), mi * u.y + 2.0 * w.y * (acc[2 * j + 1] - a.y));
            }
        } else if (PH == PH_GT) {        // dT = tril(2 A diag(g_v) B^T + (T - diag(1/T_ii))/N), Adam on T
            const double invN = 1.0 / (double)M;
            if (gr < M) {
#pragma unroll
                for (int j = 0; j < 16; j += 2) {
                    const int cc = gc0 + j;
                    const size_t idx = (size_t)gr * Mp + cc;
                    if (cc + 1 <= gr) {          // both elements in the lower triangle: 128-bit loads / stores
                        double2 p = *reinterpret_cast<const double2*>(base + lay.T + idx);
                        double2 m1 = *reinterpret_cast<const double2*>(base + lay.Tm + idx);
                        double2 m2 = *reinterpret_cast<const double2*>(base + lay.Tv + idx);
                        const double ga = 2.0 * acc[j] + p.x * invN;
                        const double gb = 2.0 * acc[j + 1] + (p.y - (cc + 1 == gr ? 1.0 / p.y : 0.0)) * invN;
                        adam_update(p.x, m1.x, m2.x, ga, prm);
                        adam_update(p.y, m1.y, m2.y, gb, prm);
                        *reinterpret_cast<double2*>(base + lay.T + idx) = p;
                        *reinterpret_cast<double2*>(base + lay.Tm + idx) = m1;
                        *reinterpret_cast<double2*>(base + lay.Tv + idx) = m2;
                    } else if (cc == gr) {       // the diagonal element alone
                        double p = base[lay.T + idx];
                        const double g = 2.0 * acc[j] + (p - 1.0 / p) * invN;
                        double m1 = base[lay.Tm + idx], m2 = base[lay.Tv + idx];
                        adam_update(p, m1, m2, g, prm);
                        base[lay.T + idx] = p;
                        base[lay.Tm + idx] = m1;
                        base[lay.Tv + idx] = m2;
                    }
                }
            }
        } else if (PH == PH_GC || PH == PH_Y) {
            double* out = base + (PH == PH_GC ? lay.GC : lay.GA) + (size_t)gr * Mp + gc0;
#pragma unroll
            for (int j = 0; j < 16; j += 2) *reinterpret_cast<double2*>(out + j) = make_double2(acc[j], acc[j + 1]);
        } else if (PH == PH_GL) {        // S = -sym(Phi(G_A A^T)) mirrored, into the B buffer
            double* out = base + lay.Bm;
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const int cc = gc0 + j;
                const double val = -0.5 * acc[j];
                if (cc <= gr) {
                    out[(size_t)gr * Wp + cc] = val;
                    if (cc < gr) out[(size_t)cc * Wp + gr] = val;
                }
            }
        } else if (PH == PH_GK) {        // G_K = L^-T Y, symmetric: lower part + mirror, into the B buffer
            double* out = base + lay.Bm;
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const int cc = gc0 + j;
                if (cc <= gr) {
                    out[(size_t)gr * Wp + cc] = acc[j];
                    if (cc < gr) out[(size_t)cc * Wp + gr] = acc[j];
                }
            }
        }
    };
    const size_t kstride = (size_t)oz_rb(R.Mp) * OZ_BLK, plane = oz_plane_bytes(R.Mp);
    oz_tile<OZ_S>(oz_smem_b, oz_buf(ws, R, abuf) + k0 * kstride + (size_t)2 * ti * OZ_BLK, kstride, plane,
                  oz_buf(ws, R, bbuf) + k0 * kstride + (size_t)tj * OZ_BLK, kstride, plane, k1 - k0, epi);
}
