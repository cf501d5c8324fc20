// Stage C — batched variational-GP regions (sm_100a), float64.
//
// Replaces fit_gp_spp (/root/reference/gapro/gaussian_process_utils.py:382-445) and the gpytorch
// machinery behind GPClassificationModel (:11-25); the arithmetic is SURVEY.md §8a-C, implemented
// with the hand-derived gradient.  Every region's matrices are padded to multiples of 64 and live
// in the caller's workspace; one training step is a fixed sequence of ragged, batched tile
// kernels over ALL regions of a chunk (tile tables built on the host), so small and large regions
// share launches and the 148 SMs see thousands of independent 64x64 tiles per launch:
//
//   build K_zz, K_zx  ->  blocked left-looking Cholesky with the inverse factor built alongside
//   ->  A = L^-1 K_zx  ->  B = T^T A  ->  column stats + Gauss-Hermite  ->  G_A  ->  dT (+Adam)
//   ->  dm (+Adam)  ->  G_C = L^-T G_A  ->  G_L  ->  sym(Phi(L^T G_L))  ->  Y  ->  G_K
//   ->  kernel-parameter / inducing-point gradients  ->  Adam on Z, c, rho_s, rho_l.
//
// All O(M^3) products run on the FP64 tensor pipe (mma.sync m8n8k4 f64, "DMMA") from shared
// memory tiles filled by cp.async double buffering.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "common.cuh"

namespace {

constexpr int TB = 64;            // tile edge; every matrix dimension is padded to a multiple of it
constexpr int BK = 16;            // k-chunk staged per pipeline stage
constexpr int LDK = BK + 2;       // smem row stride of a k-contiguous operand tile  [64][LDK]
constexpr int STAGE = TB * LDK;   // doubles per operand stage (>= BK*TB of the swizzled m/n-contiguous tile)
constexpr int GEMM_THREADS = 128;
constexpr int N_GH = 20;
constexpr double MIN_VARIANCE = 1e-6;
constexpr double MEAN_INIT_STD = 1e-3;
constexpr double BETA1 = 0.9, BETA2 = 0.999, ADAM_EPS = 1e-8;

__constant__ double c_gh_t[N_GH] = {
    -5.38748089001123276e+00, -4.60368244955074424e+00, -3.94476404011562520e+00, -3.34785456738321630e+00,
    -2.78880605842813045e+00, -2.25497400208927568e+00, -1.73853771211658614e+00, -1.23407621539532308e+00,
    -7.37473728545394391e-01, -2.45340708300901239e-01, 2.45340708300901239e-01,  7.37473728545394391e-01,
    1.23407621539532308e+00,  1.73853771211658614e+00,  2.25497400208927568e+00,  2.78880605842813045e+00,
    3.34785456738321630e+00,  3.94476404011562520e+00,  4.60368244955074424e+00,  5.38748089001123276e+00};
__constant__ double c_gh_w[N_GH] = {
    2.22939364553414471e-13, 4.39934099227317473e-10, 1.08606937076927821e-07, 7.80255647853205987e-06,
    2.28338636016353646e-04, 3.24377334223785669e-03, 2.48105208874636433e-02, 1.09017206020023294e-01,
    2.86675505362834149e-01, 4.62243669600610085e-01, 4.62243669600610085e-01, 2.86675505362834149e-01,
    1.09017206020023294e-01, 2.48105208874636433e-02, 3.24377334223785669e-03, 2.28338636016353646e-04,
    7.80255647853205987e-06, 1.08606937076927821e-07, 4.39934099227317473e-10, 2.22939364553414471e-13};

// ---------------------------------------------------------------------------------------------
// region descriptor and workspace layout
// ---------------------------------------------------------------------------------------------
struct Region {
    int M, N;          // training rows (= inducing points), test rows
    int Mp, Np, Wp;    // padded: Mp = ceil64(M), Np = ceil64(N), Wp = max(Mp, Np)
    int nb, nbw;       // Mp/64, Wp/64
    int n_b1;          // first n_b1 training rows carry label -1
    int train_off, test_off;
    int orig;          // index in the caller's region order
    int oz;            // 1: the tile products of the training steps run on tcgen05 (gp_ozaki.cuh)
    long long base;    // offset of the region's buffers in the workspace, in doubles
    long long oz_base; // offset of the digit-plane buffers (oz regions), in doubles
};

struct Layout {
    long long X, Z, Zm, Zv, gZ, Xt, y, m, mm, mv, scal, mu, var, gmu, gv, gsrow, glrow;
    long long L, Linv, T, Tm, Tv, GA, GC, Kc, Kzx, A, Bm, total;
};
enum { SC_C = 0, SC_RS = 1, SC_RL = 2, SC_M0 = 3, SC_V0 = 6, SC_N = 16 };

__host__ __device__ inline long long ev2(long long x) { return (x + 1) & ~1LL; }

__host__ __device__ inline Layout make_layout(int Mp, int Np, int Wp, int D) {
    Layout l;
    long long o = 0;
    const long long zd = ev2((long long)Mp * D);
    l.X = o; o += zd;
    l.Z = o; o += zd;
    l.Zm = o; o += zd;
    l.Zv = o; o += zd;
    l.gZ = o; o += zd;
    l.Xt = o; o += ev2((long long)Np * D);
    l.y = o; o += Mp;
    l.m = o; o += Mp;
    l.mm = o; o += Mp;
    l.mv = o; o += Mp;
    l.scal = o; o += SC_N;
    l.mu = o; o += Wp;
    l.var = o; o += Wp;
    l.gmu = o; o += Wp;
    l.gv = o; o += Wp;
    l.gsrow = o; o += Mp;
    l.glrow = o; o += Mp;
    const long long mm = (long long)Mp * Mp, mw = (long long)Mp * Wp;
    l.L = o; o += mm;
    l.Linv = o; o += mm;
    l.T = o; o += mm;
    l.Tm = o; o += mm;
    l.Tv = o; o += mm;
    l.GA = o; o += mm;
    l.GC = o; o += mm;
    l.Kc = o; o += mm;
    l.Kzx = o; o += mw;
    l.A = o; o += mw;
    l.Bm = o; o += mw;
    l.total = o;
    return l;
}

struct GpParams {
    int D;
    double jitter_zz, jitter_xx;
    double lr_over_bc1, bc2_sqrt;   // Adam scalars of the current step
    int predict;                    // 1: columns are the test rows
};

__device__ __forceinline__ double softplus_d(double x) { return log1p(exp(-fabs(x))) + fmax(x, 0.0); }
__device__ __forceinline__ double sigmoid_d(double x) { return 1.0 / (1.0 + exp(-x)); }

__device__ __forceinline__ void adam_update(double& p, double& m, double& v, double g, const GpParams& prm) {
    m = BETA1 * m + (1.0 - BETA1) * g;
    v = BETA2 * v + (1.0 - BETA2) * g * g;
    p -= prm.lr_over_bc1 * m / (sqrt(v) / prm.bc2_sqrt + ADAM_EPS);
}

// ---------------------------------------------------------------------------------------------
// 64x64xK tile product on the FP64 tensor pipe
// ---------------------------------------------------------------------------------------------
constexpr int NSTAGE = 3;
struct GemmSmem {
    double a[NSTAGE][STAGE];
    double b[NSTAGE][STAGE];
};
constexpr int GEMM_SMEM = (int)sizeof(GemmSmem);

__device__ __forceinline__ void cp_async16(double* smem_dst, const double* gmem_src) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__device__ __forceinline__ void dmma(double& d0, double& d1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(d0), "+d"(d1)
                 : "d"(a), "d"(b));
}

// Operand tile: 64 rows (m or n) x 16 k, staged so that every fragment load is a conflict-free
// 128-bit shared load.
//   KC = true : element(r,k) = g[r*ld + k]; smem [64][LDK] (k contiguous, rows padded to 18 doubles)
//   KC = false: element(r,k) = g[k*ld + r]; smem [16][64]  (r contiguous, 16-byte units XOR-swizzled
//               with swz(k) so that the four k-rows a quarter-warp touches fall into distinct banks)
// Fragment <-> matrix maps (the k order inside a chunk is free as long as A and B agree):
//   k of MMA step kk for lane (gid, tig): 4*tig + kk
//   row of sub-tile i for lane gid:       KC ? 8*i + gid : 4*gid + i
__device__ __forceinline__ int swz(int k) { return ((k >> 2) & 1) | (((k >> 3) & 1) << 2); }

template <bool KC>
__device__ __forceinline__ int frag_row(int i, int g) { return KC ? 8 * i + g : 4 * g + i; }

// Which 32x32 quadrant of the tile a warp owns.  Warp w always runs on scheduler partition w mod 4, and
// the quadrants do unequal work on triangular / padded tiles; rotating the assignment with the block
// index spreads the lighter quadrants over all four partitions of an SM instead of always the same two.
__device__ __forceinline__ int warp_quadrant() { return (int)((threadIdx.x >> 5) ^ (blockIdx.x & 3u)); }

// Thread -> data map of the loaders: every warp-wide 16-byte cp.async lands on distinct banks
// (k-contiguous tile: 4 rows x 8 units, bank = (row + unit) mod 8 with the 9-unit row stride;
//  r-contiguous tile: one k-row x 32 units, XOR-swizzle permutes banks inside each group of 8).
template <bool KC>
__device__ __forceinline__ void load_stage(double* s, const double* g, int ld, int k) {
    const int t = threadIdx.x;
    if (KC) {
        const int u = t & 7, rr = t >> 3;                 // unit (2 doubles) in the row, row in the pass
        const double* src = g + (size_t)rr * ld + k + 2 * u;
        double* dst = s + rr * LDK + 2 * u;
#pragma unroll
        for (int q = 0; q < 4; ++q) cp_async16(dst + q * 16 * LDK, src + (size_t)q * 16 * ld);
    } else {
        const int u = t & 31, kr = t >> 5;                // unit in the k-row, k-row in the pass
        const double* src = g + (size_t)(k + kr) * ld + 2 * u;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int kk = kr + 4 * q;
            cp_async16(s + kk * TB + 2 * (u ^ swz(kk)), src + (size_t)4 * q * ld);
        }
    }
}

// two MMA steps (kk = 2*h, 2*h+1) worth of fragments of one operand: f[i][0..1]
template <bool KC>
__device__ __forceinline__ void load_frags(double (&f)[4][2], const double* s, int w32, int gid, int tig, int h) {
    if (KC) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const double2 v = *reinterpret_cast<const double2*>(s + (w32 + 8 * i + gid) * LDK + 4 * tig + 2 * h);
            f[i][0] = v.x;
            f[i][1] = v.y;
        }
    } else {
        const int u0 = (w32 >> 1) + 2 * gid, x = swz(4 * tig);
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const double* row = s + (4 * tig + 2 * h + e) * TB;
            const double2 lo = *reinterpret_cast<const double2*>(row + 2 * (u0 ^ x));
            const double2 hi = *reinterpret_cast<const double2*>(row + 2 * ((u0 + 1) ^ x));
            f[0][e] = lo.x;
            f[1][e] = lo.y;
            f[2][e] = hi.x;
            f[3][e] = hi.y;
        }
    }
}

// acc[i][j][e] holds C(row, col) with row = wm*32 + frag_row<AKC>(i, gid),
//                                      col = wn*32 + frag_row<BKC>(j, 2*tig + e)
// Three-stage cp.async pipeline, one __syncthreads per 16-deep chunk.
template <bool AKC, bool BKC, int TRI = 0>
__device__ __forceinline__ void gemm_accum(double (&acc)[4][4][2], const double* __restrict__ A, int lda,
                                           const double* __restrict__ B, int ldb, int k0, int k1,
                                           const double* __restrict__ kscale, GemmSmem& sm, int mlim = TB,
                                           int nlim = TB, int tri0 = 0) {
    const int lane = threadIdx.x & 31, warp = warp_quadrant();
    const int gid = lane >> 2, tig = lane & 3;
    const int wm32 = (warp >> 1) * 32, wn32 = (warp & 1) * 32;
    // a warp whose 32x32 block lies entirely in the zero padding only helps with the loads
    const bool active = wm32 < mlim && wn32 < nlim;
    // triangular operand: the warp's 32 rows (TRI = +-1, A operand) or columns (TRI = 2, B operand) see only
    // zeros beyond / before the diagonal, so it may skip those chunks (tri0 = first row / column of the tile)
    //   TRI = +1: A(r,k) = 0 for k > r      TRI = -1: A(r,k) = 0 for k < r      TRI = 2: B(c,k) = 0 for k < c
    const int wk_hi = TRI == 1 ? tri0 + wm32 + 32 : 0x7fffffff;
    const int wk_lo = TRI == -1 ? tri0 + wm32 : (TRI == 2 ? tri0 + wn32 : 0);
    const int nchunk = (k1 - k0) / BK;
    if (nchunk <= 0) return;
#pragma unroll
    for (int s = 0; s < NSTAGE - 1; ++s) {
        if (s < nchunk) {
            load_stage<AKC>(sm.a[s], A, lda, k0 + s * BK);
            load_stage<BKC>(sm.b[s], B, ldb, k0 + s * BK);
        }
        cp_async_commit();
    }
    int stage = 0;
    for (int c = 0; c < nchunk; ++c) {
        double2 sc0 = make_double2(1.0, 1.0), sc1 = sc0;
        if (kscale) {                  // issued ahead of the barrier so the global latency is hidden
            const double2* kp = reinterpret_cast<const double2*>(kscale + k0 + c * BK + 4 * tig);
            sc0 = __ldg(kp);
            sc1 = __ldg(kp + 1);
        }
        cp_async_wait<NSTAGE - 2>();   // chunk c has landed
        __syncthreads();               // ... for every thread, and chunk c-1 is fully consumed
        {
            const int nc = c + NSTAGE - 1;
            int ns = stage + NSTAGE - 1;
            if (ns >= NSTAGE) ns -= NSTAGE;
            if (nc < nchunk) {
                load_stage<AKC>(sm.a[ns], A, lda, k0 + nc * BK);
                load_stage<BKC>(sm.b[ns], B, ldb, k0 + nc * BK);
            }
            cp_async_commit();
        }
        const double* sa = sm.a[stage];
        const double* sb = sm.b[stage];
        bool on = active;
        if (TRI != 0) {
            const int kc = k0 + c * BK;
            on = on && kc < wk_hi && kc + BK > wk_lo;
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            if (!on) break;
            double af[4][2], bf[4][2];
            load_frags<AKC>(af, sa, wm32, gid, tig, h);
            load_frags<BKC>(bf, sb, wn32, gid, tig, h);
            if (kscale) {
                const double2 sc = h ? sc1 : sc0;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    af[i][0] *= sc.x;
                    af[i][1] *= sc.y;
                }
            }
#pragma unroll
            for (int e = 0; e < 2; ++e)
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) dmma(acc[i][j][0], acc[i][j][1], af[i][e], bf[j][e]);
        }
        if (++stage == NSTAGE) stage = 0;
    }
    cp_async_wait<0>();
    __syncthreads();   // the stages may be reused (next product, or aliased scratch) right after
}

// Visits the accumulator as pairs of horizontally adjacent elements: v0 = C(row, col), v1 = C(row, col+1).
#define ACC_FOREACH(AKC_, BKC_, ROW0, COL0, ...)                                                   \
    {                                                                                              \
        const int lane_ = threadIdx.x & 31, warp_ = warp_quadrant();                               \
        const int gid_ = lane_ >> 2, tig_ = lane_ & 3;                                             \
        const int wm_ = warp_ >> 1, wn_ = warp_ & 1;                                               \
        _Pragma("unroll") for (int i_ = 0; i_ < 4; ++i_) {                                         \
            _Pragma("unroll") for (int p_ = 0; p_ < 4; ++p_) {                                     \
                const int row = (ROW0) + wm_ * 32 + frag_row<AKC_>(i_, gid_);                      \
                const int col = (COL0) + wn_ * 32 +                                                \
                                ((BKC_) ? 8 * p_ + 2 * tig_ : 8 * tig_ + 4 * (p_ >> 1) + 2 * (p_ & 1)); \
                double& v0 = (BKC_) ? acc[i_][p_][0] : acc[i_][2 * (p_ & 1)][p_ >> 1];             \
                double& v1 = (BKC_) ? acc[i_][p_][1] : acc[i_][2 * (p_ & 1) + 1][p_ >> 1];         \
                __VA_ARGS__                                                                        \
            }                                                                                      \
        }                                                                                          \
    }

enum Phase {
    PH_BUILD = 0, PH_CHOL, PH_A, PH_B, PH_COLSTATS, PH_GA, PH_GT, PH_GM, PH_GC, PH_GL, PH_SP, PH_Y, PH_GK,
    PH_KGRAD, PH_ADAM, PH_COUNT
};

template <int PH>
__global__ void __launch_bounds__(GEMM_THREADS, 4)
k_gemm(const Region* __restrict__ regs, const int4* __restrict__ tiles, GpParams prm, double* __restrict__ ws) {
    extern __shared__ __align__(16) unsigned char smem_gemm[];
    GemmSmem& sm = *reinterpret_cast<GemmSmem*>(smem_gemm);
    const int4 t = tiles[blockIdx.x];
    const Region R = regs[t.x];
    const int ti = t.y, tj = t.z;
    const Layout lay = make_layout(R.Mp, R.Np, R.Wp, prm.D);
    double* base = ws + R.base;
    const int Mp = R.Mp, Wp = R.Wp;
    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    const int r0 = ti * TB, c0 = tj * TB;
    // padding rows/columns are exact zeros in every operand of these products: clip the contraction to
    // the real size (rounded to the chunk) and skip warps that would only produce padding
    const int kend = (R.M + BK - 1) / BK * BK;
    const int ncol = prm.predict ? R.N : R.M;
    const int mlim = (R.M + 31) / 32 * 32 - r0, nlim = (ncol + 31) / 32 * 32 - c0;
#define KCLIP(k) ((k) < kend ? (k) : kend)

    if (PH == PH_A) {          // A = Linv * Kzx, Linv lower: k <= i
        gemm_accum<true, false, 1>(acc, base + lay.Linv + (size_t)r0 * Mp, Mp, base + lay.Kzx + c0, Wp, 0,
                                   KCLIP(r0 + TB), nullptr, sm, mlim, nlim, r0);
        double* out = base + lay.A;
        ACC_FOREACH(true, false, r0, c0, { *reinterpret_cast<double2*>(out + (size_t)row * Wp + col) = make_double2(v0, v1); })
    } else if (PH == PH_B) {   // B = T^T * A, T lower: k >= i
        gemm_accum<false, false, -1>(acc, base + lay.T + r0, Mp, base + lay.A + c0, Wp, r0, kend, nullptr, sm, mlim,
                                     nlim, r0);
        double* out = base + lay.Bm;
        ACC_FOREACH(false, false, r0, c0, { *reinterpret_cast<double2*>(out + (size_t)row * Wp + col) = make_double2(v0, v1); })
    } else if (PH == PH_GA) {  // G_A = m g_mu^T + 2 (T B - A) diag(g_v)
        gemm_accum<true, false, 1>(acc, base + lay.T + (size_t)r0 * Mp, Mp, base + lay.Bm + c0, Wp, 0, KCLIP(r0 + TB),
                                   nullptr, sm, mlim, nlim, r0);
        const double* Am = base + lay.A;
        const double* mv = base + lay.m;
        const double* gmu = base + lay.gmu;
        const double* gv = base + lay.gv;
        double* out = base + lay.GA;
        ACC_FOREACH(true, false, r0, c0, {
            const double2 a = *reinterpret_cast<const double2*>(Am + (size_t)row * Wp + col);
            const double mi = mv[row];
            double2 o;
            o.x = mi * gmu[col] + 2.0 * gv[col] * (v0 - a.x);
            o.y = mi * gmu[col + 1] + 2.0 * gv[col + 1] * (v1 - a.y);
            *reinterpret_cast<double2*>(out + (size_t)row * Mp + col) = o;
        })
    } else if (PH == PH_GT) {  // dT = tril(2 A diag(g_v) B^T + (T - diag(1/T_ii))/N), Adam on T
        gemm_accum<true, true>(acc, base + lay.A + (size_t)r0 * Wp, Wp, base + lay.Bm + (size_t)c0 * Wp, Wp, 0, kend,
                               base + lay.gv, sm, mlim, nlim);
        double* T = base + lay.T;
        double* Tm = base + lay.Tm;
        double* Tv = base + lay.Tv;
        const double invN = 1.0 / (double)R.M;
        ACC_FOREACH(true, true, r0, c0, {
            if (row < R.M && col + 1 <= row) {
                // both elements of the pair lie in the lower triangle (col is even; the second one may be the diagonal):
                // 128-bit loads / stores of T and its two Adam moments
                const size_t idx = (size_t)row * Mp + col;
                double2 p = *reinterpret_cast<const double2*>(T + idx);
                double2 m1 = *reinterpret_cast<const double2*>(Tm + idx), m2 = *reinterpret_cast<const double2*>(Tv + idx);
                const double ga = 2.0 * v0 + p.x * invN;
                const double gb = 2.0 * v1 + (p.y - (col + 1 == row ? 1.0 / p.y : 0.0)) * invN;
                adam_update(p.x, m1.x, m2.x, ga, prm);
                adam_update(p.y, m1.y, m2.y, gb, prm);
                *reinterpret_cast<double2*>(T + idx) = p;
                *reinterpret_cast<double2*>(Tm + idx) = m1;
                *reinterpret_cast<double2*>(Tv + idx) = m2;
            } else if (row < R.M && col <= row) {      // col == row: the diagonal element alone
                const size_t idx = (size_t)row * Mp + col;
                double p = T[idx];
                const double g = 2.0 * v0 + (p - 1.0 / p) * invN;
                double m1 = Tm[idx], m2 = Tv[idx];
                adam_update(p, m1, m2, g, prm);
                T[idx] = p;
                Tm[idx] = m1;
                Tv[idx] = m2;
            }
        })
    } else if (PH == PH_GC) {  // G_C = Linv^T * G_A: k >= i
        gemm_accum<false, false, -1>(acc, base + lay.Linv + r0, Mp, base + lay.GA + c0, Mp, r0, kend, nullptr, sm, mlim,
                                     nlim, r0);
        double* out = base + lay.GC;
        ACC_FOREACH(false, false, r0, c0, { *reinterpret_cast<double2*>(out + (size_t)row * Mp + col) = make_double2(v0, v1); })
    } else if (PH == PH_GL) {
        // Cholesky adjoint without forming G_L: with Q = G_A A^T,
        //   dLoss/dK_zz = -Linv^T sym(Phi(Q)) Linv,   sym(Phi(Q)) = 1/2 tril(Q) mirrored
        // (from dA = -Phi(L^-1 dK L^-T) A; identical to L^-T sym(Phi(L^T G_L)) L^-1 with G_L = -tril(L^-T Q)).
        // This phase writes S = -sym(Phi(Q)) into the B buffer.
        gemm_accum<true, true>(acc, base + lay.GA + (size_t)r0 * Mp, Mp, base + lay.A + (size_t)c0 * Wp, Wp, 0, kend,
                               nullptr, sm, mlim, nlim);
        double* out = base + lay.Bm;
        ACC_FOREACH(true, true, r0, c0, {
            _Pragma("unroll") for (int e = 0; e < 2; ++e) {
                const int cc = col + e;
                const double v = -0.5 * (e ? v1 : v0);
                if (cc <= row) {
                    out[(size_t)row * Wp + cc] = v;
                    if (cc < row) out[(size_t)cc * Wp + row] = v;
                }
            }
        })
    } else if (PH == PH_Y) {   // Y = S * Linv: k >= j, lower tiles only (all that G_K's lower tiles read; into the G_A buffer)
        gemm_accum<true, false, 2>(acc, base + lay.Bm + (size_t)r0 * Wp, Wp, base + lay.Linv + c0, Mp, c0, kend, nullptr,
                                   sm, mlim, nlim, c0);
        double* out = base + lay.GA;
        ACC_FOREACH(true, false, r0, c0, { *reinterpret_cast<double2*>(out + (size_t)row * Mp + col) = make_double2(v0, v1); })
    } else if (PH == PH_GK) {  // G_K = Linv^T * Y (symmetric): lower tiles, mirrored   (into the B buffer)
        gemm_accum<false, false, -1>(acc, base + lay.Linv + r0, Mp, base + lay.GA + c0, Mp, r0, kend, nullptr, sm, mlim,
                                     nlim, r0);
        double* out = base + lay.Bm;
        ACC_FOREACH(false, false, r0, c0, {
            *reinterpret_cast<double2*>(out + (size_t)row * Wp + col) = make_double2(v0, v1);
            if (ti != tj) {
                out[(size_t)col * Wp + row] = v0;
                out[(size_t)(col + 1) * Wp + row] = v1;
            }
        })
    }
}

#undef KCLIP

#include "gp_ozaki.cuh"

// ---------------------------------------------------------------------------------------------
// kernel matrices: K_zz = s exp(-r2/2) + jitter I (lower tiles), K_zx = s exp(-r2/2)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_build(const Region* __restrict__ regs, const int4* __restrict__ tiles, GpParams prm, double* __restrict__ ws) {
    extern __shared__ double smem_build[];
    const int D = prm.D;
    const int4 t = tiles[blockIdx.x];
    const Region R = regs[t.x];
    const int ti = t.y, tj = t.z;
    const Layout lay = make_layout(R.Mp, R.Np, R.Wp, D);
    double* base = ws + R.base;
    // row block [64][D] (read as broadcasts), column blocks transposed [D][65] (lanes read consecutive words)
    constexpr int LDT = TB + 1;
    double* zi = smem_build;
    double* zjT = zi + TB * D;
    double* xjT = zjT + D * LDT;
    const double* Z = base + lay.Z;
    const double* Xc = prm.predict ? base + lay.Xt : base + lay.X;
    const int ncols = prm.predict ? R.N : R.M;       // valid columns of K_zx
    const int colrows = prm.predict ? R.Np : R.Mp;   // allocated rows of the column matrix
    const bool do_zz = (tj <= ti) && (tj < R.nb);
    const bool have_x = (tj + 1) * TB <= colrows;
    for (int e = threadIdx.x; e < TB * D; e += blockDim.x) {
        const int r = e / D, d = e - r * D;
        zi[e] = Z[(size_t)ti * TB * D + e];
        zjT[d * LDT + r] = do_zz ? Z[(size_t)tj * TB * D + e] : 0.0;
        xjT[d * LDT + r] = have_x ? Xc[(size_t)tj * TB * D + e] : 0.0;
    }
    __syncthreads();
    const double* sc = base + lay.scal;
    const double ell = softplus_d(sc[SC_RL]), s = softplus_d(sc[SC_RS]);
    const double inv_l2 = 1.0 / (ell * ell);
    double* Kzx = base + lay.Kzx;
    double* Kzz = base + lay.L;
    double* Kc = base + lay.Kc;
    // thread = (column lj, 16 rows): the column's features are read once per d and reused over the rows
    const int lj = threadIdx.x & 63, lq = threadIdx.x >> 6;
    const int j = tj * TB + lj;
    double d2x[16], d2z[16];
#pragma unroll
    for (int q = 0; q < 16; ++q) d2x[q] = d2z[q] = 0.0;
    for (int d = 0; d < D; ++d) {
        const double xv = xjT[d * LDT + lj], zv = zjT[d * LDT + lj];
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const double zr = zi[(lq * 16 + q) * D + d];          // warp-uniform address: broadcast
            const double a = zr - xv, b = zr - zv;
            d2x[q] = fma(a, a, d2x[q]);
            d2z[q] = fma(b, b, d2z[q]);
        }
    }
#pragma unroll
    for (int q = 0; q < 16; ++q) {
        const int i = ti * TB + lq * 16 + q;
        Kzx[(size_t)i * R.Wp + j] = (i < R.M && j < ncols) ? s * exp(-0.5 * (d2x[q] * inv_l2)) : 0.0;
        if (do_zz) {
            double v, v0 = 0.0;
            if (i < R.M && j < R.M) {
                v0 = s * exp(-0.5 * (d2z[q] * inv_l2));
                v = v0 + (i == j ? prm.jitter_zz : 0.0);
            } else {
                v = (i == j) ? 1.0 : 0.0;
            }
            Kzz[(size_t)i * R.Mp + j] = v;
            Kc[(size_t)i * R.Mp + j] = v0;            // jitter-free copy (both halves) for the gradient kernel
            if (ti != tj) Kc[(size_t)j * R.Mp + i] = v0;
        }
    }
}

// Wide-feature variant (8 < D <= 64): the squared distances are a real dense contraction over the feature dimension,
//   r^2(i, j) = |z_i|^2 + |x_j|^2 - 2 z_i . x_j   (clamped at 0, gpytorch's `sq_dist`),
// and the dot products run on the FP64 tensor pipe: warp = 8 rows x 64 columns of the tile, mma.sync m8n8k4 over the
// features, operands staged row-major in shared memory (row stride D + 4: conflict-free fragment loads).
template <int NCH>
constexpr int build_wide_smem() { return (3 * 64 * (32 * NCH + 4) + 3 * 64) * (int)sizeof(double); }

template <int NCH>
__global__ void __launch_bounds__(256)
k_build_wide(const Region* __restrict__ regs, const int4* __restrict__ tiles, GpParams prm, double* __restrict__ ws) {
    constexpr int DP = 32 * NCH, LDZ = DP + 4;
    extern __shared__ __align__(16) double smem_bw[];
    double* zi = smem_bw;                // rows of the tile's row block     [64][LDZ]
    double* zj = zi + 64 * LDZ;          // rows of Z of the column block
    double* xj = zj + 64 * LDZ;          // rows of X (or the test rows) of the column block
    double* ni = xj + 64 * LDZ;          // squared norms
    double* nzj = ni + 64;
    double* nxj = nzj + 64;
    const int D = prm.D;
    const int4 t = tiles[blockIdx.x];
    const Region R = regs[t.x];
    const int ti = t.y, tj = t.z;
    const Layout lay = make_layout(R.Mp, R.Np, R.Wp, D);
    double* base = ws + R.base;
    const double* Z = base + lay.Z;
    const double* Xc = prm.predict ? base + lay.Xt : base + lay.X;
    const int ncols = prm.predict ? R.N : R.M;
    const int colrows = prm.predict ? R.Np : R.Mp;
    const bool do_zz = (tj <= ti) && (tj < R.nb);
    const bool have_x = (tj + 1) * TB <= colrows;
    for (int e = threadIdx.x; e < 64 * DP; e += 256) {
        const int r = e / DP, d = e - r * DP;
        const bool in = d < D;
        zi[r * LDZ + d] = in ? Z[(size_t)(ti * TB + r) * D + d] : 0.0;
        zj[r * LDZ + d] = (in && do_zz) ? Z[(size_t)(tj * TB + r) * D + d] : 0.0;
        xj[r * LDZ + d] = (in && have_x) ? Xc[(size_t)(tj * TB + r) * D + d] : 0.0;
    }
    __syncthreads();
    if (threadIdx.x < 192) {
        const double* v = (threadIdx.x < 64 ? zi : (threadIdx.x < 128 ? zj : xj)) + (threadIdx.x & 63) * LDZ;
        double n = 0.0;
        for (int d = 0; d < D; ++d) n = fma(v[d], v[d], n);
        (threadIdx.x < 64 ? ni : (threadIdx.x < 128 ? nzj : nxj))[threadIdx.x & 63] = n;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, gid = lane >> 2, tig = lane & 3;
    double az[8][2], ax[8][2];
#pragma unroll
    for (int c = 0; c < 8; ++c) az[c][0] = az[c][1] = ax[c][0] = ax[c][1] = 0.0;
#pragma unroll 2
    for (int d0 = 0; d0 < DP; d0 += 4) {
        const double a = zi[(8 * warp + gid) * LDZ + d0 + tig];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            dmma(ax[c][0], ax[c][1], a, xj[(8 * c + gid) * LDZ + d0 + tig]);
            if (do_zz) dmma(az[c][0], az[c][1], a, zj[(8 * c + gid) * LDZ + d0 + tig]);
        }
    }
    const double* sc = base + lay.scal;
    const double ell = softplus_d(sc[SC_RL]), s = softplus_d(sc[SC_RS]);
    const double inv_l2 = 1.0 / (ell * ell);
    double* Kzx = base + lay.Kzx;
    double* Kzz = base + lay.L;
    double* Kc = base + lay.Kc;
    const int lr = 8 * warp + gid, i = ti * TB + lr;
    const double nrow = ni[lr];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        const int lc = 8 * c + 2 * tig, j = tj * TB + lc;
        double kx[2], kz[2], k0[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const double r2x = fmax(nrow + nxj[lc + e] - 2.0 * ax[c][e], 0.0);
            kx[e] = (i < R.M && j + e < ncols) ? s * exp(-0.5 * (r2x * inv_l2)) : 0.0;
            if (do_zz) {
                if (i < R.M && j + e < R.M) {
                    const double r2z = (i == j + e) ? 0.0 : fmax(nrow + nzj[lc + e] - 2.0 * az[c][e], 0.0);
                    k0[e] = s * exp(-0.5 * (r2z * inv_l2));
                    kz[e] = k0[e] + (i == j + e ? prm.jitter_zz : 0.0);
                } else {
                    k0[e] = 0.0;
                    kz[e] = (i == j + e) ? 1.0 : 0.0;
                }
            }
        }
        *reinterpret_cast<double2*>(Kzx + (size_t)i * R.Wp + j) = make_double2(kx[0], kx[1]);
        if (do_zz) {
            *reinterpret_cast<double2*>(Kzz + (size_t)i * R.Mp + j) = make_double2(kz[0], kz[1]);
            *reinterpret_cast<double2*>(Kc + (size_t)i * R.Mp + j) = make_double2(k0[0], k0[1]);
            if (ti != tj) {
                Kc[(size_t)j * R.Mp + i] = k0[0];
                Kc[(size_t)(j + 1) * R.Mp + i] = k0[1];
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Blocked RIGHT-looking Cholesky with the inverse factor built alongside.  Block step kb is three
// short launches whose tiles all contract over a single 64-wide block, so the critical path of a
// region with nb blocks is nb * (diag + panel + update) instead of growing with nb^2:
//   diag  : L_kk = chol(K[kb,kb]) ; Linv_kk = L_kk^-1                      (tile already updated)
//   panel : L[i,kb]    = K[i,kb] Linv_kk^T                                 (i > kb)
//           Linv[kb,j] = -Linv_kk S[kb,j]                                  (j < kb)
//   update: K[i,j] -= L[i,kb] L[j,kb]^T                                    (i >= j > kb)
//           S[i,j] (+)= L[i,kb] Linv[kb,j]                                 (i > kb >= j; '=' when j == kb)
// S[i,j] = sum_{k=j..kb} L[i,k] Linv[k,j] accumulates in place in the strictly-lower tiles of the
// Linv buffer until step i turns it into Linv[i,j].
// ---------------------------------------------------------------------------------------------
constexpr int LDS_ = TB + 1;
constexpr int DIAG_SMEM = (2 * TB * LDS_ + TB) * (int)sizeof(double);

// 64x64 Cholesky factor (in place in sL) and its inverse (into sX, zero-initialised by the caller) in shared memory,
// 128 threads; returns (on every thread of warp 0) whether a pivot was not positive.  Row stride LD doubles.
template <int LD>
__device__ __forceinline__ bool chol_inv_64(double* __restrict__ sL, double* __restrict__ sX, double* __restrict__ dinv) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    bool bad = false;
#pragma unroll 1
    for (int p = 0; p < 4; ++p) {
        const int c0 = 16 * p;
        // (a) 16x16 diagonal block: warp 0, lane r (and its mirror r+16) owns row r
        if (warp == 0) {
            const int r = lane & 15;
            double a[16];
#pragma unroll
            for (int k = 0; k < 16; ++k) a[k] = sL[(c0 + r) * LD + c0 + k];
#pragma unroll
            for (int c = 0; c < 16; ++c) {
                double piv = __shfl_sync(0xffffffffu, a[c], c);
                if (!(piv > 0.0)) {
                    bad = true;
                    piv = 1.0;
                }
                const double rs = rsqrt(piv);
                const double l = a[c] * rs;                 // lane c: piv * rsqrt(piv) = sqrt(piv)
#pragma unroll
                for (int cc = c + 1; cc < 16; ++cc) a[cc] = fma(-l, __shfl_sync(0xffffffffu, l, cc), a[cc]);
                a[c] = l;
                if (lane == c) dinv[c0 + c] = rs;
            }
            if (lane < 16) {
#pragma unroll
                for (int k = 0; k < 16; ++k) sL[(c0 + r) * LD + c0 + k] = (k <= r) ? a[k] : 0.0;
            }
        }
        __syncthreads();
        // (b) rows below the block: one thread per row, forward substitution against the 16x16 factor
        const int nt = 48 - 16 * p;
        if (tid < nt) {
            const int r = c0 + 16 + tid;
            double x[16];
#pragma unroll
            for (int k = 0; k < 16; ++k) x[k] = sL[r * LD + c0 + k];
#pragma unroll
            for (int c = 0; c < 16; ++c) {
                double sum = x[c];
#pragma unroll
                for (int k = 0; k < c; ++k) sum = fma(-x[k], sL[(c0 + c) * LD + c0 + k], sum);
                x[c] = sum * dinv[c0 + c];
            }
#pragma unroll
            for (int k = 0; k < 16; ++k) sL[r * LD + c0 + k] = x[k];
        }
        __syncthreads();
        // (c) trailing update of the lower triangle: thread = (row, strip of columns)
        if (nt > 0) {
            const int nstrip = GEMM_THREADS / nt;
            const int rr = tid % nt, strip = tid / nt;
            if (strip < nstrip) {
                const int r = c0 + 16 + rr;
                double lr[16];
#pragma unroll
                for (int k = 0; k < 16; ++k) lr[k] = sL[r * LD + c0 + k];
                for (int cc = c0 + 16 + strip; cc <= r; cc += nstrip) {
                    double sum = sL[r * LD + cc];
#pragma unroll
                    for (int k = 0; k < 16; ++k) sum = fma(-lr[k], sL[cc * LD + c0 + k], sum);
                    sL[r * LD + cc] = sum;
                }
            }
        }
        __syncthreads();
    }
    // ---- inverse.  Diagonal 16x16 blocks: warp p, lane c (and mirror) owns column c.
    {
        const int c0 = 16 * warp, c = lane & 15;
        double x[16];
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            double sum = (q == c) ? 1.0 : 0.0;
#pragma unroll
            for (int k = 0; k < q; ++k) sum = fma(-sL[(c0 + q) * LD + c0 + k], x[k], sum);
            x[q] = sum * dinv[c0 + q];
        }
        if (lane < 16) {
#pragma unroll
            for (int q = 0; q < 16; ++q) sX[(c0 + q) * LD + c0 + c] = (q >= c) ? x[q] : 0.0;
        }
    }
    __syncthreads();
    // Off-diagonal blocks by distance d = i - j:  X_ij = -X_ii * sum_{k=j..i-1} L_ik X_kj.
    // One warp per block; lane = (row r, half h of the 16 columns).
#pragma unroll 1
    for (int d = 1; d < 4; ++d) {
        if (warp < 4 - d) {
            const int i = warp + d, j = warp;
            const int r = lane & 15, h = lane >> 4;
            double t[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) t[q] = 0.0;
            const double* Lrow = sL + (16 * i + r) * LD + 16 * j;            // L[i-block row r][cols of blocks j..i-1]
            for (int kk = 0; kk < 16 * d; ++kk) {
                const double lv = Lrow[kk];
                const double* xr = sX + (16 * j + kk) * LD + 16 * j + 8 * h;  // X[(blocks j..i-1) row kk][block j cols]
#pragma unroll
                for (int q = 0; q < 8; ++q) t[q] = fma(lv, xr[q], t[q]);
            }
            // stage T in the destination block, then out = -X_ii * T
            double* Tb = sX + (16 * i) * LD + 16 * j;
#pragma unroll
            for (int q = 0; q < 8; ++q) Tb[r * LD + 8 * h + q] = t[q];
            __syncwarp();
            double o[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) o[q] = 0.0;
            const double* Xii = sX + (16 * i + r) * LD + 16 * i;
            for (int m = 0; m <= r; ++m) {
                const double xv = Xii[m];
#pragma unroll
                for (int q = 0; q < 8; ++q) o[q] = fma(-xv, Tb[m * LD + 8 * h + q], o[q]);
            }
            __syncwarp();
#pragma unroll
            for (int q = 0; q < 8; ++q) Tb[r * LD + 8 * h + q] = o[q];
        }
        __syncthreads();
    }
    return bad;
}

// 64x64 factorisation + triangular inverse in shared memory, blocked by 16: the 16x16 diagonal blocks
// are factored / inverted by one warp entirely in registers (rows or columns per lane, pivots and
// multipliers exchanged with shuffles, no block barrier inside), the panel below is a per-row
// forward substitution, trailing and off-diagonal blocks are small register-tiled products.
// 12 block barriers for the factorisation and 4 for the inverse instead of ~320.
__global__ void __launch_bounds__(GEMM_THREADS)
k_rl_diag(const Region* __restrict__ regs, int kb, GpParams prm, double* __restrict__ ws, int32_t* __restrict__ status) {
    extern __shared__ __align__(16) unsigned char smem_diag[];
    double* sL = reinterpret_cast<double*>(smem_diag);   // [64][65] tile, then L
    double* sX = sL + TB * LDS_;                         // [64][65] L^-1
    double* dinv = sX + TB * LDS_;                       // [64] 1 / L[k][k]
    const Region R = regs[blockIdx.x];
    const Layout lay = make_layout(R.Mp, R.Np, R.Wp, prm.D);
    double* base = ws + R.base;
    const int Mp = R.Mp;
    double* Lg = base + lay.L;
    double* Li = base + lay.Linv;
    const int r0 = kb * TB;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int e = tid; e < TB * TB; e += GEMM_THREADS) {
        const int r = e >> 6, c = e & 63;
        sL[r * LDS_ + c] = __ldcg(Lg + (size_t)(r0 + r) * Mp + r0 + c);
        sX[r * LDS_ + c] = 0.0;
    }
    __syncthreads();
    const bool bad = chol_inv_64<LDS_>(sL, sX, dinv);
    if (bad && tid == 0) atomicOr(status + R.orig, GAPRO_GP_NOT_PSD);
    for (int e = tid; e < TB * TB; e += GEMM_THREADS) {
        const int rr = e >> 6, c = e & 63;
        const bool low = c <= rr;
        Lg[(size_t)(r0 + rr) * Mp + r0 + c] = low ? sL[rr * LDS_ + c] : 0.0;
        Li[(size_t)(r0 + rr) * Mp + r0 + c] = low ? sX[rr * LDS_ + c] : 0.0;
    }
}

__global__ void __launch_bounds__(GEMM_THREADS, 4)
k_rl_panel(const Region* __restrict__ regs, const int2* __restrict__ ptiles, int kb, GpParams prm,
           double* __restrict__ ws) {
    extern __shared__ __align__(16) unsigned char smem_panel[];
    GemmSmem& sm = *reinterpret_cast<GemmSmem*>(smem_panel);
    const int2 pt = ptiles[blockIdx.x];
    const Region R = regs[pt.x];
    const Layout lay = make_layout(R.Mp, R.Np, R.Wp, prm.D);
    double* base = ws + R.base;
    const int Mp = R.Mp;
    double* Lg = base + lay.L;
    double* Li = base + lay.Linv;
    const int r0 = kb * TB;
    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    if (pt.y >= kb) {
        // L[i,kb] = K[i,kb] Linv_kk^T, in place: out[r,c] = sum_k K[i0+r][r0+k] Linv_kk[c][k]
        const int i0 = (pt.y + 1) * TB;
        gemm_accum<true, true>(acc, Lg + (size_t)i0 * Mp + r0, Mp, Li + (size_t)r0 * Mp + r0, Mp, 0, TB, nullptr, sm);
        ACC_FOREACH(true, true, 0, 0, {
            *reinterpret_cast<double2*>(Lg + (size_t)(i0 + row) * Mp + r0 + col) = make_double2(v0, v1);
        })
    } else {
        // Linv[kb,j] = -Linv_kk S[kb,j], in place: out[r,c] = -sum_k Linv_kk[r][k] S[r0+k][j0+c]
        const int j0 = pt.y * TB;
        gemm_accum<true, false>(acc, Li + (size_t)r0 * Mp + r0, Mp, Li + (size_t)r0 * Mp + j0, Mp, 0, TB, nullptr, sm);
        ACC_FOREACH(true, false, 0, 0, {
            *reinterpret_cast<double2*>(Li + (size_t)(r0 + row) * Mp + j0 + col) = make_double2(-v0, -v1);
        })
    }
}

// Trailing update with the block steps kb0 .. kb0+nk-1 (contraction over nk*64).  Updates are applied a
// group of steps at a time (ChunkTables::sweep_group): after any but the last step of a group only the next
// block column / block row is brought up to date with the steps of the group so far (what the next diag and
// panel need), after the last one every remaining lower tile receives the whole group in one pass - 1/group
// of the read-modify-write traffic of a per-step update and a contraction long enough to fill the pipeline.
__global__ void __launch_bounds__(GEMM_THREADS, 4)
k_rl_update(const Region* __restrict__ regs, const int4* __restrict__ tiles, int kb0, int nk, GpParams prm,
            double* __restrict__ ws) {
    extern __shared__ __align__(16) unsigned char smem_upd[];
    GemmSmem& sm = *reinterpret_cast<GemmSmem*>(smem_upd);
    const int4 t = tiles[blockIdx.x];
    const Region R = regs[t.x];
    const Layout lay = make_layout(R.Mp, R.Np, R.Wp, prm.D);
    double* base = ws + R.base;
    const int Mp = R.Mp;
    double* Lg = base + lay.L;
    double* Li = base + lay.Linv;
    const int k0 = kb0 * TB, k1 = (kb0 + nk) * TB, i0 = t.y * TB, j0 = t.z * TB;
    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    if (t.z >= kb0 + nk) {
        // K[i,j] -= sum_k L[i,k] L[j,k]^T   (pull the read-modify-write tile towards L2 while the product runs)
        ACC_FOREACH(true, true, 0, 0, {
            (void)v0;
            (void)v1;
            asm volatile("prefetch.global.L2 [%0];" ::"l"(Lg + (size_t)(i0 + row) * Mp + j0 + col));
        })
        gemm_accum<true, true>(acc, Lg + (size_t)i0 * Mp, Mp, Lg + (size_t)j0 * Mp, Mp, k0, k1, nullptr, sm);
        ACC_FOREACH(true, true, 0, 0, {
            double2* p = reinterpret_cast<double2*>(Lg + (size_t)(i0 + row) * Mp + j0 + col);
            const double2 k = __ldcg(p);
            *p = make_double2(k.x - v0, k.y - v1);
        })
    } else {
        // S[i,j] (+)= sum_k L[i,k] Linv[k,j]; the first contribution of a block column overwrites
        const bool first = t.z >= kb0;
        if (!first) {
            ACC_FOREACH(true, false, 0, 0, {
                (void)v0;
                (void)v1;
                asm volatile("prefetch.global.L2 [%0];" ::"l"(Li + (size_t)(i0 + row) * Mp + j0 + col));
            })
        }
        gemm_accum<true, false>(acc, Lg + (size_t)i0 * Mp, Mp, Li + j0, Mp, k0, k1, nullptr, sm);
        ACC_FOREACH(true, false, 0, 0, {
            double2* p = reinterpret_cast<double2*>(Li + (size_t)(i0 + row) * Mp + j0 + col);
            double2 o = make_double2(v0, v1);
            if (!first) {
                const double2 k = __ldcg(p);
                o.x += k.x;
                o.y += k.y;
            }
            *p = o;
        })
    }
}

// ---------------------------------------------------------------------------------------------
// column statistics: mu = A^T m + c, var = s + jitter_xx + colsum(B^2) - colsum(A^2), then either
// the Gauss-Hermite gradients g_mu, g_v (training) or the outputs (prediction)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double hazard(double z) {
    // phi(z)/Phi(z) = sqrt(2/pi) / erfcx(-z/sqrt2)
    return 0.79788456080286535588 / erfcx(-z * 0.70710678118654752440);
}

struct PredictOut {
    float *prob, *conf, *mu, *var;
    uint8_t* label;
    double *mu64, *var64;
    int32_t* status;
};

__global__ void __launch_bounds__(256)
k_colstats(const Region* __restrict__ regs, const int2* __restrict__ rtiles, GpParams prm, double* __restrict__ ws,
           PredictOut po) {
    __shared__ double red[3][4][TB];
    const int2 rt = rtiles[blockIdx.x];
    const Region R = regs[rt.x];
    const Layout lay = make_layout(R.Mp, R.Np, R.Wp, prm.D);
    double* base = ws + R.base;
    const int Wp = R.Wp;
    const int cl = threadIdx.x & 63, q = threadIdx.x >> 6;
    const int n = rt.y * TB + cl;
    const double* A = base + lay.A;
    const double* Bm = base + lay.Bm;
    const double* mv = base + lay.m;
    double s_mu = 0.0, s_b = 0.0, s_a = 0.0;
    for (int k = q; k < R.Mp; k += 4) {
        const double a = A[(size_t)k * Wp + n], b = Bm[(size_t)k * Wp + n];
        s_mu += a * mv[k];
        s_b += b * b;
        s_a += a * a;
    }
    red[0][q][cl] = s_mu;
    red[1][q][cl] = s_b;
    red[2][q][cl] = s_a;
    __syncthreads();
    if (q != 0) return;
    s_mu = ((red[0][0][cl] + red[0][1][cl]) + red[0][2][cl]) + red[0][3][cl];
    s_b = ((red[1][0][cl] + red[1][1][cl]) + red[1][2][cl]) + red[1][3][cl];
    s_a = ((red[2][0][cl] + red[2][1][cl]) + red[2][2][cl]) + red[2][3][cl];
    const double* sc = base + lay.scal;
    const double s = softplus_d(sc[SC_RS]);
    const double mu = s_mu + sc[SC_C];
    const double v = s + prm.jitter_xx + s_b - s_a;
    const bool clamped = v < MIN_VARIANCE;
    const double var = clamped ? MIN_VARIANCE : v;
    if (prm.predict) {
        if (n < R.N) {
            const double link = mu / sqrt(1.0 + var);
            const double p = 0.5 * erfc(-link * 0.70710678118654752440);
            const float pf = (float)p;
            const bool lab = pf >= 0.5f;
            const int o = R.test_off + n;
            po.prob[o] = pf;
            po.label[o] = lab ? 1 : 0;
            po.conf[o] = lab ? pf : (1.0f - pf);
            po.mu[o] = (float)mu;
            po.var[o] = (float)var;
            if (po.mu64) po.mu64[o] = mu;
            if (po.var64) po.var64[o] = var;
            if (!(isfinite(mu) && isfinite(var))) atomicOr(po.status + R.orig, GAPRO_GP_NAN);
        }
        return;
    }
    double gmu = 0.0, gv = 0.0;
    if (n < R.M) {
        const double y = base[lay.y + n];
        const double sd = sqrt(2.0 * var);
        double a0 = 0.0, a1 = 0.0;
        for (int k = 0; k < N_GH; ++k) {
            const double h = hazard(y * (sd * c_gh_t[k] + mu));
            a0 += c_gh_w[k] * h;
            a1 += c_gh_w[k] * c_gh_t[k] * h;
        }
        const double pref = -(1.0 / (double)R.M) * 0.56418958354775628695;   // -(1/N)/sqrt(pi)
        gmu = pref * y * a0;
        gv = clamped ? 0.0 : pref * y * a1 / sd;
    }
    base[lay.mu + n] = mu;
    base[lay.var + n] = var;
    base[lay.gmu + n] = gmu;
    base[lay.gv + n] = gv;
}

// dm = A g_mu + m/N, Adam on m.  One warp per row.
__global__ void __launch_bounds__(256)
k_grad_m(const Region* __restrict__ regs, const int2* __restrict__ rtiles, GpParams prm, double* __restrict__ ws) {
    const int2 rt = rtiles[blockIdx.x];
    const Region R = regs[rt.x];
    const Layout lay = make_layout(R.Mp, R.Np, R.Wp, prm.D);
    double* base = ws + R.base;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const double* gmu = base + lay.gmu;
    for (int rr = 0; rr < 8; ++rr) {
        const int i = rt.y * TB + warp * 8 + rr;
        if (i >= R.M) break;
        const double* Arow = base + lay.A + (size_t)i * R.Wp;
        double s = 0.0;
        for (int n = lane; n < R.M; n += 32) s += Arow[n] * gmu[n];
        for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) {
            double p = base[lay.m + i], m1 = base[lay.mm + i], m2 = base[lay.mv + i];
            const double g = s + p / (double)R.M;
            adam_update(p, m1, m2, g, prm);
            base[lay.m + i] = p;
            base[lay.mm + i] = m1;
            base[lay.mv + i] = m2;
        }
    }
}

// Gradients w.r.t. the inducing points and the raw kernel parameters from G_K (in the B buffer,
// symmetric) and G_C.  A CTA owns 8*ROWS inducing rows (ROWS per warp) and walks over the columns in
// blocks of 32.  HBM-bound (four M x M matrices are read once): the 32 x 32 blocks of the four matrices
// and the Z / X rows of the column block are staged by a three-stage cp.async pipeline (one
// __syncthreads per block, two blocks always in flight), lanes run over the 32 columns.
constexpr int KG_STAGES = 3;
template <int DMAX>
struct KgStage {
    double gk[32][32], kz[32][32], gc[32][32], kx[32][32];   // G_K, K_zz, G_C, K_zx blocks
    double z[32 * DMAX], x[32 * DMAX];                       // rows jb..jb+31 of Z and X, [32][D] as in memory
};
template <int DMAX, int ROWS>
constexpr int kgrad_smem() { return KG_STAGES * (int)sizeof(KgStage<DMAX>) + 8 * ROWS * DMAX * (int)sizeof(double); }

template <int DMAX, int ROWS>
__global__ void __launch_bounds__(256, (DMAX <= 8) ? 2 : 1)
k_kgrad(const Region* __restrict__ regs, const int2* __restrict__ rtiles, GpParams prm, double* __restrict__ ws) {
    static_assert(8 * ROWS == 32, "one CTA stages 32 matrix rows");
    constexpr int SPLIT = TB / (8 * ROWS);           // CTAs per 64-row tile
    extern __shared__ __align__(16) unsigned char smem_kg[];
    KgStage<DMAX>* st = reinterpret_cast<KgStage<DMAX>*>(smem_kg);
    double (*Zi)[DMAX] = reinterpret_cast<double (*)[DMAX]>(smem_kg + KG_STAGES * sizeof(KgStage<DMAX>));
    const int2 rt = rtiles[blockIdx.x / SPLIT];
    const Region R = regs[rt.x];
    const int D = prm.D;
    const Layout lay = make_layout(R.Mp, R.Np, R.Wp, D);
    double* base = ws + R.base;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const double* sc = base + lay.scal;
    const double ell = softplus_d(sc[SC_RL]), s = softplus_d(sc[SC_RS]);
    const double inv_l2 = 1.0 / (ell * ell), inv_s = 1.0 / s, m2_ell = -2.0 / ell;
    const double* Z = base + lay.Z;
    const double* X = base + lay.X;
    const int row0 = rt.y * TB + (blockIdx.x % SPLIT) * 8 * ROWS;
    if (row0 >= R.M) return;
    for (int e = threadIdx.x; e < 8 * ROWS * DMAX; e += blockDim.x) {
        const int rr = e / DMAX, d = e - rr * DMAX;
        Zi[rr][d] = (d < D && row0 + rr < R.M) ? Z[(size_t)(row0 + rr) * D + d] : 0.0;
    }
    // loader: thread t moves 16-byte unit (t & 15) of row (t >> 4) + 16 * (q & 1) of matrix q >> 1, q = 0..7
    // (rows row0 .. row0+31 and columns jb .. jb+31 always exist: the matrices are padded to multiples of 64)
    const int lr = threadIdx.x >> 4, lc = 2 * (threadIdx.x & 15);
    const double* g_gk = base + lay.Bm + (size_t)(row0 + lr) * R.Wp + lc;
    const double* g_kz = base + lay.Kc + (size_t)(row0 + lr) * R.Mp + lc;
    const double* g_gc = base + lay.GC + (size_t)(row0 + lr) * R.Mp + lc;
    const double* g_kx = base + lay.Kzx + (size_t)(row0 + lr) * R.Wp + lc;
    const size_t half_w = (size_t)16 * R.Wp, half_m = (size_t)16 * R.Mp;
    const int zx_units = 16 * D;                     // 16-byte units in 32 rows of Z (or X)
    auto issue = [&](int stage, int jb) {
        KgStage<DMAX>& S = st[stage];
        cp_async16(&S.gk[lr][lc], g_gk + jb);
        cp_async16(&S.gk[lr + 16][lc], g_gk + half_w + jb);
        cp_async16(&S.kz[lr][lc], g_kz + jb);
        cp_async16(&S.kz[lr + 16][lc], g_kz + half_m + jb);
        cp_async16(&S.gc[lr][lc], g_gc + jb);
        cp_async16(&S.gc[lr + 16][lc], g_gc + half_m + jb);
        cp_async16(&S.kx[lr][lc], g_kx + jb);
        cp_async16(&S.kx[lr + 16][lc], g_kx + half_w + jb);
        const int t = threadIdx.x;
        if (t < zx_units) cp_async16(&S.z[2 * t], Z + (size_t)jb * D + 2 * t);
        else if (t < 2 * zx_units) cp_async16(&S.x[2 * (t - zx_units)], X + (size_t)jb * D + 2 * (t - zx_units));
    };
    double az[ROWS][DMAX], as[ROWS], al[ROWS], cz[ROWS];
#pragma unroll
    for (int q = 0; q < ROWS; ++q) {
        as[q] = al[q] = cz[q] = 0.0;
#pragma unroll
        for (int d = 0; d < DMAX; ++d) az[q][d] = 0.0;
    }
    const int nblk = (R.M + 31) >> 5;
#pragma unroll
    for (int p = 0; p < KG_STAGES - 1; ++p) {
        if (p < nblk) issue(p, 32 * p);
        cp_async_commit();
    }
    int stage = 0;
    for (int b = 0; b < nblk; ++b) {
        cp_async_wait<KG_STAGES - 2>();   // block b has landed
        __syncthreads();                  // ... for every thread, block b-1 is consumed, Zi is visible
        {
            const int nb = b + KG_STAGES - 1;
            int ns = stage + KG_STAGES - 1;
            if (ns >= KG_STAGES) ns -= KG_STAGES;
            if (nb < nblk) issue(ns, 32 * nb);
            cp_async_commit();
        }
        const KgStage<DMAX>& S = st[stage];
        const int j = 32 * b + lane;
        if (j < R.M) {
            // the adjoint weights do not depend on the distances: read them first, then ONE pass over d
            double grz2[ROWS], grx[ROWS], d2z[ROWS], d2x[ROWS];
#pragma unroll
            for (int q = 0; q < ROWS; ++q) {
                const int r = warp * ROWS + q;
                grz2[q] = grx[q] = d2z[q] = d2x[q] = 0.0;
                if (row0 + r < R.M) {
                    const double gk = S.gk[r][lane], kz = S.kz[r][lane];
                    const double gc = S.gc[r][lane], kx = S.kx[r][lane];
                    // zz: W = Gr + Gr^T = 2 Gr (G_K, K_zz symmetric);  zx: Gr once.
                    // sum_j [2 grz (z_i - z_j) + grx (z_i - x_j)] = z_i * cz - sum_j (2 grz z_j + grx x_j)
                    grz2[q] = -gk * kz;
                    grx[q] = -0.5 * gc * kx;
                    as[q] += (gk * kz + gc * kx) * inv_s;
                    cz[q] += grz2[q] + grx[q];
                }
            }
#pragma unroll
            for (int d = 0; d < DMAX; ++d) {
                if (d < D) {
                    const double zjd = S.z[lane * D + d], xjd = S.x[lane * D + d];
#pragma unroll
                    for (int q = 0; q < ROWS; ++q) {
                        const double zi = Zi[warp * ROWS + q][d];
                        const double dz = zi - zjd, dx = zi - xjd;
                        d2z[q] = fma(dz, dz, d2z[q]);
                        d2x[q] = fma(dx, dx, d2x[q]);
                        az[q][d] = fma(-grz2[q], zjd, fma(-grx[q], xjd, az[q][d]));
                    }
                }
            }
#pragma unroll
            for (int q = 0; q < ROWS; ++q) al[q] += (0.5 * grz2[q] * d2z[q] + grx[q] * d2x[q]) * (inv_l2 * m2_ell);
        }
        if (++stage == KG_STAGES) stage = 0;
    }
    cp_async_wait<0>();
#pragma unroll
    for (int q = 0; q < ROWS; ++q) {
        const int i = row0 + warp * ROWS + q;
        double a0 = as[q], a1 = al[q], a2 = cz[q];
        for (int o = 16; o; o >>= 1) {
            a0 += __shfl_xor_sync(0xffffffffu, a0, o);
            a1 += __shfl_xor_sync(0xffffffffu, a1, o);
            a2 += __shfl_xor_sync(0xffffffffu, a2, o);
#pragma unroll
            for (int d = 0; d < DMAX; ++d) az[q][d] += __shfl_xor_sync(0xffffffffu, az[q][d], o);
        }
        if (lane == 0 && i < R.M) {
            base[lay.gsrow + i] = a0;
            base[lay.glrow + i] = a1;
#pragma unroll
            for (int d = 0; d < DMAX; ++d)
                if (d < D) base[lay.gZ + (size_t)i * D + d] = 2.0 * inv_l2 * fma(a2, Zi[warp * ROWS + q][d], az[q][d]);
        }
    }
}

// Wide-feature variant (8 < D <= 64, e.g. the 32-d deep features of --use_deepfeat).  With D = 32 the
// inducing-point gradient  dZ = -(W_zz Z + W_zx X),  W_zz = -G_K o K_zz,  W_zx = -1/2 G_C o K_zx,  is a real dense
// contraction (K = M, N = D: 4 D / 32 = 4 flop per byte of the four M x M matrices it reads once) and runs on the
// FP64 tensor pipe: a CTA owns 64 inducing rows, walks over the columns in chunks of 32, forms the two weight
// blocks element-wise (thread = row quarter: 8 consecutive columns, so the global loads are 64-byte runs and the
// per-row sums stay in registers), stages them and the Z / X rows of the chunk in shared memory and issues
// mma.sync m8n8k4 (warp = 8 rows x all feature columns).  The next chunk's 4 x 8 values are loaded into registers
// before the MMAs of the current one.  The squared distance for the lengthscale gradient is recovered from the stored
// kernel value, r^2 = -2 ln(K / s).
template <int NCH>
constexpr int kgrad_wide_smem() { return (2 * 64 * 36 + 2 * 32 * (32 * NCH + 4) + 64) * (int)sizeof(double); }

template <int NCH>
__global__ void __launch_bounds__(256)
k_kgrad_wide(const Region* __restrict__ regs, const int2* __restrict__ rtiles, GpParams prm, double* __restrict__ ws) {
    constexpr int DP = 32 * NCH, LDW = 36, LDF = DP + 4, NCB = DP / 8;
    extern __shared__ __align__(16) double smem_kw[];
    double* Wz = smem_kw;                               // weight blocks [64 rows][32 columns of the chunk]
    double* Wx = Wz + 64 * LDW;
    double* Zs = Wx + 64 * LDW;                         // rows jb .. jb+31 of Z and X, [32][D]
    double* Xs = Zs + 32 * LDF;
    double* s_cz = Xs + 32 * LDF;
    const int2 rt = rtiles[blockIdx.x];
    const Region R = regs[rt.x];
    const int D = prm.D, M = R.M;
    const Layout lay = make_layout(R.Mp, R.Np, R.Wp, D);
    double* base = ws + R.base;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, gid = lane >> 2, tig = lane & 3;
    const double* sc = base + lay.scal;
    const double ell = softplus_d(sc[SC_RL]), s = softplus_d(sc[SC_RS]);
    const double inv_l2 = 1.0 / (ell * ell), inv_s = 1.0 / s, m2_ell = -2.0 / ell;
    const double* Z = base + lay.Z;
    const double* X = base + lay.X;
    const int row0 = rt.y * TB;
    if (row0 >= M) return;
    // element-wise role: row er, columns 8 * eq .. 8 * eq + 7 of the chunk
    const int er = tid >> 2, eq = tid & 3;
    const int i = row0 + er;
    const double* g_gk = base + lay.Bm + (size_t)i * R.Wp + 8 * eq;
    const double* g_kz = base + lay.Kc + (size_t)i * R.Mp + 8 * eq;
    const double* g_gc = base + lay.GC + (size_t)i * R.Mp + 8 * eq;
    const double* g_kx = base + lay.Kzx + (size_t)i * R.Wp + 8 * eq;
    double2 pre[4][4];                                  // next chunk: 4 matrices x 8 doubles
    auto fetch = [&](int jb) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {                   // rows and columns exist up to Mp (padded to 64): always in bounds
            pre[0][u] = *reinterpret_cast<const double2*>(g_gk + jb + 2 * u);
            pre[1][u] = *reinterpret_cast<const double2*>(g_kz + jb + 2 * u);
            pre[2][u] = *reinterpret_cast<const double2*>(g_gc + jb + 2 * u);
            pre[3][u] = *reinterpret_cast<const double2*>(g_kx + jb + 2 * u);
        }
    };
    double acc[NCB][2];
#pragma unroll
    for (int c = 0; c < NCB; ++c) acc[c][0] = acc[c][1] = 0.0;
    double as = 0.0, al = 0.0, cz = 0.0;
    const int nblk = (M + 31) >> 5;
    fetch(0);
    for (int b = 0; b < nblk; ++b) {
        const int jb = 32 * b;
        __syncthreads();                                // the previous chunk's MMAs have read the shared tiles
        // Z / X rows of the chunk
        for (int e = tid; e < 32 * DP; e += 256) {
            const int jj = e / DP, d = e - jj * DP;
            const bool ok = (jb + jj < M) && d < D;
            Zs[jj * LDF + d] = ok ? Z[(size_t)(jb + jj) * D + d] : 0.0;
            Xs[jj * LDF + d] = ok ? X[(size_t)(jb + jj) * D + d] : 0.0;
        }
        // weights of this thread's 8 elements
#pragma unroll
        for (int u = 0; u < 4; ++u) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int j = jb + 8 * eq + 2 * u + h;
                const double gk = h ? pre[0][u].y : pre[0][u].x, kz = h ? pre[1][u].y : pre[1][u].x;
                const double gc = h ? pre[2][u].y : pre[2][u].x, kx = h ? pre[3][u].y : pre[3][u].x;
                double wz = 0.0, wx = 0.0;
                if (i < M && j < M) {
                    wz = -gk * kz;
                    wx = -0.5 * gc * kx;
                    as += (gk * kz + gc * kx) * inv_s;
                    cz += wz + wx;
                    const double r2z = kz > 0.0 ? -2.0 * log(kz * inv_s) : 0.0;     // r^2 (already divided by l^2)
                    const double r2x = kx > 0.0 ? -2.0 * log(kx * inv_s) : 0.0;
                    al += (0.5 * wz * r2z + wx * r2x) * m2_ell;
                }
                Wz[er * LDW + 8 * eq + 2 * u + h] = wz;
                Wx[er * LDW + 8 * eq + 2 * u + h] = wx;
            }
        }
        if (b + 1 < nblk) fetch(jb + 32);
        __syncthreads();
        // acc(rows 8 warp + gid, feature columns) += Wz * Zs + Wx * Xs
#pragma unroll
        for (int k0 = 0; k0 < 32; k0 += 4) {
            const double az_ = Wz[(8 * warp + gid) * LDW + k0 + tig], ax_ = Wx[(8 * warp + gid) * LDW + k0 + tig];
#pragma unroll
            for (int c = 0; c < NCB; ++c) {
                dmma(acc[c][0], acc[c][1], az_, Zs[(k0 + tig) * LDF + 8 * c + gid]);
                dmma(acc[c][0], acc[c][1], ax_, Xs[(k0 + tig) * LDF + 8 * c + gid]);
            }
        }
    }
    // per-row sums: the four threads of a row are consecutive lanes
#pragma unroll
    for (int o = 1; o < 4; o <<= 1) {
        as += __shfl_xor_sync(0xffffffffu, as, o);
        al += __shfl_xor_sync(0xffffffffu, al, o);
        cz += __shfl_xor_sync(0xffffffffu, cz, o);
    }
    if (eq == 0) {
        s_cz[er] = cz;
        if (i < M) {
            base[lay.gsrow + i] = as;
            base[lay.glrow + i] = al;
        }
    }
    __syncthreads();
    // dZ[i][d] = 2 / l^2 * (cz_i z_i[d] - acc): this lane holds row 8 warp + gid, columns 8 c + 2 tig + {0, 1}
    const int oi = row0 + 8 * warp + gid;
    if (oi < M) {
        const double czi = s_cz[8 * warp + gid];
#pragma unroll
        for (int c = 0; c < NCB; ++c)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int d = 8 * c + 2 * tig + e;
                if (d < D) base[lay.gZ + (size_t)oi * D + d] = 2.0 * inv_l2 * fma(czi, Z[(size_t)oi * D + d], -acc[c][e]);
            }
    }
}

// Adam on Z and on the three scalars (c, rho_s, rho_l).  One CTA per region.
__device__ double block_sum(double v, double* red) {
    const int tid = threadIdx.x;
    __syncthreads();
    red[tid] = v;
    __syncthreads();
    for (int s = blockDim.x >> 1; s > 0; s >>= 1) {
        if (tid < s) red[tid] += red[tid + s];
        __syncthreads();
    }
    return red[0];
}

__global__ void __launch_bounds__(256)
k_adam_small(const Region* __restrict__ regs, GpParams prm, double* __restrict__ ws) {
    __shared__ double red[256];
    const Region R = regs[blockIdx.x];
    const Layout lay = make_layout(R.Mp, R.Np, R.Wp, prm.D);
    double* base = ws + R.base;
    const int tid = threadIdx.x;
    const int MD = R.M * prm.D;
    for (int e = tid; e < MD; e += blockDim.x) {
        double p = base[lay.Z + e], m1 = base[lay.Zm + e], m2 = base[lay.Zv + e];
        adam_update(p, m1, m2, base[lay.gZ + e], prm);
        base[lay.Z + e] = p;
        base[lay.Zm + e] = m1;
        base[lay.Zv + e] = m2;
    }
    double a = 0.0, b = 0.0, c = 0.0, d = 0.0;
    for (int i = tid; i < R.M; i += blockDim.x) {
        a += base[lay.gmu + i];
        b += base[lay.gv + i];
        c += base[lay.gsrow + i];
        d += base[lay.glrow + i];
    }
    const double g_c = block_sum(a, red);
    const double g_v = block_sum(b, red);
    const double g_sr = block_sum(c, red);
    const double g_lr = block_sum(d, red);
    if (tid == 0) {
        double* sc = base + lay.scal;
        const double g[3] = {g_c, (g_v + g_sr) * sigmoid_d(sc[SC_RS]), g_lr * sigmoid_d(sc[SC_RL])};
        for (int k = 0; k < 3; ++k) {
            double p = sc[k], m1 = sc[SC_M0 + k], m2 = sc[SC_V0 + k];
            adam_update(p, m1, m2, g[k], prm);
            sc[k] = p;
            sc[SC_M0 + k] = m1;
            sc[SC_V0 + k] = m2;
        }
    }
}

#include "gp_small.cuh"

// initial state: X, Z <- training rows (float32 widened), Xt <- test rows, y, m <- 1e-3 * noise, T <- I
__global__ void __launch_bounds__(256)
k_region_init(const Region* __restrict__ regs, int D, const float* __restrict__ feats, const int32_t* __restrict__ train_idx,
              const int32_t* __restrict__ test_idx, const float* __restrict__ noise, double* __restrict__ ws) {
    const Region R = regs[blockIdx.x];
    const Layout lay = make_layout(R.Mp, R.Np, R.Wp, D);
    double* base = ws + R.base;
    for (int e = threadIdx.x; e < R.M * D; e += blockDim.x) {
        const int i = e / D, d = e % D;
        const double v = (double)feats[(size_t)train_idx[R.train_off + i] * D + d];
        base[lay.X + e] = v;
        base[lay.Z + e] = v;
    }
    for (int e = threadIdx.x; e < R.N * D; e += blockDim.x) {
        const int i = e / D, d = e % D;
        base[lay.Xt + e] = (double)feats[(size_t)test_idx[R.test_off + i] * D + d];
    }
    for (int i = threadIdx.x; i < R.Mp; i += blockDim.x) {
        base[lay.T + (size_t)i * R.Mp + i] = 1.0;
        if (i < R.M) {
            base[lay.y + i] = i < R.n_b1 ? -1.0 : 1.0;
            base[lay.m + i] = MEAN_INIT_STD * (double)noise[R.train_off + i];
        }
    }
}

// ---------------------------------------------------------------------------------------------
// host driver
// ---------------------------------------------------------------------------------------------
inline int ceil64(int x) { return (x + 63) / 64 * 64; }

// ---- tcgen05 path configuration (development knobs; defaults are what the parity suite runs with) -----------
static int oz_min_rows() {
    // GAPRO_GP_OZAKI=1: regions with at least this many padded training rows run their tile products on tcgen05
    // (8 digits).  Opt-in: the digit-plane products are accurate relative to row-max x column-max x K, float64 is
    // accurate componentwise, and the 50-step Adam trajectory amplifies the difference.  Measured against the fp64
    // oracle: 4.4e-7 on the 8k-superpoint golden region and 8e-7 on the whole configs[3] scene (same as DMMA, 1.28x
    // faster), but 7.8e-5 (worst element 1.6e-4) on the worst-conditioned region of the configs[4] scene, where DMMA
    // itself is at 8e-6 - past the 1e-4 bar, so it is not the default (DESIGN.md section 4.1).
    int on = 0, m = 2048;
    if (const char* e = getenv("GAPRO_GP_OZAKI")) on = atoi(e);
    if (const char* e = getenv("GAPRO_GP_OZAKI_MIN_M")) m = atoi(e);
    return on ? m : (1 << 30);
}

Region make_region(int M, int N, int n_b1, int train_off, int test_off, int orig) {
    Region r;
    r.M = M;
    r.N = N;
    r.Mp = ceil64(M);
    r.Np = ceil64(N);
    r.Wp = std::max(r.Mp, r.Np);
    r.nb = r.Mp / TB;
    r.nbw = r.Wp / TB;
    r.n_b1 = n_b1;
    r.train_off = train_off;
    r.test_off = test_off;
    r.orig = orig;
    r.oz = (r.Mp >= oz_min_rows() && M <= 8192) ? 1 : 0;      // K <= 8192 keeps the int32 accumulators exact
                                                              // (cleared again for D > 8, see restrict_oz)
    r.base = 0;
    r.oz_base = 0;
    return r;
}

// The digit-plane products are accurate relative to row-max x column-max x K.  With the 32-d deep features the
// kernel matrices span tens of decades inside a row and the fit then needs float64's componentwise accuracy
// (measured: 1e-2 differences after 50 steps at ANY digit count, DESIGN.md section 4): raw 6-d features only.
void restrict_oz(std::vector<Region>& rs, int D) {
    if (D > 8)
        for (Region& r : rs) r.oz = 0;
}

size_t region_core_doubles(const Region& r, int D) {
    return (size_t)gapro_align_up((size_t)make_layout(r.Mp, r.Np, r.Wp, D).total, 32);
}
size_t region_doubles(const Region& r, int D) {
    size_t d = region_core_doubles(r, D);
    if (r.oz) d += (size_t)gapro_align_up((size_t)oz_region_doubles(r.Mp), 32);
    return d;
}


// Trailing updates of the sweep are applied `group` block steps at a time (contraction depth group * 64);
// between two full passes only the next block column / block row is brought up to date.
static int sweep_group_size() {
    int g = 4;      // measured on the bench batch: 2 -> 1563 ms, 4 -> 1544 ms, 8 -> 1559 ms per step
    if (const char* e = getenv("GAPRO_GP_SWEEP_GROUP")) g = atoi(e);
    return g < 1 ? 1 : (g > 8 ? 8 : g);
}

// entries of every descriptor / tile table of a set of regions (exact; additive over regions)
enum { TC_REGS = 0, TC_FULL, TC_LOWER, TC_WIDE, TC_ROWS, TC_ROWSP, TC_PANEL, TC_UPD, TC_FULL_S, TC_LOWER_S, TC_OZ_VB,
       TC_OZ_BLK, TC_OZ_FULL, TC_OZ_LOWER, TC_COUNT };
static const size_t TC_ELEM[TC_COUNT] = {sizeof(Region), 16, 16, 16, 8, 8, 8, 16, 16, 16, 8, 16, 16, 16};

void count_tables(const std::vector<Region>& rs, size_t (&n)[TC_COUNT]) {
    for (int i = 0; i < TC_COUNT; ++i) n[i] = 0;
    const int sg = sweep_group_size();
    n[TC_REGS] = rs.size();
    for (const Region& r : rs) {
        const size_t full = (size_t)r.nb * r.nb, lower = (size_t)r.nb * (r.nb + 1) / 2;
        n[TC_FULL] += full;
        n[TC_LOWER] += lower;
        n[TC_WIDE] += (size_t)r.nb * r.nbw;
        n[TC_ROWS] += r.nb;
        for (int t = 0; t < r.Np / TB; ++t) n[TC_ROWSP] += (t * TB < r.N);
        n[TC_PANEL] += r.nb - 1;
        for (int kb = 0; kb < r.nb; ++kb) {
            if (kb % sg == sg - 1) {
                for (int i = r.nb - 1; i > kb; --i) n[TC_UPD] += i + 1;
            } else if (kb + 1 < r.nb) {
                n[TC_UPD] += (r.nb - 1 - kb) + (kb + 1);
            }
        }
        if (!r.oz) {
            n[TC_FULL_S] += full;
            n[TC_LOWER_S] += lower;
        } else {
            const int kbt = (r.M + 63) / 64, t128 = (r.M + 127) / 128;
            n[TC_OZ_VB] += kbt;
            n[TC_OZ_BLK] += (size_t)kbt * kbt;
            n[TC_OZ_FULL] += (size_t)t128 * kbt;
            for (int ti = 0; ti < t128; ++ti)
                for (int tj = 0; tj < kbt; ++tj) n[TC_OZ_LOWER] += (tj * 64 <= ti * 128 + 127);
        }
    }
}
size_t tables_bytes(const size_t (&n)[TC_COUNT]) {
    size_t b = 0;
    for (int i = 0; i < TC_COUNT; ++i) b += gapro_align_up(n[i] ? n[i] * TC_ELEM[i] : 1, 256);
    return b;
}

// bytes of descriptors + tile tables for a set of regions that run_regions may split into up to MAX_GROUPS = 8
// stream groups: the counts are additive over regions, every group pays its own per-table alignment
size_t aux_bytes(const std::vector<Region>& rs) {
    size_t n[TC_COUNT];
    count_tables(rs, n);
    return tables_bytes(n) + (size_t)8 * TC_COUNT * 256;
}

thread_local int64_t g_launches = 0;

struct ChunkTables {
    Region* regs;
    int4 *full, *lower, *wide;
    int2 *rows, *rowsp, *panel;
    int4* upd;                      // update tiles of all block steps, step-major
    std::vector<int> upd_off;       // upd_off[kb] .. upd_off[kb+1]: tiles of step kb
    int n_full, n_lower, n_wide, n_rows, n_rowsp;
    // the tile products of the training steps: small regions (DMMA tiles) / large regions (tcgen05, gp_ozaki.cuh)
    int4 *full_s, *lower_s, *oz_blk, *oz_full, *oz_lower;
    int2* oz_vb;
    int n_full_s, n_lower_s, n_oz_vb, n_oz_blk, n_oz_full, n_oz_lower, oz_max_m = 0;
    std::vector<int> cnt_gt;        // cnt_gt[kb] = #regions with nb > kb
    std::vector<int> panel_prefix;  // panel tiles of the first cnt_gt[kb] regions
    int nbmax;
    int sweep_group;                // block steps whose trailing updates are applied in one pass
    int n_small = 0;                // trailing single-tile regions trained by k_small_fit (they are the LAST regions of
                                    // the size-sorted list and own exactly one entry of full / lower / rows / *_s)
};



// ---- opt-in per-phase profiling with CUDA events on the launching stream ------------------
constexpr int PROF_PREDICT = PH_COUNT, PROF_SETUP = PH_COUNT + 1, PROF_SLOTS = PH_COUNT + 2;
struct ProfSpan {
    int slot, group;
    cudaEvent_t a, b;
};
thread_local int g_prof_group = 0;
struct ProfState {
    bool on = false;
    std::vector<ProfSpan> spans;
    double flops_alg[PROF_SLOTS] = {0};   // algorithmic flops (unpadded sizes, FMA = 2)
    double flops_exe[PROF_SLOTS] = {0};   // flops actually issued by the tile kernels (padding, whole tiles)
    int64_t launches[PROF_SLOTS] = {0};
};
thread_local ProfState g_prof;

void prof_begin(int slot, cudaStream_t st) {
    if (!g_prof.on) return;
    ProfSpan sp;
    sp.slot = slot;
    sp.group = g_prof_group;
    cudaEventCreate(&sp.a);
    cudaEventCreate(&sp.b);
    cudaEventRecord(sp.a, st);
    g_prof.spans.push_back(sp);
}
void prof_end(cudaStream_t st) {
    if (!g_prof.on) return;
    cudaEventRecord(g_prof.spans.back().b, st);
}

// flops of one training step of one region, per phase
void prof_account_train(const Region& r, int steps) {
    if (!g_prof.on) return;
    const double M = r.M, Mp = r.Mp, m3 = M * M * M, nb = r.nb, t3 = 2.0 * 64 * 64 * 64;
    const double tri = nb * (nb + 1) / 2;               // lower tiles
    const double kfull_tri = t3 * nb * tri;             // triangular operand x full: sum_ti (ti+1) * nb tiles
    auto add = [&](int ph, double alg, double exe) {
        g_prof.flops_alg[ph] += steps * alg;
        g_prof.flops_exe[ph] += steps * exe;
    };
    add(PH_CHOL, 2.0 * m3 / 3.0, t3 * (nb * (nb - 1) + (nb - 1) * nb * (nb + 1) / 3.0));
    add(PH_A, m3, kfull_tri);
    add(PH_B, m3, kfull_tri);
    add(PH_GA, m3, kfull_tri);
    add(PH_GT, m3, t3 * tri * nb);
    add(PH_GC, m3, kfull_tri);
    add(PH_GL, m3, t3 * tri * nb);
    add(PH_Y, 2.0 * m3 / 3.0, t3 * nb * (nb + 1) * (2 * nb + 1) / 6.0);
    add(PH_GK, m3 / 3.0, t3 * nb * (nb + 1) * (nb + 2) / 6.0);
    (void)Mp;
}

struct Driver {
    cudaStream_t stream;
    int D;
    double lr, jitter_zz, jitter_xx;
    double* ws;
    int n_regs;
    ChunkTables tb;
    PredictOut po;
    // two-priority scheme: the latency-bound part of a step (kernel matrices + block sweep) runs on a
    // high-priority stream, the throughput-bound tile products on a low-priority one, so that the block
    // chain of one group is scheduled ahead of the other groups' tile products instead of behind them
    cudaStream_t s_hi = nullptr, s_lo = nullptr;
    cudaEvent_t ev_swept = nullptr, ev_stepped = nullptr;
    cudaEvent_t ev_prev_swept = nullptr;   // first sweep of the previous group: staggers the groups by one sweep
    cudaEvent_t ev_small = nullptr;        // k_small_fit of this group has finished (it runs on its own stream)
    // careful mode (ONE region on the caller's stream, after the batched pass flagged it): every Cholesky is
    // checked on the host and retried with psd_safe_cholesky's jitter ladder
    bool careful = false;
    int retries = 0;
    bool failed = false;

    // gpytorch.utils.cholesky.psd_safe_cholesky: plain attempt, then +1e-8 * 10^k on the diagonal for k = 0, 1, 2
    // (float64 `cholesky_jitter`, max_tries 3), NotPSDError after that
    int factor_careful(const GpParams& p) {
        for (int level = 0;; ++level) {
            GpParams q = p;
            if (level) q.jitter_zz = p.jitter_zz + 1e-8 * pow(10.0, (double)(level - 1));
            GAPRO_CUDA_TRY(cudaMemsetAsync(po.status + tb_orig, 0, 4, stream));
            build(q);
            cholesky(q);
            int32_t h = 0;
            GAPRO_CUDA_TRY(cudaMemcpyAsync(&h, po.status + tb_orig, 4, cudaMemcpyDeviceToHost, stream));
            GAPRO_CUDA_TRY(cudaStreamSynchronize(stream));
            if (!(h & GAPRO_GP_NOT_PSD)) {
                retries += level;
                return GAPRO_OK;
            }
            if (level == 3) {
                retries += level;
                failed = true;
                return GAPRO_OK;
            }
        }
    }
    int tb_orig = 0;                       // careful mode: index of the region in the caller's order

    void to_hi() {
        if (!s_hi) return;
        cudaStreamWaitEvent(s_hi, ev_stepped, 0);      // (a never-recorded event is complete)
        stream = s_hi;
    }
    void to_lo() {
        if (!s_hi) return;
        cudaEventRecord(ev_swept, s_hi);
        cudaStreamWaitEvent(s_lo, ev_swept, 0);
        stream = s_lo;
    }
    void step_done() {
        if (s_hi) cudaEventRecord(ev_stepped, s_lo);
    }

    GpParams params(int step, int predict) const {
        GpParams p;
        p.D = D;
        p.jitter_zz = jitter_zz;
        p.jitter_xx = jitter_xx;
        p.predict = predict;
        if (step > 0) {
            p.lr_over_bc1 = lr / (1.0 - pow(BETA1, (double)step));
            p.bc2_sqrt = sqrt(1.0 - pow(BETA2, (double)step));
        } else {
            p.lr_over_bc1 = 0.0;
            p.bc2_sqrt = 1.0;
        }
        return p;
    }

    void oz_slice(int mat, int flags, int buf, const GpParams& p) {
        k_oz_zero_b<<<tb.n_oz_vb, 64, 0, stream>>>(tb.regs, tb.oz_vb, ws, buf);
        k_oz_vecmax_b<<<dim3(tb.n_oz_vb, (tb.oz_max_m + OZ_KCH - 1) / OZ_KCH), 256, 0, stream>>>(tb.regs, tb.oz_vb, p, ws,
                                                                                                mat, flags, buf);
        k_oz_slice_b<<<tb.n_oz_blk, 256, 0, stream>>>(tb.regs, tb.oz_blk, p, ws, mat, flags, buf);
        g_launches += 3;
    }
    template <int PH>
    void oz_gemm(bool lower, int abuf, int bbuf, const GpParams& p) {
        const int4* tiles = lower ? tb.oz_lower : tb.oz_full;
        const int n = lower ? tb.n_oz_lower : tb.n_oz_full;
        k_oz_gemm_b<PH><<<n, oz::OZ_THREADS, oz::oz_smem_bytes(OZ_S), stream>>>(tb.regs, tiles, p, ws, abuf, bbuf);
        ++g_launches;
    }
    // phase PH of the large regions: slice the operands it contracts, then the tcgen05 tile product
    template <int PH>
    void oz_phase(const GpParams& p) {
        if (tb.n_oz_vb <= 0) return;
        if (PH == PH_A) {            // A = L^-1 K_zx
            oz_slice(OM_LINV, 0, OB_LR, p);
            oz_slice(OM_LINV, OZF_TRANS, OB_LC, p);      // columns of L^-1: G_C, Y, G_K
            oz_slice(OM_KZX, OZF_TRANS, OB_X1, p);
            oz_gemm<PH_A>(false, OB_LR, OB_X1, p);
        } else if (PH == PH_B) {     // B = T^T A
            oz_slice(OM_T, OZF_TRANS, OB_X2, p);
            oz_slice(OM_A, OZF_TRANS, OB_X3, p);
            oz_gemm<PH_B>(false, OB_X2, OB_X3, p);
        } else if (PH == PH_GA) {    // T B
            oz_slice(OM_T, 0, OB_X1, p);
            oz_slice(OM_BM, OZF_TRANS, OB_X2, p);
            oz_gemm<PH_GA>(false, OB_X1, OB_X2, p);
        } else if (PH == PH_GT) {    // A diag(g_v) B^T
            oz_slice(OM_A, OZF_GV, OB_X1, p);
            oz_slice(OM_BM, 0, OB_X2, p);
            oz_gemm<PH_GT>(true, OB_X1, OB_X2, p);
        } else if (PH == PH_GC) {    // L^-T G_A
            oz_slice(OM_GA, OZF_TRANS, OB_X1, p);
            oz_gemm<PH_GC>(false, OB_LC, OB_X1, p);
        } else if (PH == PH_GL) {    // G_A A^T
            oz_slice(OM_GA, 0, OB_X1, p);
            oz_slice(OM_A, 0, OB_X2, p);
            oz_gemm<PH_GL>(true, OB_X1, OB_X2, p);
        } else if (PH == PH_Y) {     // S L^-1   (S in the B buffer)
            oz_slice(OM_BM, 0, OB_X1, p);
            oz_gemm<PH_Y>(true, OB_X1, OB_LC, p);
        } else if (PH == PH_GK) {    // L^-T Y   (Y in the G_A buffer, lower tiles only)
            oz_slice(OM_GA, OZF_TRANS | OZF_YTRI, OB_X1, p);
            oz_gemm<PH_GK>(true, OB_LC, OB_X1, p);
        }
    }

    template <int PH>
    void gemm(const int4* tiles, int n, const GpParams& p) {
        if (n <= 0) return;
        k_gemm<PH><<<n, GEMM_THREADS, GEMM_SMEM, stream>>>(tb.regs, tiles, p, ws);
        ++g_launches;
    }

    void build(const GpParams& p) {
        const int4* tiles = p.predict ? tb.wide : tb.full;
        const int n = p.predict ? tb.n_wide : tb.n_full - tb.n_small;
        if (n <= 0) return;
        if (D > 32)
            k_build_wide<2><<<n, 256, build_wide_smem<2>(), stream>>>(tb.regs, tiles, p, ws);
        else if (D > 8)
            k_build_wide<1><<<n, 256, build_wide_smem<1>(), stream>>>(tb.regs, tiles, p, ws);
        else
            k_build<<<n, 256, (TB * D + 2 * D * (TB + 1)) * sizeof(double), stream>>>(tb.regs, tiles, p, ws);
        ++g_launches;
    }

    void cholesky(const GpParams& p) {
        for (int kb = 0; kb < tb.nbmax; ++kb) {
            const int live = tb.cnt_gt[kb] - ((kb == 0 && !p.predict) ? tb.n_small : 0);
            if (live <= 0) break;
            k_rl_diag<<<live, GEMM_THREADS, DIAG_SMEM, stream>>>(tb.regs, kb, p, ws, po.status);
            ++g_launches;
            const int np = tb.panel_prefix[kb];
            if (np > 0) {
                k_rl_panel<<<np, GEMM_THREADS, GEMM_SMEM, stream>>>(tb.regs, tb.panel, kb, p, ws);
                ++g_launches;
            }
            const int nu = tb.upd_off[kb + 1] - tb.upd_off[kb];
            if (nu > 0) {
                const int kb0 = kb - kb % tb.sweep_group, nk = kb - kb0 + 1;
                k_rl_update<<<nu, GEMM_THREADS, GEMM_SMEM, stream>>>(tb.regs, tb.upd + tb.upd_off[kb], kb0, nk, p, ws);
                ++g_launches;
            }
        }
    }

    void kgrad(const GpParams& p) {
        const int nr = tb.n_rows - tb.n_small;
        if (nr <= 0) return;
        if (D <= 6)
            k_kgrad<6, 4><<<nr * 2, 256, kgrad_smem<6, 4>(), stream>>>(tb.regs, tb.rows, p, ws);
        else if (D <= 8)
            k_kgrad<8, 4><<<nr * 2, 256, kgrad_smem<8, 4>(), stream>>>(tb.regs, tb.rows, p, ws);
        else if (D <= 32)
            k_kgrad_wide<1><<<nr, 256, kgrad_wide_smem<1>(), stream>>>(tb.regs, tb.rows, p, ws);
        else
            k_kgrad_wide<2><<<nr, 256, kgrad_wide_smem<2>(), stream>>>(tb.regs, tb.rows, p, ws);
        ++g_launches;
    }

    // one training step; stop_phase < PH_COUNT truncates it (debug)
    void train_step(int step, int stop_phase) {
        const GpParams p = params(step, 0);
        int ph = 0;
#define PHASE(X)                     \
    if (ph >= stop_phase) return;    \
    prof_begin(ph, stream);          \
    X;                               \
    prof_end(stream);                \
    ++ph;
        to_hi();
        if (step == 1 && s_hi && ev_prev_swept) cudaStreamWaitEvent(s_hi, ev_prev_swept, 0);
        if (careful) {
            if (failed || factor_careful(p) != GAPRO_OK || failed) return;
            ph = 2;
        } else {
            PHASE(build(p))
            PHASE(cholesky(p))
        }
        to_lo();
        const int nfs = tb.n_full_s - tb.n_small, nls = tb.n_lower_s - tb.n_small, nrw = tb.n_rows - tb.n_small;
        const int nrg = n_regs - tb.n_small;
        PHASE((gemm<PH_A>(tb.full_s, nfs, p), oz_phase<PH_A>(p)))
        PHASE((gemm<PH_B>(tb.full_s, nfs, p), oz_phase<PH_B>(p)))
        PHASE((nrw > 0 ? (k_colstats<<<nrw, 256, 0, stream>>>(tb.regs, tb.rows, p, ws, po), ++g_launches) : 0))
        PHASE((gemm<PH_GA>(tb.full_s, nfs, p), oz_phase<PH_GA>(p)))
        PHASE((gemm<PH_GT>(tb.lower_s, nls, p), oz_phase<PH_GT>(p)))
        PHASE((nrw > 0 ? (k_grad_m<<<nrw, 256, 0, stream>>>(tb.regs, tb.rows, p, ws), ++g_launches) : 0))
        PHASE((gemm<PH_GC>(tb.full_s, nfs, p), oz_phase<PH_GC>(p)))
        PHASE((gemm<PH_GL>(tb.lower_s, nls, p), oz_phase<PH_GL>(p)))
        PHASE((void)0)   // (slot of the former L^T G_L product, folded into the previous phase)
        PHASE((gemm<PH_Y>(tb.lower_s, nls, p), oz_phase<PH_Y>(p)))   // G_K's lower tiles read only Y[k >= j]
        PHASE((gemm<PH_GK>(tb.lower_s, nls, p), oz_phase<PH_GK>(p)))
        PHASE(kgrad(p))
        PHASE((nrg > 0 ? (k_adam_small<<<nrg, 256, 0, stream>>>(tb.regs, p, ws), ++g_launches) : 0))
#undef PHASE
        step_done();
    }

    void predict() {
        const GpParams p = params(0, 1);
        prof_begin(PROF_PREDICT, stream);
        to_hi();
        if (ev_small) cudaStreamWaitEvent(stream, ev_small, 0);      // the small regions' trained state
        if (careful) {
            if (failed || factor_careful(p) != GAPRO_OK || failed) return;
        } else {
            build(p);
            cholesky(p);
        }
        to_lo();
        gemm<PH_A>(tb.wide, tb.n_wide, p);
        gemm<PH_B>(tb.wide, tb.n_wide, p);
        if (tb.n_rowsp > 0) {
            k_colstats<<<tb.n_rowsp, 256, 0, stream>>>(tb.regs, tb.rowsp, p, ws, po);
            ++g_launches;
        }
        prof_end(stream);
    }
};

// lays out one chunk (regions already carry .base), uploads descriptors and tile tables
int setup_chunk(std::vector<Region>& rs, char* aux, const char* aux_end, cudaStream_t stream, ChunkTables& tb,
                size_t* consumed) {
    std::vector<int4> full, lower, wide, full_s, lower_s, oz_blk, oz_full, oz_lower;
    std::vector<int2> rows, rowsp, panel, oz_vb;
    tb.nbmax = 0;
    tb.oz_max_m = 0;
    for (size_t r = 0; r < rs.size(); ++r) tb.nbmax = std::max(tb.nbmax, rs[r].nb);
    tb.cnt_gt.assign(tb.nbmax + 1, 0);
    tb.panel_prefix.assign(tb.nbmax + 1, 0);
    std::vector<int> panel_before(rs.size() + 1, 0);
    for (size_t r = 0; r < rs.size(); ++r) {
        const Region& R = rs[r];
        for (int ti = 0; ti < R.nb; ++ti) {
            for (int tj = 0; tj < R.nb; ++tj) full.push_back(make_int4((int)r, ti, tj, 0));
            for (int tj = 0; tj <= ti; ++tj) lower.push_back(make_int4((int)r, ti, tj, 0));
            for (int tj = 0; tj < R.nbw; ++tj) wide.push_back(make_int4((int)r, ti, tj, 0));
            rows.push_back(make_int2((int)r, ti));
            if (!R.oz) {
                for (int tj = 0; tj < R.nb; ++tj) full_s.push_back(make_int4((int)r, ti, tj, 0));
                for (int tj = 0; tj <= ti; ++tj) lower_s.push_back(make_int4((int)r, ti, tj, 0));
            }
        }
        if (R.oz) {
            const int kbt = (R.M + 63) / 64, t128 = (R.M + 127) / 128;
            tb.oz_max_m = std::max(tb.oz_max_m, R.M);
            for (int vb = 0; vb < kbt; ++vb) oz_vb.push_back(make_int2((int)r, vb));
            for (int kb = 0; kb < kbt; ++kb)
                for (int rb = 0; rb < kbt; ++rb) oz_blk.push_back(make_int4((int)r, kb, rb, 0));
            for (int ti = 0; ti < t128; ++ti)
                for (int tj = 0; tj < kbt; ++tj) {
                    oz_full.push_back(make_int4((int)r, ti, tj, 0));
                    if (tj * 64 <= ti * 128 + 127) oz_lower.push_back(make_int4((int)r, ti, tj, 0));
                }
        }
        for (int t = 0; t < R.Np / TB; ++t)
            if (t * TB < R.N) rowsp.push_back(make_int2((int)r, t));
        for (int t = 0; t < R.nb - 1; ++t) panel.push_back(make_int2((int)r, t));
        panel_before[r + 1] = (int)panel.size();
        for (int kb = 0; kb < R.nb; ++kb) tb.cnt_gt[kb]++;
    }
    // regions are sorted by nb descending, so {nb > kb} is the prefix of length cnt_gt[kb]
    for (int kb = 0; kb <= tb.nbmax; ++kb) tb.panel_prefix[kb] = panel_before[tb.cnt_gt[kb]];
    // update tiles, step-major.  Steps are grouped by sweep_group.  Last step of a group: every lower tile
    // (i, j <= i) with i > kb receives all steps of the group in one pass; any other step kb: only block
    // column kb+1 (K tiles) and block row kb+1 (S tiles) receive the steps of the group so far.
    std::vector<int4> upd;
    tb.sweep_group = sweep_group_size();
    tb.upd_off.assign(tb.nbmax + 1, 0);
    for (int kb = 0; kb < tb.nbmax; ++kb) {
        tb.upd_off[kb] = (int)upd.size();
        const int live = tb.cnt_gt[kb];
        for (int r = 0; r < live; ++r) {
            const int nb = rs[r].nb;
            if (kb % tb.sweep_group == tb.sweep_group - 1) {
                for (int i = nb - 1; i > kb; --i)
                    for (int j = 0; j <= i; ++j) upd.push_back(make_int4(r, i, j, 0));
            } else if (kb + 1 < nb) {
                for (int i = nb - 1; i > kb; --i) upd.push_back(make_int4(r, i, kb + 1, 0));
                for (int j = 0; j <= kb; ++j) upd.push_back(make_int4(r, kb + 1, j, 0));
            }
        }
    }
    tb.upd_off[tb.nbmax] = (int)upd.size();
    // table bytes of this group before anything is copied: the chunk was sized with aux_bytes(chunk), which
    // covers the tables of all its groups and their per-table alignment
    {
        size_t n[TC_COUNT];
        count_tables(rs, n);
        const size_t need = tables_bytes(n);
        const size_t have[TC_COUNT] = {rs.size(), full.size(), lower.size(), wide.size(), rows.size(), rowsp.size(),
                                       panel.size(), upd.size(), full_s.size(), lower_s.size(), oz_vb.size(),
                                       oz_blk.size(), oz_full.size(), oz_lower.size()};
        for (int i = 0; i < TC_COUNT; ++i)
            if (have[i] != n[i]) {
                gapro_set_error("gapro_gp_fit_batch: tile table %d has %zu entries, the layout counted %zu", i, have[i], n[i]);
                return GAPRO_ERR_WORKSPACE;
            }
        if (aux + need > aux_end) {
            gapro_set_error("gapro_gp_fit_batch: tile tables (%zu bytes) overrun the workspace by %zu bytes", need,
                            (size_t)(aux + need - aux_end));
            return GAPRO_ERR_WORKSPACE;
        }
    }
    size_t o = 0;
    auto put = [&](const void* src, size_t bytes) -> char* {
        char* dst = aux + o;
        o += gapro_align_up(bytes ? bytes : 1, 256);
        if (bytes) cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream);
        return dst;
    };
    tb.regs = (Region*)put(rs.data(), rs.size() * sizeof(Region));
    tb.full = (int4*)put(full.data(), full.size() * 16);
    tb.lower = (int4*)put(lower.data(), lower.size() * 16);
    tb.wide = (int4*)put(wide.data(), wide.size() * 16);
    tb.rows = (int2*)put(rows.data(), rows.size() * 8);
    tb.rowsp = (int2*)put(rowsp.data(), rowsp.size() * 8);
    tb.panel = (int2*)put(panel.data(), panel.size() * 8);
    tb.upd = (int4*)put(upd.data(), upd.size() * 16);
    tb.full_s = (int4*)put(full_s.data(), full_s.size() * 16);
    tb.lower_s = (int4*)put(lower_s.data(), lower_s.size() * 16);
    tb.oz_vb = (int2*)put(oz_vb.data(), oz_vb.size() * 8);
    tb.oz_blk = (int4*)put(oz_blk.data(), oz_blk.size() * 16);
    tb.oz_full = (int4*)put(oz_full.data(), oz_full.size() * 16);
    tb.oz_lower = (int4*)put(oz_lower.data(), oz_lower.size() * 16);
    tb.n_full_s = (int)full_s.size();
    tb.n_lower_s = (int)lower_s.size();
    tb.n_oz_vb = (int)oz_vb.size();
    tb.n_oz_blk = (int)oz_blk.size();
    tb.n_oz_full = (int)oz_full.size();
    tb.n_oz_lower = (int)oz_lower.size();
    *consumed = o;
    tb.n_full = (int)full.size();
    tb.n_lower = (int)lower.size();
    tb.n_wide = (int)wide.size();
    tb.n_rows = (int)rows.size();
    tb.n_rowsp = (int)rowsp.size();
    // the host vectors die at return: the copies above must have been consumed
    GAPRO_CUDA_TRY(cudaStreamSynchronize(stream));
    return GAPRO_OK;
}

int check_device() {
    int dev = 0;
    GAPRO_CUDA_TRY(cudaGetDevice(&dev));
    return GAPRO_OK;
}

std::vector<Region> sorted_regions(int n_regions, const int32_t* train_off, const int32_t* n_b1,
                                   const int32_t* test_off) {
    std::vector<Region> rs;
    rs.reserve(n_regions);
    for (int r = 0; r < n_regions; ++r)
        rs.push_back(make_region(train_off[r + 1] - train_off[r], test_off[r + 1] - test_off[r], n_b1 ? n_b1[r] : 0,
                                 train_off[r], test_off[r], r));
    std::stable_sort(rs.begin(), rs.end(), [](const Region& a, const Region& b) {
        if (a.nb != b.nb) return a.nb > b.nb;
        return a.nbw > b.nbw;
    });
    return rs;
}

}  // namespace

extern "C" size_t gapro_gp_workspace_bytes(int32_t n_regions, const int32_t* train_off, const int32_t* test_off,
                                           int32_t D) {
    if (n_regions <= 0 || !train_off || !test_off || D <= 0) return 0;
    std::vector<Region> rs = sorted_regions(n_regions, train_off, nullptr, test_off);
    restrict_oz(rs, D);
    size_t doubles = 0;
    for (const Region& r : rs) doubles += region_doubles(r, D);
    return doubles * 8 + aux_bytes(rs);
}

extern "C" size_t gapro_gp_min_workspace_bytes(int32_t n_regions, const int32_t* train_off, const int32_t* test_off,
                                               int32_t D) {
    if (n_regions <= 0 || !train_off || !test_off || D <= 0) return 0;
    std::vector<Region> rs = sorted_regions(n_regions, train_off, nullptr, test_off);
    restrict_oz(rs, D);
    size_t best = 0;
    for (const Region& r : rs) {
        std::vector<Region> one(1, r);
        best = std::max(best, region_doubles(r, D) * 8 + aux_bytes(one));
    }
    return best;
}

extern "C" int64_t gapro_gp_last_launch_count(void) { return g_launches; }

// Host-only replay of the workspace arithmetic (no CUDA call): the regions are split round-robin over `groups`
// stream groups exactly as run_regions does; returns (bytes aux_bytes() reserves for the whole chunk) - (bytes the
// groups' tile tables take with their per-table alignment).  Negative = the tables would overrun the workspace.
extern "C" int64_t gapro_gp_debug_aux_slack(int32_t n_regions, const int32_t* train_off, const int32_t* test_off,
                                            int32_t groups) {
    if (n_regions <= 0 || !train_off || !test_off || groups < 1) return 0;
    std::vector<Region> rs = sorted_regions(n_regions, train_off, nullptr, test_off);
    std::vector<std::vector<Region>> gs(groups);
    for (size_t i = 0; i < rs.size(); ++i) gs[i % groups].push_back(rs[i]);
    int64_t used = 0;
    for (const std::vector<Region>& g : gs) {
        if (g.empty()) continue;
        size_t n[TC_COUNT];
        count_tables(g, n);
        used += (int64_t)tables_bytes(n);
    }
    return (int64_t)aux_bytes(rs) - used;
}

// ---- side streams: independent region groups run concurrently so that the latency-bound
// Cholesky sweep of one group overlaps the tile products of the others --------------------------------
constexpr int MAX_GROUPS = 8;
struct StreamPool {
    cudaStream_t hi[MAX_GROUPS] = {};
    cudaStream_t lo[MAX_GROUPS] = {};
    cudaEvent_t fork = nullptr, join[MAX_GROUPS] = {};
    cudaEvent_t swept[MAX_GROUPS] = {};
    cudaEvent_t stepped[MAX_GROUPS] = {};
    cudaStream_t aux[MAX_GROUPS] = {};                       // the one-CTA-per-small-region kernel of a group
    cudaEvent_t small_fork[MAX_GROUPS] = {}, small_done[MAX_GROUPS] = {};
    bool ready = false;
};
// streams and events belong to the device that was current when they were created: one pool per device
constexpr int MAX_DEVICES = 64;
thread_local StreamPool g_pools[MAX_DEVICES];
thread_local StreamPool* g_pool_ptr = &g_pools[0];
#define g_pool (*g_pool_ptr)

static int ensure_pool() {
    int dev = 0;
    GAPRO_CUDA_TRY(cudaGetDevice(&dev));
    GAPRO_REQUIRE(dev >= 0 && dev < MAX_DEVICES, "gp: device ordinal %d not supported", dev);
    g_pool_ptr = &g_pools[dev];
    if (g_pool.ready) return GAPRO_OK;
    int least = 0, greatest = 0;
    GAPRO_CUDA_TRY(cudaDeviceGetStreamPriorityRange(&least, &greatest));
    for (int i = 0; i < MAX_GROUPS; ++i) {
        GAPRO_CUDA_TRY(cudaStreamCreateWithPriority(&g_pool.hi[i], cudaStreamNonBlocking, greatest));
        GAPRO_CUDA_TRY(cudaStreamCreateWithPriority(&g_pool.lo[i], cudaStreamNonBlocking, least));
        GAPRO_CUDA_TRY(cudaEventCreateWithFlags(&g_pool.join[i], cudaEventDisableTiming));
        GAPRO_CUDA_TRY(cudaEventCreateWithFlags(&g_pool.swept[i], cudaEventDisableTiming));
        GAPRO_CUDA_TRY(cudaEventCreateWithFlags(&g_pool.stepped[i], cudaEventDisableTiming));
        GAPRO_CUDA_TRY(cudaStreamCreateWithPriority(&g_pool.aux[i], cudaStreamNonBlocking, least));
        GAPRO_CUDA_TRY(cudaEventCreateWithFlags(&g_pool.small_fork[i], cudaEventDisableTiming));
        GAPRO_CUDA_TRY(cudaEventCreateWithFlags(&g_pool.small_done[i], cudaEventDisableTiming));
    }
    GAPRO_CUDA_TRY(cudaEventCreateWithFlags(&g_pool.fork, cudaEventDisableTiming));
    g_pool.ready = true;
    return GAPRO_OK;
}

static int n_groups_for(const std::vector<Region>& chunk) {
    // default 4.  Measured: 1602 / 1596 / 1548 ms per step with 1 / 2 / 4 groups on the 8-scene bench batch; one
    // configs[1] scene (93 regions): 82.1 / 81.9 / 75.5 ms with 2000 / 3828 / 7484 launches - even the single scene
    // is bound by the dependent chain of small kernels on the GPU, not by the host's launch rate.
    const size_t n_regions = chunk.size();
    int g = 4;
    if (const char* e = getenv("GAPRO_GP_STREAMS")) g = atoi(e);
    if (g < 1) g = 1;
    if (g > MAX_GROUPS) g = MAX_GROUPS;
    // per-phase event timing needs a single stream (GAPRO_GP_TIMELINE keeps the groups: overlapping spans)
    if (g_prof.on && !getenv("GAPRO_GP_TIMELINE")) g = 1;
    while (g > 1 && n_regions < (size_t)4 * g) --g;
    return g;
}

template <typename K>
static int allow_smem(K kernel, int bytes) {
    if (bytes > 0) GAPRO_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    // one shared-memory carve-out for every kernel of the stage: CTAs of kernels running concurrently on
    // different streams can then be co-resident on an SM
    GAPRO_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                        (int)cudaSharedmemCarveoutMaxShared));
    return GAPRO_OK;
}

static int set_kernel_attributes() {
    // cudaFuncSetAttribute is per device (several engines may live in one process)
    static bool done_dev[MAX_DEVICES] = {};
    int dev = 0;
    GAPRO_CUDA_TRY(cudaGetDevice(&dev));
    GAPRO_REQUIRE(dev >= 0 && dev < MAX_DEVICES, "gp: device ordinal %d not supported", dev);
    bool& done = done_dev[dev];
    if (done) return GAPRO_OK;
    int rc = allow_smem(k_build, (TB * 64 + 2 * 64 * (TB + 1)) * 8);
    if (rc == GAPRO_OK) rc = allow_smem(k_build_wide<1>, build_wide_smem<1>());
    if (rc == GAPRO_OK) rc = allow_smem(k_build_wide<2>, build_wide_smem<2>());
    if (rc == GAPRO_OK) rc = allow_smem(k_rl_diag, DIAG_SMEM);
    if (rc == GAPRO_OK) rc = allow_smem(k_small_fit, SM_SMEM);
    if (rc == GAPRO_OK) rc = allow_smem(k_rl_panel, GEMM_SMEM);
    if (rc == GAPRO_OK) rc = allow_smem(k_rl_update, GEMM_SMEM);
    if (rc == GAPRO_OK) rc = allow_smem(k_gemm<PH_A>, GEMM_SMEM);
    if (rc == GAPRO_OK) rc = allow_smem(k_gemm<PH_B>, GEMM_SMEM);
    if (rc == GAPRO_OK) rc = allow_smem(k_gemm<PH_GA>, GEMM_SMEM);
    if (rc == GAPRO_OK) rc = allow_smem(k_gemm<PH_GT>, GEMM_SMEM);
    if (rc == GAPRO_OK) rc = allow_smem(k_gemm<PH_GC>, GEMM_SMEM);
    if (rc == GAPRO_OK) rc = allow_smem(k_gemm<PH_GL>, GEMM_SMEM);
    if (rc == GAPRO_OK) rc = allow_smem(k_gemm<PH_Y>, GEMM_SMEM);
    if (rc == GAPRO_OK) rc = allow_smem(k_gemm<PH_GK>, GEMM_SMEM);
    if (rc == GAPRO_OK) rc = allow_smem(k_oz_gemm_b<PH_A>, oz::oz_smem_bytes(OZ_S));
    if (rc == GAPRO_OK) rc = allow_smem(k_oz_gemm_b<PH_B>, oz::oz_smem_bytes(OZ_S));
    if (rc == GAPRO_OK) rc = allow_smem(k_oz_gemm_b<PH_GA>, oz::oz_smem_bytes(OZ_S));
    if (rc == GAPRO_OK) rc = allow_smem(k_oz_gemm_b<PH_GT>, oz::oz_smem_bytes(OZ_S));
    if (rc == GAPRO_OK) rc = allow_smem(k_oz_gemm_b<PH_GC>, oz::oz_smem_bytes(OZ_S));
    if (rc == GAPRO_OK) rc = allow_smem(k_oz_gemm_b<PH_GL>, oz::oz_smem_bytes(OZ_S));
    if (rc == GAPRO_OK) rc = allow_smem(k_oz_gemm_b<PH_Y>, oz::oz_smem_bytes(OZ_S));
    if (rc == GAPRO_OK) rc = allow_smem(k_oz_gemm_b<PH_GK>, oz::oz_smem_bytes(OZ_S));
    if (rc == GAPRO_OK) rc = allow_smem(k_oz_vecmax_b, 0);
    if (rc == GAPRO_OK) rc = allow_smem(k_oz_zero_b, 0);
    if (rc == GAPRO_OK) rc = allow_smem(k_oz_slice_b, 0);
    if (rc == GAPRO_OK) rc = allow_smem(k_kgrad<6, 4>, kgrad_smem<6, 4>());
    if (rc == GAPRO_OK) rc = allow_smem(k_kgrad<8, 4>, kgrad_smem<8, 4>());
    if (rc == GAPRO_OK) rc = allow_smem(k_kgrad_wide<1>, kgrad_wide_smem<1>());
    if (rc == GAPRO_OK) rc = allow_smem(k_kgrad_wide<2>, kgrad_wide_smem<2>());
    if (!getenv("GAPRO_GP_DEFAULT_CARVEOUT")) {
        // the element-wise kernels too: a kernel that prefers a large L1 cannot share an SM with the tile
        // kernels of another group, which would serialise the side streams
        if (rc == GAPRO_OK) rc = allow_smem(k_colstats, 0);
        if (rc == GAPRO_OK) rc = allow_smem(k_grad_m, 0);
        if (rc == GAPRO_OK) rc = allow_smem(k_adam_small, 0);
        if (rc == GAPRO_OK) rc = allow_smem(k_region_init, 0);
    }
    done = rc == GAPRO_OK;
    return rc;
}

static int run_regions(const float* feats_spp, int32_t D, std::vector<Region>& all, const int32_t* train_idx,
                       const int32_t* test_idx, const float* init_noise, int32_t iters, int32_t stop_phase, double lr,
                       double jitter_zz, double jitter_xx, PredictOut po, void* ws, size_t ws_bytes, bool do_predict,
                       cudaStream_t stream, bool careful = false, int* retries_out = nullptr, bool* failed_out = nullptr) {
    GAPRO_REQUIRE(D >= 1 && D <= 64, "gp: feature dimension %d not in [1, 64]", D);
    restrict_oz(all, D);
    int rc = set_kernel_attributes();
    if (rc != GAPRO_OK) return rc;
    size_t pos = 0;
    while (pos < all.size()) {
        // greedy chunk: as many regions (already sorted by size) as fit in the workspace
        std::vector<Region> chunk;
        size_t doubles = 0;
        while (pos + chunk.size() < all.size()) {
            Region r = all[pos + chunk.size()];
            r.base = (long long)doubles;
            r.oz_base = (long long)(doubles + region_core_doubles(r, D));
            chunk.push_back(r);
            size_t nd = doubles + region_doubles(r, D);
            if (nd * 8 + aux_bytes(chunk) > ws_bytes) {
                chunk.pop_back();
                break;
            }
            doubles = nd;
        }
        if (chunk.empty()) {
            gapro_set_error("gapro_gp_fit_batch: workspace of %zu bytes cannot hold a region with M=%d N=%d", ws_bytes,
                            all[pos].M, all[pos].N);
            return GAPRO_ERR_WORKSPACE;
        }
        const int G = careful ? 1 : n_groups_for(chunk);
        const bool small_path = !(getenv("GAPRO_GP_SMALL") && atoi(getenv("GAPRO_GP_SMALL")) == 0);
        if (G > 1 && (rc = ensure_pool()) != GAPRO_OK) return rc;
        // round-robin over the size-sorted list: every group sees the same size distribution
        std::vector<std::vector<Region>> groups(G);
        for (size_t i = 0; i < chunk.size(); ++i) groups[i % G].push_back(chunk[i]);
        std::vector<Driver> drv(G);
        prof_begin(PROF_SETUP, stream);
        GAPRO_CUDA_TRY(cudaMemsetAsync(ws, 0, doubles * 8, stream));
        char* aux = (char*)ws + doubles * 8;
        for (int g = 0; g < G; ++g) {
            Driver& d = drv[g];
            d.stream = stream;
            if (G > 1) {
                d.s_hi = g_pool.hi[g];
                d.s_lo = g_pool.lo[g];
                d.ev_swept = g_pool.swept[g];
                d.ev_stepped = g_pool.stepped[g];
                d.stream = d.s_hi;
                if (g > 0 && !getenv("GAPRO_GP_NO_STAGGER")) d.ev_prev_swept = g_pool.swept[g - 1];
            }
            d.careful = careful;
            if (careful) d.tb_orig = groups[g][0].orig;
            d.D = D;
            d.lr = lr;
            d.jitter_zz = jitter_zz;
            d.jitter_xx = jitter_xx;
            d.ws = (double*)ws;
            d.n_regs = (int)groups[g].size();
            d.po = po;
            size_t used = 0;
            rc = setup_chunk(groups[g], aux, (const char*)ws + ws_bytes, stream, d.tb, &used);   // uploads, then syncs
            if (rc != GAPRO_OK) return rc;
            aux += used;
        }
        if (G > 1) {
            GAPRO_CUDA_TRY(cudaEventRecord(g_pool.fork, stream));
            for (int g = 0; g < G; ++g) {
                GAPRO_CUDA_TRY(cudaStreamWaitEvent(drv[g].s_hi, g_pool.fork, 0));
                GAPRO_CUDA_TRY(cudaStreamWaitEvent(drv[g].s_lo, g_pool.fork, 0));
                // a fresh "previous step finished" marker, so that the first to_hi() does not wait on a stale one
                GAPRO_CUDA_TRY(cudaEventRecord(drv[g].ev_stepped, drv[g].s_lo));
            }
        }
        for (int g = 0; g < G; ++g) {
            k_region_init<<<drv[g].n_regs, 256, 0, drv[g].stream>>>(drv[g].tb.regs, D, feats_spp, train_idx, test_idx,
                                                                    init_noise, drv[g].ws);
            ++g_launches;
            // single-tile regions: all training steps in one launch, state in shared memory (gp_small.cuh).  They
            // are the tail of the size-sorted list; the batched training kernels then skip them, prediction does not.
            int n_small = 0;
            if (small_path && D <= SM_DMAX && iters > 0 && stop_phase == 0 && !careful)
                for (size_t i = groups[g].size(); i-- > 0 && groups[g][i].nb == 1;) ++n_small;
            drv[g].tb.n_small = n_small;
            if (n_small > 0) {
                // on its own stream: ~50 dependent steps of one CTA each must not sit in front of the batched sweep
                if ((rc = ensure_pool()) != GAPRO_OK) return rc;
                GAPRO_CUDA_TRY(cudaEventRecord(g_pool.small_fork[g], drv[g].stream));
                GAPRO_CUDA_TRY(cudaStreamWaitEvent(g_pool.aux[g], g_pool.small_fork[g], 0));
                k_small_fit<<<n_small, SM_THREADS, SM_SMEM, g_pool.aux[g]>>>(drv[g].tb.regs, drv[g].n_regs - n_small,
                                                                            drv[g].params(1, 0), lr, iters, drv[g].ws,
                                                                            po.status);
                GAPRO_CUDA_TRY(cudaEventRecord(g_pool.small_done[g], g_pool.aux[g]));
                drv[g].ev_small = g_pool.small_done[g];
                ++g_launches;
            }
        }
        prof_end(stream);
        for (int g = 0; g < G; ++g) {      // flops of the batched tile kernels: not the regions k_small_fit trains
            const size_t n_batched = groups[g].size() - (size_t)drv[g].tb.n_small;
            for (size_t i = 0; i < n_batched; ++i) prof_account_train(groups[g][i], iters);
        }
        for (int it = 1; it <= iters; ++it)
            for (int g = 0; g < G; ++g) {
                g_prof_group = g;
                drv[g].train_step(it, PH_COUNT);
            }
        g_prof_group = 0;
        if (stop_phase > 0)
            for (int g = 0; g < G; ++g) drv[g].train_step(iters + 1, stop_phase);
        if (do_predict)
            for (int g = 0; g < G; ++g) drv[g].predict();
        for (int g = 0; g < G; ++g)
            if (drv[g].ev_small) GAPRO_CUDA_TRY(cudaStreamWaitEvent(stream, drv[g].ev_small, 0));
        if (G > 1)
            for (int g = 0; g < G; ++g) {
                // whatever ran last on either stream of the group must be done
                GAPRO_CUDA_TRY(cudaEventRecord(g_pool.join[g], drv[g].s_hi));
                GAPRO_CUDA_TRY(cudaStreamWaitEvent(drv[g].s_lo, g_pool.join[g], 0));
                GAPRO_CUDA_TRY(cudaEventRecord(g_pool.join[g], drv[g].s_lo));
                GAPRO_CUDA_TRY(cudaStreamWaitEvent(stream, g_pool.join[g], 0));
            }
        GAPRO_KERNEL_CHECK();
        if (careful) {
            if (retries_out) *retries_out = drv[0].retries;
            if (failed_out) *failed_out = drv[0].failed;
        }
        pos += chunk.size();
        if (pos < all.size()) GAPRO_CUDA_TRY(cudaStreamSynchronize(stream));   // workspace is reused
    }
    return GAPRO_OK;
}

extern "C" int gapro_gp_fit_batch(const float* feats_spp, int32_t D, int32_t n_regions, const int32_t* train_off,
                                  const int32_t* n_b1, const int32_t* test_off, const int32_t* train_idx,
                                  const int32_t* test_idx, const float* init_noise, int32_t iters, double lr,
                                  double jitter_zz, double jitter_xx, float* out_prob, float* out_conf,
                                  uint8_t* out_label, float* out_mu, float* out_var, double* out_mu64,
                                  double* out_var64, int32_t* status, void* ws, size_t ws_bytes, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    g_launches = 0;
    if (n_regions == 0) return GAPRO_OK;
    GAPRO_REQUIRE(n_regions > 0 && feats_spp && train_off && n_b1 && test_off && train_idx && test_idx && init_noise &&
                      out_prob && out_conf && out_label && out_mu && out_var && status && ws,
                  "gapro_gp_fit_batch: null pointer");
    GAPRO_REQUIRE(iters >= 0, "gapro_gp_fit_batch: iters < 0");
    for (int r = 0; r < n_regions; ++r) {
        const int M = train_off[r + 1] - train_off[r], N = test_off[r + 1] - test_off[r];
        GAPRO_REQUIRE(M >= 1 && N >= 1 && n_b1[r] >= 0 && n_b1[r] <= M,
                      "gapro_gp_fit_batch: region %d has M=%d N=%d n_b1=%d", r, M, N, n_b1[r]);
    }
    if (check_device() != GAPRO_OK) return GAPRO_ERR_CUDA;
    GAPRO_CUDA_TRY(cudaMemsetAsync(status, 0, (size_t)n_regions * 4, stream));
    std::vector<Region> all = sorted_regions(n_regions, train_off, n_b1, test_off);
    PredictOut po{out_prob, out_conf, out_mu, out_var, out_label, out_mu64, out_var64, status};
    int rc = run_regions(feats_spp, D, all, train_idx, test_idx, init_noise, iters, 0, lr, jitter_zz, jitter_xx, po, ws,
                         ws_bytes, true, stream);
    if (rc != GAPRO_OK) return rc;
    // The batched pass has no host round trip inside its 50 steps, so a non-positive pivot is only flagged there.
    // Regions it flagged (none in practice at jitter 1e-4 in float64) are fitted again one at a time with the retry
    // ladder of psd_safe_cholesky; status then carries the retry count, and GAPRO_GP_NOT_PSD only if the ladder
    // was exhausted (where gpytorch raises NotPSDError).
    std::vector<int32_t> h(n_regions);
    GAPRO_CUDA_TRY(cudaMemcpyAsync(h.data(), status, (size_t)n_regions * 4, cudaMemcpyDeviceToHost, stream));
    GAPRO_CUDA_TRY(cudaStreamSynchronize(stream));
    for (const Region& r : all) {
        if (!(h[r.orig] & GAPRO_GP_NOT_PSD)) continue;
        std::vector<Region> one(1, r);
        int retries = 0;
        bool failed = false;
        rc = run_regions(feats_spp, D, one, train_idx, test_idx, init_noise, iters, 0, lr, jitter_zz, jitter_xx, po, ws,
                         ws_bytes, true, stream, true, &retries, &failed);
        if (rc != GAPRO_OK) return rc;
        int32_t w = 0;
        GAPRO_CUDA_TRY(cudaMemcpyAsync(&w, status + r.orig, 4, cudaMemcpyDeviceToHost, stream));
        GAPRO_CUDA_TRY(cudaStreamSynchronize(stream));
        w = (w & GAPRO_GP_NAN) | (failed ? GAPRO_GP_NOT_PSD : 0) |
            ((retries > 0xffff ? 0xffff : retries) << GAPRO_GP_RETRY_SHIFT);
        GAPRO_CUDA_TRY(cudaMemcpyAsync(status + r.orig, &w, 4, cudaMemcpyHostToDevice, stream));
        GAPRO_CUDA_TRY(cudaStreamSynchronize(stream));
    }
    return GAPRO_OK;
}


// ---- profiling API ---------------------------------------------------------------------------
extern "C" int gapro_gp_set_profiling(int enable) {
    for (ProfSpan& sp : g_prof.spans) {
        cudaEventDestroy(sp.a);
        cudaEventDestroy(sp.b);
    }
    g_prof = ProfState();
    g_prof.on = enable != 0;
    return GAPRO_OK;
}

extern "C" const char* gapro_gp_phase_names(void) {
    return "build,chol,A,B,colstats,GA,GT,GM,GC,GL,SP,Y,GK,kgrad,adam,predict,setup";
}

// ms / flops per phase slot accumulated since gapro_gp_set_profiling(1).  SYNCHRONISES on the events.
extern "C" int gapro_gp_get_profile(double* ms, double* flops_alg, double* flops_exe, int32_t cap) {
    GAPRO_REQUIRE(ms && flops_alg && flops_exe && cap >= PROF_SLOTS, "gapro_gp_get_profile: need %d slots", PROF_SLOTS);
    for (int i = 0; i < PROF_SLOTS; ++i) {
        ms[i] = 0.0;
        flops_alg[i] = g_prof.flops_alg[i];
        flops_exe[i] = g_prof.flops_exe[i];
    }
    for (ProfSpan& sp : g_prof.spans) {
        GAPRO_CUDA_TRY(cudaEventSynchronize(sp.b));
        float t = 0.f;
        GAPRO_CUDA_TRY(cudaEventElapsedTime(&t, sp.a, sp.b));
        ms[sp.slot] += t;
    }
    if (const char* path = getenv("GAPRO_GP_TIMELINE")) {
        // development aid: every span as "slot group start_ms end_ms" relative to the first one
        if (FILE* f = fopen(path, "w")) {
            for (ProfSpan& sp : g_prof.spans) {
                float t0 = 0.f, t1 = 0.f;
                cudaEventElapsedTime(&t0, g_prof.spans.front().a, sp.a);
                cudaEventElapsedTime(&t1, g_prof.spans.front().a, sp.b);
                fprintf(f, "%d %d %.4f %.4f\n", sp.slot, sp.group, t0, t1);
            }
            fclose(f);
        }
    }
    return PROF_SLOTS;
}

// ---- FP64 pipe peak microbenchmark (the roofline denominator for the GP kernels) -------------------
namespace {
template <bool DMMA>
__global__ void __launch_bounds__(256) k_fp64_peak(double* out, int iters) {
    double acc[8][2];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j][0] = acc[j][1] = 0.0;
    const double a = 1.0 + 1e-9 * threadIdx.x, b = 1.0 - 1e-9 * threadIdx.x;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (DMMA) {
                dmma(acc[j][0], acc[j][1], a, b);
            } else {
                acc[j][0] = fma(a, b, acc[j][0]);
                acc[j][1] = fma(b, a, acc[j][1]);
            }
        }
    }
    double s = 0.0;
#pragma unroll
    for (int j = 0; j < 8; ++j) s += acc[j][0] + acc[j][1];
    if (s == 12345.678) out[0] = s;
}

// both at once: 4 DMMA (1024 FMA per warp) and 32 DFMA (1024 FMA per warp) per iteration, independent
// accumulators - do the tensor sub-pipe and the FP64 FMA pipe add up, or do they share the datapath?
__global__ void __launch_bounds__(256) k_fp64_peak_mixed(double* out, int iters) {
    double acc[4][2], f[16];
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[j][0] = acc[j][1] = 0.0;
#pragma unroll
    for (int j = 0; j < 16; ++j) f[j] = 0.0;
    const double a = 1.0 + 1e-9 * threadIdx.x, b = 1.0 - 1e-9 * threadIdx.x;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int r = 0; r < 2; ++r) {
#pragma unroll
            for (int j = 0; j < 2; ++j) dmma(acc[2 * r + j][0], acc[2 * r + j][1], a, b);
#pragma unroll
            for (int j = 0; j < 16; ++j) f[j] = fma(a, b, f[j]);
        }
    }
    double s = 0.0;
#pragma unroll
    for (int j = 0; j < 4; ++j) s += acc[j][0] + acc[j][1];
#pragma unroll
    for (int j = 0; j < 16; ++j) s += f[j];
    if (s == 12345.678) out[0] = s;
}
}  // namespace

// Returns the sustained FP64 rate in TFLOP/s of a register-resident DMMA (use_dmma=1), DFMA (0) or mixed (2) loop.
extern "C" int gapro_fp64_peak(int use_dmma, int iters, double* tflops, double* scratch_dev, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    GAPRO_REQUIRE(tflops && scratch_dev && iters > 0, "gapro_fp64_peak: bad arguments");
    int dev = 0, sms = 0;
    GAPRO_CUDA_TRY(cudaGetDevice(&dev));
    GAPRO_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int blocks = sms * 4, threads = 256;
    cudaEvent_t a, b;
    GAPRO_CUDA_TRY(cudaEventCreate(&a));
    GAPRO_CUDA_TRY(cudaEventCreate(&b));
    for (int rep = 0; rep < 2; ++rep) {   // first pass warms up
        GAPRO_CUDA_TRY(cudaEventRecord(a, stream));
        if (use_dmma == 2)
            k_fp64_peak_mixed<<<blocks, threads, 0, stream>>>(scratch_dev, iters);
        else if (use_dmma)
            k_fp64_peak<true><<<blocks, threads, 0, stream>>>(scratch_dev, iters);
        else
            k_fp64_peak<false><<<blocks, threads, 0, stream>>>(scratch_dev, iters);
        GAPRO_CUDA_TRY(cudaEventRecord(b, stream));
        GAPRO_CUDA_TRY(cudaEventSynchronize(b));
    }
    float ms = 0.f;
    GAPRO_CUDA_TRY(cudaEventElapsedTime(&ms, a, b));
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    // DMMA m8n8k4: 256 FMA per warp instruction; DFMA: 2 per thread per j
    const double fma_per_block_iter = use_dmma == 2 ? (threads / 32) * 2048.0
                                      : use_dmma  ? (threads / 32) * 8.0 * 256.0 : threads * 8.0 * 2.0;
    *tflops = 2.0 * fma_per_block_iter * blocks * (double)iters / (ms * 1e-3) / 1e12;
    return GAPRO_OK;
}

extern "C" const char* gapro_gp_debug_layout_names(void) {
    return "X,Z,Zm,Zv,gZ,Xt,y,m,mm,mv,scal,mu,var,gmu,gv,gsrow,glrow,L,Linv,T,Tm,Tv,GA,GC,Kzx,A,Bm,total,Mp,Np,Wp,Kc";
}

extern "C" int gapro_gp_debug_run(const float* feats_spp, int32_t D, int32_t M, int32_t n_b1, int32_t N,
                                  const int32_t* train_idx, const int32_t* test_idx, const float* init_noise,
                                  int32_t iters, int32_t stop_phase, double lr, double jitter_zz, double jitter_xx,
                                  void* ws, size_t ws_bytes, int64_t* layout, int32_t layout_cap, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    g_launches = 0;
    GAPRO_REQUIRE(feats_spp && train_idx && test_idx && init_noise && ws && layout, "gapro_gp_debug_run: null pointer");
    GAPRO_REQUIRE(M >= 1 && N >= 1 && layout_cap >= 32, "gapro_gp_debug_run: bad sizes");
    std::vector<Region> all(1, make_region(M, N, n_b1, 0, 0, 0));
    const Layout l = make_layout(all[0].Mp, all[0].Np, all[0].Wp, D);
    const long long vals[32] = {l.X,  l.Z,   l.Zm,    l.Zv,    l.gZ, l.Xt,   l.y, l.m,  l.mm, l.mv, l.scal,
                                l.mu, l.var, l.gmu,   l.gv,    l.gsrow, l.glrow, l.L, l.Linv, l.T, l.Tm, l.Tv,
                                l.GA, l.GC,  l.Kzx,   l.A,     l.Bm, l.total, all[0].Mp, all[0].Np, all[0].Wp, l.Kc};
    for (int i = 0; i < 32; ++i) layout[i] = vals[i];
    // status lives at the very end of the workspace for the debug run
    GAPRO_REQUIRE(ws_bytes >= 64, "gapro_gp_debug_run: workspace too small");
    int32_t* status = (int32_t*)((char*)ws + ws_bytes - 64);
    GAPRO_CUDA_TRY(cudaMemsetAsync(status, 0, 4, stream));
    PredictOut po{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, status};
    return run_regions(feats_spp, D, all, train_idx, test_idx, init_noise, iters, stop_phase, lr, jitter_zz, jitter_xx,
                       po, ws, ws_bytes - 64, false, stream);
}
