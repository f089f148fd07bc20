// Direct kriging on a dense Cholesky factor of a square kernel-covariance operator: A = L L' (nugget included), the
// solves A^-1 B and L^-1 B, log det A, and the kriging variance of C(T, S) targets.  For the n of most kriging problems
// (thousands to tens of thousands of observations) the n^3 / 3 flops of one factorisation cost less than one CG solve
// (cov_solve.cu) and serve any number of right-hand sides; the variance needs one triangular solve per target, which
// CG cannot offer at a useful price.
//
// Storage: the factor's order is rounded up to np = a multiple of CH_B = 128 and the padding is the identity,
// A_pad = [A 0; 0 I] = [L 0; 0 I][L 0; 0 I]', so every kernel works on whole 128 x 128 tiles.  L is column-major with
// pitch np (a multiple of 128 doubles: 16-byte aligned columns for cp.async), lower triangle only; the inverses of the
// np / 128 diagonal blocks are kept beside it (128 x 128 each) for the triangular solves.
//
// Blocked right-looking factorisation, for each 128-column block k:
//   1. chol_diag_kernel: L11 = chol(A11) and X11 = L11^-1, one CTA, the block resident in shared memory
//   2. panel:            L21 = A21 X11'                  (chol_gemm_kernel, set)
//   3. trailing update:  A22 -= L21 L21', lower tiles only (chol_gemm_kernel, subtract) -- the n^3 / 3 flops
// chol_gemm_kernel is one "C = / -= A B'" kernel on FP64 tensor cores (mma.sync.m8n8k4.f64 -> DMMA.8x8x4) with the
// 16-warp structure of the product kernels: a 128 x 128 tile per CTA, warps 4 x 4 over it, 32 x 32 each; k-tiles of 32
// staged through a double-buffered shared tile [k][row] (pitch 136 = 8 mod 16 doubles: the four k rows of a fragment
// load fall into the two halves of the banks -- two wavefronts for 32 doubles, the minimum).  Operand layouts are
// template parameters, so the same kernel serves the solves: forward B_j = X_jj B_j, B_(>j) -= L_(>j, j) B_j; backward
// B_j = X_jj' B_j, B_(<j) -= L_(j, <j)' B_j, on a row-major work block of width 128 .. 1024.
// Every reduction has a fixed order (no atomics): factor, solve, log-determinant and variance are bit-reproducible.
//
// Conditional Gaussian simulation (chol_simulate; LU simulation).  The N points are ordered sources first,
// P = [S (ns points); T (m = N - ns)], and the factor is that of the joint matrix A = C(P, P) + diag(d), d_i = the nugget
// for i < ns (observation noise) and tau for the targets (tau = 0: the noise-free field of krige / variance; a small
// tau > 0 is jitter for smooth kernels and close targets).  Its leading ns x ns block L_SS is the factor of
// C(S, S) + nugget I, and A_TS = L_TS L_SS'.  For k realisations from host standard normals Xi = [Xi_S; Xi_T] (N x k) and
// a drift F_s (ns x p), F_t (m x p), 0 <= p <= 32:
//   g = L_SS^-1 y,  G = L_SS^-1 F_s,  B = (G'G)^-1 G' (g 1' - Xi_S)   (p x k)
//   V = [g 1' - G B; Xi_T]   (N x k),   Z = F_t B + L(T, :) V   (m x k)
// This is "unconditional sample plus kriging of its residual" arranged so that a batch needs one triangular product and
// no triangular solve.  Xi = 0 gives the dual-form estimate (beta = (G'G)^-1 G'g, yhat = F_t beta + L_TS (g - G beta));
// Cov(Z) = L_TT L_TT' + (F_t - L_TS G)(G'G)^-1(F_t - L_TS G)', whose diagonal is the kriging variance + tau; p = 0 gives
// Z = L_TS g + L_TT Xi_T, independent of Xi_S; ns = 0 gives Z = L Xi.  The product Z = L(T, :) V is chol_trmm_kernel;
// g and G come from a forward sweep that stops after the source blocks, G'G and G' Xi_S from chol_gemm_kernel.
//
// Gaussian log-likelihood of the covariance parameters and its exact gradient (chol_loglik).  A = C(S, S) + nugget I is
// the square operator exactly as built, y the n observations, F the n x p drift (0 <= p <= 32), A = L L'.  With
// g = L^-1 y, G = L^-1 F, R'R = G'G (R upper triangular), beta = (G'G)^-1 G'g, e = g - G beta and q = ||e||^2:
//   ML (beta profiled by GLS):  l = -1/2 (n log 2 pi + log det A + q)
//   REML:                       l = -1/2 ((n - p) log 2 pi + log det A + 2 sum_k log R_kk + q)
// The REML form leaves out log det F'F, so its value depends on the scaling of F (its gradient and maximiser do not).
// With alpha = L^-T e (= A^-1 (y - F beta)) and H = L^-T G R^-1 (H H' = A^-1 F (F'A^-1 F)^-1 F'A^-1):
//   W = alpha alpha' - A^-1 (ML),  W = alpha alpha' - A^-1 + H H' (REML),  dl / dtheta = 1/2 sum_ij W_ij dA_ij / dtheta
// (for ML the envelope theorem makes this the gradient of the profile likelihood).  The parameters are, per structure s,
// sill_s then range_(s,a), a = 0 .. d - 1, then the nugget; dA / dnugget = I, the others as in kcov_grad_kernel.
// Device work: the factor (chol_factor); one forward sweep of [F | y] as a row-major np x 128 block, G'G and G'g on
// chol_gemm_kernel, R on chol_upper_kernel, beta and log det R, e (and G R^-1), q in fixed-order kernels; for the gradient
// one backward sweep of [G R^-1 | e] gives [H | alpha].  A^-1 is never held whole: for each chunk of <= 1024 columns from
// block column j0 the identity columns are swept forward from block j0 (the rows above are zero) and backward down to
// block j0, which gives rows >= j0 of A^-1(:, chunk) bit for bit as the full sweeps would (2 n^3 / 3 flops in all, as a
// triangular inverse plus L^-T L^-1, in one np x 1024 block).  The rank-(p + 1) term is applied to the chunk first as one
// chol_gemm_kernel update, Z = A^-1 - [H alpha][H alpha]' = -W on rows >= j0, with K = p + 1 rounded up to 32: on the
// tensor cores it costs about 2 n^2 K flops in all (1 ms at n = 20 000), where folding it into the contraction would add
// 2 (p + 1) loads and p + 1 FMAs per entry to an FP64-pipe-bound kernel.  kcov_grad_kernel then contracts each chunk.
//
// Cross-validation (chol_crossval; Dubrule 1983).  With P = A^-1 - A^-1 F (F'A^-1 F)^-1 F'A^-1 = L^-T (I - G^ G^') L^-1,
// G^ = G R^-1 (orthonormal columns), and alpha = P y = L^-T e, a held-out set B has err_B = P_BB^-1 alpha_B,
// var_B = diag(P_BB^-1) and log p(y_B | y_-B) = -1/2 (alpha_B' err_B + |B| log 2 pi - log det P_BB).  The groups are packed
// into chunks of <= 1024 columns; per chunk W = (I - G^ G^') L^-1 E_chunk (forward from the chunk's first block row, two
// chol_gemm_kernel launches for the projection) and Q = W'W on chol_gemm_kernel, so P_BB = Q_BB is a Gram;
// chol_cv_group_kernel factors each P_BB.
#include "common.cuh"
#include "algos.h"
#include "ptx.cuh"
#include <algorithm>
#include <cmath>

namespace gsi {

constexpr int CH_B = 128;              // block width of the factorisation and GEMM tile (rows and columns)
constexpr int CH_K = 32;               // k values per pipeline stage of chol_gemm_kernel
constexpr int CH_P = CH_B + 8;         // pitch of a [k][128] shared operand tile
constexpr int CH_THREADS = 512;
constexpr int CH_TILE = CH_K * CH_P;   // doubles of one operand tile
constexpr size_t CH_GEMM_SMEM = (size_t)2 * 2 * CH_TILE * sizeof(double);     // 2 stages x (A, B)
constexpr int CD_P = CH_B + 1;         // pitch of the diagonal block in shared memory
constexpr size_t CH_DIAG_SMEM = ((size_t)CH_B * CD_P + CH_B) * sizeof(double);
constexpr int CH_MAX_DRIFT = 32;       // drift columns of the universal-kriging variance
constexpr int CH_MAX_CHUNK = kMaxWideCols;

// C (+)= A B' on 128 x 128 tiles.  A(m, k) = A_KC ? A[m * lda + k] : A[k * lda + m];  B(n, k) likewise with B_KC;
// C(m, n) = C_ROW ? C[m * ldc + n] : C[n * ldc + m].  K is a multiple of CH_K.  lower: only the tiles (i, j), j <= i,
// of an mt x mt grid, blockIdx.x = i (i + 1) / 2 + j; otherwise blockIdx = (column tile, row tile).
struct ChGemm {
    const double* A; int64_t lda;
    const double* B; int64_t ldb;
    double* C; int64_t ldc;
    int64_t K;
    int sub;       // 1: C -= A B'   0: C = A B'
    int lower;
};

__device__ __forceinline__ void cp_async16(void* s, const void* g) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(smem_u32(s)), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" :: "n"(N) : "memory"); }

// one operand tile, 128 rows (m or n) x CH_K k values, into s[k * CH_P + row]
template <bool KC>
__device__ __forceinline__ void ch_load_tile(double* s, const double* g, int64_t ld, int64_t row0, int64_t k0, int tid) {
    if constexpr (!KC) {
        // (row, k) at g[k * ld + row]: 16-byte asynchronous copies along the rows
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int c = tid + q * CH_THREADS;
            const int k = c >> 6, r2 = (c & 63) * 2;
            cp_async16(s + k * CH_P + r2, g + (k0 + k) * ld + row0 + r2);
        }
    } else {
        // (row, k) at g[row * ld + k]: pairs along k through registers, transposed into shared memory (a lane per row:
        // conflict-free stores)
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int c = tid + q * CH_THREADS;
            const int r = c & (CH_B - 1), k2 = (c >> 7) * 2;
            const double2 v = __ldg(reinterpret_cast<const double2*>(g + (row0 + r) * ld + k0 + k2));
            s[k2 * CH_P + r] = v.x;
            s[(k2 + 1) * CH_P + r] = v.y;
        }
    }
}

template <bool A_KC, bool B_KC, bool C_ROW>
__global__ void __launch_bounds__(CH_THREADS, 1) chol_gemm_kernel(const ChGemm a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double* sm = reinterpret_cast<double*>(smem_raw);
    int64_t ti, tj;
    if (a.lower) {
        const int64_t t = blockIdx.x;
        int64_t i = (int64_t)((sqrt(8.0 * (double)t + 1.0) - 1.0) * 0.5);
        while ((i + 1) * (i + 2) / 2 <= t) ++i;
        while (i * (i + 1) / 2 > t) --i;
        ti = i;
        tj = t - i * (i + 1) / 2;
    } else {
        ti = blockIdx.y;
        tj = blockIdx.x;
    }
    const int64_t m0 = ti * CH_B, n0 = tj * CH_B;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const int wm = warp & 3, wn = warp >> 2;
    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }
    const int nk = (int)(a.K / CH_K);
    auto load = [&](int st, int kt) {
        double* sa = sm + (size_t)st * 2 * CH_TILE;
        ch_load_tile<A_KC>(sa, a.A, a.lda, m0, (int64_t)kt * CH_K, tid);
        ch_load_tile<B_KC>(sa + CH_TILE, a.B, a.ldb, n0, (int64_t)kt * CH_K, tid);
        cp_async_commit();
    };
    load(0, 0);
    for (int kt = 0; kt < nk; ++kt) {
        if (kt + 1 < nk) {
            load((kt + 1) & 1, kt + 1);
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
        const double* sa = sm + (size_t)(kt & 1) * 2 * CH_TILE;
        const double* sb = sa + CH_TILE;
#pragma unroll
        for (int ks = 0; ks < CH_K / 4; ++ks) {
            const double* ar = sa + (ks * 4 + t) * CH_P + wm * 32 + g;
            const double* br = sb + (ks * 4 + t) * CH_P + wn * 32 + g;
            double af[4], bf[4];
#pragma unroll
            for (int f = 0; f < 4; ++f) { af[f] = ar[f * 8]; bf[f] = br[f * 8]; }
#pragma unroll
            for (int fm = 0; fm < 4; ++fm)
#pragma unroll
                for (int fn = 0; fn < 4; ++fn) dmma884(acc[fm][fn][0], acc[fm][fn][1], af[fm], bf[fn]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int fm = 0; fm < 4; ++fm) {
        const int64_t m = m0 + wm * 32 + fm * 8 + g;
#pragma unroll
        for (int fn = 0; fn < 4; ++fn) {
            const int64_t n = n0 + wn * 32 + fn * 8 + 2 * t;
            if constexpr (C_ROW) {
                double2* c = reinterpret_cast<double2*>(a.C + m * a.ldc + n);
                double2 v = make_double2(acc[fm][fn][0], acc[fm][fn][1]);
                if (a.sub) { const double2 o = *c; v.x = o.x - v.x; v.y = o.y - v.y; }
                *c = v;
            } else {
                double* c0 = a.C + n * a.ldc + m;
                double* c1 = c0 + a.ldc;
                if (a.sub) { *c0 -= acc[fm][fn][0]; *c1 -= acc[fm][fn][1]; }
                else { *c0 = acc[fm][fn][0]; *c1 = acc[fm][fn][1]; }
            }
        }
    }
}

// Diagonal block (k0, k0) of the column-major A (pitch lda): L11 = chol(A11) into A's lower triangle, X11 = L11^-1 into
// inv (column-major 128 x 128, zero above the diagonal).  Shared S[r * CD_P + c]: the strict lower triangle holds L, the
// upper triangle X transposed (S[c][r] = X(r, c), r > c), dg the diagonal of L.  A pivot that is not positive (or NaN)
// records the 1-based global column in *info (the first failure wins; later launches return at once).
__global__ void __launch_bounds__(CH_THREADS, 1) chol_diag_kernel(double* __restrict__ A, int64_t lda, int64_t k0,
                                                                  double* __restrict__ inv, int* __restrict__ info) {
    extern __shared__ __align__(16) double S[];
    double* dg = S + CH_B * CD_P;
    if (*info != 0) return;
    const int tid = threadIdx.x;
    for (int e = tid; e < CH_B * CH_B; e += CH_THREADS) {
        const int r = e & (CH_B - 1), c = e >> 7;
        if (r >= c) S[r * CD_P + c] = A[(k0 + c) * lda + k0 + r];
    }
    __syncthreads();
    // right-looking, column by column: thread (r = tid & 127, phase tid >> 7) updates row r, columns phase, phase + 4, ..
    const int r = tid & (CH_B - 1), ph = tid >> 7;
    for (int j = 0; j < CH_B; ++j) {
        const double d = S[j * CD_P + j];
        __syncthreads();                                        // every thread has read the pivot
        if (!(d > 0.0)) {
            if (tid == 0) atomicCAS(info, 0, (int)(k0 + j + 1));
            return;                                             // uniform: all threads saw the same d
        }
        const double s = sqrt(d);
        if (tid == 0) dg[j] = s;
        if (ph == 0 && r > j) S[r * CD_P + j] /= s;
        __syncthreads();
        if (r > j) {
            const double lr = S[r * CD_P + j];
            for (int c = j + 1 + ph; c <= r; c += 4) S[r * CD_P + c] -= lr * S[c * CD_P + j];
        }
        __syncthreads();
    }
    // X = L^-1 row by row: X(i, i) = 1 / L(i, i), X(i, c) = -(sum_{c <= k < i} L(i, k) X(k, c)) / L(i, i); thread
    // (c = tid >> 2, q = tid & 3) adds k = c + q, c + q + 4, .. and the four quarters meet by shuffles (fixed order)
    const int c = tid >> 2, q = tid & 3;
    for (int i = 1; i < CH_B; ++i) {
        double sum = 0.0;
        if (c < i)
            for (int k = c + q; k < i; k += 4) sum += S[i * CD_P + k] * (k == c ? 1.0 / dg[c] : S[c * CD_P + k]);
        sum += __shfl_xor_sync(0xffffffffu, sum, 1);
        sum += __shfl_xor_sync(0xffffffffu, sum, 2);
        if (q == 0 && c < i) S[c * CD_P + i] = -sum / dg[i];
        __syncthreads();
    }
    for (int e = tid; e < CH_B * CH_B; e += CH_THREADS) {
        const int rr = e & (CH_B - 1), cc = e >> 7;
        if (rr > cc) A[(k0 + cc) * lda + k0 + rr] = S[rr * CD_P + cc];
        else if (rr == cc) A[(k0 + cc) * lda + k0 + rr] = dg[rr];
        inv[cc * CH_B + rr] = rr > cc ? S[cc * CD_P + rr] : (rr == cc ? 1.0 / dg[rr] : 0.0);
    }
}

// log det = 2 sum_i log L(i, i) over the n true rows: one CTA, thread t adds i = t, t + 1024, .. in order, then a fixed
// tree
__global__ void chol_logdet_kernel(const double* __restrict__ L, int64_t ld, int64_t n, double* __restrict__ out) {
    __shared__ double red[1024];
    double s = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += 1024) s += log(L[i * ld + i]);
    red[threadIdx.x] = s;
    __syncthreads();
    for (int w = 512; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[0] = 2.0 * red[0];
}

// *flag = 1 when an entry of the rows x cols TALL block (pitch ld) is not finite
__global__ void chol_nonfinite_kernel(const double* __restrict__ X, int64_t ld, int64_t rows, int64_t cols, int* flag) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows * cols) return;
    const int64_t i = idx / cols, c = idx - i * cols;
    if (!isfinite(X[i * ld + c])) *flag = 1;
}

// var[c] = c(t, t) - ||L^-1 c_t||^2 (+ r' (G'G)^-1 r, r = f_t - G' L^-1 c_t, with R'R = G'G: r' (G'G)^-1 r = ||R^-T r||^2)
// H: G' W (row-major, pitch ldh), Ft: the chunk's drift rows (column-major, pitch ldf), R: upper p x p (pitch p)
__global__ void chol_variance_kernel(const double* __restrict__ colsq, const double* __restrict__ ctt, int64_t mc, int p,
                                     const double* __restrict__ H, int64_t ldh, const double* __restrict__ Ft, int64_t ldf,
                                     const double* __restrict__ R, double* __restrict__ var) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= mc) return;
    double v = ctt[0] - colsq[c];
    if (p > 0) {
        double z[CH_MAX_DRIFT];
        double acc = 0.0;
#pragma unroll
        for (int i = 0; i < CH_MAX_DRIFT; ++i) {
            z[i] = 0.0;
            if (i < p) {
                double s = Ft[c + i * ldf] - H[i * ldh + c];
#pragma unroll
                for (int k = 0; k < i; ++k) s -= R[k + i * p] * z[k];
                z[i] = s / R[i + i * p];
                acc += z[i] * z[i];
            }
        }
        v += acc;
    }
    var[c] = v;
}

// A(i, i) += d[i] after the fill, rounded once as the fill adds the nugget (a constant d on an operator without nugget
// gives the bits of that nugget inside the operator)
__global__ void chol_add_diag_kernel(double* __restrict__ A, int64_t lda, const double* __restrict__ d, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) A[i * lda + i] = __dadd_rn(A[i * lda + i], d[i]);
}

// Z = L(rows, :) V for the lower-triangular factor: L column-major (pitch np), V row-major np x kp (pitch kp), Z row-major
// (pitch kp) holding rows r0 .. np.  One CTA per 128 x 128 tile (row tile i >= r0 / 128, column tile c) reduces over the
// k-blocks j = 0 .. i in order; tiles are issued heaviest first (i descending), so the ragged K leaves no long tail.  The
// strict upper triangle of L's storage is not zero (the fill skips whole tiles only, the diagonal blocks are written on
// and below the diagonal), so the diagonal block j = i is masked to its lower triangle in shared memory.
struct ChTrmm {
    const double* L; int64_t np;
    const double* V; int64_t kp;
    double* Z; int64_t r0;
    int64_t nct;   // column tiles: kp / 128
};

__global__ void __launch_bounds__(CH_THREADS, 1) chol_trmm_kernel(const ChTrmm a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double* sm = reinterpret_cast<double*>(smem_raw);
    const int64_t t0 = blockIdx.x / a.nct;
    const int64_t ti = a.np / CH_B - 1 - t0, tj = blockIdx.x - t0 * a.nct;
    const int64_t m0 = ti * CH_B, n0 = tj * CH_B;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const int wm = warp & 3, wn = warp >> 2;
    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }
    const int kdiag = (int)(ti * (CH_B / CH_K));                 // first k-tile of the diagonal block
    const int nk = kdiag + CH_B / CH_K;
    auto load = [&](int st, int kt) {
        double* sa = sm + (size_t)st * 2 * CH_TILE;
        ch_load_tile<false>(sa, a.L, a.np, m0, (int64_t)kt * CH_K, tid);
        ch_load_tile<false>(sa + CH_TILE, a.V, a.kp, n0, (int64_t)kt * CH_K, tid);
        cp_async_commit();
    };
    load(0, 0);
    for (int kt = 0; kt < nk; ++kt) {
        if (kt + 1 < nk) {
            load((kt + 1) & 1, kt + 1);
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
        double* sa = sm + (size_t)(kt & 1) * 2 * CH_TILE;
        if (kt >= kdiag) {                                        // L(m0 + r, m0 + kb + k) = 0 where kb + k > r
            const int kb = (kt - kdiag) * CH_K;
            for (int e = tid; e < CH_K * CH_B; e += CH_THREADS) {
                const int k = e >> 7, r = e & (CH_B - 1);
                if (kb + k > r) sa[k * CH_P + r] = 0.0;
            }
            __syncthreads();
        }
        const double* sb = sa + CH_TILE;                           // chol_gemm_kernel's k-tile step
#pragma unroll
        for (int ks = 0; ks < CH_K / 4; ++ks) {
            const double* ar = sa + (ks * 4 + t) * CH_P + wm * 32 + g;
            const double* br = sb + (ks * 4 + t) * CH_P + wn * 32 + g;
            double af[4], bf[4];
#pragma unroll
            for (int f = 0; f < 4; ++f) { af[f] = ar[f * 8]; bf[f] = br[f * 8]; }
#pragma unroll
            for (int fm = 0; fm < 4; ++fm)
#pragma unroll
                for (int fn = 0; fn < 4; ++fn) dmma884(acc[fm][fn][0], acc[fm][fn][1], af[fm], bf[fn]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int fm = 0; fm < 4; ++fm) {
        const int64_t m = m0 + wm * 32 + fm * 8 + g - a.r0;
#pragma unroll
        for (int fn = 0; fn < 4; ++fn) {
            const int64_t n = n0 + wn * 32 + fn * 8 + 2 * t;
            *reinterpret_cast<double2*>(a.Z + m * a.kp + n) = make_double2(acc[fm][fn][0], acc[fm][fn][1]);
        }
    }
}

// The drift terms of conditional simulation for a 32-column strip of the k realisations.  W: row-major (pitch 128) with
// G = L_SS^-1 F_s in columns 0 .. p - 1 and g = L_SS^-1 y in column p; GtG = W'W (row-major, pitch 128; G'g in its
// column p); H: G' Xi_S (row-major p x kp); R: upper p x p with R'R = G'G (column-major, pitch p).
//   B(:, c) = R^-1 R^-T (G'g - H(:, c))   (p x kp row-major in Bm, written by the CTAs of the first row strip)
//   V(i, c) = g_i - sum_q G(i, q) B(q, c) for the source rows i < ns  (p = 0: V(i, c) = g_i)
constexpr int SIM_ROWS = 64;   // source rows per CTA
__global__ void __launch_bounds__(256) chol_sim_drift_kernel(const double* __restrict__ W, const double* __restrict__ GtG,
                                                             const double* __restrict__ H, const double* __restrict__ R,
                                                             int p, int64_t ns, double* __restrict__ Bm,
                                                             double* __restrict__ V, int64_t kp) {
    __shared__ double sB[CH_MAX_DRIFT][32];
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int64_t c = (int64_t)blockIdx.x * 32 + tx;
    if (p > 0 && ty == 0) {
        for (int i = 0; i < p; ++i) {                             // R' z = G'g - G' xi_c
            double s = GtG[i * CH_B + p] - H[i * kp + c];
            for (int k = 0; k < i; ++k) s -= R[k + i * p] * sB[k][tx];
            sB[i][tx] = s / R[i + i * p];
        }
        for (int i = p - 1; i >= 0; --i) {                        // R b = z
            double s = sB[i][tx];
            for (int k = i + 1; k < p; ++k) s -= R[i + k * p] * sB[k][tx];
            sB[i][tx] = s / R[i + i * p];
        }
        if (blockIdx.y == 0)
            for (int i = 0; i < p; ++i) Bm[i * kp + c] = sB[i][tx];
    }
    __syncthreads();
    const int64_t r1 = min(ns, (int64_t)(blockIdx.y + 1) * SIM_ROWS);
    for (int64_t i = (int64_t)blockIdx.y * SIM_ROWS + ty; i < r1; i += 8) {
        const double* wi = W + i * CH_B;
        double v = wi[p];
        for (int q = 0; q < p; ++q) v -= wi[q] * sB[q][tx];
        V[i * kp + c] = v;
    }
}

// Z (TALL m x k, pitch ldz) = the TRMM rows off .. off + m of Zw (pitch kp) + F_t B (F_t column-major m x p; B row-major
// p x kp); p = 0 copies
__global__ void chol_sim_out_kernel(const double* __restrict__ Zw, int64_t kp, int64_t off, const double* __restrict__ Ft,
                                    int64_t m, int p, const double* __restrict__ Bm, double* __restrict__ Z, int64_t ldz,
                                    int64_t k) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= m * k) return;
    const int64_t r = idx / k, c = idx - r * k;
    double fb = 0.0;
    for (int q = 0; q < p; ++q) fb += Ft[r + q * m] * Bm[q * kp + c];
    const double z = Zw[(off + r) * kp + c];
    Z[r * ldz + c] = p > 0 ? fb + z : z;
}

// Likelihood value, drift part.  GtG: [G | g]'[G | g] (row-major, pitch 128), R: upper p x p with R'R = G'G (column-major,
// pitch p).  out[0 .. p - 1] = beta = R^-1 R^-T G'g, out[CH_MAX_DRIFT] = sum_k log R_kk, in order (one thread)
__global__ void chol_lik_beta_kernel(const double* __restrict__ GtG, const double* __restrict__ R, int p,
                                     double* __restrict__ out) {
    double z[CH_MAX_DRIFT];
    double ld = 0.0;
    for (int i = 0; i < p; ++i) {                                 // R' z = G'g
        double s = GtG[i * CH_B + p];
        for (int k = 0; k < i; ++k) s -= R[k + i * p] * z[k];
        z[i] = s / R[i + i * p];
        ld += log(R[i + i * p]);
    }
    for (int i = p - 1; i >= 0; --i) {                            // R beta = z
        double s = z[i];
        for (int k = i + 1; k < p; ++k) s -= R[i + k * p] * z[k];
        z[i] = s / R[i + i * p];
    }
    for (int i = 0; i < p; ++i) out[i] = z[i];
    out[CH_MAX_DRIFT] = ld;
}

// Row i of W = [G | g] (row-major np x 128): g_i <- e_i = g_i - G_i beta.  mode 1 (ML gradient): G_i <- 0; mode 2 (REML
// gradient): G_i <- G_i R^-1 (the row solve h R = G_i); mode 0 leaves G
__global__ void chol_lik_resid_kernel(double* __restrict__ W, int64_t np, int p, const double* __restrict__ beta,
                                      const double* __restrict__ R, int mode) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= np) return;
    double* w = W + i * CH_B;
    double e = w[p];
    for (int q = 0; q < p; ++q) e -= w[q] * beta[q];
    w[p] = e;
    if (mode == 1) {
        for (int q = 0; q < p; ++q) w[q] = 0.0;
    } else if (mode == 2) {
        double h[CH_MAX_DRIFT];
        for (int k = 0; k < p; ++k) {
            double s = w[k];
            for (int q = 0; q < k; ++q) s -= h[q] * R[q + k * p];
            h[k] = s / R[k + k * p];
        }
        for (int k = 0; k < p; ++k) w[k] = h[k];
    }
}

// *out = sum_i W[i * 128 + col]^2 over the n true rows: one CTA, the order of chol_logdet_kernel
__global__ void chol_lik_sumsq_kernel(const double* __restrict__ W, int64_t n, int col, double* __restrict__ out) {
    __shared__ double red[1024];
    double s = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += 1024) {
        const double v = W[i * CH_B + col];
        s = fma(v, v, s);
    }
    red[threadIdx.x] = s;
    __syncthreads();
    for (int w = 512; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[0] = red[0];
}

// Z(j0 + c, c) = 1, c < w: the identity columns of a chunk (row-major, pitch ldz; the rest was zeroed)
__global__ void chol_eye_kernel(double* __restrict__ Z, int64_t ldz, int64_t j0, int64_t w) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c < w) Z[(j0 + c) * ldz + c] = 1.0;
}

// Z(cidx[c], c) = 1, c < w: the held-out points of a cross-validation chunk (row-major, pitch ldz; the rest was zeroed)
__global__ void chol_cv_scatter_kernel(double* __restrict__ Z, int64_t ldz, const int64_t* __restrict__ cidx, int64_t w) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c < w) Z[cidx[c] * ldz + c] = 1.0;
}

// One held-out group of a cross-validation chunk: its points are the chunk columns col .. col + size - 1, in the caller's
// order, and its results go to entries pos .. pos + size - 1 of the outputs and to entry g of the log-densities
struct CvGroup {
    int64_t pos;
    int32_t size, col, g, pad;
};
constexpr int CV_THREADS = 128;
// A pivot of P_BB at or below CV_PIVOT_TOL (A^-1)_jj counts as zero: the projection and the Gram leave an error of a few
// units of roundoff times (A^-1)_jj on a pivot that is zero in exact arithmetic, and a group whose drift the remaining
// points cannot identify has such a pivot
constexpr double CV_PIVOT_TOL = 0x1p-36;

// The groups of a chunk, SMAX = 32 (a warp per group of <= 32 points, four per CTA) or 128 (a CTA per group).  From the
// chunk Gram Q = P(chunk, chunk) (lower triangle, row-major, pitch ldq), ref (the unprojected (A^-1)_jj of the chunk's
// columns) and alpha (alpha_i at alpha[i * CH_B]): P_BB = L_B L_B' and X = L_B^-1 in shared memory (S[r * SP + c]: L
// strictly below the diagonal, X transposed above it, dg the diagonal of L, rf its reciprocals), then with z = X alpha_B
//   err = X' z = P_BB^-1 alpha_B,  var = the squared column norms of X = diag(P_BB^-1),
//   logpdf = -1/2 (||z||^2 + size log 2 pi - 2 sum log dg)
// Thread t of a team owns row t in the factorisation and column t of X; every sum runs in a fixed order, so a group's
// results depend only on its own P_BB, alpha_B and ref.  A pivot at or below the tolerance records the 1-based group in
// *failed (atomicMin: the lowest failing group wins whatever the launch order).
template <int SMAX>
__global__ void __launch_bounds__(CV_THREADS) chol_cv_group_kernel(const CvGroup* __restrict__ grp, int ng,
                                                                   const double* __restrict__ Q, int64_t ldq,
                                                                   const double* __restrict__ ref,
                                                                   const int64_t* __restrict__ cidx,
                                                                   const double* __restrict__ alpha,
                                                                   double* __restrict__ err, double* __restrict__ var,
                                                                   double* __restrict__ logpdf, int* __restrict__ failed) {
    constexpr int TEAMS = CV_THREADS / SMAX, SP = SMAX + 1;
    extern __shared__ __align__(16) double cv_smem[];
    const int team = threadIdx.x / SMAX, t = threadIdx.x % SMAX;
    const int gi = blockIdx.x * TEAMS + team;
    if (gi >= ng) return;                                        // uniform over the team
    auto bar = [] { if constexpr (SMAX == CV_THREADS) __syncthreads(); else __syncwarp(); };
    double* S = cv_smem + (size_t)team * (SMAX * SP + 4 * SMAX);
    double* dg = S + SMAX * SP;
    double* a = dg + SMAX;
    double* z = a + SMAX;
    double* rf = z + SMAX;
    const CvGroup G = grp[gi];
    const int s = G.size;
    for (int e = t; e < s * s; e += SMAX) {
        const int r = e / s, c = e - r * s;
        if (r >= c) S[r * SP + c] = Q[(int64_t)(G.col + r) * ldq + G.col + c];
    }
    if (t < s) {
        a[t] = alpha[cidx[G.col + t] * CH_B];
        rf[t] = ref[G.col + t];
    }
    bar();
    for (int j = 0; j < s; ++j) {
        const double d = S[j * SP + j];
        if (!(d > CV_PIVOT_TOL * rf[j])) {                       // uniform: the team saw the same d and rf[j]
            if (t == 0) atomicMin(failed, G.g + 1);
            return;
        }
        const double sq = sqrt(d), rq = 1.0 / sq;
        if (t > j && t < s) S[t * SP + j] *= rq;
        bar();                                                   // every thread has also read rf[j]
        if (t == j) {
            dg[j] = sq;
            rf[j] = rq;                                          // 1 / L(j, j) from here on
        }
        if (t > j && t < s) {
            const double l = S[t * SP + j];
            for (int c = j + 1; c <= t; ++c) S[t * SP + c] -= l * S[c * SP + j];
        }
        bar();
    }
    // column t of X: X(t, t) = 1 / L(t, t), X(i, t) = -(sum_{t <= k < i} L(i, k) X(k, t)) / L(i, i)
    if (t < s) {
        const double xt = rf[t];
        double v = xt * xt;
        for (int i = t + 1; i < s; ++i) {
            double sum = S[i * SP + t] * xt;
            for (int k = t + 1; k < i; ++k) sum = fma(S[i * SP + k], S[t * SP + k], sum);
            const double x = -sum * rf[i];
            S[t * SP + i] = x;
            v = fma(x, x, v);
        }
        var[G.pos + t] = v;
    }
    bar();
    if (t < s) {                                                  // z_t = sum_{j <= t} X(t, j) alpha_j
        double zt = 0.0;
        for (int j = 0; j < t; ++j) zt = fma(S[j * SP + t], a[j], zt);
        z[t] = fma(a[t], rf[t], zt);
    }
    bar();
    if (t < s) {                                                  // err_t = sum_{i >= t} X(i, t) z_i
        double et = z[t] * rf[t];
        for (int i = t + 1; i < s; ++i) et = fma(S[t * SP + i], z[i], et);
        err[G.pos + t] = et;
    }
    if (logpdf && t == 0) {
        double q = 0.0, ld = 0.0;
        for (int i = 0; i < s; ++i) {
            q = fma(z[i], z[i], q);
            ld += log(dg[i]);
        }
        logpdf[G.g] = -0.5 * (q + s * 1.83787706640934548356 - 2.0 * ld);
    }
}

template <int SMAX>
constexpr size_t cv_group_smem() { return (size_t)(CV_THREADS / SMAX) * (SMAX * (SMAX + 1) + 4 * SMAX) * sizeof(double); }

namespace {

template <bool AK, bool BK, bool CR>
void gemm(gsi_ctx* ctx, const ChGemm& a, int64_t mt, int64_t nt) {
    if (mt <= 0 || nt <= 0) return;
    auto kfn = chol_gemm_kernel<AK, BK, CR>;
    GSI_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CH_GEMM_SMEM));
    const dim3 grid = a.lower ? dim3((unsigned)(mt * (mt + 1) / 2)) : dim3((unsigned)nt, (unsigned)mt);
    kfn<<<grid, CH_THREADS, CH_GEMM_SMEM, ctx->stream>>>(a);
    GSI_CUDA(cudaGetLastError());
    count_launch(ctx);
}

ChGemm gm(const double* A, int64_t lda, const double* B, int64_t ldb, double* C, int64_t ldc, int64_t K, int sub, int lower) {
    ChGemm a;
    a.A = A; a.lda = lda; a.B = B; a.ldb = ldb; a.C = C; a.ldc = ldc; a.K = K; a.sub = sub; a.lower = lower;
    return a;
}

// W (row-major np x kp, pitch ldw; kp a multiple of 128) <- L^-1 W on the leading nb block rows (nb = np / 128: all of
// W; a smaller nb leaves the rows from nb * 128 on unchanged, and the rows above are those of the full solve).  kb0 > 0
// starts at block row kb0 for a W whose rows above kb0 * 128 are zero: those rows are neither read nor written, and the
// rows below are bit for bit those of the full sweep (which would only subtract exact zeros from them)
void forward(const gsi_chol* f, double* W, int64_t ldw, int64_t kp, int64_t nb, int64_t kb0 = 0) {
    gsi_ctx* ctx = f->ctx;
    const int64_t nt = kp / CH_B;
    for (int64_t kb = kb0; kb < nb; ++kb) {
        const int64_t j0 = kb * CH_B;
        double* Wj = W + j0 * ldw;
        gemm<false, false, true>(ctx, gm(f->inv + kb * CH_B * CH_B, CH_B, Wj, ldw, Wj, ldw, CH_B, 0, 0), 1, nt);
        gemm<false, false, true>(ctx, gm(f->L + j0 * f->np + j0 + CH_B, f->np, Wj, ldw, Wj + CH_B * ldw, ldw, CH_B, 1, 0),
                                 nb - kb - 1, nt);
    }
}

// W <- L^-T W.  kb1 > 0 stops after block row kb1: the rows from kb1 * 128 on are those of the full sweep (they do not
// depend on the rows above), the rows above are neither read nor written
void backward(const gsi_chol* f, double* W, int64_t ldw, int64_t kp, int64_t kb1 = 0) {
    gsi_ctx* ctx = f->ctx;
    const int64_t nb = f->np / CH_B, nt = kp / CH_B;
    for (int64_t kb = nb - 1; kb >= kb1; --kb) {
        const int64_t j0 = kb * CH_B;
        double* Wj = W + j0 * ldw;
        gemm<true, false, true>(ctx, gm(f->inv + kb * CH_B * CH_B, CH_B, Wj, ldw, Wj, ldw, CH_B, 0, 0), 1, nt);
        gemm<true, false, true>(ctx, gm(f->L + j0 + kb1 * CH_B * f->np, f->np, Wj, ldw, W + kb1 * CH_B * ldw, ldw, CH_B, 1, 0),
                                kb - kb1, nt);
    }
}

struct DevMem {
    void* p = nullptr;
    explicit DevMem(size_t bytes) { GSI_CUDA(cudaMalloc(&p, bytes)); }
    ~DevMem() { if (p) cudaFree(p); }
    double* d() const { return static_cast<double*>(p); }
};

// The drift part of the likelihood and of cross-validation, enqueued without a synchronisation: [G | g] = L^-1 [F | y]
// into W (row-major np x 128, zero padded; Wh is its host staging block and must live until the stream has passed the
// copy), then with p > 0 GtG = [G | g]'[G | g], R'R = G'G (a failed factor sets flag[1]), beta and sum log R_kk into res
// and chol_lik_resid_kernel in `mode`.  res must be zeroed by the caller
void drift_residual(const gsi_chol* f, const double* y, const double* F, int64_t p, int mode, double* W, double* GtG,
                    double* R, double* res, int* flag, std::vector<double>& Wh) {
    gsi_ctx* ctx = f->ctx;
    cudaStream_t st = ctx->stream;
    const int64_t n = f->n, np = f->np;
    Wh.assign((size_t)np * CH_B, 0.0);
    for (int64_t i = 0; i < n; ++i) {
        for (int64_t q = 0; q < p; ++q) Wh[(size_t)i * CH_B + q] = F[q * n + i];
        Wh[(size_t)i * CH_B + p] = y[i];
    }
    GSI_CUDA(cudaMemcpyAsync(W, Wh.data(), Wh.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    forward(f, W, CH_B, CH_B, np / CH_B);
    GSI_CUDA(cudaMemsetAsync(flag, 0, 2 * sizeof(int), st));
    if (p > 0) {
        gemm<false, false, true>(ctx, gm(W, CH_B, W, CH_B, GtG, CH_B, np, 0, 0), 1, 1);
        tall_head_to_cm_kernel<<<(unsigned)((p * p + 255) / 256), 256, 0, st>>>(GtG, CH_B, (int)p, R);
        chol_upper_kernel<<<1, 1024, 0, st>>>(R, (int)p, flag + 1);
        chol_lik_beta_kernel<<<1, 1, 0, st>>>(GtG, R, (int)p, res);
        chol_lik_resid_kernel<<<(unsigned)((np + 255) / 256), 256, 0, st>>>(W, np, (int)p, res, R, mode);
        GSI_CUDA(cudaGetLastError());
        count_launch(ctx, 4);
    }
}

// device memory of a call that needs `need` bytes besides what it holds, checked before any allocation
void require_free(gsi_ctx* ctx, double need, const char* what, int64_t n) {
    size_t fr = 0, tot = 0;
    GSI_CUDA(cudaMemGetInfo(&fr, &tot));
    if (need > (double)fr) {
        pool_release(ctx);
        GSI_CUDA(cudaMemGetInfo(&fr, &tot));
    }
    if (need > (double)fr) {
        char msg[256];
        snprintf(msg, sizeof(msg), "%s: n = %lld needs %.0f bytes of device memory, %zu are free", what, (long long)n,
                 need, fr);
        throw Error(GSI_ERR_UNSUPPORTED, msg);
    }
}

}  // namespace

void chol_destroy(gsi_chol* f) {
    if (!f) return;
    cudaSetDevice(f->ctx->device);
    if (f->L) cudaFree(f->L);
    if (f->inv) cudaFree(f->inv);
    if (f->info) cudaFree(f->info);
    delete f;
}

gsi_chol* chol_factor(gsi_op* op, const double* diag, int64_t* failed_column) {
    gsi_ctx* ctx = op->ctx;
    cudaStream_t st = ctx->stream;
    if (failed_column) *failed_column = 0;
    GSI_REQUIRE(op->type == OP_KERNELCOV, GSI_ERR_UNSUPPORTED,
                "kernelcov_chol needs a square kernel-covariance operator (gsi_op_kernelcov, _grid, _model or _model_grid)");
    GSI_REQUIRE(ctx->world == 1, GSI_ERR_UNSUPPORTED, "kernelcov_chol is single-GPU: the dense factor is not distributed");
    const int64_t n = op->n, np = round_up(n, CH_B);
    if (diag)
        for (int64_t i = 0; i < n; ++i)
            GSI_REQUIRE(std::isfinite(diag[i]), GSI_ERR_INVALID_ARGUMENT, "kernelcov_chol_diag: diag has a non-finite entry");
    const double need = (double)np * (double)np * 8.0 + (double)np * CH_B * 8.0 + 4096.0 + (diag ? (double)n * 8.0 : 0.0);
    size_t fr = 0, tot = 0;
    GSI_CUDA(cudaMemGetInfo(&fr, &tot));
    if (need > (double)fr) {
        pool_release(ctx);                                        // cached iterate blocks count as free
        GSI_CUDA(cudaMemGetInfo(&fr, &tot));
    }
    if (need > (double)fr) {
        char msg[256];
        snprintf(msg, sizeof(msg), "kernelcov_chol: the dense factor of n = %lld needs %.0f bytes of device memory, %zu are "
                 "free (use gsi_kernelcov_solve)", (long long)n, need, fr);
        throw Error(GSI_ERR_UNSUPPORTED, msg);
    }
    std::unique_ptr<gsi_chol, void (*)(gsi_chol*)> f(new gsi_chol(), chol_destroy);
    f->ctx = ctx; f->n = n; f->np = np;
    GSI_CUDA(cudaMalloc(&f->L, (size_t)np * np * sizeof(double)));
    GSI_CUDA(cudaMalloc(&f->inv, (size_t)np * CH_B * sizeof(double)));
    GSI_CUDA(cudaMalloc(&f->info, 4 * sizeof(double)));
    GSI_CUDA(cudaMemsetAsync(f->info, 0, 4 * sizeof(double), st));
    int* info = reinterpret_cast<int*>(f->info);
    f->flags = reinterpret_cast<int*>(f->info + 2);
    double* ld_out = f->info + 1;
    // 1. the lower triangle of A, padding included
    phase_begin(ctx);
    KcovBlock b;
    b.r0 = 0; b.rows = np; b.c0 = 0; b.cols = np; b.nr_valid = n; b.nc_valid = n; b.nugget_diag = 1; b.lower = 1;
    b.out = f->L; b.rs = 1; b.cs = np;
    kcov_block(op, KB_SQUARE, b);
    if (diag) {                                                   // + diag(d), one rounding per entry as the nugget's
        DevMem dd((size_t)n * sizeof(double));
        GSI_CUDA(cudaMemcpyAsync(dd.d(), diag, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, st));
        chol_add_diag_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(f->L, np, dd.d(), n);
        GSI_CUDA(cudaGetLastError());
        count_launch(ctx);
        GSI_CUDA(cudaStreamSynchronize(st));                      // dd is freed on return
    }
    phase_end(ctx, PH_CHOL_FILL);
    // 2. blocked right-looking factorisation
    GSI_CUDA(cudaFuncSetAttribute(chol_diag_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CH_DIAG_SMEM));
    const int64_t nb = np / CH_B;
    for (int64_t kb = 0; kb < nb; ++kb) {
        const int64_t k0 = kb * CH_B, mt = nb - kb - 1;
        double* invk = f->inv + kb * CH_B * CH_B;
        phase_begin(ctx);
        chol_diag_kernel<<<1, CH_THREADS, CH_DIAG_SMEM, st>>>(f->L, np, k0, invk, info);
        GSI_CUDA(cudaGetLastError());
        count_launch(ctx);
        phase_end(ctx, PH_CHOL_DIAG);
        if (mt == 0) break;
        double* A21 = f->L + k0 * np + k0 + CH_B;
        phase_begin(ctx);
        gemm<false, false, false>(ctx, gm(A21, np, invk, CH_B, A21, np, CH_B, 0, 0), mt, 1);
        phase_end(ctx, PH_CHOL_PANEL);
        phase_begin(ctx);
        gemm<false, false, false>(ctx, gm(A21, np, A21, np, f->L + (k0 + CH_B) * np + k0 + CH_B, np, CH_B, 1, 1), mt, mt);
        phase_end(ctx, PH_GEMM);
        if (ctx->time_gemm) {
            ctx->gemm_launches += 1;
            ctx->gemm_flops_accum += 2.0 * CH_B * CH_B * CH_B * (double)(mt * (mt + 1) / 2);
        }
    }
    int h = 0;
    GSI_CUDA(cudaMemcpyAsync(&h, info, sizeof(int), cudaMemcpyDeviceToHost, st));
    GSI_CUDA(cudaStreamSynchronize(st));
    if (h != 0) {
        if (failed_column) *failed_column = h;
        throw Error(GSI_ERR_NOT_POSDEF, "PosDefException(" + std::to_string(h) + "): the covariance matrix is not numerically "
                                        "positive definite at column " + std::to_string(h) + " (add a nugget)");
    }
    chol_logdet_kernel<<<1, 1024, 0, st>>>(f->L, np, n, ld_out);
    GSI_CUDA(cudaGetLastError());
    count_launch(ctx);
    GSI_CUDA(cudaMemcpyAsync(&f->logdet, ld_out, sizeof(double), cudaMemcpyDeviceToHost, st));
    GSI_CUDA(cudaStreamSynchronize(st));
    return f.release();
}

void chol_download(const gsi_chol* f, double* host, int64_t ldh) {
    const int64_t n = f->n;
    GSI_REQUIRE(host != nullptr && ldh >= n, GSI_ERR_INVALID_ARGUMENT, "chol_download: null host array or ldh < n");
    GSI_CUDA(cudaMemcpy2DAsync(host, (size_t)ldh * 8, f->L, (size_t)f->np * 8, (size_t)n * 8, (size_t)n,
                               cudaMemcpyDeviceToHost, f->ctx->stream));
    GSI_CUDA(cudaStreamSynchronize(f->ctx->stream));
    for (int64_t c = 1; c < n; ++c) std::memset(host + c * ldh, 0, (size_t)c * sizeof(double));   // strict upper triangle
}

void chol_solve(const gsi_chol* f, int half, const gsi_buf* B, gsi_buf* X) {
    gsi_ctx* ctx = f->ctx;
    cudaStream_t st = ctx->stream;
    const int64_t n = f->n;
    GSI_REQUIRE(half == 0 || half == 1, GSI_ERR_INVALID_ARGUMENT, "chol_solve: half must be 0 (A^-1 B) or 1 (L^-1 B)");
    GSI_REQUIRE(B->layout == GSI_LAYOUT_TALL && B->rows == n, GSI_ERR_DIMENSION_MISMATCH, "chol_solve: B must be TALL n x k");
    GSI_REQUIRE(X->layout == GSI_LAYOUT_TALL && X->rows == n && X->cols == B->cols, GSI_ERR_DIMENSION_MISMATCH,
                "chol_solve: X must be TALL with B's shape");
    GSI_REQUIRE(B->ctx == ctx && X->ctx == ctx, GSI_ERR_INVALID_ARGUMENT, "chol_solve: buffers of another context");
    const int64_t k = B->cols;
    int* flag = f->flags;
    GSI_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), st));
    chol_nonfinite_kernel<<<(unsigned)((n * k + 255) / 256), 256, 0, st>>>(B->d, B->ld, n, k, flag);
    GSI_CUDA(cudaGetLastError());
    count_launch(ctx);
    int h = 0;
    GSI_CUDA(cudaMemcpyAsync(&h, flag, sizeof(int), cudaMemcpyDeviceToHost, st));
    GSI_CUDA(cudaStreamSynchronize(st));
    GSI_REQUIRE(h == 0, GSI_ERR_INVALID_ARGUMENT, "chol_solve: B has a non-finite entry");
    const int64_t kw = k < CH_MAX_CHUNK ? k : CH_MAX_CHUNK;
    const int64_t kp = round_up(kw, CH_B);
    DevMem W((size_t)f->np * kp * sizeof(double));
    for (int64_t c0 = 0; c0 < k; c0 += CH_MAX_CHUNK) {
        const int64_t w = k - c0 < CH_MAX_CHUNK ? k - c0 : CH_MAX_CHUNK;
        const int64_t wp = round_up(w, CH_B);
        GSI_CUDA(cudaMemsetAsync(W.d(), 0, (size_t)f->np * kp * sizeof(double), st));
        tall_cols_copy(ctx, B->d + c0, B->ld, W.d(), kp, n, w);
        forward(f, W.d(), kp, wp, f->np / CH_B);
        if (half == 0) backward(f, W.d(), kp, wp);
        tall_cols_copy(ctx, W.d(), kp, X->d + c0, X->ld, n, w);
    }
    GSI_CUDA(cudaStreamSynchronize(st));
}

void chol_variance(const gsi_chol* f, gsi_op* cross, const double* Fs, const double* Ft, int64_t p, double* var_out) {
    gsi_ctx* ctx = f->ctx;
    cudaStream_t st = ctx->stream;
    const int64_t n = f->n, np = f->np;
    GSI_REQUIRE(cross->type == OP_KERNELCROSS, GSI_ERR_INVALID_ARGUMENT,
                "chol_krige_variance needs a cross-covariance operator C(T, S) (gsi_op_kernelcov_cross or _cross_grid)");
    GSI_REQUIRE(cross->ctx == ctx, GSI_ERR_INVALID_ARGUMENT, "chol_krige_variance: the operator belongs to another context");
    GSI_REQUIRE(cross->n == n, GSI_ERR_DIMENSION_MISMATCH,
                "chol_krige_variance: the operator's sources must be the factor's n points");
    GSI_REQUIRE(p >= 0 && p <= CH_MAX_DRIFT, GSI_ERR_INVALID_ARGUMENT, "chol_krige_variance: p must be in 0..32");
    GSI_REQUIRE(p == 0 || (Fs && Ft), GSI_ERR_INVALID_ARGUMENT, "chol_krige_variance: F_s and F_t are needed when p > 0");
    const int64_t m = cross->mloc;
    if (m == 0) return;
    const int64_t kp0 = round_up(m < CH_MAX_CHUNK ? m : CH_MAX_CHUNK, CH_B);
    DevMem W((size_t)np * kp0 * sizeof(double));
    DevMem small((size_t)(CS_PARTS_MAX * CH_MAX_CHUNK + CH_MAX_CHUNK + m + 8) * sizeof(double));
    double* part = small.d();
    double* colsq = part + (size_t)CS_PARTS_MAX * CH_MAX_CHUNK;
    double* var = colsq + CH_MAX_CHUNK;
    double* ctt = var + m;
    // the prior variance c(t, t): the generator's value at zero offset (a 1 x 1 block of C(T, T))
    KcovBlock b0;
    b0.r0 = 0; b0.rows = 1; b0.c0 = 0; b0.cols = 1; b0.nr_valid = m; b0.nc_valid = m; b0.nugget_diag = 0; b0.lower = 0;
    b0.out = ctt; b0.rs = 1; b0.cs = 1;
    kcov_block(cross, KB_TARGETS, b0);
    // drift: G = L^-1 F_s (row-major np x 128), R'R = G'G (R upper p x p), F_t on the device
    std::unique_ptr<DevMem> G, Rm, Ftd, H;
    if (p > 0) {
        G.reset(new DevMem((size_t)np * CH_B * sizeof(double)));
        Rm.reset(new DevMem((size_t)(CH_B * CH_B + p * p) * sizeof(double) + 16));
        Ftd.reset(new DevMem((size_t)m * p * sizeof(double)));
        H.reset(new DevMem((size_t)CH_B * kp0 * sizeof(double)));
        // F_s (host column-major n x p) as the row-major np x 128 block G, zero padded
        std::vector<double> Gh((size_t)np * CH_B, 0.0);
        for (int64_t q = 0; q < p; ++q)
            for (int64_t i = 0; i < n; ++i) Gh[(size_t)i * CH_B + q] = Fs[q * n + i];
        GSI_CUDA(cudaMemcpyAsync(G->d(), Gh.data(), Gh.size() * sizeof(double), cudaMemcpyHostToDevice, st));
        GSI_CUDA(cudaMemcpyAsync(Ftd->d(), Ft, (size_t)m * p * sizeof(double), cudaMemcpyHostToDevice, st));
        int* flag = f->flags;
        GSI_CUDA(cudaMemsetAsync(flag, 0, 2 * sizeof(int), st));
        chol_nonfinite_kernel<<<(unsigned)((np * CH_B + 255) / 256), 256, 0, st>>>(G->d(), CH_B, np, CH_B, flag);
        chol_nonfinite_kernel<<<(unsigned)((m * p + 255) / 256), 256, 0, st>>>(Ftd->d(), p, m, p, flag);
        GSI_CUDA(cudaGetLastError());
        count_launch(ctx, 2);
        forward(f, G->d(), CH_B, CH_B, np / CH_B);
        double* GtG = Rm->d();
        double* R = GtG + CH_B * CH_B;
        gemm<false, false, true>(ctx, gm(G->d(), CH_B, G->d(), CH_B, GtG, CH_B, np, 0, 0), 1, 1);
        tall_head_to_cm_kernel<<<(unsigned)((p * p + 255) / 256), 256, 0, st>>>(GtG, CH_B, (int)p, R);
        chol_upper_kernel<<<1, 1024, 0, st>>>(R, (int)p, flag + 1);
        GSI_CUDA(cudaGetLastError());
        count_launch(ctx, 2);
        int hf[2] = {0, 0};
        GSI_CUDA(cudaMemcpyAsync(hf, flag, 2 * sizeof(int), cudaMemcpyDeviceToHost, st));
        GSI_CUDA(cudaStreamSynchronize(st));
        GSI_REQUIRE(hf[0] == 0, GSI_ERR_INVALID_ARGUMENT, "chol_krige_variance: F_s or F_t has a non-finite entry");
        if (hf[1] != 0)
            throw Error(GSI_ERR_NOT_POSDEF, "chol_krige_variance: F_s' C^-1 F_s is not positive definite (the drift columns "
                                            "at the sources are linearly dependent)");
    }
    for (int64_t t0 = 0; t0 < m; t0 += CH_MAX_CHUNK) {
        const int64_t w = m - t0 < CH_MAX_CHUNK ? m - t0 : CH_MAX_CHUNK;
        const int64_t wp = round_up(w, CH_B);
        GSI_CUDA(cudaMemsetAsync(W.d(), 0, (size_t)np * kp0 * sizeof(double), st));
        KcovBlock b;                                               // W = C(S, T_chunk), row-major
        b.r0 = 0; b.rows = n; b.c0 = t0; b.cols = w; b.nr_valid = n; b.nc_valid = m; b.nugget_diag = 0; b.lower = 0;
        b.out = W.d(); b.rs = kp0; b.cs = 1;
        kcov_block(cross, KB_CROSS_T, b);
        forward(f, W.d(), kp0, wp, np / CH_B);                     // W = L^-1 C(S, T_chunk)
        col_dot(ctx, W.d(), W.d(), kp0, n, w, part, colsq, nullptr);
        if (p > 0)                                                 // H = G' W
            gemm<false, false, true>(ctx, gm(G->d(), CH_B, W.d(), kp0, H->d(), kp0, np, 0, 0), 1, wp / CH_B);
        chol_variance_kernel<<<(unsigned)((w + 127) / 128), 128, 0, st>>>(colsq, ctt, w, (int)p, p > 0 ? H->d() : nullptr, kp0,
                                                                         p > 0 ? Ftd->d() + t0 : nullptr, m,
                                                                         p > 0 ? Rm->d() + CH_B * CH_B : nullptr, var + t0);
        GSI_CUDA(cudaGetLastError());
        count_launch(ctx);
    }
    GSI_CUDA(cudaMemcpyAsync(var_out, var, (size_t)m * sizeof(double), cudaMemcpyDeviceToHost, st));
    GSI_CUDA(cudaStreamSynchronize(st));
}

void chol_simulate(const gsi_chol* f, int64_t ns, const double* y, const double* Fs, const double* Ft, int64_t p,
                   const gsi_buf* Xi, gsi_buf* Z) {
    gsi_ctx* ctx = f->ctx;
    cudaStream_t st = ctx->stream;
    const int64_t n = f->n, np = f->np, m = n - ns;
    GSI_REQUIRE(ns >= 0 && ns < n, GSI_ERR_INVALID_ARGUMENT, "chol_simulate: ns must be in 0 .. n - 1");
    GSI_REQUIRE(p >= 0 && p <= CH_MAX_DRIFT, GSI_ERR_INVALID_ARGUMENT, "chol_simulate: p must be in 0..32");
    GSI_REQUIRE(p == 0 || ns > 0, GSI_ERR_INVALID_ARGUMENT, "chol_simulate: a drift needs conditioning data (ns > 0)");
    GSI_REQUIRE(ns == 0 || y, GSI_ERR_INVALID_ARGUMENT, "chol_simulate: y is needed when ns > 0");
    GSI_REQUIRE(p == 0 || (Fs && Ft), GSI_ERR_INVALID_ARGUMENT, "chol_simulate: F_s and F_t are needed when p > 0");
    GSI_REQUIRE(Xi->layout == GSI_LAYOUT_TALL && Xi->rows == n && Xi->cols >= 1 && Xi->cols <= CH_MAX_CHUNK,
                GSI_ERR_DIMENSION_MISMATCH, "chol_simulate: Xi must be TALL n x k, 1 <= k <= 1024");
    GSI_REQUIRE(Z->layout == GSI_LAYOUT_TALL && Z->rows == m && Z->cols == Xi->cols, GSI_ERR_DIMENSION_MISMATCH,
                "chol_simulate: Z must be TALL (n - ns) x k");
    GSI_REQUIRE(Xi->ctx == ctx && Z->ctx == ctx, GSI_ERR_INVALID_ARGUMENT, "chol_simulate: buffers of another context");
    bool finite = true;
    for (int64_t i = 0; i < ns; ++i) finite = finite && std::isfinite(y[i]);
    for (int64_t i = 0; i < ns * p; ++i) finite = finite && std::isfinite(Fs[i]);
    for (int64_t i = 0; i < m * p; ++i) finite = finite && std::isfinite(Ft[i]);
    GSI_REQUIRE(finite, GSI_ERR_INVALID_ARGUMENT, "chol_simulate: y, F_s or F_t has a non-finite entry");
    const int64_t k = Xi->cols, kp = round_up(k, CH_B);
    int* flag = f->flags;
    GSI_CUDA(cudaMemsetAsync(flag, 0, 2 * sizeof(int), st));
    chol_nonfinite_kernel<<<(unsigned)((n * k + 255) / 256), 256, 0, st>>>(Xi->d, Xi->ld, n, k, flag);
    GSI_CUDA(cudaGetLastError());
    count_launch(ctx);
    // V = [g 1' - G B; Xi_T] (row-major np x kp, zero padded), the TRMM rows from the tile that holds row ns
    const int64_t r0 = ns / CH_B * CH_B;
    DevMem V((size_t)np * kp * sizeof(double));
    DevMem Zw((size_t)(np - r0) * kp * sizeof(double));
    GSI_CUDA(cudaMemsetAsync(V.d(), 0, (size_t)np * kp * sizeof(double), st));
    tall_cols_copy(ctx, Xi->d, Xi->ld, V.d(), kp, n, k);
    std::unique_ptr<DevMem> W, small;
    double *GtG = nullptr, *R = nullptr, *H = nullptr, *Bm = nullptr, *Ftd = nullptr;
    if (ns > 0) {
        // [G | g] = L_SS^-1 [F_s | y]: rows below ns of L^-1 [F_s y; 0] are L_SS^-1 [F_s y], so the sweep stops after
        // the block rows that hold sources; the rows from ns on are zeroed for the reductions over the sources
        const int64_t nbs = (ns + CH_B - 1) / CH_B;
        W.reset(new DevMem((size_t)np * CH_B * sizeof(double)));
        small.reset(new DevMem((size_t)(CH_B * CH_B + CH_MAX_DRIFT * CH_MAX_DRIFT + (CH_B + CH_MAX_DRIFT) * kp + m * p) *
                               sizeof(double)));
        GtG = small->d(); R = GtG + CH_B * CH_B; H = R + CH_MAX_DRIFT * CH_MAX_DRIFT; Bm = H + CH_B * kp;
        Ftd = Bm + CH_MAX_DRIFT * kp;
        std::vector<double> Wh((size_t)np * CH_B, 0.0);
        for (int64_t i = 0; i < ns; ++i) {
            for (int64_t q = 0; q < p; ++q) Wh[(size_t)i * CH_B + q] = Fs[q * ns + i];
            Wh[(size_t)i * CH_B + p] = y[i];
        }
        GSI_CUDA(cudaMemcpyAsync(W->d(), Wh.data(), Wh.size() * sizeof(double), cudaMemcpyHostToDevice, st));
        if (p > 0)
            GSI_CUDA(cudaMemcpyAsync(Ftd, Ft, (size_t)m * p * sizeof(double), cudaMemcpyHostToDevice, st));
        forward(f, W->d(), CH_B, CH_B, nbs);
        GSI_CUDA(cudaMemsetAsync(W->d() + ns * CH_B, 0, (size_t)(np - ns) * CH_B * sizeof(double), st));
        if (p > 0) {
            gemm<false, false, true>(ctx, gm(W->d(), CH_B, W->d(), CH_B, GtG, CH_B, nbs * CH_B, 0, 0), 1, 1);   // W'W
            gemm<false, false, true>(ctx, gm(W->d(), CH_B, V.d(), kp, H, kp, nbs * CH_B, 0, 0), 1, kp / CH_B); // W'Xi
            tall_head_to_cm_kernel<<<(unsigned)((p * p + 255) / 256), 256, 0, st>>>(GtG, CH_B, (int)p, R);
            chol_upper_kernel<<<1, 1024, 0, st>>>(R, (int)p, flag + 1);
            GSI_CUDA(cudaGetLastError());
            count_launch(ctx, 2);
        }
    }
    int hf[2] = {0, 0};
    GSI_CUDA(cudaMemcpyAsync(hf, flag, 2 * sizeof(int), cudaMemcpyDeviceToHost, st));
    GSI_CUDA(cudaStreamSynchronize(st));
    GSI_REQUIRE(hf[0] == 0, GSI_ERR_INVALID_ARGUMENT, "chol_simulate: Xi has a non-finite entry");
    if (hf[1] != 0)
        throw Error(GSI_ERR_NOT_POSDEF, "chol_simulate: F_s' C^-1 F_s is not positive definite (the drift columns at the "
                                        "sources are linearly dependent)");
    if (ns > 0) {
        chol_sim_drift_kernel<<<dim3((unsigned)(kp / 32), (unsigned)((ns + SIM_ROWS - 1) / SIM_ROWS)), dim3(32, 8), 0, st>>>(
            W->d(), GtG, H, R, (int)p, ns, Bm, V.d(), kp);
        GSI_CUDA(cudaGetLastError());
        count_launch(ctx);
    }
    // Zw = L(r0 .., :) V: the n^2 k flops
    const int64_t nrt = (np - r0) / CH_B, nct = kp / CH_B;
    ChTrmm a;
    a.L = f->L; a.np = np; a.V = V.d(); a.kp = kp; a.Z = Zw.d(); a.r0 = r0; a.nct = nct;
    GSI_CUDA(cudaFuncSetAttribute(chol_trmm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CH_GEMM_SMEM));
    phase_begin(ctx);
    chol_trmm_kernel<<<(unsigned)(nrt * nct), CH_THREADS, CH_GEMM_SMEM, st>>>(a);
    GSI_CUDA(cudaGetLastError());
    count_launch(ctx);
    phase_end(ctx, PH_GEMM);
    if (ctx->time_gemm) {
        const int64_t nb = np / CH_B, i0 = r0 / CH_B;
        ctx->gemm_launches += 1;
        ctx->gemm_flops_accum += 2.0 * CH_B * CH_B * CH_B * (double)nct * (double)((nb * (nb + 1) - i0 * (i0 + 1)) / 2);
    }
    chol_sim_out_kernel<<<(unsigned)((m * k + 255) / 256), 256, 0, st>>>(Zw.d(), kp, ns - r0, Ftd, m, (int)p, Bm, Z->d,
                                                                         Z->ld, k);
    GSI_CUDA(cudaGetLastError());
    count_launch(ctx);
    GSI_CUDA(cudaStreamSynchronize(st));
}

void chol_loglik(gsi_op* op, const double* y, const double* F, int64_t p, int reml, double* loglik, double* beta_out,
                 double* grad_out, int64_t* failed_column) {
    gsi_ctx* ctx = op->ctx;
    cudaStream_t st = ctx->stream;
    if (failed_column) *failed_column = 0;
    GSI_REQUIRE(op->type == OP_KERNELCOV, GSI_ERR_UNSUPPORTED,
                "kernelcov_loglik needs a square kernel-covariance operator (gsi_op_kernelcov, _grid, _model or _model_grid)");
    GSI_REQUIRE(ctx->world == 1, GSI_ERR_UNSUPPORTED, "kernelcov_loglik is single-GPU: the dense factor is not distributed");
    const int64_t n = op->n, np = round_up(n, CH_B), nb = np / CH_B;
    GSI_REQUIRE(p >= 0 && p <= CH_MAX_DRIFT, GSI_ERR_INVALID_ARGUMENT, "kernelcov_loglik: p must be in 0..32");
    GSI_REQUIRE((p == 0) == (F == nullptr), GSI_ERR_INVALID_ARGUMENT, "kernelcov_loglik: F must be given iff p > 0");
    GSI_REQUIRE(!reml || p < n, GSI_ERR_INVALID_ARGUMENT, "kernelcov_loglik: REML needs fewer drift columns than points");
    bool finite = true;
    for (int64_t i = 0; i < n; ++i) finite = finite && std::isfinite(y[i]);
    for (int64_t i = 0; i < n * p; ++i) finite = finite && std::isfinite(F[i]);
    GSI_REQUIRE(finite, GSI_ERR_INVALID_ARGUMENT, "kernelcov_loglik: y or F has a non-finite entry");
    const bool want_grad = grad_out != nullptr;
    GSI_REQUIRE(!want_grad || op->table == nullptr, GSI_ERR_UNSUPPORTED,
                "kernelcov_loglik: the gradient needs an operator on coordinates (a grid operator's lattice table has no "
                "derivative; pass the grid nodes' coordinates to gsi_op_kernelcov / _model)");
    // device memory of the whole call, checked before the factor is allocated: the factor (as chol_factor counts it),
    // the [F | y] block and, for the gradient, one chunk of A^-1 and the partial sums of the contraction
    const int64_t ldz = np < CH_MAX_CHUNK ? np : CH_MAX_CHUNK;
    const int64_t nchunks = (n + CH_MAX_CHUNK - 1) / CH_MAX_CHUNK;
    const int64_t max_parts = (n + KG_ROWS - 1) / KG_ROWS * (CH_MAX_CHUNK / KG_COLS);
    const size_t small_doubles = (size_t)CH_B * CH_B + CH_MAX_DRIFT * CH_MAX_DRIFT + 2 * CH_MAX_DRIFT;
    double need = (double)np * np * 8.0 + (double)np * CH_B * 8.0 + 4096.0 + (double)np * CH_B * 8.0 + small_doubles * 8.0;
    if (want_grad) need += (double)np * ldz * 8.0 + (double)(max_parts + nchunks + 1) * KG_SLOTS * 8.0;
    require_free(ctx, need, "kernelcov_loglik", n);
    std::unique_ptr<gsi_chol, void (*)(gsi_chol*)> f(chol_factor(op, nullptr, failed_column), chol_destroy);
    // value: [G | g] = L^-1 [F | y] (row-major np x 128, zero padded), beta, e, q
    DevMem W((size_t)np * CH_B * sizeof(double));
    DevMem small(small_doubles * sizeof(double));
    double* GtG = small.d();
    double* R = GtG + CH_B * CH_B;
    double* res = R + CH_MAX_DRIFT * CH_MAX_DRIFT;             // beta (p), log det R, q
    int* flag = f->flags;
    std::vector<double> Wh;
    GSI_CUDA(cudaMemsetAsync(res, 0, 2 * CH_MAX_DRIFT * sizeof(double), st));
    drift_residual(f.get(), y, F, p, !want_grad ? 0 : (reml ? 2 : 1), W.d(), GtG, R, res, flag, Wh);
    chol_lik_sumsq_kernel<<<1, 1024, 0, st>>>(W.d(), n, (int)p, res + CH_MAX_DRIFT + 1);
    GSI_CUDA(cudaGetLastError());
    count_launch(ctx);
    double hres[2 * CH_MAX_DRIFT];
    int hf[2] = {0, 0};
    GSI_CUDA(cudaMemcpyAsync(hres, res, sizeof(hres), cudaMemcpyDeviceToHost, st));
    GSI_CUDA(cudaMemcpyAsync(hf, flag, 2 * sizeof(int), cudaMemcpyDeviceToHost, st));
    GSI_CUDA(cudaStreamSynchronize(st));
    if (hf[1] != 0)
        throw Error(GSI_ERR_NOT_POSDEF, "kernelcov_loglik: F' A^-1 F is not positive definite (the drift columns are "
                                        "linearly dependent)");
    const double log2pi = 1.83787706640934548356;
    const double q = hres[CH_MAX_DRIFT + 1];
    *loglik = reml ? -0.5 * ((double)(n - p) * log2pi + f->logdet + 2.0 * hres[CH_MAX_DRIFT] + q)
                   : -0.5 * ((double)n * log2pi + f->logdet + q);
    if (beta_out)
        for (int64_t k = 0; k < p; ++k) beta_out[k] = hres[k];
    if (!want_grad) return;
    // gradient: [H | alpha] = L^-T [G R^-1 | e] (ML: H = 0), then per chunk of A^-1 the rank update and the contraction
    backward(f.get(), W.d(), CH_B, CH_B);
    DevMem Z((size_t)np * ldz * sizeof(double));
    DevMem part((size_t)max_parts * KG_SLOTS * sizeof(double));
    DevMem csum((size_t)(nchunks + 1) * KG_SLOTS * sizeof(double));
    const int64_t K = round_up(p + 1, CH_K);
    int64_t c = 0;
    for (int64_t j0 = 0; j0 < n; j0 += CH_MAX_CHUNK, ++c) {
        const int64_t wp = np - j0 < CH_MAX_CHUNK ? np - j0 : CH_MAX_CHUNK, kb0 = j0 / CH_B;
        double* Zc = Z.d() + j0 * ldz;
        GSI_CUDA(cudaMemsetAsync(Zc, 0, (size_t)(np - j0) * ldz * sizeof(double), st));
        chol_eye_kernel<<<(unsigned)((wp + 255) / 256), 256, 0, st>>>(Z.d(), ldz, j0, wp);
        GSI_CUDA(cudaGetLastError());
        count_launch(ctx);
        forward(f.get(), Z.d(), ldz, wp, nb, kb0);
        backward(f.get(), Z.d(), ldz, wp, kb0);
        const double* Wj = W.d() + j0 * CH_B;
        gemm<true, true, true>(ctx, gm(Wj, CH_B, Wj, CH_B, Zc, ldz, K, 1, 0), (np - j0) / CH_B, wp / CH_B);
        const int64_t nparts = kcov_grad(op, Z.d(), ldz, j0, wp, part.d());
        kcov_grad_reduce(ctx, part.d(), nparts, csum.d() + c * KG_SLOTS);
    }
    double* total = csum.d() + nchunks * KG_SLOTS;
    kcov_grad_reduce(ctx, csum.d(), nchunks, total);
    double S[KG_SLOTS];
    GSI_CUDA(cudaMemcpyAsync(S, total, sizeof(S), cudaMemcpyDeviceToHost, st));
    GSI_CUDA(cudaStreamSynchronize(st));
    const bool model = op->kind == KC_KIND_MODEL;
    const int ns = model ? op->nstruct : 1, d = op->dim;
    for (int s = 0; s < ns; ++s) {
        const double sill = model ? op->msills[s] : op->sigma2;
        grad_out[s * (1 + d)] = 0.5 * S[4 * s];
        for (int a = 0; a < d; ++a) grad_out[s * (1 + d) + 1 + a] = -(sill / op->mranges[s][a]) * S[4 * s + 1 + a];
    }
    grad_out[ns * (1 + d)] = 0.5 * S[KG_SLOTS - 1];
}

void chol_crossval(const gsi_chol* f, const double* y, const double* F, int64_t p, int64_t ngroups,
                   const int64_t* group_ptr, const int64_t* group_idx, double* err_out, double* var_out,
                   double* logpdf_out, int64_t* failed_group) {
    gsi_ctx* ctx = f->ctx;
    cudaStream_t st = ctx->stream;
    const int64_t n = f->n, np = f->np, nb = np / CH_B;
    if (failed_group) *failed_group = 0;
    // ---- arguments, all on the host before any device work
    GSI_REQUIRE(p >= 0 && p <= CH_MAX_DRIFT, GSI_ERR_INVALID_ARGUMENT, "chol_crossval: p must be in 0..32");
    GSI_REQUIRE((p == 0) == (F == nullptr), GSI_ERR_INVALID_ARGUMENT, "chol_crossval: F must be given iff p > 0");
    bool finite = true;
    for (int64_t i = 0; i < n; ++i) finite = finite && std::isfinite(y[i]);
    for (int64_t i = 0; i < n * p; ++i) finite = finite && std::isfinite(F[i]);
    GSI_REQUIRE(finite, GSI_ERR_INVALID_ARGUMENT, "chol_crossval: y or F has a non-finite entry");
    std::vector<int64_t> loo_ptr, loo_idx;
    if (!group_ptr) {                                            // leave-one-out: n singletons in index order
        GSI_REQUIRE(group_idx == nullptr && ngroups == n, GSI_ERR_INVALID_ARGUMENT,
                    "chol_crossval: leave-one-out (group_ptr NULL) takes group_idx NULL and ngroups = n");
        loo_ptr.resize(n + 1);
        loo_idx.resize(n);
        for (int64_t i = 0; i <= n; ++i) loo_ptr[i] = i;
        for (int64_t i = 0; i < n; ++i) loo_idx[i] = i;
        group_ptr = loo_ptr.data();
        group_idx = loo_idx.data();
    }
    GSI_REQUIRE(ngroups >= 1 && ngroups <= n && group_idx != nullptr && group_ptr[0] == 0, GSI_ERR_INVALID_ARGUMENT,
                "chol_crossval: the groups need 1 <= ngroups <= n, group_idx and group_ptr[0] = 0");
    std::vector<char> seen(n, 0);
    for (int64_t g = 0; g < ngroups; ++g) {
        const int64_t s = group_ptr[g + 1] - group_ptr[g];
        GSI_REQUIRE(s >= 1 && s <= CH_B, GSI_ERR_INVALID_ARGUMENT,
                    "chol_crossval: group " + std::to_string(g) + " has " + std::to_string(s) +
                        " points (group_ptr must increase by 1..128)");
        for (int64_t k = group_ptr[g]; k < group_ptr[g + 1]; ++k) {
            const int64_t i = group_idx[k];
            GSI_REQUIRE(i >= 0 && i < n, GSI_ERR_INVALID_ARGUMENT,
                        "chol_crossval: group " + std::to_string(g) + " has the point index " + std::to_string(i) +
                            " outside 0 .. n - 1");
            GSI_REQUIRE(!seen[i], GSI_ERR_INVALID_ARGUMENT,
                        "chol_crossval: the point index " + std::to_string(i) + " is held out twice");
            seen[i] = 1;
        }
    }
    const int64_t m = group_ptr[ngroups];
    // ---- chunks: the groups by their smallest index, packed whole into <= 1024 columns.  cidx: the point of every
    // chunk column; desc: per chunk its groups of <= 32 points, then the larger ones
    std::vector<int64_t> order(ngroups), gmin(ngroups);
    for (int64_t g = 0; g < ngroups; ++g) {
        order[g] = g;
        gmin[g] = *std::min_element(group_idx + group_ptr[g], group_idx + group_ptr[g + 1]);
    }
    std::sort(order.begin(), order.end(), [&](int64_t a, int64_t b) { return gmin[a] < gmin[b]; });
    struct Chunk { int64_t c0, w, kb0, d0, nsmall, nlarge; };
    std::vector<Chunk> chunks;
    std::vector<int64_t> cidx(m);
    std::vector<CvGroup> desc(ngroups);
    {
        int64_t c0 = 0, gpos = 0;
        for (int64_t k = 0; k < ngroups;) {
            Chunk ch{c0, 0, gmin[order[k]] / CH_B, gpos, 0, 0};
            int64_t k1 = k;
            while (k1 < ngroups && ch.w + (group_ptr[order[k1] + 1] - group_ptr[order[k1]]) <= CH_MAX_CHUNK)
                ch.w += group_ptr[order[k1] + 1] - group_ptr[order[k1]], ++k1;
            for (int pass = 0; pass < 2; ++pass) {                 // small groups first, then the large ones
                int64_t col = 0;
                for (int64_t q = k; q < k1; ++q) {
                    const int64_t g = order[q], s = group_ptr[g + 1] - group_ptr[g];
                    if ((s > 32) == (pass == 1)) {
                        desc[gpos++] = CvGroup{group_ptr[g], (int32_t)s, (int32_t)col, (int32_t)g, 0};
                        (pass ? ch.nlarge : ch.nsmall) += 1;
                    }
                    if (pass == 0)
                        for (int64_t r = 0; r < s; ++r) cidx[c0 + col + r] = group_idx[group_ptr[g] + r];
                    col += s;
                }
            }
            chunks.push_back(ch);
            c0 += ch.w;
            k = k1;
        }
    }
    int64_t wmax = 0;
    for (const Chunk& ch : chunks) wmax = std::max(wmax, ch.w);
    const int64_t ld = round_up(wmax, CH_B);
    // ---- device memory: [G^ | e] and its backward copy, the chunk block, its Gram and G^'W, the column norms, the
    // drift scalars, the index and group tables, the outputs
    const size_t small_doubles = (size_t)CH_B * CH_B + CH_MAX_DRIFT * CH_MAX_DRIFT + 2 * CH_MAX_DRIFT;
    const size_t tail_doubles = (size_t)CS_PARTS_MAX * ld + ld + 2 * (size_t)m + (size_t)ngroups + 1;
    const double need = 2.0 * np * CH_B * 8.0 + (double)np * ld * 8.0 + (double)ld * ld * 8.0 + (double)CH_B * ld * 8.0 +
                        (double)(small_doubles + tail_doubles) * 8.0 + (double)m * 8.0 + (double)ngroups * sizeof(CvGroup);
    require_free(ctx, need, "chol_crossval", n);
    DevMem W((size_t)np * CH_B * sizeof(double)), Wa((size_t)np * CH_B * sizeof(double));
    DevMem Z((size_t)np * ld * sizeof(double)), Q((size_t)ld * ld * sizeof(double)), H((size_t)CH_B * ld * sizeof(double));
    DevMem small(small_doubles * sizeof(double)), tail(tail_doubles * sizeof(double));
    DevMem cidx_d((size_t)m * sizeof(int64_t)), desc_d((size_t)ngroups * sizeof(CvGroup));
    double* GtG = small.d();
    double* R = GtG + CH_B * CH_B;
    double* res = R + CH_MAX_DRIFT * CH_MAX_DRIFT;
    double* part = tail.d();
    double* colsq = part + (size_t)CS_PARTS_MAX * ld;
    double* err = colsq + ld;
    double* var = err + m;
    double* lpd = var + m;
    int* failed = reinterpret_cast<int*>(lpd + ngroups);
    const int64_t* cidx_dev = static_cast<const int64_t*>(cidx_d.p);
    const CvGroup* desc_dev = static_cast<const CvGroup*>(desc_d.p);
    GSI_CUDA(cudaMemcpyAsync(cidx_d.p, cidx.data(), (size_t)m * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    GSI_CUDA(cudaMemcpyAsync(desc_d.p, desc.data(), (size_t)ngroups * sizeof(CvGroup), cudaMemcpyHostToDevice, st));
    GSI_CUDA(cudaMemsetAsync(failed, 0x7f, sizeof(int), st));  // 0x7f7f7f7f: no group failed
    // ---- 1. [G^ | e] = [G R^-1 | g - G beta] in W (kept for the projection), alpha = L^-T e from a copy
    int* flag = f->flags;
    std::vector<double> Wh;
    GSI_CUDA(cudaMemsetAsync(res, 0, 2 * CH_MAX_DRIFT * sizeof(double), st));
    drift_residual(f, y, F, p, 2, W.d(), GtG, R, res, flag, Wh);
    int hf[2] = {0, 0};
    GSI_CUDA(cudaMemcpyAsync(hf, flag, 2 * sizeof(int), cudaMemcpyDeviceToHost, st));
    GSI_CUDA(cudaStreamSynchronize(st));
    if (hf[1] != 0)
        throw Error(GSI_ERR_NOT_POSDEF, "chol_crossval: F' A^-1 F is not positive definite (the drift columns are "
                                        "linearly dependent)");
    GSI_CUDA(cudaMemcpyAsync(Wa.d(), W.d(), (size_t)np * CH_B * sizeof(double), cudaMemcpyDeviceToDevice, st));
    backward(f, Wa.d(), CH_B, CH_B);
    const double* alpha = Wa.d() + p;
    // ---- 2. per chunk: W = (I - G^ G^') L^-1 E_chunk, Q = W'W, then the groups
    const int64_t K = round_up(p, CH_K);
    GSI_CUDA(cudaFuncSetAttribute(chol_cv_group_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)cv_group_smem<32>()));
    GSI_CUDA(cudaFuncSetAttribute(chol_cv_group_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)cv_group_smem<128>()));
    for (const Chunk& ch : chunks) {
        const int64_t wp = round_up(ch.w, CH_B), mt = wp / CH_B;
        // the whole block is zeroed: rows above kb0 stay exact zeros through the sweep, and the column norms and the
        // projection read every row (a column's norm then has the same bits in every chunk: col_dot's row partition
        // depends on the row count only).  The Gram of p = 0 skips those zero rows
        const int64_t r0 = p > 0 ? 0 : ch.kb0 * CH_B;
        GSI_CUDA(cudaMemsetAsync(Z.d(), 0, (size_t)np * ld * sizeof(double), st));
        chol_cv_scatter_kernel<<<(unsigned)((ch.w + 255) / 256), 256, 0, st>>>(Z.d(), ld, cidx_dev + ch.c0, ch.w);
        GSI_CUDA(cudaGetLastError());
        count_launch(ctx);
        forward(f, Z.d(), ld, wp, nb, ch.kb0);
        col_dot(ctx, Z.d(), Z.d(), ld, n, ch.w, part, colsq, nullptr);   // (A^-1)_jj, the pivot scale
        if (p > 0) {
            gemm<false, false, true>(ctx, gm(W.d(), CH_B, Z.d(), ld, H.d(), ld, np, 0, 0), 1, mt);   // H = [G^ | e]' W
            if (K > p) GSI_CUDA(cudaMemsetAsync(H.d() + p * ld, 0, (size_t)(K - p) * ld * sizeof(double), st));
            gemm<true, false, true>(ctx, gm(W.d(), CH_B, H.d(), ld, Z.d(), ld, K, 1, 0), nb, mt);   // W -= G^ H
        }
        gemm<false, false, true>(ctx, gm(Z.d() + r0 * ld, ld, Z.d() + r0 * ld, ld, Q.d(), ld, np - r0, 0, 1), mt, mt);
        const double* Qc = Q.d();
        if (ch.nsmall > 0) {
            chol_cv_group_kernel<32><<<(unsigned)((ch.nsmall + 3) / 4), CV_THREADS, cv_group_smem<32>(), st>>>(
                desc_dev + ch.d0, (int)ch.nsmall, Qc, ld, colsq, cidx_dev + ch.c0, alpha, err, var,
                logpdf_out ? lpd : nullptr, failed);
            GSI_CUDA(cudaGetLastError());
            count_launch(ctx);
        }
        if (ch.nlarge > 0) {
            chol_cv_group_kernel<128><<<(unsigned)ch.nlarge, CV_THREADS, cv_group_smem<128>(), st>>>(
                desc_dev + ch.d0 + ch.nsmall, (int)ch.nlarge, Qc, ld, colsq, cidx_dev + ch.c0, alpha, err, var,
                logpdf_out ? lpd : nullptr, failed);
            GSI_CUDA(cudaGetLastError());
            count_launch(ctx);
        }
    }
    int hfail = 0;
    GSI_CUDA(cudaMemcpyAsync(&hfail, failed, sizeof(int), cudaMemcpyDeviceToHost, st));
    GSI_CUDA(cudaMemcpyAsync(err_out, err, (size_t)m * sizeof(double), cudaMemcpyDeviceToHost, st));
    GSI_CUDA(cudaMemcpyAsync(var_out, var, (size_t)m * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (logpdf_out)
        GSI_CUDA(cudaMemcpyAsync(logpdf_out, lpd, (size_t)ngroups * sizeof(double), cudaMemcpyDeviceToHost, st));
    GSI_CUDA(cudaStreamSynchronize(st));
    if (hfail != 0x7f7f7f7f) {
        if (failed_group) *failed_group = hfail;
        throw Error(GSI_ERR_NOT_POSDEF, "chol_crossval: P_BB of group " + std::to_string(hfail) + " (1-based) is not "
                                        "positive definite (the remaining points do not identify the drift, or the "
                                        "block is numerically singular)");
    }
}

}  // namespace gsi
