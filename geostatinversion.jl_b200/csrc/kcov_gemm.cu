// Matrix-free covariance-kernel operator  W[I, :] = C[I, :] * X   (SURVEY.md §8 a8).
//
// C[i,j] = sigma2 * k(r2(u_i, u_j)) + nugget * (i == j) is never materialised.  Per
// 32-point k-tile, the four warps that share a 16-row group generate that group's
// 16 x 32 block of kernel values ONCE (4 entries per thread, FP64 DFMA/exp) into a
// double-buffered shared-memory tile laid out for conflict-free DMMA A-fragment loads,
// synchronise through a per-row-group mbarrier (arrive after publishing, wait right before
// the first read, so stragglers are covered by the next tile's generation work), and then each warp multiplies it against its
// quarter of the X tile with FP64 tensor-core MMAs (mma.sync.m8n8k4.f64 -> DMMA.8x8x4),
// accumulating a 16 x (8*NB/4) strip in registers.  X tiles (TALL layout, a k-tile is one
// contiguous chunk) and the scaled coordinates arrive by 1-D bulk async copies (UBLKCP)
// completing on mbarriers; thread 0 issues them `lookahead` tiles ahead.
//
// Why this shape (profiles/r01): a single warp can issue a DMMA only every ~32 cycles
// while the pipe retires one per 16, and DFMA shares that pipe -- so the SM needs >= 3-4
// warps per scheduler (16 warps/SM, <= 128 registers each) and every kernel value must be
// generated exactly once per CTA.  The 8-warp / A-in-registers first version stalled 43 %
// of samples in `wait` with the DMMA pipe 71 % busy.
//
// CTA = 16 warps = 4 row groups (16 rows) x 4 column groups: 64 rows x 8*NB columns.
// Persistent grid: one CTA per SM (x occupancy), static schedule: full rounds of 64-row
// tiles plus one tail round at 16-row-group granularity (see the schedule comment below).
#include "common.cuh"
#include "algos.h"
#include "ptx.cuh"
#include "nb_list.h"

namespace gsi {

constexpr int KC_BM = 64;          // rows per CTA tile
constexpr int KC_BK = 32;          // j-points (GEMM K) per pipeline stage
constexpr int KC_AP = KC_BK + 4;   // pitch of the generated A tile (4 mod 16 doubles)
constexpr int KC_WARPS = 16;
constexpr int KC_THREADS = KC_WARPS * 32;
constexpr int KC_CG = 4;           // column groups (warps sharing one row group)
constexpr long long KC_SPIN_LIMIT = 400000;   // cycles (~0.2 ms) a producer waits on the sweep window before giving it up

struct KcovBase {
    const double* X;       // TALL, all n rows (zero padded), pitch ld
    double* W;             // TALL, local rows, pitch ldw
    const double* u;       // scaled coordinates [3][n_pad]              (arithmetic generation)
    const int* lat;        // lattice indices [3][n_pad]                 (structured grid: table lookup)
    const double* table;   // k(r2) for every lattice offset: table[dx + nx*(dy + ny*dz)]
    int nx, ny;
    int sweep_groups, sweep_div, l2_hint;   // k-sweep de-synchronisation (power-of-two groups, spread = groups/div of X)
    int pad0;
    unsigned int* sync_cnt;                 // sweep window: arrivals per epoch (zeroed before the launch)
    int win_epochs, epoch_shift;            // a CTA runs at most win_epochs epochs of 2^epoch_shift k-tiles ahead of the slowest
    int64_t n;             // columns of C (= rows of X)
    int64_t n_pad;
    int64_t row0;          // first global row of this rank's block
    int64_t mloc;          // local rows
    int64_t ld, ldw;
    double sigma2, nugget, beta;
    int stages;
    // stream-K tail (see the schedule comment in the kernel): the 64-row tiles left over after the full rounds
    // are split along k into equal shares of tail_u k-tiles per CTA; partial sums go to `partial`
    int64_t tail_u;        // k-tiles of tail work per CTA (0: no tail)
    double* partial;       // [2 * grid][KC_BM][ldw] raw accumulators of the tail segments (slot 2b + s)
};
// the product kernel's parameters: KcovBase (all the tail fix-up reads) with the nested model appended
struct KcovParams : KcovBase {
    // nested model (KC_KIND_MODEL): u is [nstruct][3][n_pad], value = sum_s sill_s * k_{kind_s}(r2_s)
    int nstruct;
    int mkinds[GSI_MODEL_MAX_STRUCTURES];
    double msills[GSI_MODEL_MAX_STRUCTURES], mbetas[GSI_MODEL_MAX_STRUCTURES];
    // row side: the points of the output rows, the same layouts as u / lat with their own stride.  A square operator
    // passes u / lat themselves; a cross-covariance operator C(T, S) passes the other point set (row0 = 0 then)
    const double* ur;      // scaled coordinates of the row points [nstruct][3][nr_pad]
    const int* latr;       // lattice indices of the row points [3][nr_pad]
    int64_t nr_pad;
    int64_t nr;            // row points: a generated row beyond the last one is clamped to it (never stored)
};

template <int KIND>
__host__ __device__ constexpr bool kind_is_table() { return KIND == KC_KIND_TABLE || KIND == KC_KIND_TABLE_SIGNED; }
// coordinate doubles of one k-tile in a pipeline stage (the model carries up to GSI_MODEL_MAX_STRUCTURES sets)
template <int KIND>
__host__ __device__ constexpr int kc_coord_doubles() { return (KIND == KC_KIND_MODEL ? GSI_MODEL_MAX_STRUCTURES : 1) * 3 * KC_BK; }

// 2^(j/64), j = 0..63, correctly rounded (generated with 200-bit arithmetic)
__constant__ double kExp2Table[64] = {
    0x1.0000000000000p+0, 0x1.02c9a3e778061p+0, 0x1.059b0d3158574p+0, 0x1.0874518759bc8p+0,
    0x1.0b5586cf9890fp+0, 0x1.0e3ec32d3d1a2p+0, 0x1.11301d0125b51p+0, 0x1.1429aaea92de0p+0,
    0x1.172b83c7d517bp+0, 0x1.1a35beb6fcb75p+0, 0x1.1d4873168b9aap+0, 0x1.2063b88628cd6p+0,
    0x1.2387a6e756238p+0, 0x1.26b4565e27cddp+0, 0x1.29e9df51fdee1p+0, 0x1.2d285a6e4030bp+0,
    0x1.306fe0a31b715p+0, 0x1.33c08b26416ffp+0, 0x1.371a7373aa9cbp+0, 0x1.3a7db34e59ff7p+0,
    0x1.3dea64c123422p+0, 0x1.4160a21f72e2ap+0, 0x1.44e086061892dp+0, 0x1.486a2b5c13cd0p+0,
    0x1.4bfdad5362a27p+0, 0x1.4f9b2769d2ca7p+0, 0x1.5342b569d4f82p+0, 0x1.56f4736b527dap+0,
    0x1.5ab07dd485429p+0, 0x1.5e76f15ad2148p+0, 0x1.6247eb03a5585p+0, 0x1.6623882552225p+0,
    0x1.6a09e667f3bcdp+0, 0x1.6dfb23c651a2fp+0, 0x1.71f75e8ec5f74p+0, 0x1.75feb564267c9p+0,
    0x1.7a11473eb0187p+0, 0x1.7e2f336cf4e62p+0, 0x1.82589994cce13p+0, 0x1.868d99b4492edp+0,
    0x1.8ace5422aa0dbp+0, 0x1.8f1ae99157736p+0, 0x1.93737b0cdc5e5p+0, 0x1.97d829fde4e50p+0,
    0x1.9c49182a3f090p+0, 0x1.a0c667b5de565p+0, 0x1.a5503b23e255dp+0, 0x1.a9e6b5579fdbfp+0,
    0x1.ae89f995ad3adp+0, 0x1.b33a2b84f15fbp+0, 0x1.b7f76f2fb5e47p+0, 0x1.bcc1e904bc1d2p+0,
    0x1.c199bdd85529cp+0, 0x1.c67f12e57d14bp+0, 0x1.cb720dcef9069p+0, 0x1.d072d4a07897cp+0,
    0x1.d5818dcfba487p+0, 0x1.da9e603db3285p+0, 0x1.dfc97337b9b5fp+0, 0x1.e502ee78b3ff6p+0,
    0x1.ea4afa2a490dap+0, 0x1.efa1bee615a27p+0, 0x1.f50765b6e4540p+0, 0x1.fa7c1819e90d8p+0,
};

// exp(-y) for y >= 0 with a 64-entry table and a degree-5 polynomial: 10 FP64 pipe
// instructions instead of the ~17 of the library exp() -- the kernel generation shares the
// FP64 pipe with the DMMAs (a register-resident DMMA loop drops from 37.1 to 31.6 TF/s when
// one library-exp Gaussian value is generated per 28 DMMAs, tools/mma_lds_peak.cu), so
// every DFMA removed here is tensor throughput.  Error <= 2.5 ulp (library exp: 1 ulp), asserted
// value by value by tests/test_gpu_product_exact.py; largest error measured on a B200 (1000 W):
// 1.91 ulp over 12 600 arguments, and 2.20 ulp (y = 4.1859874635335022) in a host emulation of this
// exact instruction sequence over 2e7 arguments -- so "2 ulp" is not a bound.  Results below 2^-1000
// are flushed to zero.  `tab` is the table staged in shared memory.
__device__ __forceinline__ double fast_exp_neg(double y, const double* __restrict__ tab) {
    const double L = 92.33248261689366;                    // 64 / ln 2
    const double MAGIC = 6755399441055744.0;               // 1.5 * 2^52: round-to-nearest integer trick
    const double LN2_64_HI = 0x1.62e42fef80000p-7;         // ln2/64, 34 significant bits (k * HI exact)
    const double LN2_64_LO = 0x1.1cf79abc9e3b4p-42;
    const double t = fma(y, -L, MAGIC);
    const int k = __double2loint(t);                       // k = round(-y * 64 / ln2) <= 0
    const double kf = t - MAGIC;
    double r = fma(kf, -LN2_64_HI, -y);
    r = fma(kf, -LN2_64_LO, r);                            // |r| <= ln2/128
    double p = 1.0 / 120.0;
    p = fma(p, r, 1.0 / 24.0);
    p = fma(p, r, 1.0 / 6.0);
    p = fma(p, r, 0.5);
    p = fma(p, r, 1.0);
    p = fma(p, r, 1.0);
    const double v = tab[k & 63] * p;                      // in [1/2 .. 2)
    const int e = k >> 6;                                  // floor(k / 64) <= 0
    const int hi = __double2hiint(v) + (e << 20);
    const double res = __hiloint2double(hi, __double2loint(v));
    // y >= 1024 (hi word >= 0x40900000; also inf/NaN): k would wrap for y >~ 2.3e7 -- flush by the
    // integer compare on y itself (no FP64-pipe instruction)
    return (e < -1000 || __double2hiint(y) >= 0x40900000) ? 0.0 : res;
}

// sqrt(x) for x > 0 (callers add 1e-300 so the diagonal r2 = 0 stays finite): hardware
// rsqrt seed (MUFU, 2^-22) + two Goldschmidt steps = 6 FP64 pipe instructions, about 2 ulp.  Not
// observable on its own: the tests bound exp(-sqrt(r2)) by 2.5 + 4 y ulp (y = sqrt(r2); the 4 y term is
// 2 ulp of y times the conditioning y); largest error measured on a B200 for y < 1: 1.87 ulp.
__device__ __forceinline__ double fast_sqrt_pos(double x) {
    double rs;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(rs) : "d"(x));
    double h = __hiloint2double(__double2hiint(rs) - 0x00100000, __double2loint(rs));   // rs / 2
    double g = x * rs;
    double r = fma(-g, h, 0.5);
    g = fma(g, r, g);
    h = fma(h, r, h);
    r = fma(-g, h, 0.5);
    g = fma(g, r, g);
    return g;
}

// kinds whose value is a function of sqrt(r2): r2 gets a 1e-300 offset so that fast_sqrt_pos stays finite
// on the diagonal (sqrt(1e-300) = 1e-150 leaves every one of these values at exactly 1)
template <int KIND>
__device__ __forceinline__ constexpr bool kind_takes_sqrt() {
    return KIND == GSI_KERNEL_EXPONENTIAL || KIND == GSI_KERNEL_MATERN32 || KIND == GSI_KERNEL_MATERN52 ||
           KIND == GSI_KERNEL_SPHERICAL;
}

// kind-specific value from r2.  For the Gaussian kernel the coordinates handed to the
// kernel are pre-scaled by 1/sqrt(2) so that r2 already carries the factor 1/2; for the Matern
// kernels by sqrt(3) / sqrt(5), so that s = sqrt(r2) is the argument sqrt(2 nu) r of the Matern form.
// Relative error, in units of 2^-52 (measured in ulps of the exact value of the device's r2 this is at most twice
// as much, as a value and its rounding error can sit at opposite ends of a binade), with k = the conditioning
// |s k'(s) / k(s)| and 2 ulp of s from fast_sqrt_pos (each contributing at most 2 k * 2^-52):
//   matern32   fma(s, e, e) = RN(e (1 + s)):     2.5 (fast_exp_neg) + 0.5 (fma)                       = 3    + 2 k
//   matern52   RN(RN(fma(r2, RN(1/3), RN(s + 1))) e): 2.5 + 0.5 (s + 1) + 0.25 (1/3) + 0.5 (fma) + 0.5 = 4.25 + 2 k
//   spherical  RN(RN(0.5 t * t) RN(2 + s)), t = 1 - s (exact for s >= 0.5, 2^-53 relative below,
//              doubled by the square): 1 + 0.5 + 0.5 + 0.5                                            = 2.5  + 2 k
// tests/test_gpu_matern.py asserts 6 + 4 k, 8.5 + 4 k and 5 + 4 k ulp.  Largest errors measured on a B200
// (1000 W), d = 1..3, about 4200 arguments each: matern32 2.31 ulp for s < 1 (worst against the bound 2.05 of
// 6.25 ulp), matern52 3.07 ulp for s < 1 (3.07 of 8.71), spherical 4.15 ulp for s < 0.5 (worst against the bound
// 2.40 of 5.09).  Every term of the Matern polynomials is positive (no cancellation); the clamp of matern52
// to 1 only moves a value towards the exact one (<= 1).  The spherical form 0.5 (1 - s)^2 (2 + s) avoids the
// cancellation of 1 - 1.5 s + 0.5 s^3 as s -> 1.  The Matern values are flushed to zero with their exp factor
// (below 2^-1000).
template <int KIND>
__device__ __forceinline__ double kern_eval(double r2, double beta, const double* __restrict__ tab) {
    if (KIND == GSI_KERNEL_EXPONENTIAL) return fast_exp_neg(fast_sqrt_pos(r2), tab);
    if (KIND == GSI_KERNEL_GAUSSIAN) return fast_exp_neg(r2, tab);
    if (KIND == GSI_KERNEL_MATERN32) {
        const double s = fast_sqrt_pos(r2);
        const double e = fast_exp_neg(s, tab);
        return fma(s, e, e);                                   // (1 + s) e^-s
    }
    if (KIND == GSI_KERNEL_MATERN52) {
        const double s = fast_sqrt_pos(r2);
        const double e = fast_exp_neg(s, tab);
        // (1 + s + s^2/3) e^-s.  For s around 2e-8 the exact value is 1 - s^3/30 and the rounding errors of e and
        // of the product can leave 1 + 2^-52 (host emulation of this sequence), so the value is clamped to 1
        return fmin(fma(r2, 1.0 / 3.0, s + 1.0) * e, 1.0);
    }
    if (KIND == GSI_KERNEL_SPHERICAL) {
        const double s = fast_sqrt_pos(r2);
        const double t = 1.0 - s;
        return s < 1.0 ? (0.5 * t) * t * (2.0 + s) : 0.0;      // 0.5 (1 - s)^2 (2 + s)
    }
    if (kind_is_table<KIND>() || KIND == KC_KIND_MODEL) return 0.0;
    return exp(-beta * log1p(r2));
}

// Nested model (KC_KIND_MODEL): v = sum_s fma(c_s, kern_eval<kind_s>(r2_s), v), s = 0..nstruct-1, the kind decided at run
// time (warp-uniform: one model per launch).  r2_s = sum_k (ui[s][k] - uj[s][k])^2 by the same fma chain as the single
// kinds.  Error bound: every term is >= 0 (c_s > 0, k >= 0), so nothing cancels.  With b_s the bound of kind_s in ulps of
// its own exact value k_s (above; 2.5 + 4 y exponential, 2.5 Gaussian, 2 + 4 |z| power law, 6 / 8.5 / 5 + 4 k Matern 3/2,
// 5/2, spherical) each term carries a relative error b_s 2^-52 and the S roundings of the fma chain add gamma_S <= S 2^-53
// relative to the sum v:  |v_hat - v| <= 2^-52 sum_s c_s k_s b_s + gamma_S v,  i.e. in ulps of v at most
// 2 sum_s (c_s k_s / v) b_s + S <= 2 max_s b_s + S.  tests/test_gpu_kcov_model.py asserts the weighted form value by value.
// Two identical structures with c = 0.5 give 0.5 k + 0.5 k = k exactly, the single kind's value bit for bit.
__device__ __forceinline__ double kern_eval_runtime(int kind, double r2, double beta, const double* __restrict__ tab) {
    switch (kind) {
        case GSI_KERNEL_EXPONENTIAL: return kern_eval<GSI_KERNEL_EXPONENTIAL>(r2, beta, tab);
        case GSI_KERNEL_GAUSSIAN: return kern_eval<GSI_KERNEL_GAUSSIAN>(r2, beta, tab);
        case GSI_KERNEL_MATERN32: return kern_eval<GSI_KERNEL_MATERN32>(r2, beta, tab);
        case GSI_KERNEL_MATERN52: return kern_eval<GSI_KERNEL_MATERN52>(r2, beta, tab);
        case GSI_KERNEL_SPHERICAL: return kern_eval<GSI_KERNEL_SPHERICAL>(r2, beta, tab);
        default: return kern_eval<GSI_KERNEL_POWERLAW>(r2, beta, tab);
    }
}
__device__ __forceinline__ bool kind_takes_sqrt_runtime(int kind) { return kind != GSI_KERNEL_GAUSSIAN && kind != GSI_KERNEL_POWERLAW; }

// ui: the row's coordinates [nstruct][DIM] (shared memory); uj: column point of structure 0, coordinate k, at
// uj[k * kstride], structure s at + s * sstride
template <int DIM>
__device__ __forceinline__ double model_value(const KcovParams& p, const double* ui, const double* uj, int64_t kstride,
                                              int64_t sstride, const double* __restrict__ tab) {
    double v = 0.0;
    for (int s = 0; s < p.nstruct; ++s) {
        const int kind = p.mkinds[s];
        double r2 = kind_takes_sqrt_runtime(kind) ? 1e-300 : 0.0;
#pragma unroll
        for (int k = 0; k < DIM; ++k) {
            const double dk = ui[s * DIM + k] - uj[s * sstride + k * kstride];
            r2 = fma(dk, dk, r2);
        }
        v = fma(p.msills[s], kern_eval_runtime(kind, r2, p.mbetas[s], tab), v);
    }
    return v;
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" :: "r"(id), "r"(nthreads) : "memory");
}

// (Two probes of the first round -- the X tile fetched as four paced bulk copies, and an L2 bulk
// prefetch a few k-tiles ahead of every CTA's sweep -- were run on hardware in round 2
// (profiles/r02/l2_question.md): both bit-identical, the paced fetch 19 % slower, the prefetch
// within 0.1 % of the default although it turns every shared-memory fill into an L2 hit.  So an
// L2-served X stream is not slower as such; both variants were removed.  A third probe, round 2: the tile fetched
// as 4 / 8 / 32 bulk copies in an order rotated by the CTA index -- the idea being that CTAs sweeping X in step
// (sweep window) hammer the same L2 lines in the same order -- made every schedule slower (windowed front 563 ->
// 623 / 652 / 836 ms, default 516 -> 559 ms: the per-copy cost outweighs any spreading; gpurun_out r03_chunks.log);
// removed as well.)
// Signed lattice table (KC_KIND_TABLE_SIGNED): index of the offset li - lj, folded by central symmetry -- the last axis
// stored as |delta|, every component negated when that delta is negative, the other axes shifted by n - 1 into
// 0 .. 2n - 2.  Integer ALU only; unsigned because 2 n - 1 may reach 2^31 - 1 (the index itself is < 2^31).  Column
// point c: lattice index k at col[k * stride + c]
template <int DIM>
__device__ __forceinline__ int signed_table_index(const int (&li)[DIM], const int* col, int64_t stride, int c, int nx, int ny) {
    const int dl = li[DIM - 1] - col[(DIM - 1) * stride + c];
    const bool neg = dl < 0;
    unsigned idx = (unsigned)(neg ? -dl : dl);
#pragma unroll
    for (int k = DIM - 2; k >= 0; --k) {
        const int dk = li[k] - col[k * stride + c];
        const unsigned nk = (unsigned)(k == 0 ? nx : ny);
        idx = idx * (2u * nk - 1u) + (unsigned)(neg ? -dk : dk) + (nk - 1u);
    }
    return (int)idx;
}

template <int NB, int KIND, int DIM>
__global__ void __launch_bounds__(KC_THREADS, 1) kcov_gemm_kernel(const __grid_constant__ KcovParams p) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int ld = NB * 8 + 4;
    constexpr int NBW = (NB + KC_CG - 1) / KC_CG;                // n-blocks per warp
    constexpr int stage_doubles = KC_BK * ld + kc_coord_doubles<KIND>();   // X tile + coordinate tile
    constexpr int a_doubles = KC_BM * KC_AP;
    double* smem = reinterpret_cast<double*>(smem_raw);
    double* a_tiles = smem + (size_t)p.stages * stage_doubles;   // [2][KC_BM][KC_AP]
    uint64_t* full = reinterpret_cast<uint64_t*>(a_tiles + 2 * a_doubles);
    uint64_t* empty = full + p.stages;
    uint64_t* abar = empty + p.stages;                            // one per row group, 4 warp arrivals
    double* etab = reinterpret_cast<double*>(abar + 4);           // 2^(j/64) table for fast_exp_neg

    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const int lane = tid & 31;
    const int nstages = p.stages;
    const int rg = warp >> 2;                 // row group: rows rg*16 .. rg*16+15 of the tile
    const int cg = (warp + rg) & 3;           // column group, rotated per row group so that each SM
                                              // sub-partition (warp % 4) hosts all four column groups
                                              // (the last group may own fewer n-blocks)
    const int nb0 = cg * NBW;                 // first n-block of this warp

    if (tid < 64) etab[tid] = kExp2Table[tid];
    if (tid == 0) {
        for (int s = 0; s < nstages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], KC_WARPS);
        }
        for (int r = 0; r < 4; ++r) mbar_init(&abar[r], KC_CG);
        mbar_fence_init();
    }
    __syncthreads();

    // Work schedule.  Full rounds: CTA b takes the 64-row tile (round*grid + b), i.e. four consecutive
    // 16-row groups, and sweeps all nkt k-tiles (cyclically, from its own start tile kt0).  The tiles left
    // over after the full rounds (< grid of them) form the STREAM-K TAIL: their tail_tiles * nkt k-tile
    // units are cut into equal contiguous shares of p.tail_u units, one share per CTA, so a share is a k
    // range of one tile or the end of one tile plus the start of the next -- at most two SEGMENTS.  A tail
    // segment stores its raw accumulators to p.partial (slot 2b + s); kcov_tail_fixup_kernel adds the
    // pieces of a tile in ascending CTA order (deterministic) and applies sigma2 / nugget.  Every SM thus
    // ends within one k-tile of every other whatever the row count (round 1 spread the leftover 16-row
    // groups over the CTAs with full k sweeps: 4.5 % of a C3 product at 8 GPUs, where a rank's 1568 row
    // groups are 2.65 rounds).
    const int64_t total_rg = (p.mloc + 15) / 16;
    const int64_t per_round = (int64_t)gridDim.x * 4;
    const int64_t full_rounds = total_rg / per_round;
    const int64_t tail_rg0 = full_rounds * per_round;                         // first row group of the tail
    const int64_t tail_tiles = (total_rg - tail_rg0 + 3) / 4;
    const int64_t nkt = (p.n + KC_BK - 1) / KC_BK;
    // De-synchronised (cyclic) k sweeps (gsi_ctx_set_option "kcov.sweep_*" / GSI_SWEEP): CTA b starts
    // its sweep (b mod groups) * separation tiles into X (default 64 groups over a quarter of X).
    // Measured on C3 (profiles/r01): +2.5 % over lock-step starts.  In this mode the X stream
    // (366 MB > L2) is served mostly from HBM -- ncu: 610-716 GB read per launch (L2 hit rate
    // 26-33 %, 17 % of HBM bandwidth) -- with the DMMA pipe 91-93 % busy, 3.95 us per k-tile.
    const int64_t kt_sep = p.sweep_div < 0 ? -(int64_t)p.sweep_div
                           : p.sweep_div == 0 ? 0
                           : (nkt >= p.sweep_div ? nkt / p.sweep_div : (nkt >= 16 ? 1 : 0));
    const int64_t kt0 = ((int64_t)(blockIdx.x & (p.sweep_groups - 1)) * kt_sep) % nkt;
    // Sweep window (p.win_epochs > 0, default off): the persistent CTAs all stream the same X, but
    // left alone they drift apart by more than an L2's worth of k-tiles.  The schedule is static --
    // the launch ends with its slowest CTA anyway -- so the producer can hold a CTA that is more than
    // win_epochs epochs ahead of the slowest one: every 2^epoch_shift k-tiles it counts itself into
    // the epoch's arrival counter and waits until the epoch win_epochs back has been reached by every
    // CTA that will ever reach it (all CTAs during the full rounds, the tail CTAs afterwards).  The
    // wait is bounded (KC_SPIN_LIMIT): a CTA that times out -- co-tenancy, a debugger -- drops the
    // window for the rest of the launch, so the window can cost time but never progress.
    // MEASURED (profiles/r01/sweep_schedules_c3_summary.csv, 22 schedules): one coherent front cuts
    // DRAM traffic 611 GB -> 8.0 GB per launch (= X once per round, L2 hit rate 98.6 %) and products
    // stay bit-identical, but EVERY L2-served variant -- any window, lock-step or de-phased CTAs,
    // 2..32 fronts, evict_last -- runs at 589-612 ms (4.5 us per k-tile) against 528-532 ms streamed
    // from HBM, and so does a problem whose X fits L2 outright; the pacing itself is free (same
    // window over the quarter-of-X spread: 530 ms).  The HBM-streamed schedule therefore stays the
    // default; the window is the knob for deployments that must spare HBM bandwidth.  Why the
    // L2-served stream costs the DMMA pipe ~13 % is the first ncu question of the next round.
    const int64_t full_it = full_rounds * nkt;
    // my share of the tail: units [u0, u1) -> segment A = (tile tA, k-tiles [kA, kA + lenA)), segment B = (tile tA + 1, [0, lenB))
    const int64_t tail_units = tail_tiles * nkt;
    int64_t u0 = (int64_t)blockIdx.x * p.tail_u, u1 = u0 + p.tail_u;
    if (u0 > tail_units) u0 = tail_units;
    if (u1 > tail_units) u1 = tail_units;
    const int64_t tA = u0 / nkt, kA = u0 - tA * nkt;
    const int64_t lenA = (u1 - u0 < nkt - kA) ? u1 - u0 : nkt - kA;
    const int64_t lenB = (u1 - u0) - lenA;
    const int nseg_tail = (lenA > 0 ? 1 : 0) + (lenB > 0 ? 1 : 0);
    const int64_t nseg = full_rounds + nseg_tail;
    // segment j: first row group, active row groups, first k-tile, k-tiles, partial slot (-1: direct output)
    struct Seg { int64_t base_rg; int nact; int64_t kbeg; int64_t klen; int slot; };
    auto seg_info = [&](int64_t j) -> Seg {
        Seg g;
        if (j < full_rounds) { g.base_rg = (j * gridDim.x + blockIdx.x) * 4; g.nact = 4; g.kbeg = 0; g.klen = nkt; g.slot = -1; return g; }
        const int sidx = (int)(j - full_rounds);
        const int64_t tile = tA + sidx;
        g.base_rg = tail_rg0 + tile * 4;
        const int64_t left = total_rg - g.base_rg;
        g.nact = (int)(left < 4 ? left : 4);
        g.kbeg = sidx == 0 ? kA : 0;
        g.klen = sidx == 0 ? lenA : lenB;
        g.slot = 2 * (int)blockIdx.x + sidx;
        return g;
    };
    // iteration `it` of this CTA -> its segment and global k-tile
    auto locate = [&](int64_t it_, int64_t& j, int64_t& kt) {
        if (it_ < full_it) {
            j = it_ / nkt;
            kt = it_ - j * nkt + kt0;
            if (kt >= nkt) kt -= nkt;
        } else {
            const int64_t r = it_ - full_it;
            if (r < lenA) { j = full_rounds; kt = kA + r; }
            else { j = full_rounds + 1; kt = r - lenA; }
        }
    };
    // CTAs that execute iteration x of the tail (x >= 0): those whose share is longer than x
    auto tail_ctas_beyond = [&](int64_t x) -> unsigned {
        if (p.tail_u <= 0 || x >= p.tail_u) return 0u;
        int64_t c = (tail_units - x + p.tail_u - 1) / p.tail_u;
        if (c > (int64_t)gridDim.x) c = gridDim.x;
        return c < 0 ? 0u : (unsigned)c;
    };
    bool window_on = p.win_epochs > 0;            // thread 0 only
    const uint64_t xpolicy = l2_policy_evict_last();
    const uint32_t stage_bytes = (uint32_t)(KC_BK * ld * sizeof(double) +
                                            (KIND == KC_KIND_MODEL ? p.nstruct : 1) * DIM * KC_BK *
                                                (kind_is_table<KIND>() ? sizeof(int) : sizeof(double)));

    // ---------------- producer (thread 0): streams X / coordinate tiles ----------------------
    const int64_t total_it = full_it + (u1 - u0);
    const int lookahead = nstages > 2 ? nstages - 2 : 1;
    // Producer state, advanced incrementally (no 64-bit divisions on thread 0's path: its warp is an MMA
    // warp too, and what the producer spends per k-tile is added to the whole CTA's iteration time):
    //   p_it     next iteration to produce      p_s / p_ph   its pipeline stage / mbarrier phase
    //   p_kt     its global k-tile              p_left       k-tiles left in its segment (incl. itself)
    //   p_seg    its segment (0 .. nseg-1)
    int64_t p_it = 0, p_kt = 0, p_left = 0, p_seg = -1;
    int p_s = 0;
    uint32_t p_ph = 0;
    // first k-tile and length of segment j
    auto seg_first_kt = [&](int64_t j, int64_t& len) -> int64_t {
        if (j < full_rounds) { len = nkt; return kt0; }
        if (j == full_rounds) { len = lenA; return kA; }
        len = lenB; return 0;
    };
    auto produce_next = [&]() {
        if (p_left == 0) {                                        // enter the next segment
            ++p_seg;
            p_kt = seg_first_kt(p_seg, p_left);
        }
        const int64_t kt = p_kt;
        // k-tile of the iteration after this one (its coordinates ride along with this stage)
        int64_t ktn;
        if (p_left > 1) {
            ktn = kt + 1;
            if (p_seg < full_rounds && ktn == nkt) ktn = 0;
        } else if (p_seg + 1 < nseg) {
            int64_t len_unused;
            ktn = seg_first_kt(p_seg + 1, len_unused);
        } else {
            ktn = kt;
        }
        if (p.win_epochs > 0 && (p_it & (((int64_t)1 << p.epoch_shift) - 1)) == 0) {
            const int64_t e = p_it >> p.epoch_shift;
            atomicAdd(p.sync_cnt + e, 1u);
            const int64_t ew = e - p.win_epochs;
            if (window_on && ew >= 0) {
                const unsigned target = ((ew << p.epoch_shift) < full_it) ? gridDim.x : tail_ctas_beyond((ew << p.epoch_shift) - full_it);
                const volatile unsigned int* c = p.sync_cnt + ew;
                const long long t0 = clock64();
                while (*c < target) {
                    if (clock64() - t0 > KC_SPIN_LIMIT) { window_on = false; break; }
                }
            }
        }
        mbar_wait(&empty[p_s], p_ph ^ 1u);
        double* xs = smem + (size_t)p_s * stage_doubles;
        double* us = xs + KC_BK * ld;
        mbar_expect_tx(&full[p_s], stage_bytes);
        if (p.l2_hint) bulk_g2s_hint(xs, p.X + kt * KC_BK * p.ld, KC_BK * ld * 8, &full[p_s], xpolicy);
        else bulk_g2s(xs, p.X + kt * KC_BK * p.ld, KC_BK * ld * 8, &full[p_s]);
        if (kind_is_table<KIND>()) {
            int* usi = reinterpret_cast<int*>(us);
            for (int k = 0; k < DIM; ++k)
                bulk_g2s(usi + k * KC_BK, p.lat + k * p.n_pad + ktn * KC_BK, KC_BK * 4, &full[p_s]);
        } else if (KIND == KC_KIND_MODEL) {
            for (int s = 0; s < p.nstruct; ++s)
                for (int k = 0; k < DIM; ++k)
                    bulk_g2s(us + (s * DIM + k) * KC_BK, p.u + (s * 3 + k) * p.n_pad + ktn * KC_BK, KC_BK * 8, &full[p_s]);
        } else {
            for (int k = 0; k < DIM; ++k)
                bulk_g2s(us + k * KC_BK, p.u + k * p.n_pad + ktn * KC_BK, KC_BK * 8, &full[p_s]);
        }
        // advance
        ++p_it;
        --p_left;
        p_kt = kt + 1;
        if (p_seg < full_rounds && p_kt == nkt) p_kt = 0;
        if (++p_s == nstages) { p_s = 0; p_ph ^= 1u; }
    };
    if (tid == 0) {
        for (int64_t i = 0; i < lookahead && i < total_it; ++i) produce_next();
    }

    const int g = lane >> 2;      // fragment row (A, C) / column (B)
    const int t = lane & 3;       // fragment k index (A, B) / column pair (C)
    // generation role inside the row group: 128 threads x 4 entries = 16 rows x 32 points
    const int gtid = tid & 127;                  // thread index within the row group
    const int grow_in_tile = rg * 16 + (gtid >> 3);
    // my four points of the k-tile: columns gj0, gj0+1 and gj0+16, gj0+17 (gcol(e)).  The eight threads of a row
    // then publish 16-byte pairs at units 0..7 and 8..15 of the row: conflict-free 128-bit stores (round 1 used
    // four adjacent columns per thread: units 0,2,..,14 -> every quarter-warp store 2-way conflicted, 56 % of all
    // shared-store wavefronts of the kernel).
    const int gj0 = (gtid & 7) * 2;
    auto gcol = [&](int e) -> int { return gj0 + (e & 1) + ((e >> 1) << 4); };
    int li[DIM];
    auto row_coords = [&](int64_t base_rg, double (&ui)[DIM]) {
        int64_t gpt = p.row0 + base_rg * 16 + grow_in_tile;           // row point of my generated row
        if (gpt > p.nr - 1) gpt = p.nr - 1;                           // tail rows: clamp (never stored)
        if constexpr (KIND == KC_KIND_MODEL) {
            // the row's nstruct * DIM coordinates go to shared memory, [KC_BM][GSI_MODEL_MAX_STRUCTURES * DIM] after
            // etab (they do not fit the register budget): the 8 threads of a row, all in this warp, load them
            // together; only this warp reads them
            __syncwarp();
            for (int q = gtid & 7; q < p.nstruct * DIM; q += 8) {
                const int s = q / DIM, k = q - s * DIM;
                etab[64 + grow_in_tile * (GSI_MODEL_MAX_STRUCTURES * DIM) + q] = p.ur[(s * 3 + k) * p.nr_pad + gpt];
            }
            __syncwarp();
        } else {
#pragma unroll
            for (int k = 0; k < DIM; ++k) {
                if (kind_is_table<KIND>()) li[k] = p.latr[k * p.nr_pad + gpt];
                else ui[k] = p.ur[k * p.nr_pad + gpt];
            }
        }
    };

    // table variant: lattice offset of (my row, column point e of the tile) -> table index
    auto table_index = [&](const int* usi, int e) -> int {
        int idx = 0;
#pragma unroll
        for (int k = DIM - 1; k >= 0; --k) {
            int dk = li[k] - usi[k * KC_BK + gcol(e)];
            dk = dk < 0 ? -dk : dk;
            idx = (k == DIM - 1) ? dk : idx * (k == 0 ? p.nx : p.ny) + dk;
        }
        return idx;
    };
    auto gen4 = [&](const double (&ui)[DIM], const double* u0, int64_t ustride, double (&v)[4]) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            double r2 = kind_takes_sqrt<KIND>() ? 1e-300 : 0.0;
#pragma unroll
            for (int k = 0; k < DIM; ++k) {
                const double dk = ui[k] - u0[k * ustride + gcol(e)];
                r2 = fma(dk, dk, r2);
            }
            v[e] = kern_eval<KIND>(r2, p.beta, etab);
        }
    };
    auto store4 = [&](double* as, const double (&v)[4]) {
        double2* dst = reinterpret_cast<double2*>(as + grow_in_tile * KC_AP + gj0);
        dst[0] = make_double2(v[0], v[1]);
        dst[8] = make_double2(v[2], v[3]);          // + 16 columns
    };

    int c_s = 0;                       // consumer pipeline stage / mbarrier phase of iteration `it`
    uint32_t c_ph = 0;
    double ui[DIM];
    if (nseg > 0) {
        // prologue: kernel values of (first segment, its first k-tile) straight from global coordinates
        const Seg g0 = seg_info(0);
        int64_t j0, ktf;
        locate(0, j0, ktf);
        row_coords(g0.base_rg, ui);
        if (rg < g0.nact) {
            double v[4];
            if (KIND == KC_KIND_TABLE) {
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    int idx = 0;
#pragma unroll
                    for (int k = DIM - 1; k >= 0; --k) {
                        int dk = li[k] - p.lat[k * p.n_pad + ktf * KC_BK + gcol(e)];
                        dk = dk < 0 ? -dk : dk;
                        idx = (k == DIM - 1) ? dk : idx * (k == 0 ? p.nx : p.ny) + dk;
                    }
                    v[e] = __ldg(p.table + idx);
                }
            } else if constexpr (KIND == KC_KIND_TABLE_SIGNED) {
#pragma unroll
                for (int e = 0; e < 4; ++e)
                    v[e] = __ldg(p.table + signed_table_index<DIM>(li, p.lat + ktf * KC_BK, p.n_pad, gcol(e), p.nx, p.ny));
            } else if constexpr (KIND == KC_KIND_MODEL) {
                const double* urow = etab + 64 + grow_in_tile * (GSI_MODEL_MAX_STRUCTURES * DIM);
#pragma unroll
                for (int e = 0; e < 4; ++e)
                    v[e] = model_value<DIM>(p, urow, p.u + ktf * KC_BK + gcol(e), p.n_pad, 3 * p.n_pad, etab);
            } else {
                gen4(ui, p.u + ktf * KC_BK, p.n_pad, v);
            }
            store4(a_tiles, v);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&abar[rg]);
    }
    // (loop state is kept small on purpose: the kernel sits at the 128-register limit and every value that
    //  lives across the k loop costs the generation / MMA interleave its scheduling freedom)
    int par = 0;                                                      // parity of the A-tile buffer of this iteration
    for (int64_t j = 0; j < nseg; ++j) {
        int klen;
        bool active;
        {
            const Seg sg = seg_info(j);
            klen = (int)sg.klen;
            active = rg < sg.nact;                                    // warp-uniform
        }
        double acc[2][NBW][2];
#pragma unroll
        for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int nb = 0; nb < NBW; ++nb) { acc[h][nb][0] = 0.0; acc[h][nb][1] = 0.0; }

        for (int ktl = 0; ktl < klen; ++ktl, par ^= 1) {
            if (tid == 0 && p_it < total_it) produce_next();           // (p_it == it + lookahead)
            const int s = c_s;
            mbar_wait(&full[s], c_ph);
            if (++c_s == nstages) { c_s = 0; c_ph ^= 1u; }
            __syncwarp();
            const double* xs = smem + (size_t)s * stage_doubles;
            const double* us = xs + KC_BK * ld;                       // coordinates of the next iteration's k-tile
            const double* as = a_tiles + (size_t)par * a_doubles;
            // ---- kernel values of the NEXT iteration's block (independent of the MMAs below: the two
            //      instruction streams overlap on the shared FP64 pipe)
            bool gen_next = active;
            if (ktl + 1 == klen) {                                    // the next block belongs to the next segment
                gen_next = false;
                if (j + 1 < nseg) {
                    const Seg sn = seg_info(j + 1);
                    row_coords(sn.base_rg, ui);
                    gen_next = rg < sn.nact;
                }
            }
            double* anext = a_tiles + (size_t)(par ^ 1) * a_doubles + grow_in_tile * KC_AP + gj0;
            double tv[4] = {0.0, 0.0, 0.0, 0.0};
            if (kind_is_table<KIND>() && gen_next) {
                // structured grid: the four kernel values are table look-ups (L1/L2 hits, no FP64 pipe
                // work); issued now, consumed after the MMA loop
                const int* usi = reinterpret_cast<const int*>(us);
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    if constexpr (KIND == KC_KIND_TABLE_SIGNED)
                        tv[e] = __ldg(p.table + signed_table_index<DIM>(li, usi, KC_BK, gcol(e), p.nx, p.ny));
                    else
                        tv[e] = __ldg(p.table + table_index(usi, e));
                }
            }
            // ---- tensor-core phase on the current k-tile: wait until the whole row group has
            //      published this block (and has stopped reading the other buffer)
            mbar_wait(&abar[rg], (uint32_t)par);
            __syncwarp();
            const double* arow0 = as + (rg * 16 + g) * KC_AP + t;
            const double* arow1 = arow0 + 8 * KC_AP;
#pragma unroll
            for (int ks = 0; ks < KC_BK / 4; ++ks) {
                // one kernel value of the NEXT block every second k-step: a single exp chain
                // is live at a time and its DFMAs interleave with this step's DMMAs
                if constexpr (KIND == KC_KIND_MODEL) {
                    if ((ks & 1) == 0 && gen_next) {
                        const int e = ks >> 1;
                        const double* urow = etab + 64 + grow_in_tile * (GSI_MODEL_MAX_STRUCTURES * DIM);
                        anext[(e & 1) + ((e >> 1) << 4)] = model_value<DIM>(p, urow, us + gcol(e), KC_BK, DIM * KC_BK, etab);
                    }
                }
                if (!kind_is_table<KIND>() && KIND != KC_KIND_MODEL && (ks & 1) == 0 && gen_next) {
                    const int e = ks >> 1;
                    double r2 = kind_takes_sqrt<KIND>() ? 1e-300 : 0.0;
#pragma unroll
                    for (int k = 0; k < DIM; ++k) {
                        const double dk = ui[k] - us[k * KC_BK + gcol(e)];
                        r2 = fma(dk, dk, r2);
                    }
                    anext[(e & 1) + ((e >> 1) << 4)] = kern_eval<KIND>(r2, p.beta, etab);
                }
                if (active) {
                    const double a0 = arow0[ks * 4];
                    const double a1 = arow1[ks * 4];
                    const double* xrow = xs + (ks * 4 + t) * ld + nb0 * 8 + g;
#pragma unroll
                    for (int nb = 0; nb < NBW; ++nb) {
                        if (nb0 + nb < NB) {
                            const double b = xrow[nb * 8];
                            dmma884(acc[0][nb][0], acc[0][nb][1], a0, b);
                            dmma884(acc[1][nb][0], acc[1][nb][1], a1, b);
                        }
                    }
                }
            }
            if (kind_is_table<KIND>() && gen_next) {
                double2* dst = reinterpret_cast<double2*>(anext);
                dst[0] = make_double2(tv[0], tv[1]);
                dst[8] = make_double2(tv[2], tv[3]);
            }
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(&empty[s]);
                mbar_arrive(&abar[rg]);           // next block published; current block no longer read
            }
        }

        const Seg sg = seg_info(j);
        if (sg.slot < 0) {
            // epilogue of a full round: W = sigma2 * acc + nugget * X[global row]
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int64_t lrow = (sg.base_rg + rg) * 16 + h * 8 + g;
                if (active && lrow < p.mloc) {
                    double* wrow = p.W + lrow * p.ldw + nb0 * 8 + 2 * t;
                    const double* xg = p.X + (p.row0 + lrow) * p.ld + nb0 * 8 + 2 * t;
#pragma unroll
                    for (int nb = 0; nb < NBW; ++nb) {
                        if (nb0 + nb < NB) {
                            double2 v;
                            v.x = p.sigma2 * acc[h][nb][0];
                            v.y = p.sigma2 * acc[h][nb][1];
                            if (p.nugget != 0.0) {
                                const double2 xv = *reinterpret_cast<const double2*>(xg + nb * 8);
                                v.x += p.nugget * xv.x;
                                v.y += p.nugget * xv.y;
                            }
                            *reinterpret_cast<double2*>(wrow + nb * 8) = v;
                        }
                    }
                }
            }
        } else if (active) {
            // tail segment: raw partial sums of this k range -> slot (kcov_tail_fixup_kernel combines them)
            double* part = p.partial + (size_t)sg.slot * KC_BM * p.ldw;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                double* prow = part + (size_t)(rg * 16 + h * 8 + g) * p.ldw + nb0 * 8 + 2 * t;
#pragma unroll
                for (int nb = 0; nb < NBW; ++nb)
                    if (nb0 + nb < NB) *reinterpret_cast<double2*>(prow + nb * 8) = make_double2(acc[h][nb][0], acc[h][nb][1]);
            }
        }
    }
}

// Tail tiles: W[rows of tile t] = sigma2 * (sum of the k-range pieces in ascending CTA order) + nugget * X[rows].
// Piece of CTA b for tile t lives in slot 2b (tile t is the first tile of b's share) or 2b + 1.
// Grid: (tail tiles, KC_BM / KF_ROWS row chunks); the slot list of the tile is built once per CTA (the
// round-2 version divided 64-bit integers per piece and element on 9 CTAs: 141 us for 9 tiles at n = 10 000).
constexpr int KF_ROWS = 8;
constexpr int KF_MAX_PIECES = 160;     // pieces of one tile <= CTAs of the main grid (<= SMs, checked at launch)
__global__ void kcov_tail_fixup_kernel(KcovBase p, int64_t nkt, int64_t tail_rg0, int grid_main, int cols) {
    __shared__ int s_slot[KF_MAX_PIECES];
    const int64_t tile = blockIdx.x;
    const int64_t ulo = tile * nkt, uhi = ulo + nkt;                  // this tile's units
    const int b_first = (int)(ulo / p.tail_u);
    int b_last = (int)((uhi - 1) / p.tail_u);
    if (b_last > grid_main - 1) b_last = grid_main - 1;
    const int npieces = b_last - b_first + 1;
    for (int k = threadIdx.x; k < npieces; k += blockDim.x) {
        const int b = b_first + k;
        const int64_t first_tile = ((int64_t)b * p.tail_u) / nkt;
        s_slot[k] = 2 * b + (tile == first_tile ? 0 : 1);
    }
    __syncthreads();
    const int64_t row_base = tail_rg0 * 16 + tile * KC_BM;
    const int r_lo = blockIdx.y * KF_ROWS;
    for (int idx = threadIdx.x; idx < KF_ROWS * cols; idx += blockDim.x) {
        const int r = r_lo + idx / cols, c = idx % cols;
        const int64_t lrow = row_base + r;
        if (lrow >= p.mloc) continue;
        const double* src = p.partial + (size_t)r * p.ldw + c;
        double s = 0.0;
        for (int k = 0; k < npieces; ++k) s += src[(size_t)s_slot[k] * KC_BM * p.ldw];
        double v = p.sigma2 * s;
        if (p.nugget != 0.0) v += p.nugget * p.X[(p.row0 + lrow) * p.ld + c];
        p.W[lrow * p.ldw + c] = v;
    }
}

// all_sms: the cross-covariance operator launches the full persistent grid even when the output has fewer than
// 4 x grid row groups.  C(obs, grid) X has few rows and a long k range (200 x 200 704); a grid capped at its 13 row
// groups would leave 135 of 148 SMs idle, while the stream-K tail spreads the k range over every CTA (CTAs past the
// last unit own no work).  The tail invariants hold for any grid: tail tiles <= grid, so a share of
// ceil(tiles * nkt / grid) <= nkt units spans at most two segments, and a tile's pieces <= grid <= KF_MAX_PIECES.
// The square operators keep the capped grid (a different grid reorders their sums).
template <int NB, int KIND, int DIM>
static void launch_kcov(gsi_ctx* ctx, const KcovParams& p0, bool all_sms) {
    KcovParams p = p0;
    const int ld = NB * 8 + 4;
    const size_t stage_bytes = (size_t)(KC_BK * ld + kc_coord_doubles<KIND>()) * sizeof(double);
    const size_t a_bytes = (size_t)2 * KC_BM * KC_AP * sizeof(double);
    int stages = (int)((224 * 1024 - a_bytes - 1024) / stage_bytes);
    if (stages > 4) stages = 4;
    if (stages < 2) stages = 2;
    p.stages = stages;
    const size_t urow_bytes = KIND == KC_KIND_MODEL ? (size_t)KC_BM * GSI_MODEL_MAX_STRUCTURES * DIM * sizeof(double) : 0;
    const size_t smem = stages * stage_bytes + a_bytes + (2 * stages + 4) * sizeof(uint64_t) + 64 * sizeof(double) + urow_bytes;
    auto kfn = kcov_gemm_kernel<NB, KIND, DIM>;
    GSI_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0;
    GSI_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kfn, KC_THREADS, smem));
    if (occ < 1) occ = 1;
    const int64_t total_rg = (p.mloc + 15) / 16;                 // 16-row groups; a CTA runs up to 4 at a time
    int64_t grid = (int64_t)ctx->num_sms * occ;
    if (!all_sms && grid > total_rg) grid = total_rg;
    if (grid < 1) grid = 1;
    p.pad0 = 0;
    p.win_epochs = ctx->kcov_window > 0 ? ctx->kcov_window : 0;
    p.epoch_shift = ctx->kcov_epoch_shift;
    p.sync_cnt = nullptr;
    if (p.win_epochs > 0) {
        // one arrival counter per epoch of the longest CTA schedule (full rounds + tail round)
        const int64_t nkt = (p.n + KC_BK - 1) / KC_BK;
        const int64_t rounds = total_rg / (grid * 4) + (total_rg % (grid * 4) != 0 ? 1 : 0);
        const size_t n_epochs = (size_t)((rounds * nkt) >> p.epoch_shift) + 2;
        if (n_epochs > ctx->sweep_cnt_n) {
            if (ctx->sweep_cnt) GSI_CUDA(cudaFree(ctx->sweep_cnt));
            ctx->sweep_cnt = nullptr; ctx->sweep_cnt_n = 0;
            GSI_CUDA(cudaMalloc(&ctx->sweep_cnt, n_epochs * sizeof(unsigned int)));
            ctx->sweep_cnt_n = n_epochs;
        }
        GSI_CUDA(cudaMemsetAsync(ctx->sweep_cnt, 0, n_epochs * sizeof(unsigned int), ctx->stream));
        p.sync_cnt = ctx->sweep_cnt;
    }
    // stream-K tail: tiles left over after the full rounds, cut into equal k shares (one per CTA)
    const int64_t nkt_h = (p.n + KC_BK - 1) / KC_BK;
    const int64_t full_rounds_h = total_rg / (grid * 4);
    const int64_t tail_rg0_h = full_rounds_h * grid * 4;
    const int64_t tail_tiles_h = (total_rg - tail_rg0_h + 3) / 4;
    p.tail_u = tail_tiles_h > 0 ? (tail_tiles_h * nkt_h + grid - 1) / grid : 0;
    p.partial = nullptr;
    size_t part_bytes = 0;
    if (tail_tiles_h > 0) {
        part_bytes = (size_t)2 * grid * KC_BM * p.ldw * sizeof(double);
        p.partial = static_cast<double*>(pool_alloc(ctx, part_bytes));
    }
    struct PartGuard { gsi_ctx* c; void* q; size_t b; ~PartGuard() { if (q) pool_free(c, q, b); } } pguard{ctx, p.partial, part_bytes};
    kfn<<<(unsigned)grid, KC_THREADS, smem, ctx->stream>>>(p);
    GSI_CUDA(cudaGetLastError());
    count_launch(ctx);
    if (tail_tiles_h > 0) {
        GSI_REQUIRE(grid <= KF_MAX_PIECES, GSI_ERR_UNSUPPORTED, "kernelcov apply: more CTAs than the tail fix-up handles");
        kcov_tail_fixup_kernel<<<dim3((unsigned)tail_tiles_h, KC_BM / KF_ROWS), 256, 0, ctx->stream>>>(p, nkt_h, tail_rg0_h,
                                                                                                      (int)grid, 8 * NB);
        GSI_CUDA(cudaGetLastError());
        count_launch(ctx);
    }
}

template <int NB, int KIND>
static void dispatch_dim(gsi_ctx* ctx, const KcovParams& p, int dim, bool all_sms) {
    if (dim <= 2) launch_kcov<NB, KIND, 2>(ctx, p, all_sms);
    else launch_kcov<NB, KIND, 3>(ctx, p, all_sms);
}

template <int NB>
static void dispatch_kind(gsi_ctx* ctx, const KcovParams& p, int kind, int dim, bool all_sms) {
    switch (kind) {
        case GSI_KERNEL_EXPONENTIAL: dispatch_dim<NB, GSI_KERNEL_EXPONENTIAL>(ctx, p, dim, all_sms); break;
        case GSI_KERNEL_GAUSSIAN: dispatch_dim<NB, GSI_KERNEL_GAUSSIAN>(ctx, p, dim, all_sms); break;
        case GSI_KERNEL_POWERLAW: dispatch_dim<NB, GSI_KERNEL_POWERLAW>(ctx, p, dim, all_sms); break;
        case GSI_KERNEL_MATERN32: dispatch_dim<NB, GSI_KERNEL_MATERN32>(ctx, p, dim, all_sms); break;
        case GSI_KERNEL_MATERN52: dispatch_dim<NB, GSI_KERNEL_MATERN52>(ctx, p, dim, all_sms); break;
        case GSI_KERNEL_SPHERICAL: dispatch_dim<NB, GSI_KERNEL_SPHERICAL>(ctx, p, dim, all_sms); break;
        case KC_KIND_TABLE: dispatch_dim<NB, KC_KIND_TABLE>(ctx, p, dim, all_sms); break;
        case KC_KIND_TABLE_SIGNED: dispatch_dim<NB, KC_KIND_TABLE_SIGNED>(ctx, p, dim, all_sms); break;
        case KC_KIND_MODEL: dispatch_dim<NB, KC_KIND_MODEL>(ctx, p, dim, all_sms); break;
        default: throw Error(GSI_ERR_INVALID_ARGUMENT, "unknown covariance kernel kind");
    }
}

// Square operator (OP_KERNELCOV): W = C[row0 .. row0 + mloc, :] X, trans ignored (C is symmetric).
// Cross-covariance operator (OP_KERNELCROSS, C = C(T, S), targets compacted to this rank's mloc points):
//   trans = 0: W (mloc rows) = C X,  X: all n source rows   -- target rows x source columns
//   trans = 1: W (n rows) = C' X,    X: this rank's mloc target rows (zero padded beyond them: the last k-tile's
//              padded columns multiply them)                -- source rows x target columns
void kcov_apply(gsi_op* op, int trans, const gsi_buf* X, gsi_buf* W) {
    gsi_ctx* ctx = op->ctx;
    const bool cross = op->type == OP_KERNELCROSS;
    const bool tr = cross && trans;
    const int64_t krows = tr ? op->mloc : op->n;               // rows of X (the product's k range)
    const int64_t orows = tr ? op->n : op->mloc;               // rows of W
    GSI_REQUIRE(X->layout == GSI_LAYOUT_TALL && W->layout == GSI_LAYOUT_TALL, GSI_ERR_INVALID_ARGUMENT,
                "kernelcov apply needs TALL buffers");
    GSI_REQUIRE(X->rows == krows, GSI_ERR_DIMENSION_MISMATCH, "kernelcov apply: X must have n rows");
    GSI_REQUIRE(W->rows == orows, GSI_ERR_DIMENSION_MISMATCH, "kernelcov apply: W must have mloc rows");
    GSI_REQUIRE(X->cols == W->cols, GSI_ERR_DIMENSION_MISMATCH, "kernelcov apply: X/W column mismatch");
    if (cross && (orows == 0 || krows == 0)) {                 // a rank without target rows: no rows, or C' X = 0
        if (orows > 0) tall_zero(ctx, W);
        return;
    }
    if (X->cols > kMaxCols) {
        // wide iterate (K + p > 256): the product runs on 256-column chunks packed into compact buffers
        for (int64_t c0 = 0; c0 < X->cols; c0 += kMaxCols) {
            const int64_t w = (X->cols - c0 < kMaxCols) ? X->cols - c0 : kMaxCols;
            BufPtr xc = make_buf(ctx, GSI_LAYOUT_TALL, X->rows, w);
            BufPtr wc = make_buf(ctx, GSI_LAYOUT_TALL, W->rows, w);
            tall_cols_copy(ctx, X->d + c0, X->ld, xc->d, xc->ld, X->rows, w);
            kcov_apply(op, trans, xc.get(), wc.get());
            tall_cols_copy(ctx, wc->d, wc->ld, W->d + c0, W->ld, W->rows, w);
        }
        return;
    }
    const int nb = nb_for_cols(X->cols);
    GSI_REQUIRE(X->ld == 8 * nb + 4 && W->ld == X->ld, GSI_ERR_INVALID_ARGUMENT, "kernelcov apply: bad pitch");
    KcovParams p;
    p.X = X->d; p.W = W->d; p.u = op->ucoords;
    p.lat = op->lattice; p.table = op->table; p.nx = op->grid_nx; p.ny = op->grid_ny;
    p.sweep_groups = ctx->kcov_sweep_groups; p.sweep_div = ctx->kcov_sweep_div; p.l2_hint = ctx->kcov_l2_hint;
    p.n = op->n; p.n_pad = op->n_pad; p.row0 = op->row0; p.mloc = op->mloc;
    p.ld = X->ld; p.ldw = W->ld;
    p.sigma2 = op->sigma2; p.nugget = op->nugget; p.beta = op->beta;
    p.stages = 0;
    p.nstruct = op->nstruct;
    for (int s = 0; s < GSI_MODEL_MAX_STRUCTURES; ++s) {
        p.mkinds[s] = op->mkinds[s]; p.msills[s] = op->msills[s]; p.mbetas[s] = op->mbetas[s];
    }
    p.ur = op->ucoords; p.latr = op->lattice; p.nr_pad = op->n_pad; p.nr = op->n;
    if (cross) {
        // sources: ucoords / lattice (n points); targets: ucoords_t / lattice_t (this rank's mloc points)
        p.row0 = 0;
        if (!tr) {
            p.ur = op->ucoords_t; p.latr = op->lattice_t; p.nr_pad = op->nt_pad; p.nr = op->mloc;
        } else {
            p.u = op->ucoords_t; p.lat = op->lattice_t; p.n = op->mloc; p.n_pad = op->nt_pad;
            p.mloc = op->n;
        }
    }
    const int kind = op->table ? (op->table_signed ? KC_KIND_TABLE_SIGNED : KC_KIND_TABLE) : op->kind;
    switch (nb) {
#define GSI_CASE(N) case N: dispatch_kind<N>(ctx, p, kind, op->dim, cross); break;
        GSI_NB_LIST(GSI_CASE)
#undef GSI_CASE
        default: throw Error(GSI_ERR_UNSUPPORTED, "kernelcov apply: unsupported column-block count");
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Materialised covariance blocks (cov_chol.cu: the dense Cholesky factor and the kriging-variance chunks).
// out[(i - r0) * rs + (j - c0) * cs] = C[i, j] for rows [r0, r0 + rows) x columns [c0, c0 + cols), from the product
// kernel's own value code: the same r2 fma chain, kern_eval / model_value, table and signed-table look-ups, and the
// sigma2 / nugget epilogue (sigma2 * value, then + nugget where i == j).  The product on an identity column adds exact
// zeros to value * 1, so an entry equals (C I[:, j])[i] bit for bit.  The arithmetic kinds use the same DIM
// instantiation as the product (d = 1 runs as DIM = 2 on a zero second coordinate).
// Row points: p.ur / p.latr (pitch p.nr_pad); column points: p.u / p.lat (pitch p.n_pad).  Entries with i >= nr_valid
// or j >= nc_valid are padding (the factor rounds its order up to a multiple of its block): 1 where i == j, else 0.
// lower != 0: CTA tiles entirely above the diagonal are skipped (the factor reads the lower triangle only).
constexpr int KB_ROWS = 64;       // rows of a CTA tile (one per threadIdx.x)
constexpr int KB_COLS = 64;       // columns of a CTA tile
constexpr int KB_TY = 4;          // threadIdx.y: column phases

// |lattice offset| table index of row lattice point li and column point c (lattice index k at col[k * stride + c]):
// the index the product kernel's table_index forms, |dx| + nx * (|dy| + ny * |dz|)
template <int DIM>
__device__ __forceinline__ int abs_table_index(const int (&li)[DIM], const int* col, int64_t stride, int64_t c, int nx, int ny) {
    int idx = 0;
#pragma unroll
    for (int k = DIM - 1; k >= 0; --k) {
        int dk = li[k] - col[k * stride + c];
        dk = dk < 0 ? -dk : dk;
        idx = (k == DIM - 1) ? dk : idx * (k == 0 ? nx : ny) + dk;
    }
    return idx;
}

template <int KIND, int DIM>
__global__ void __launch_bounds__(KB_ROWS * KB_TY) kcov_block_kernel(const __grid_constant__ KcovParams p, int64_t r0,
                                                                     int64_t rows, int64_t c0, int64_t cols,
                                                                     int64_t nr_valid, int64_t nc_valid, int nugget_diag,
                                                                     int lower, double* __restrict__ out, int64_t rs,
                                                                     int64_t cs) {
    __shared__ double etab[64 + (KIND == KC_KIND_MODEL ? KB_ROWS * GSI_MODEL_MAX_STRUCTURES * DIM : 0)];
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int64_t ti = r0 + (int64_t)blockIdx.x * KB_ROWS, tj = c0 + (int64_t)blockIdx.y * KB_COLS;
    if (lower && tj > ti + KB_ROWS - 1) return;                  // the whole CTA
    const int tid = ty * KB_ROWS + tx;
    if (tid < 64) etab[tid] = kExp2Table[tid];
    const int64_t i = ti + tx;
    const int64_t gpt = i < nr_valid ? i : nr_valid - 1;        // padding rows: any valid point (never stored)
    double ui[DIM];
    int li[DIM];
    double* urow = etab + 64 + tx * (GSI_MODEL_MAX_STRUCTURES * DIM);
    if constexpr (KIND == KC_KIND_MODEL) {
        if (ty == 0)
            for (int q = 0; q < p.nstruct * DIM; ++q) {
                const int s = q / DIM, k = q - s * DIM;
                urow[q] = p.ur[(s * 3 + k) * p.nr_pad + gpt];
            }
    } else {
#pragma unroll
        for (int k = 0; k < DIM; ++k) {
            if (kind_is_table<KIND>()) li[k] = p.latr[k * p.nr_pad + gpt];
            else ui[k] = p.ur[k * p.nr_pad + gpt];
        }
    }
    __syncthreads();
    if (i >= r0 + rows) return;
    for (int q = ty; q < KB_COLS; q += KB_TY) {
        const int64_t j = tj + q;
        if (j >= c0 + cols) break;
        double v;
        if (i >= nr_valid || j >= nc_valid) {
            v = i == j ? 1.0 : 0.0;
        } else {
            double kv;
            if constexpr (KIND == KC_KIND_TABLE) {
                kv = __ldg(p.table + abs_table_index<DIM>(li, p.lat, p.n_pad, j, p.nx, p.ny));
            } else if constexpr (KIND == KC_KIND_TABLE_SIGNED) {
                kv = __ldg(p.table + signed_table_index<DIM>(li, p.lat + j, p.n_pad, 0, p.nx, p.ny));
            } else if constexpr (KIND == KC_KIND_MODEL) {
                kv = model_value<DIM>(p, urow, p.u + j, p.n_pad, 3 * p.n_pad, etab);
            } else {
                double r2 = kind_takes_sqrt<KIND>() ? 1e-300 : 0.0;
#pragma unroll
                for (int k = 0; k < DIM; ++k) {
                    const double dk = ui[k] - p.u[k * p.n_pad + j];
                    r2 = fma(dk, dk, r2);
                }
                kv = kern_eval<KIND>(r2, p.beta, etab);
            }
            // the product's epilogue: sigma2 * acc, then + nugget * x (x = 1 on the diagonal) -- two roundings, no fma
            v = __dmul_rn(p.sigma2, kv);
            if (nugget_diag && i == j && p.nugget != 0.0) v = __dadd_rn(v, p.nugget);
        }
        out[(i - r0) * rs + (j - c0) * cs] = v;
    }
}

template <int KIND, int DIM>
static void launch_block(gsi_ctx* ctx, const KcovParams& p, const KcovBlock& b) {
    const dim3 grid((unsigned)((b.rows + KB_ROWS - 1) / KB_ROWS), (unsigned)((b.cols + KB_COLS - 1) / KB_COLS));
    kcov_block_kernel<KIND, DIM><<<grid, dim3(KB_ROWS, KB_TY), 0, ctx->stream>>>(
        p, b.r0, b.rows, b.c0, b.cols, b.nr_valid, b.nc_valid, b.nugget_diag, b.lower, b.out, b.rs, b.cs);
    GSI_CUDA(cudaGetLastError());
    count_launch(ctx);
}

template <int KIND>
static void block_dim(gsi_ctx* ctx, const KcovParams& p, const KcovBlock& b, int dim) {
    if (dim <= 2) launch_block<KIND, 2>(ctx, p, b);
    else launch_block<KIND, 3>(ctx, p, b);
}

// rows index the row point set and columns the column point set of `side`:
//   KB_SQUARE        square operator: both are its n points (the nugget on the diagonal)
//   KB_CROSS         cross-covariance C(T, S): rows are the targets, columns the sources (the operator's orientation)
//   KB_CROSS_T       its transpose C(S, T): rows are the sources, columns the targets
//   KB_TARGETS       C(T, T) without nugget (the prior variance c(t, t) on the diagonal)
void kcov_block(gsi_op* op, int side, const KcovBlock& b) {
    gsi_ctx* ctx = op->ctx;
    if (b.rows <= 0 || b.cols <= 0) return;
    KcovParams p;
    std::memset(&p, 0, sizeof(p));
    p.u = op->ucoords; p.lat = op->lattice; p.table = op->table; p.nx = op->grid_nx; p.ny = op->grid_ny;
    p.n = op->n; p.n_pad = op->n_pad; p.row0 = 0; p.mloc = op->mloc;
    p.sigma2 = op->sigma2; p.nugget = op->nugget; p.beta = op->beta;
    p.nstruct = op->nstruct;
    for (int s = 0; s < GSI_MODEL_MAX_STRUCTURES; ++s) {
        p.mkinds[s] = op->mkinds[s]; p.msills[s] = op->msills[s]; p.mbetas[s] = op->mbetas[s];
    }
    p.ur = op->ucoords; p.latr = op->lattice; p.nr_pad = op->n_pad; p.nr = op->n;
    if (side == KB_CROSS) {
        p.ur = op->ucoords_t; p.latr = op->lattice_t; p.nr_pad = op->nt_pad; p.nr = op->mloc;
    } else if (side == KB_CROSS_T) {
        p.u = op->ucoords_t; p.lat = op->lattice_t; p.n_pad = op->nt_pad; p.n = op->mloc;
    } else if (side == KB_TARGETS) {
        p.ur = p.u = op->ucoords_t; p.latr = p.lat = op->lattice_t; p.nr_pad = p.n_pad = op->nt_pad; p.nr = p.n = op->mloc;
        p.nugget = 0.0;
    }
    const int kind = op->table ? (op->table_signed ? KC_KIND_TABLE_SIGNED : KC_KIND_TABLE) : op->kind;
    switch (kind) {
        case GSI_KERNEL_EXPONENTIAL: block_dim<GSI_KERNEL_EXPONENTIAL>(ctx, p, b, op->dim); break;
        case GSI_KERNEL_GAUSSIAN: block_dim<GSI_KERNEL_GAUSSIAN>(ctx, p, b, op->dim); break;
        case GSI_KERNEL_POWERLAW: block_dim<GSI_KERNEL_POWERLAW>(ctx, p, b, op->dim); break;
        case GSI_KERNEL_MATERN32: block_dim<GSI_KERNEL_MATERN32>(ctx, p, b, op->dim); break;
        case GSI_KERNEL_MATERN52: block_dim<GSI_KERNEL_MATERN52>(ctx, p, b, op->dim); break;
        case GSI_KERNEL_SPHERICAL: block_dim<GSI_KERNEL_SPHERICAL>(ctx, p, b, op->dim); break;
        case KC_KIND_TABLE: block_dim<KC_KIND_TABLE>(ctx, p, b, op->dim); break;
        case KC_KIND_TABLE_SIGNED: block_dim<KC_KIND_TABLE_SIGNED>(ctx, p, b, op->dim); break;
        case KC_KIND_MODEL: block_dim<KC_KIND_MODEL>(ctx, p, b, op->dim); break;
        default: throw Error(GSI_ERR_INVALID_ARGUMENT, "unknown covariance kernel kind");
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Likelihood gradient (cov_chol.cu, chol_loglik): the contraction sum_ij w_ij W_ij dA_ij / dtheta over one chunk of
// columns of W = alpha alpha' - A^-1 (+ H H'), the chunk held as Z = -W (row-major, pitch ldz, row i at Z + i * ldz).
// Every parameter's dA / dtheta comes from the operator's own scaled coordinates u (layout [nstruct][3][n_pad]; a single
// kind is the one-structure case of that layout):
//   dA_ij / dsill_s        = k_s(r2_s)                        (the value kern_eval gives the factor's fill, bit for bit)
//   dA_ij / drange_(s,a)   = sill_s k_s'(r2_s) (-2 du_(s,a)^2) / range_(s,a),   k' = dk / dr2 in the kernel's own units
// The kernel sums w W k_s and w W k_s' du_(s,a)^2 (w = 2 below the diagonal, 1 on it) per structure and axis; the host
// applies sill_s, -2 / range_(s,a) and the factor 1/2.  A single kind with d = 1 runs as DIM = 2 on a zero second
// coordinate: its axis-1 sums are exact zeros.
//
// dk / dr2 per kind (s = sqrt(r2) by fast_sqrt_pos; the 1e-300 offset of r2 makes du = 0 give 0 * finite = 0 for the
// kinds that divide by s, and du_a^2 / s <= s keeps them finite near the diagonal).  Relative error of the derivative
// value in units of 2^-52, in the style of the bounds beside kern_eval (2.5 for fast_exp_neg, 2 ulp of s entering with
// the conditioning of the expression in s, 0.5 per rounding):
//   exponential  RN(RN(-0.5 e) / s), e = e^-s:        2.5 + 2 s (s in e) + 2 (s in the divisor) + 0.5          = 5 + 2 s
//   gaussian     -e^-r2:                              2.5                                                      = 2.5
//   powerlaw     RN(RN(-beta v) / RN(1 + r2)), v the library value (2 + 4 |z|, z = beta log1p r2): + 1.5  = 3.5 + 4 |z|
//   matern32     RN(-0.5 e):                          2.5 + 2 s                                                = 2.5 + 2 s
//   matern52     RN(RN(RN(s + 1) e) RN(-1/6)):        2.5 + 2 s + 2 s / (1 + s) + 0.5 + 0.5 + 0.25 + 0.5      = 6.25 + 4 s
//   spherical    RN(RN(RN(-0.75 t) RN(1 + s)) / s), t = 1 - s (exact for s >= 0.5, 2^-53 below):
//                0.5 + 0.5 + 0.5 + 0.5 + 0.5 + 2 c, c = 1 + s / (1 - s) + s / (1 + s)                        = 2.5 + 2 c
// (c grows as s -> 1, where the derivative itself goes to 0 and its absolute error with it.)  Each summed term adds
// the roundings of w W k' du^2 (3 products and one fma: < 2 units) to these.  The derivative bounds are asserted
// argument by argument by tests/test_gpu_kcov_lik_exact.py::test_derivative_per_argument (one pair of points per call,
// so each range component is a single term).  The full sums cancel near the optimum (W = alpha alpha' - A^-1), so
// tests/test_gpu_kcov_lik.py bounds each gradient component by 1e-11 S_theta, S_theta = 1/2 sum_ij |W_ij| |dA_ij / dtheta|,
// the conditioning of the sum.
// Cost: one kern_eval-sized evaluation plus the derivative (one more FP64 multiply, a division for the exponential and
// spherical kinds) and 2 + d FMAs per structure per entry: FP64-pipe bound, about 30 FP64 instructions per entry and
// structure.  Every partial sum has a fixed order (thread: rows in order; warp: a fixed xor tree; CTA: warps in order;
// then kcov_grad_reduce over the CTAs and the chunks), so the gradient is bit-reproducible.
constexpr int KG_TY = 4;          // threadIdx.y: row phases (a thread takes rows ty, ty + 4, .. of the tile)

struct KcovGrad {
    const double* u; int64_t n_pad, n;
    int nstruct;
    int kinds[GSI_MODEL_MAX_STRUCTURES];
    double betas[GSI_MODEL_MAX_STRUCTURES];
    const double* Z; int64_t ldz, j0, w;
    double* part;
};

// k(r2) exactly as kern_eval<kind> computes it, and dk / dr2 in the same scaled units
__device__ __forceinline__ double kern_value_deriv(int kind, double r2, double beta, const double* __restrict__ tab,
                                                   double& dk) {
    if (kind == GSI_KERNEL_GAUSSIAN) {
        const double e = fast_exp_neg(r2, tab);
        dk = -e;
        return e;
    }
    if (kind == GSI_KERNEL_POWERLAW) {
        const double v = exp(-beta * log1p(r2));
        dk = (-beta * v) / (1.0 + r2);
        return v;
    }
    const double s = fast_sqrt_pos(r2);
    if (kind == GSI_KERNEL_SPHERICAL) {
        const double t = 1.0 - s;
        dk = s < 1.0 ? (-0.75 * t) * (1.0 + s) / s : 0.0;      // -3/4 (1 - s)(1 + s) / s
        return s < 1.0 ? (0.5 * t) * t * (2.0 + s) : 0.0;
    }
    const double e = fast_exp_neg(s, tab);
    if (kind == GSI_KERNEL_EXPONENTIAL) {
        dk = (-0.5 * e) / s;                                    // -e^-s / (2 s)
        return e;
    }
    if (kind == GSI_KERNEL_MATERN32) {
        dk = -0.5 * e;                                          // -e^-s / 2
        return fma(s, e, e);
    }
    dk = ((s + 1.0) * e) * (-1.0 / 6.0);                        // -(1 + s) e^-s / 6
    return fmin(fma(r2, 1.0 / 3.0, s + 1.0) * e, 1.0);
}

// One CTA per KG_ROWS x KG_COLS tile of the chunk (rows from j0, chunk columns c = blockIdx.y * KG_COLS + threadIdx.x);
// tiles wholly above the diagonal write zero partials.  part[(blockIdx.y * gridDim.x + blockIdx.x) * KG_SLOTS + slot].
template <int DIM>
__global__ void __launch_bounds__(KG_COLS * KG_TY) kcov_grad_kernel(const __grid_constant__ KcovGrad a) {
    constexpr int UP = GSI_MODEL_MAX_STRUCTURES * DIM;            // row coordinates per point in shared memory
    __shared__ double etab[64];
    __shared__ double urow[KG_ROWS * UP];
    __shared__ double red[KG_COLS * KG_TY / 32][KG_SLOTS];
    const int tx = threadIdx.x, ty = threadIdx.y, tid = ty * KG_COLS + tx;
    const int ns = a.nstruct;
    const int64_t i0 = a.j0 + (int64_t)blockIdx.x * KG_ROWS;
    const int64_t c = (int64_t)blockIdx.y * KG_COLS + tx;
    const int64_t j = a.j0 + c;
    if (tid < 64) etab[tid] = kExp2Table[tid];
    for (int e = tid; e < KG_ROWS * ns * DIM; e += KG_COLS * KG_TY) {
        const int r = e / (ns * DIM), q = e - r * (ns * DIM), s = q / DIM, k = q - s * DIM;
        const int64_t gi = i0 + r < a.n ? i0 + r : a.n - 1;
        urow[r * UP + q] = a.u[(s * 3 + k) * a.n_pad + gi];
    }
    const int64_t jc = j < a.n ? j : a.n - 1;
    double uj[GSI_MODEL_MAX_STRUCTURES][DIM];
#pragma unroll
    for (int s = 0; s < GSI_MODEL_MAX_STRUCTURES; ++s)
#pragma unroll
        for (int k = 0; k < DIM; ++k) uj[s][k] = s < ns ? a.u[(s * 3 + k) * a.n_pad + jc] : 0.0;
    double acc[KG_SLOTS];
#pragma unroll
    for (int q = 0; q < KG_SLOTS; ++q) acc[q] = 0.0;
    __syncthreads();
    const bool col_ok = c < a.w && j < a.n;
    if (a.j0 + (int64_t)blockIdx.y * KG_COLS <= i0 + KG_ROWS - 1) {      // the tile reaches the lower triangle
        for (int r = ty; r < KG_ROWS; r += KG_TY) {
            const int64_t i = i0 + r;
            if (!col_ok || i < j || i >= a.n) continue;
            const double wv = -a.Z[i * a.ldz + c];
            const double wt = i == j ? wv : 2.0 * wv;
            const double* ur = urow + r * UP;
#pragma unroll
            for (int s = 0; s < GSI_MODEL_MAX_STRUCTURES; ++s) {
                if (s < ns) {
                    const int kind = a.kinds[s];
                    double du[DIM];
                    double r2 = kind_takes_sqrt_runtime(kind) ? 1e-300 : 0.0;
#pragma unroll
                    for (int k = 0; k < DIM; ++k) {                       // model_value's r2 chain, row minus column
                        du[k] = ur[s * DIM + k] - uj[s][k];
                        r2 = fma(du[k], du[k], r2);
                    }
                    double dk;
                    const double kv = kern_value_deriv(kind, r2, a.betas[s], etab, dk);
                    acc[4 * s] = fma(wt, kv, acc[4 * s]);
                    const double g = wt * dk;
#pragma unroll
                    for (int k = 0; k < DIM; ++k) acc[4 * s + 1 + k] = fma(g, du[k] * du[k], acc[4 * s + 1 + k]);
                }
            }
            if (i == j) acc[KG_SLOTS - 1] += wv;
        }
    }
    const int warp = tid >> 5, lane = tid & 31;
#pragma unroll
    for (int q = 0; q < KG_SLOTS; ++q) {
        double v = acc[q];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) red[warp][q] = v;
    }
    __syncthreads();
    if (tid < KG_SLOTS) {
        double v = 0.0;
#pragma unroll
        for (int w = 0; w < KG_COLS * KG_TY / 32; ++w) v += red[w][tid];
        a.part[((int64_t)blockIdx.y * gridDim.x + blockIdx.x) * KG_SLOTS + tid] = v;
    }
}

// out[slot] = sum over the nparts rows of part: lane l adds rows l, l + 32, .. in order, then a fixed xor tree
__global__ void __launch_bounds__(32 * KG_SLOTS) kcov_grad_reduce_kernel(const double* __restrict__ part, int64_t nparts,
                                                                         double* __restrict__ out) {
    const int lane = threadIdx.x, slot = threadIdx.y;
    double v = 0.0;
    for (int64_t k = lane; k < nparts; k += 32) v += part[k * KG_SLOTS + slot];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) out[slot] = v;
}

int64_t kcov_grad(gsi_op* op, const double* Z, int64_t ldz, int64_t j0, int64_t w, double* part) {
    gsi_ctx* ctx = op->ctx;
    KcovGrad a;
    std::memset(&a, 0, sizeof(a));
    a.u = op->ucoords; a.n_pad = op->n_pad; a.n = op->n;
    const bool model = op->kind == KC_KIND_MODEL;
    a.nstruct = model ? op->nstruct : 1;
    for (int s = 0; s < GSI_MODEL_MAX_STRUCTURES; ++s) {
        a.kinds[s] = model ? op->mkinds[s] : op->kind;
        a.betas[s] = model ? op->mbetas[s] : op->beta;
    }
    a.Z = Z; a.ldz = ldz; a.j0 = j0; a.w = w; a.part = part;
    const int64_t rows = op->n - j0, cols = w < rows ? w : rows;
    const dim3 grid((unsigned)((rows + KG_ROWS - 1) / KG_ROWS), (unsigned)((cols + KG_COLS - 1) / KG_COLS));
    if (op->dim <= 2) kcov_grad_kernel<2><<<grid, dim3(KG_COLS, KG_TY), 0, ctx->stream>>>(a);
    else kcov_grad_kernel<3><<<grid, dim3(KG_COLS, KG_TY), 0, ctx->stream>>>(a);
    GSI_CUDA(cudaGetLastError());
    count_launch(ctx);
    return (int64_t)grid.x * grid.y;
}

void kcov_grad_reduce(gsi_ctx* ctx, const double* part, int64_t nparts, double* out) {
    kcov_grad_reduce_kernel<<<1, dim3(32, KG_SLOTS), 0, ctx->stream>>>(part, nparts, out);
    GSI_CUDA(cudaGetLastError());
    count_launch(ctx);
}

}  // namespace gsi
