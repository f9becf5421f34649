// Fused per-layer row pass of the MFDGP (forward and backward) for sm_100a.
//
// Replaces, for one sparse-GP layer and a batch of R rows, what the reference reaches through
//   MFDGPHiddenLayer.__call__        (mobocmf/layers/mfdgp_hidden_layer.py:245-286)  sample propagation + concat
//   MFDGPHiddenLayer.forward         (mobocmf/layers/mfdgp_hidden_layer.py:232-243)  K(Z_l, X), diag K(X, X)
//   UnwhitenedVariationalStrategy.forward [upstream gpytorch]                        mean / variance of q(f)
// and the autograd backward of those (loss.backward(), mobocmf/util/blackbox_mfdgp_fitter.py:168).
//
// Per row x (with propagated input f) and the per-step operators W = L_p^-1, H = W L_q, beta = W m:
//   k = K(Z_l, x);  t = W k;  u = H^T t;  mu = beta.t;  v = clamp(k_xx - |t|^2, 0) + |u|^2   (train; eval: no clamp)
// which is the reference's  mean = m^T P^-1 k,  var = clamp(k_xx - |L_p^-1 k|^2, 0) + |L_q^T P^-1 k|^2.
// K(Z_l, X) lives only in shared memory (it is written to HBM only when the backward needs it).
//
// Tile: 32 rows x MP inducing points per CTA, 8 warps, two CTAs per SM (so that one CTA's covariance build on the
// DFMA side overlaps the other's products; DMMA and DFMA share the FP64 pipe, profiles/r01c_fp64_probe_*.log, so
// the gain is in the barriers and pipeline drains, not in the arithmetic).  The two triangular M x M products run on
// the DMMA pipe (mma.sync.m8n8k4.f64); each warp owns two 16-row slabs (p, ns-1-p) of the triangular operator so
// that the triangular work is balanced, and streams its slab of the operator from L2 straight into A fragments.
#include "common.cuh"

namespace mobo {

// ---- optional per-phase cycle accounting of the row kernels (tools/row_bench.cu builds with -DROW_TIMING) ----
#ifdef ROW_TIMING
__device__ unsigned long long row_times[3][512][16];
// RT_DECL: thread 0 of the CTA keeps the clock; RT_DECL_ROLE(cond): the thread for which cond holds (one per role of the
// warp-specialised kernel, each with its own accumulators in shared memory)
#define RT_DECL_ROLE(cond) __shared__ unsigned long long rt_acc_[3][16]; const bool rt_me = (cond); unsigned long long rt_prev = clock64(); \
  if (threadIdx.x < 48) rt_acc_[threadIdx.x / 16][threadIdx.x % 16] = 0ull;
#define RT_DECL RT_DECL_ROLE(threadIdx.x == 0)
#define RT_TICKW(w, k) do { if (rt_me) { const unsigned long long n_ = clock64(); rt_acc_[w][k] += n_ - rt_prev; rt_prev = n_; } } while (0)
#define RT_TICK(k) RT_TICKW(0, k)
#define RT_FLUSH(which) do { if (rt_me && blockIdx.x < 512) for (int k_ = 0; k_ < 16; ++k_) row_times[which][blockIdx.x][k_] = rt_acc_[which][k_]; } while (0)
#else
#define RT_DECL
#define RT_DECL_ROLE(cond)
#define RT_TICK(k)
#define RT_TICKW(w, k)
#define RT_FLUSH(which)
#endif

constexpr int TR = 32;             // rows per tile
constexpr int ROW_THREADS = 256;   // 8 warps: one per pair of 16-row operator slabs at MP = 256
constexpr int ROW_WARPS = ROW_THREADS / 32;
constexpr int NHALF = TR / 32;     // 32-column groups of the tile; warps = NHALF x (MP / 32) slab pairs
constexpr int ROW_CTAS_PER_SM = 2; // two CTAs per SM fill each other's phase boundaries (K build <-> DMMA products)
constexpr int MAX_MP = 256;        // slab scheme: (MP/32) warp pairs <= 8
constexpr int NCH_MAX = MAX_MP / 32;

struct RowArgs {
  int kind, d, M, MP;
  const double* Zx;        // M x d inducing inputs (x part)
  const double* zf;        // M: propagated column of the inducing inputs (kind 1): m_{l-1}
  const double* theta;     // constrained kernel hyper-parameters
  const double* ops;       // operator buffer (common.cuh)
  const double* x;         // n x d
  int xrep;                // row r reads x[r / xrep]
  const double* mu_prev;   // previous layer's q(f) moments; row r reads [r / prep]
  const double* var_prev;
  int prep;
  const double* eps;       // normals; row r reads eps[r % eps_mod]
  long long eps_mod;
  const double* f_direct;  // optional explicit propagated input (overrides mu_prev/var_prev/eps)
  long long R;
  int training;            // 1: clamp(k_xx - q, 0) branch; 0: eval branch
  // forward outputs
  double* mu;
  double* var;
  double* craw;            // optional: k_xx - |t|^2 before the clamp (mask for the backward)
  unsigned int* clamp_count; // optional: number of rows whose k_xx - |t|^2 was clamped
  double* Tsave;           // optional row-major [R][MP]: whitened rows t = W k
  double* Usave;           // optional row-major [R][MP]: u = H^T t
  // backward inputs / outputs
  const double* dmu;
  const double* dvar;
  double* dk;              // scratch [R][MP]: d loss / d K(z_j, row r), written by the product kernel, read by kgrad
  double* df;              // R: d loss / d f_r   (kind 1)
  double* dxrow;           // optional R x d: d loss / d x of each row
  double* part_theta;      // [grid][kMaxTheta]
  double* part_zf;         // [grid][MP]
  int want_param_grads;
  int want_x_grads;
  int sm_reserve;          // backward product kernel: SMs to leave free for concurrent side-stream kernels
};

// Covariance parameters in the form the row kernels evaluate them: every exponential is 2^y with the -1/2 log2(e) / l^2
// factors folded into the coefficients and log2 of the amplitude folded into the exponent, so
//   kind 0: k = 2^(la1 + sum_c c1_c (x_c - z_c)^2)
//   kind 1: k = 2^(la1 + sum_c c1_c D_c^2) * (v f f' + 2^(laf + cf (f - f')^2)) + 2^(la2 + sum_c c2_c D_c^2)
struct KernFast {
  int kind, d;
  double la1, laf, la2, vlin, cf, ilf;
  double a1, af, a2, lf;
  double c1[kMaxD], c2[kMaxD];     // -0.5 log2(e) / l^2
  double2 cc[kMaxD];               // (c1, c2) interleaved: one 16-byte broadcast load per dimension
  double il1[kMaxD], il2[kMaxD];   // 1 / l^2
};

constexpr double kExp2Magic = 6755399441055744.0;   // 1.5 * 2^52: adding it rounds to the nearest integer
constexpr int kExp2TabBits = 8, kExp2Tab = 1 << kExp2TabBits;

// 2^y to ~1.5 ulp: y = n / 256 + r, |r| <= 1/512; 2^y = 2^(n >> 8) * tab[n & 255] * p4(r) (truncation 3.8e-17).
// 8 FP64-pipe operations against ~22 for libdevice exp(): the row kernels evaluate up to 3 of these per (row, inducing
// point) pair, DFMA shares the FP64 pipe with the DMMA products (profiles/r01c_fp64_probe_*.log), and next to warps
// that stream DMMAs every FP64 instruction of another warp waits for an arbitration slot (row_fwd_ws_kernel), so the
// count matters more than the pipe time: the clamp is done on the integer pipe (arguments below -1000 give 0 for every
// purpose here; they are never NaN), and a 256-entry table buys one polynomial degree.
__device__ __forceinline__ double exp2_tab(double y, const double* __restrict__ tab) {
  // y < -1000 (sign bit set, magnitude above 1000.0 = 0x408F4000_00000000): clamp, comparing the high word as unsigned
  if ((unsigned)__double2hiint(y) > 0xC08F4000u) y = -1000.0;
  const double t = fma(y, (double)kExp2Tab, kExp2Magic);
  const int n = __double2loint(t);
  const double nf = t - kExp2Magic;
  const double r = fma(nf, -1.0 / kExp2Tab, y);         // exact
  double p = 9.618129107628477e-3;                       // ln2^4 / 4!
  p = fma(p, r, 5.550410866482158e-2);                   // ln2^3 / 3!
  p = fma(p, r, 2.402265069591007e-1);                   // ln2^2 / 2!
  p = fma(p, r, 6.931471805599453e-1);                   // ln2
  p = fma(p, r, 1.0);
  const double res = tab[n & (kExp2Tab - 1)] * p;
  return __hiloint2double(__double2hiint(res) + ((n >> kExp2TabBits) << 20), __double2loint(res));
}
__device__ __forceinline__ void fill_exp2_tab(double* tab, int tid, int nthreads) {
  for (int i = tid; i < kExp2Tab; i += nthreads) tab[i] = exp2((double)i / kExp2Tab);
}

constexpr int RPW = 4;   // tile rows per warp in the covariance phases (independent exponent chains per thread)

// Shared state of the covariance phases for NW warps (NW * RPW rows per tile).  BWD adds the per-warp accumulators.
template <int NW, bool BWD>
struct CovSmem {
  static constexpr int WARPS = NW, ROWS = NW * RPW, THREADS = NW * 32;
  KernFast kf;
  double e2tab[kExp2Tab];
  double xs[ROWS][kMaxD];
  double fs[ROWS];
  double kxx[ROWS];
  double dvar[ROWS], mask[ROWS];
  double zsT[kMaxD][MAX_MP];
  double zfs[MAX_MP];
  double acc_zf[BWD ? NW : 1][BWD ? MAX_MP : 1];   // backward: per-warp d zf accumulators
  double acc_th[BWD ? NW : 1][kMaxTheta];   // backward: per-warp d theta accumulators (scalars | l1 | l2)
};

struct RowSmem : CovSmem<ROW_WARPS, false> {
  double red[3][NCH_MAX][TR];     // per warp-pair partial column sums: q1, mu, q2
};
static_assert(ROW_WARPS * RPW == TR, "the covariance build maps RPW rows to each warp of the row tile");

__device__ __forceinline__ double* tile_ptr(unsigned char* smem) {
  return reinterpret_cast<double*>(smem + ((sizeof(RowSmem) + 127) / 128) * 128);
}

constexpr int FWD_NST = 4, BWD_NST = 4;   // A-fragment ring depth (k-steps) of the forward / backward product kernels
// (frag_group below is written for exactly 4 slots: the fragment of k-step q lives in slot q & 3)
__host__ __device__ inline size_t tile_bytes(int MP) { return (size_t)TR * (MP + 4) * sizeof(double); }
__host__ inline size_t row_smem_bytes(int MP) {
  return ((sizeof(RowSmem) + 127) / 128) * 128 + tile_bytes(MP) + (size_t)ROW_WARPS * FWD_NST * 32 * sizeof(double2);
}

// 16-byte asynchronous global -> shared copy (L2 only) and its group bookkeeping.  The "memory" clobbers keep the
// compiler from moving shared-memory reads across the wait.
__device__ __forceinline__ void cp_async16_cg(void* smem, const void* gmem) {
  const unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit_group() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ void zero_acc(double (&acc)[2][2][4][2]) {
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int b = 0; b < 2; ++b)
#pragma unroll
      for (int c = 0; c < 4; ++c) { acc[a][b][c][0] = 0.0; acc[a][b][c][1] = 0.0; }
}

// acc fragment (sl, ib, ct, e) <-> operator row i = 16 s + 8 ib + g, tile column r = 32 half + 8 ct + 2 t + e
__device__ __forceinline__ void store_acc_to_tile(const double (&acc)[2][2][4][2], double* Ks, int ldb, int sA,
                                                  int sB, int half, int lane) {
  const int g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int sl = 0; sl < 2; ++sl) {
    const int s = sl == 0 ? sA : sB;
#pragma unroll
    for (int ib = 0; ib < 2; ++ib)
#pragma unroll
      for (int ct = 0; ct < 4; ++ct)
#pragma unroll
        for (int e = 0; e < 2; ++e)
          Ks[(size_t)(32 * half + 8 * ct + 2 * t + e) * ldb + 16 * s + 8 * ib + g] = acc[sl][ib][ct][e];
  }
}

// accumulator fragments -> row-major [R][MP] rows in global memory (row r of the tile, operator index i): per store
// instruction a warp writes 4 rows x 64 contiguous bytes (full 32-byte sectors); stores are fire-and-forget
__device__ __forceinline__ void store_acc_rows(const double (&acc)[2][2][4][2], double* __restrict__ dst, long long row0,
                                               int nvalid, int MP, int sA, int sB, int half, int lane) {
  const int g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int sl = 0; sl < 2; ++sl) {
    const int s = sl == 0 ? sA : sB;
#pragma unroll
    for (int ct = 0; ct < 4; ++ct)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int r = 32 * half + 8 * ct + 2 * t + e;
        if (r < nvalid) {
          double* p = dst + (size_t)(row0 + r) * MP + 16 * s + g;
          p[0] = acc[sl][0][ct][e];
          p[8] = acc[sl][1][ct][e];
        }
      }
  }
}

__device__ inline void load_kern_fast(KernFast& kf, int kind, int d, const double* __restrict__ theta) {
  const double nhl2e = -0.5 * 1.4426950408889634074;     // -1/2 log2(e)
  kf.kind = kind; kf.d = d;
  for (int c = 0; c < kMaxD; ++c) { kf.c1[c] = 0.0; kf.c2[c] = 0.0; kf.il1[c] = 0.0; kf.il2[c] = 0.0; }
  if (kind == 0) {
    kf.a1 = theta[0]; kf.la1 = log2(kf.a1);
    kf.vlin = 0.0; kf.af = 0.0; kf.a2 = 0.0; kf.laf = -INFINITY; kf.la2 = -INFINITY; kf.cf = 0.0; kf.ilf = 0.0; kf.lf = 1.0;
    for (int c = 0; c < d; ++c) { const double l = theta[1 + c]; kf.il1[c] = 1.0 / (l * l); kf.c1[c] = nhl2e * kf.il1[c]; }
  } else {
    kf.a1 = theta[0]; kf.vlin = theta[1]; kf.af = theta[2]; kf.lf = theta[3]; kf.a2 = theta[4];
    kf.la1 = log2(kf.a1); kf.laf = log2(kf.af); kf.la2 = log2(kf.a2);
    kf.ilf = 1.0 / (kf.lf * kf.lf); kf.cf = nhl2e * kf.ilf;
    for (int c = 0; c < d; ++c) {
      const double l1 = theta[5 + c], l2 = theta[5 + d + c];
      kf.il1[c] = 1.0 / (l1 * l1); kf.il2[c] = 1.0 / (l2 * l2);
      kf.c1[c] = nhl2e * kf.il1[c]; kf.c2[c] = nhl2e * kf.il2[c];
    }
  }
  for (int c = 0; c < kMaxD; ++c) kf.cc[c] = make_double2(kf.c1[c], kf.c2[c]);
}

template <class SM>
__device__ __forceinline__ void load_inducing(const RowArgs& a, SM& sm) {
  const int tid = threadIdx.x;
  if (tid == 0) load_kern_fast(sm.kf, a.kind, a.d, a.theta);
  fill_exp2_tab(sm.e2tab, tid, SM::THREADS);
  for (int idx = tid; idx < a.MP * a.d; idx += SM::THREADS) {
    const int j = idx / a.d, c = idx - j * a.d;
    sm.zsT[c][j] = j < a.M ? a.Zx[(size_t)j * a.d + c] : 0.0;
  }
  for (int j = tid; j < a.MP; j += SM::THREADS) sm.zfs[j] = (a.kind == 1 && j < a.M) ? a.zf[j] : 0.0;
}

// K(Z_l, rows of the tile) into shared memory: Ks[r][j].  Warp <-> RPW rows, lane <-> inducing point of a 32-chunk;
// the inducing point stays in registers while the warp's rows (kept in registers too) run past it, which gives RPW
// independent exponent chains per thread.
// SHX: the warp's RPW rows are MC samples of the same point (same x, different propagated f): the two x-kernels
// a1 E1 and a2 E2 are then evaluated once per inducing point instead of once per row (the S-sample tiling of
// models/mfdgp.py:248 makes this the common case for layers >= 1).
template <int KIND, int D, bool SHX>
__device__ __forceinline__ void build_k_tile(const RowSmem& sm, double* __restrict__ Ks, int ldb, int M, int MP,
                                             int nvalid, int warp, int lane) {
  const KernFast& kf = sm.kf;
  const double* tab = sm.e2tab;
  const int rbase = warp * RPW;
  constexpr int NX = SHX ? 1 : RPW;
  double x[NX][D], f[RPW], vf[RPW], c1[D], c2[D];
#pragma unroll
  for (int i = 0; i < NX; ++i)
#pragma unroll
    for (int c = 0; c < D; ++c) x[i][c] = sm.xs[rbase + i][c];
#pragma unroll
  for (int i = 0; i < RPW; ++i) { f[i] = sm.fs[rbase + i]; vf[i] = kf.vlin * f[i]; }
#pragma unroll
  for (int c = 0; c < D; ++c) { c1[c] = kf.c1[c]; c2[c] = kf.c2[c]; }
  const double la1 = kf.la1, la2 = kf.la2, laf = kf.laf, cf = kf.cf;
  for (int ch = 0; ch < MP / 32; ++ch) {
    const int j = 32 * ch + lane;
    double z[D];
#pragma unroll
    for (int c = 0; c < D; ++c) z[c] = sm.zsT[c][j];
    const double zf = sm.zfs[j];
    const bool jok = j < M;
    double s1 = 0.0, s2 = 0.0;
#pragma unroll
    for (int i = 0; i < RPW; ++i) {
      if (!SHX || i == 0) {
        double D1 = la1, D2 = la2;
#pragma unroll
        for (int c = 0; c < D; ++c) {
          const double df = x[SHX ? 0 : i][c] - z[c];
          const double d2 = df * df;
          D1 = fma(d2, c1[c], D1);
          if (KIND == 1) D2 = fma(d2, c2[c], D2);
        }
        s1 = exp2_tab(D1, tab);
        if (KIND == 1) s2 = exp2_tab(D2, tab);
      }
      double k;
      if (KIND == 0) {
        k = s1;
      } else {
        const double dff = f[i] - zf;
        const double Ef = exp2_tab(fma(dff * dff, cf, laf), tab);
        k = fma(s1, fma(vf[i], zf, Ef), s2);
      }
      Ks[(size_t)(rbase + i) * ldb + j] = (jok && rbase + i < nvalid) ? k : 0.0;
    }
  }
}

template <int KIND, bool SHX>
__device__ __forceinline__ void build_k_tile_d(const RowSmem& sm, double* Ks, int ldb, int M, int MP, int nvalid,
                                               int warp, int lane) {
  switch (sm.kf.d) {
    case 1: build_k_tile<KIND, 1, SHX>(sm, Ks, ldb, M, MP, nvalid, warp, lane); break;
    case 2: build_k_tile<KIND, 2, SHX>(sm, Ks, ldb, M, MP, nvalid, warp, lane); break;
    case 3: build_k_tile<KIND, 3, SHX>(sm, Ks, ldb, M, MP, nvalid, warp, lane); break;
    case 4: build_k_tile<KIND, 4, SHX>(sm, Ks, ldb, M, MP, nvalid, warp, lane); break;
    case 5: build_k_tile<KIND, 5, SHX>(sm, Ks, ldb, M, MP, nvalid, warp, lane); break;
    case 6: build_k_tile<KIND, 6, SHX>(sm, Ks, ldb, M, MP, nvalid, warp, lane); break;
    case 7: build_k_tile<KIND, 7, SHX>(sm, Ks, ldb, M, MP, nvalid, warp, lane); break;
    default: build_k_tile<KIND, 8, SHX>(sm, Ks, ldb, M, MP, nvalid, warp, lane); break;
  }
}

// true when the RPW rows of this warp read the same x row (row r reads x[r / xrep])
__device__ __forceinline__ bool warp_rows_share_x(const RowArgs& a, long long row0, int warp) {
  const long long r0 = row0 + (long long)warp * RPW;
  return a.xrep > 1 && r0 / a.xrep == (r0 + RPW - 1) / a.xrep;
}

// The general covariance build of the forward kernel (layer 0, and upper layers whose rows do not share x in large
// groups: single-sample training, small S).  Kept out of line: its per-dimension register arrays (up to 8 dimensions
// x 4 rows) would otherwise set the register allocation of the whole kernel, whose DMMA products need none of them.
__device__ __noinline__ void build_k_tile_generic(const RowArgs& a, const RowSmem& sm, double* Ks, int ldb, unsigned row0,
                                                  int nvalid, int warp, int lane) {
  if (a.kind == 0) build_k_tile_d<0, false>(sm, Ks, ldb, a.M, a.MP, nvalid, warp, lane);
  else if (warp_rows_share_x(a, row0, warp)) build_k_tile_d<1, true>(sm, Ks, ldb, a.M, a.MP, nvalid, warp, lane);
  else build_k_tile_d<1, false>(sm, Ks, ldb, a.M, a.MP, nvalid, warp, lane);
}

// ---- A-fragment stream of the forward kernel ------------------------------------------------------------------------
// A tile's two triangular products are four "segments" per warp (W slab A, W slab B, H^T slab A, H^T slab B), each a run
// of k-steps whose A fragments this lane streams from L2 through its private cp.async ring.  The ring never drains: the
// last k-steps of a segment already fetch the first fragments of the NEXT segment (and the last segment of a tile those
// of the next tile's first), so a segment starts with its first NST - 1 fragments in flight instead of paying an L2
// round trip (4 per tile in the first version).  Every segment is a multiple of NST = 4 k-steps, so the slot of k-step q
// is q & 3 in every segment.  One k-step: 1 fragment copy issued, 1 fragment read, 4 B loads, 8 DMMAs.
// The 16 x 16 diagonal block of a slab is half zeros (the operators are triangular): its two k-steps that only touch
// the zero half of one 8-row group skip that group's DMMAs (LOWER: rows 0-7 x k 8-15, the slab's last k-steps; UPPER:
// rows 8-15 x k 0-7, its first ones): 16 of a slab pair's 544 DMMAs per product.
constexpr int SKIP_NONE = 0, SKIP_LOW_DIAG = 1, SKIP_UP_DIAG = 2;

template <int SKIP, bool CHAIN>
__device__ __forceinline__ void frag_group(double (&acc)[2][4][2], const double2* __restrict__ ap,
                                           const double2* __restrict__ nextp, const double* __restrict__ bp,
                                           size_t ct_stride, double2* slot) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    // k-step j + 3 of this run: in this segment, or (CHAIN: the segment's last group) fragment j - 1 of the next one
    const double2* src = (CHAIN && j >= 1) ? nextp + (j - 1) * 32 : ap + (j + 3) * 32;
    cp_async16_cg(slot + ((j + 3) & 3) * 32, src);
    cp_async_commit_group();
    cp_async_wait_group<3>();
    const double2 av = slot[j * 32];
    const bool do0 = !(SKIP == SKIP_LOW_DIAG && j >= 2), do1 = !(SKIP == SKIP_UP_DIAG && j < 2);
#pragma unroll
    for (int ct = 0; ct < 4; ++ct) {
      const double b = bp[ct * ct_stride + 4 * j];
      if (do0) dmma884(acc[0][ct][0], acc[0][ct][1], av.x, b);
      if (do1) dmma884(acc[1][ct][0], acc[1][ct][1], av.y, b);
    }
  }
}

// one segment: acc(16 rows x 32 cols) += A[slab s, its triangular k-range] * B.  The ring must already hold (or have in
// flight) the segment's first 3 fragments; on return it holds those of the segment starting at `nextp`.
template <bool UPPER>
__device__ __forceinline__ void frag_segment(double (&acc)[2][4][2], const double* __restrict__ Af, int MP, const double* Bs,
                                             int ldb, int s, int half, int lane, double2* ring,
                                             const double2* __restrict__ nextp) {
  const int g = lane >> 2, t = lane & 3;
  const int kbeg = UPPER ? 16 * s : 0;
  const int nq = (UPPER ? MP - 16 * s : 16 * (s + 1)) >> 2;        // k-steps: a multiple of 4
  double2* slot = ring + lane;
  const double2* ap = reinterpret_cast<const double2*>(Af) + ((size_t)s * (MP >> 2) + (kbeg >> 2)) * 32 + lane;
  const double* bp = Bs + (size_t)(32 * half + g) * ldb + t + kbeg;
  const size_t ct_stride = (size_t)8 * ldb;
  if (UPPER) {
    if (nq == 4) { frag_group<SKIP_UP_DIAG, true>(acc, ap, nextp, bp, ct_stride, slot); return; }
    frag_group<SKIP_UP_DIAG, false>(acc, ap, nextp, bp, ct_stride, slot);
    ap += 4 * 32; bp += 16;
    for (int q0 = 4; q0 < nq - 4; q0 += 4) {
      frag_group<SKIP_NONE, false>(acc, ap, nextp, bp, ct_stride, slot);
      ap += 4 * 32; bp += 16;
    }
    frag_group<SKIP_NONE, true>(acc, ap, nextp, bp, ct_stride, slot);
  } else {
    for (int q0 = 0; q0 < nq - 4; q0 += 4) {
      frag_group<SKIP_NONE, false>(acc, ap, nextp, bp, ct_stride, slot);
      ap += 4 * 32; bp += 16;
    }
    frag_group<SKIP_LOW_DIAG, true>(acc, ap, nextp, bp, ct_stride, slot);
  }
}

__device__ __forceinline__ const double2* frag_start(const double* Af, int MP, int s, bool upper, int lane) {
  return reinterpret_cast<const double2*>(Af) + ((size_t)s * (MP >> 2) + (upper ? 4 * s : 0)) * 32 + lane;
}

// Forward row pass of the rows that are not MC samples of few points (layer 0, single-sample training, small S; the
// others go to row_fwd_ws_kernel below).  Per 32-row tile (two CTAs per SM, 8 warps each):
//   row data (prefetched one tile ahead into registers) and x -> shared;  K(Z_l, rows) into the tile buffer
//   (build_k_tile_generic);  t = W k (DMMA);  t -> tile buffer (bulk-stored to Tsave from there);  u = H^T t (DMMA),
//   stored from the accumulators;  mean / variance.
__global__ void __launch_bounds__(ROW_THREADS, ROW_CTAS_PER_SM) row_fwd_kernel(const __grid_constant__ RowArgs a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  RowSmem& sm = *reinterpret_cast<RowSmem*>(smem_raw);
  double* Ks = tile_ptr(smem_raw);
  const int MP = a.MP, ldb = MP + 4;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double2* ring = reinterpret_cast<double2*>(reinterpret_cast<unsigned char*>(Ks) + tile_bytes(MP)) + warp * FWD_NST * 32;
  const int half = warp % NHALF, p = warp / NHALF;
  const int npairs = MP / 32, ns = MP / 16;
  const bool active = p < npairs;
  const int sA = p, sB = ns - 1 - p;
  const int g = lane >> 2, t = lane & 3;
  const double* W = a.ops + ops_block(MP, OPS_WF);
  const double* G = a.ops + ops_block(MP, OPS_HTF);
  const double* beta = a.ops + ops_beta(MP);

  RT_DECL
  load_inducing(a, sm);
  double bi[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
  if (active) {
#pragma unroll
    for (int sl = 0; sl < 2; ++sl)
#pragma unroll
      for (int ib = 0; ib < 2; ++ib) bi[sl][ib] = __ldg(beta + 16 * (sl == 0 ? sA : sB) + 8 * ib + g);
  }

  // ---- row data, prefetched one tile ahead: threads 0..31 hold a row's (mean, variance, normal) or its direct f ----
  // (row indices are 32-bit here: the launcher refuses R >= 2^31, callers chunk long before that)
  const unsigned R = (unsigned)a.R, ntiles = (R + TR - 1) / TR;
  const unsigned uxrep = (unsigned)a.xrep, uprep = (unsigned)a.prep;
  const unsigned ueps = a.eps_mod >= a.R ? 0u : (unsigned)a.eps_mod;       // 0: eps index == row
  double pf_a = 0.0, pf_b = 1.0, pf_c = 0.0;
  auto prefetch = [&](unsigned tile) {
    if (tile >= ntiles || tid >= TR) return;
    const unsigned row = tile * TR + tid;
    pf_a = 0.0; pf_b = 1.0; pf_c = 0.0;
    if (row < R && a.kind == 1) {
      if (a.f_direct) {
        pf_a = a.f_direct[row];
      } else {
        const unsigned pr = row / uprep;
        pf_a = a.mu_prev[pr];
        pf_b = a.var_prev[pr];
        pf_c = a.eps[ueps ? row % ueps : row];
      }
    }
  };
  prefetch(blockIdx.x);
  // ring: the first 3 fragments of the first segment (every later segment is primed by its predecessor)
  if (active) {
    const double2* first = frag_start(W, MP, sA, false, lane);
#pragma unroll
    for (int j = 0; j < 3; ++j) { cp_async16_cg(ring + lane + j * 32, first + j * 32); cp_async_commit_group(); }
  }
  __syncthreads();
  RT_TICK(0);

  for (unsigned tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const unsigned row0 = tile * TR;
    const int nvalid = (int)min((unsigned)TR, R - row0);
    // ---- this tile's rows: registers -> shared ----
    if (tid < TR) {
      double f = 0.0;
      if (tid < nvalid && a.kind == 1) f = a.f_direct ? pf_a : pf_a + sqrt(fmax(pf_b, kMinVariance)) * pf_c;
      sm.fs[tid] = f;
      sm.kxx[tid] = sm.kf.kind == 0 ? sm.kf.a1 : sm.kf.a1 * (sm.kf.vlin * f * f + sm.kf.af) + sm.kf.a2;
    }
    for (int idx = tid; idx < TR * a.d; idx += ROW_THREADS) {
      const int r = idx / a.d, c = idx - r * a.d;
      sm.xs[r][c] = r < nvalid ? a.x[(size_t)((row0 + r) / uxrep) * a.d + c] : 0.0;
    }
    __syncthreads();
    prefetch(tile + gridDim.x);         // lands during the products
    RT_TICK(1);
    // ---- K(Z_l, rows) into shared memory ----
    build_k_tile_generic(a, sm, Ks, ldb, row0, nvalid, warp, lane);
    RT_TICK(2);
    __syncthreads();
    RT_TICK(3);
    // ---- t = W k ----
    double acc[2][2][4][2];
    zero_acc(acc);
    if (active) {
      frag_segment<false>(acc[0], W, MP, Ks, ldb, sA, half, lane, ring, frag_start(W, MP, sB, false, lane));
      frag_segment<false>(acc[1], W, MP, Ks, ldb, sB, half, lane, ring, frag_start(G, MP, sA, true, lane));
      RT_TICK(4);
      double pq[4][2], pm[4][2];
#pragma unroll
      for (int ct = 0; ct < 4; ++ct)
#pragma unroll
        for (int e = 0; e < 2; ++e) { pq[ct][e] = 0.0; pm[ct][e] = 0.0; }
#pragma unroll
      for (int sl = 0; sl < 2; ++sl)
#pragma unroll
        for (int ib = 0; ib < 2; ++ib) {
#pragma unroll
          for (int ct = 0; ct < 4; ++ct)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const double v = acc[sl][ib][ct][e];
              pq[ct][e] = fma(v, v, pq[ct][e]);
              pm[ct][e] = fma(bi[sl][ib], v, pm[ct][e]);
            }
        }
#pragma unroll
      for (int ct = 0; ct < 4; ++ct)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          double q = pq[ct][e], m = pm[ct][e];
#pragma unroll
          for (int o = 4; o < 32; o <<= 1) {
            q += __shfl_xor_sync(0xffffffffu, q, o);
            m += __shfl_xor_sync(0xffffffffu, m, o);
          }
          if (g == 0) {
            sm.red[0][p][32 * half + 8 * ct + 2 * t + e] = q;
            sm.red[1][p][32 * half + 8 * ct + 2 * t + e] = m;
          }
        }
    }
    RT_TICK(5);
    __syncthreads();   // every warp is done reading K
    RT_TICK(6);
    if (active) store_acc_to_tile(acc, Ks, ldb, sA, sB, half, lane);
    __syncthreads();
    RT_TICK(7);
    // whitened rows t = W k, row-major [R][MP], for the backward (SYRK statistics and dt): one bulk (TMA engine)
    // shared -> global copy per row, issued by warp 0, instead of 32 shared loads + 32 global stores per thread; the
    // copies read the tile while the second product does, and are waited for before the tile is rebuilt
    if (a.Tsave && warp == 0) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // generic writes of t -> async-proxy reads
      if (lane < nvalid)
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(
                         a.Tsave + (size_t)(row0 + (unsigned)lane) * MP),
                     "r"((unsigned)__cvta_generic_to_shared(Ks + (size_t)lane * ldb)),
                     "r"((unsigned)(MP * sizeof(double))) : "memory");
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
    // ---- u = H^T t ----
    if (active) {
      zero_acc(acc);
      frag_segment<true>(acc[0], G, MP, Ks, ldb, sA, half, lane, ring, frag_start(G, MP, sB, true, lane));
      frag_segment<true>(acc[1], G, MP, Ks, ldb, sB, half, lane, ring, frag_start(W, MP, sA, false, lane));
      RT_TICK(8);
#pragma unroll
      for (int ct = 0; ct < 4; ++ct)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          double q = 0.0;
#pragma unroll
          for (int sl = 0; sl < 2; ++sl)
#pragma unroll
            for (int ib = 0; ib < 2; ++ib) q = fma(acc[sl][ib][ct][e], acc[sl][ib][ct][e], q);
#pragma unroll
          for (int o = 4; o < 32; o <<= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
          if (g == 0) sm.red[2][p][32 * half + 8 * ct + 2 * t + e] = q;
        }
      if (a.Usave) store_acc_rows(acc, a.Usave, row0, nvalid, MP, sA, sB, half, lane);
    }
    RT_TICK(9);
    __syncthreads();
    RT_TICK(10);
    if (tid < nvalid) {
      double q1 = 0.0, mu = 0.0, q2 = 0.0;
      for (int pp = 0; pp < npairs; ++pp) {
        q1 += sm.red[0][pp][tid];
        mu += sm.red[1][pp][tid];
        q2 += sm.red[2][pp][tid];
      }
      const double c = sm.kxx[tid] - q1;
      const double v = (a.training ? fmax(c, 0.0) : c) + q2;
      a.mu[row0 + tid] = mu;
      a.var[row0 + tid] = v;
      if (a.craw) a.craw[row0 + tid] = c;
      if (a.training && c < 0.0 && a.clamp_count) atomicAdd(a.clamp_count, 1u);
    }
    if (a.Tsave && warp == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    __syncthreads();
    RT_TICK(11);
  }
  cp_async_wait_group<0>();     // the chained look-ahead of the last segment
  RT_FLUSH(0);
}

// ---------------------------------------------------------------------------------------------------------------
// Warp-specialised forward kernel: the hot configuration (upper layers whose rows are MC samples of few points: the
// S-sample training tiles and the acquisition tiles).
//
// Sample-shared covariance build: with xrep >= XSHARE_MIN_REP = 11 a 32-row tile holds at most XMAX = 4 distinct x (the
// S = 64 training tiles one, the S = 25 acquisition tiles two or three).  The two x-kernels a1 E1, a2 E2 depend on
// (x, z_j) only, so they are evaluated ONCE per tile and distinct x, and the per-(row, j) work shrinks to the f-kernel:
// one exponential instead of three, and no per-dimension arithmetic.  At S = 64 that is 8x fewer x-kernel evaluations
// than build_k_tile's one per warp of RPW rows.
//
// What the measurements said (tools/row_bench -DROW_TIMING, profiles/r02_row_fwd_phases.txt):
//  * DFMA and DMMA share the FP64 pipe and the schedulers arbitrate between warps, not work: next to warps that stream
//    DMMAs (16 pipe cycles each) every FP64 instruction of another warp waits 60 - 700 cycles for its turn, however
//    little of the pipe its 2-cycle DFMAs need and whatever else that warp has in flight (4 independent exponent chains
//    per thread ran no faster than 1).  With two co-resident CTAs the build was 23 - 30 % of a CTA's time and the pipe
//    idled 26 % of the time - whenever both CTAs were outside their products at once.
//  * a lone CTA's products run at 89 % of the pipe.
//  * 8 product + 8 support warps doing build / row sums / stores in sequence: the product warps waited 16 % of the time
//    for the support group (~4700 FP64 warp-instructions per tile, ~600 per warp).
// So: ONE CTA per SM and three roles; `setmaxnreg` moves the registers to the product warps:
//   8 PRODUCT warps (128 registers): nothing but the two triangular DMMA products, tile after tile, and the accumulator
//     -> shared-memory hand-overs:  t = W k | t -> tile (in place of K) | u = H^T t | u -> tile (in place of t)
//   16 BUILD warps (48 registers), the covariance build spread evenly over them, in two stages one tile apart so that
//     no warp waits for another inside a stage:  K(Z, rows of tile i) from the x-kernel values (2 rows per warp), THEN
//     - off the path the product warps wait on - the x-kernel values and row data of tile i + 1
//   4 FINISH warps (48 registers): |t|^2, beta.t and the bulk store of t as soon as t is in the buffer (this is what the
//     product warps wait for before u may replace t); then |u|^2, bulk store of u, mean / variance; buffer released
// Two tile buffers, each cycling K -> t -> u; ten named barriers hand them over (arrive by the producer role, sync by
// the consumer role).  The row sums are taken from shared memory (the first kernel reduced them from the accumulators
// with 48 shuffles per thread inside the product warps), and t / u leave as one bulk (TMA engine) copy per row.
// Tried on top of this and measured, not kept (all within 0.65 - 0.69 of the DMMA peak; the support side's FP64
// instructions get through at ~1 per 40 cycles and scheduler whatever their organisation, and that rate, not the
// dependencies, sets the tile time once the products themselves are down to 41k cycles): row sums pre-reduced by the
// product warps from their accumulators (what the finish warps saved the product warps lost in their hand-overs); 16
// symmetric support warps that own two rows of every tile for build, sums and stores; the product warps building a
// quarter of K themselves between two tiles.
// ---------------------------------------------------------------------------------------------------------------
constexpr int XMAX = 4, XSHARE_MIN_REP = 11;     // distinct x rows per tile, and the xrep that bounds them by XMAX
constexpr int WS_PROD_WARPS = ROW_WARPS, WS_BUILD_WARPS = 16, WS_FIN_WARPS = 4;
constexpr int WS_PROD_THREADS = WS_PROD_WARPS * 32, WS_BUILD_THREADS = WS_BUILD_WARPS * 32, WS_FIN_THREADS = WS_FIN_WARPS * 32;
constexpr int WS_THREADS = WS_PROD_THREADS + WS_BUILD_THREADS + WS_FIN_THREADS;      // 896: launched with 72 registers
// 8 x 32 x 128 + 20 x 32 x 48 = 63488 <= 896 x 72 = 64512 (an exact fit of the whole file, tried as 128 + 64 with 24
// warps, never gets its registers: the kernel hangs in setmaxnreg.inc)
constexpr int WS_PROD_REGS = 128, WS_SUPPORT_REGS = 48;
constexpr int WS_ROWS_PER_WARP = TR / WS_BUILD_WARPS;       // K build: tile rows per build warp
static_assert(WS_PROD_WARPS % 4 == 0 && WS_BUILD_WARPS % 4 == 0 && WS_FIN_WARPS % 4 == 0, "setmaxnreg is per warpgroup");
static_assert(WS_ROWS_PER_WARP * WS_BUILD_WARPS == TR && WS_BUILD_THREADS == 2 * MAX_MP && XMAX == 4, "build thread mapping");
// per-tile scratch of the build role, double-buffered: stage 1 fills tile i + 1's after stage 2 has read tile i's
struct WsScratch {
  double fs[TR], vfs[TR];                       // propagated input f of the tile's rows, v_lin f
  int xsel[TR];                                 // which of the tile's distinct x a row reads
  double s12[2 * XMAX][MAX_MP];                 // [0, XMAX): a1 E1(x_c, z_j);  [XMAX, 2 XMAX): a2 E2(x_c, z_j)
};
struct WsSmem {
  KernFast kf;
  double e2tab[kExp2Tab];
  double zfs[MAX_MP];
  double beta[MAX_MP];
  double zsT[kMaxD][MAX_MP];                    // Z^T (x part of the inducing inputs)
  double kxx[4][TR];                            // per tile, slot i & 3 (written a tile before the finish warps read it)
  double q1[2][TR], mu[2][TR];                  // per tile buffer
  WsScratch scr[2];
};
__host__ __device__ inline size_t ws_head_bytes() { return ((sizeof(WsSmem) + 127) / 128) * 128; }
__host__ inline size_t ws_smem_bytes(int MP) {
  return ws_head_bytes() + 2 * tile_bytes(MP) + (size_t)ROW_WARPS * FWD_NST * 32 * sizeof(double2);
}
__device__ __forceinline__ void bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void bar_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }
// named barriers: one per role, then per tile buffer b (0 / 1):
constexpr int WS_BAR_PROD = 1, WS_BAR_BUILD = 2;
constexpr int WS_K_READY = 4;    // + b  build -> product:  K(Z, rows) is in the buffer
constexpr int WS_T_READY = 6;    // + b  product -> finish: t has replaced K
constexpr int WS_T_DONE = 8;     // + b  finish -> product: t's row sums and bulk store are done, u may replace it
constexpr int WS_U_READY = 10;   // + b  product -> finish: u has replaced t
constexpr int WS_BUF_FREE = 12;  // + b  finish -> build:   u's row sums and bulk store are done, the buffer is free
constexpr int WS_N_K = WS_BUILD_THREADS + WS_PROD_THREADS, WS_N_PF = WS_PROD_THREADS + WS_FIN_THREADS,
              WS_N_FB = WS_FIN_THREADS + WS_BUILD_THREADS;

__global__ void __launch_bounds__(WS_THREADS, 1) row_fwd_ws_kernel(const __grid_constant__ RowArgs a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  WsSmem& sm = *reinterpret_cast<WsSmem*>(smem_raw);
  const int MP = a.MP, ldb = MP + 4;
  const int role = threadIdx.x < WS_PROD_THREADS ? 0 : (threadIdx.x < WS_PROD_THREADS + WS_BUILD_THREADS ? 1 : 2);
  const int tid = role == 0 ? threadIdx.x : (role == 1 ? threadIdx.x - WS_PROD_THREADS
                                                        : threadIdx.x - WS_PROD_THREADS - WS_BUILD_THREADS);
  const int lane = tid & 31, warp = tid >> 5;
  double* tiles = reinterpret_cast<double*>(smem_raw + ws_head_bytes());
  auto tile_buf = [&](int b) { return tiles + (size_t)b * (tile_bytes(MP) / sizeof(double)); };
  const unsigned R = (unsigned)a.R, ntiles = (R + TR - 1) / TR;
  const unsigned n = blockIdx.x < ntiles ? (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0u;   // this CTA's tiles
  auto tile_of = [&](unsigned i) { return blockIdx.x + i * gridDim.x; };

  RT_DECL_ROLE(tid == 0)
  // ---- data shared by the roles ----
  if (threadIdx.x == 0) load_kern_fast(sm.kf, a.kind, a.d, a.theta);
  fill_exp2_tab(sm.e2tab, threadIdx.x, WS_THREADS);
  for (int j = threadIdx.x; j < MP; j += WS_THREADS) {
    sm.zfs[j] = j < a.M ? a.zf[j] : 0.0;
    sm.beta[j] = (a.ops + ops_beta(MP))[j];
  }
  for (int idx = threadIdx.x; idx < MP * a.d; idx += WS_THREADS) {
    const int j = idx / a.d, c = idx - j * a.d;
    sm.zsT[c][j] = j < a.M ? a.Zx[(size_t)j * a.d + c] : 0.0;
  }
  __syncthreads();
  RT_TICK(0);

  if (role == 0) {
    // =========================== product warps ===========================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(WS_PROD_REGS));
    double2* ring = reinterpret_cast<double2*>(smem_raw + ws_head_bytes() + 2 * tile_bytes(MP)) + warp * FWD_NST * 32;
    const int p = warp, npairs = MP / 32, ns = MP / 16;
    const bool active = p < npairs;
    const int sA = p, sB = ns - 1 - p;
    const double* W = a.ops + ops_block(MP, OPS_WF);
    const double* G = a.ops + ops_block(MP, OPS_HTF);
    if (active) {
      const double2* f0 = frag_start(W, MP, sA, false, lane);
#pragma unroll
      for (int j = 0; j < 3; ++j) { cp_async16_cg(ring + lane + j * 32, f0 + j * 32); cp_async_commit_group(); }
    }
    for (unsigned i = 0; i < n; ++i) {
      const int b = i & 1;
      double* Ks = tile_buf(b);
      double acc[2][2][4][2];
      bar_sync(WS_K_READY + b, WS_N_K);
      RT_TICK(1);
      // ---- t = W k ----
      zero_acc(acc);
      if (active) {
        frag_segment<false>(acc[0], W, MP, Ks, ldb, sA, 0, lane, ring, frag_start(W, MP, sB, false, lane));
        frag_segment<false>(acc[1], W, MP, Ks, ldb, sB, 0, lane, ring, frag_start(G, MP, sA, true, lane));
      }
      RT_TICK(2);
      bar_sync(WS_BAR_PROD, WS_PROD_THREADS);   // every product warp is done reading K
      if (active) store_acc_to_tile(acc, Ks, ldb, sA, sB, 0, lane);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // t is bulk-copied out by the finish warps
      bar_sync(WS_BAR_PROD, WS_PROD_THREADS);
      bar_arrive(WS_T_READY + b, WS_N_PF);
      RT_TICK(3);
      // ---- u = H^T t ----
      zero_acc(acc);
      if (active) {
        frag_segment<true>(acc[0], G, MP, Ks, ldb, sA, 0, lane, ring, frag_start(G, MP, sB, true, lane));
        frag_segment<true>(acc[1], G, MP, Ks, ldb, sB, 0, lane, ring, frag_start(W, MP, sA, false, lane));
      }
      RT_TICK(4);
      bar_sync(WS_T_DONE + b, WS_N_PF);     // all product warps are done reading t, and so are the finish warps
      RT_TICK(5);
      if (active) store_acc_to_tile(acc, Ks, ldb, sA, sB, 0, lane);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      bar_arrive(WS_U_READY + b, WS_N_PF);
      RT_TICK(6);
    }
    cp_async_wait_group<0>();     // the chained look-ahead of the last segment
    RT_FLUSH(0);
    return;
  }
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(WS_SUPPORT_REGS));
  if (n == 0) return;

  if (role == 1) {
    // =========================== build warps ===========================
    //   stage 2, tile i:      K(Z, rows): warp <-> 2 rows, lane <-> inducing point of a 32-chunk:
    //                         k = s1 (v f z_f + a_f E_f) + s2
    //   stage 1, tile i + 1:  thread (j, half): a1 E1 and a2 E2 between inducing point j and two of the tile's (at most
    //                         four) distinct x, read straight from global memory;  warp 15 also: the tile's rows -> f,
    //                         v f, k_xx, which x (row data prefetched into registers one iteration earlier)
    const unsigned uxrep = (unsigned)a.xrep, uprep = (unsigned)a.prep;
    const unsigned ueps = a.eps_mod >= a.R ? 0u : (unsigned)a.eps_mod;       // 0: eps index == row
    auto bsync = [&]() { bar_sync(WS_BAR_BUILD, WS_BUILD_THREADS); };
    const bool rows_warp = warp == WS_BUILD_WARPS - 1;
    // row data of the tile after the one being prepared: lane <-> row: (mean, variance, normal) or its direct f
    double pf_a = 0.0, pf_b = 1.0, pf_c = 0.0;
    auto prefetch = [&](unsigned i) {
      if (i >= n || !rows_warp) return;
      const unsigned row = tile_of(i) * TR + lane;
      pf_a = 0.0; pf_b = 1.0; pf_c = 0.0;
      if (row < R) {
        if (a.f_direct) {
          pf_a = a.f_direct[row];
        } else {
          const unsigned pr = row / uprep;
          pf_a = a.mu_prev[pr];
          pf_b = a.var_prev[pr];
          pf_c = a.eps[ueps ? row % ueps : row];
        }
      }
    };
    auto stage1 = [&](unsigned i) {
      WsScratch& sc = sm.scr[i & 1];
      const unsigned row0 = tile_of(i) * TR;
      const int nvalid = (int)min((unsigned)TR, R - row0);
      const unsigned xi0 = row0 / uxrep;
      const int nx = (int)((row0 + nvalid - 1) / uxrep - xi0) + 1;
      {
        const int j = tid & (MAX_MP - 1), q0 = 2 * (tid / MAX_MP);       // this thread's inducing point and first x
        if (j < MP && q0 < nx) {
          const KernFast& kf = sm.kf;
          const bool jok = j < a.M, two = q0 + 1 < nx;
          const double* x0 = a.x + (size_t)(xi0 + q0) * a.d;
          const double* x1 = two ? x0 + a.d : x0;
          double D1[2] = {kf.la1, kf.la1}, D2[2] = {kf.la2, kf.la2};
          for (int c = 0; c < a.d; ++c) {          // dimensions in ascending order, like every other build of K
            const double2 cc = kf.cc[c];
            const double z = sm.zsT[c][j];
            const double da = __ldg(x0 + c) - z, db = __ldg(x1 + c) - z;
            const double da2 = da * da, db2 = db * db;
            D1[0] = fma(da2, cc.x, D1[0]); D2[0] = fma(da2, cc.y, D2[0]);
            D1[1] = fma(db2, cc.x, D1[1]); D2[1] = fma(db2, cc.y, D2[1]);
          }
          sc.s12[q0][j] = jok ? exp2_tab(D1[0], sm.e2tab) : 0.0;
          sc.s12[XMAX + q0][j] = jok ? exp2_tab(D2[0], sm.e2tab) : 0.0;
          if (two) {
            sc.s12[q0 + 1][j] = jok ? exp2_tab(D1[1], sm.e2tab) : 0.0;
            sc.s12[XMAX + q0 + 1][j] = jok ? exp2_tab(D2[1], sm.e2tab) : 0.0;
          }
        }
      }
      if (rows_warp) {
        double f = 0.0;
        if (lane < nvalid) f = a.f_direct ? pf_a : pf_a + sqrt(fmax(pf_b, kMinVariance)) * pf_c;
        sc.fs[lane] = f;
        sc.vfs[lane] = sm.kf.vlin * f;
        sm.kxx[i & 3][lane] = sm.kf.a1 * (sm.kf.vlin * f * f + sm.kf.af) + sm.kf.a2;
        sc.xsel[lane] = lane < nvalid ? (int)((row0 + lane) / uxrep - xi0) : 0;
        prefetch(i + 1);
      }
    };
    auto stage2 = [&](unsigned i) {
      const WsScratch& sc = sm.scr[i & 1];
      double* Ks = tile_buf(i & 1);
      const int nvalid = (int)min((unsigned)TR, R - tile_of(i) * TR);
      const double laf = sm.kf.laf, cf = sm.kf.cf;
      const int r0 = warp * WS_ROWS_PER_WARP;
      double f[WS_ROWS_PER_WARP], vf[WS_ROWS_PER_WARP];
      int so[WS_ROWS_PER_WARP];                      // offset of the row's x-kernel values in s12
#pragma unroll
      for (int r = 0; r < WS_ROWS_PER_WARP; ++r) {
        f[r] = sc.fs[r0 + r]; vf[r] = sc.vfs[r0 + r];
        so[r] = sc.xsel[r0 + r] * MAX_MP + lane;
      }
      const double* s12 = &sc.s12[0][0];
      for (int ch = 0; ch < MP / 32; ++ch) {
        const int j = 32 * ch + lane;
        const double zf = sm.zfs[j];
        double k[WS_ROWS_PER_WARP];
#pragma unroll
        for (int r = 0; r < WS_ROWS_PER_WARP; ++r) {
          const double dff = f[r] - zf;
          const double Ef = exp2_tab(fma(dff * dff, cf, laf), sm.e2tab);
          k[r] = fma(s12[so[r] + 32 * ch], fma(vf[r], zf, Ef), s12[so[r] + 32 * ch + XMAX * MAX_MP]);
        }
#pragma unroll
        for (int r = 0; r < WS_ROWS_PER_WARP; ++r) Ks[(size_t)(r0 + r) * ldb + j] = r0 + r < nvalid ? k[r] : 0.0;
      }
    };
    prefetch(0);
    stage1(0);
    bsync();
    for (unsigned i = 0; i < n; ++i) {
      const int b = i & 1;
      RT_TICKW(1, 0);
      if (i >= 2) bar_sync(WS_BUF_FREE + b, WS_N_FB);      // u of tile i - 2 has left the buffer
      RT_TICKW(1, 1);
      stage2(i);
      RT_TICKW(1, 2);
      bsync();      // K(i) complete, scratch of tile i free
      bar_arrive(WS_K_READY + b, WS_N_K);
      RT_TICKW(1, 3);
      if (i + 1 < n) stage1(i + 1);      // off the path the product warps wait on: runs while u(i - 1) leaves its buffer
      RT_TICKW(1, 4);
      bsync();      // scratch of tile i + 1 complete
      RT_TICKW(1, 5);
    }
    RT_FLUSH(1);
    return;
  }

  // =========================== finish warps ===========================
  // row sums over the tile in shared memory: thread <-> (row = tid / 4, columns tid % 4 + 4 k): a half-warp's 16
  // addresses fall into 16 different 8-byte banks (ldb % 16 == 4); 4-lane fold
  const int srow = tid >> 2, spart = tid & 3;
  auto fold4 = [&](double v) {
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    return v;
  };
  // bulk (TMA engine) copies of the tile's valid rows to dst[R][MP]: every finish warp issues a quarter of them (a
  // bulk-copy instruction costs its warp ~80 cycles; one warp issuing all 32 fell 2.7k cycles behind the others) and
  // waits until the engine has read its own (the buffer is rewritten next)
  constexpr int ROWS_PER_FIN_WARP = TR / WS_FIN_WARPS;
  auto bulk_rows_out = [&](double* dst, const double* Ks, unsigned row0, int nvalid) {
    if (lane < ROWS_PER_FIN_WARP) {
      const int r = warp * ROWS_PER_FIN_WARP + lane;
      if (r < nvalid)
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(
                         dst + (size_t)(row0 + (unsigned)r) * MP),
                     "r"((unsigned)__cvta_generic_to_shared(Ks + (size_t)r * ldb)),
                     "r"((unsigned)(MP * sizeof(double))) : "memory");
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
  };
  auto bulk_wait_read = [&]() { if (lane < ROWS_PER_FIN_WARP) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); };
  for (unsigned i = 0; i < n; ++i) {
    const int b = i & 1;
    const double* Ks = tile_buf(b);
    const unsigned row0 = tile_of(i) * TR;
    const int nvalid = (int)min((unsigned)TR, R - row0);
    const double* rowp = Ks + (size_t)srow * ldb + spart;
    // ---- t is in the buffer: |t|^2 and beta . t per row, bulk store of t; then u may replace it ----
    RT_TICKW(2, 0);
    bar_sync(WS_T_READY + b, WS_N_PF);
    RT_TICKW(2, 1);
    if (a.Tsave) bulk_rows_out(a.Tsave, Ks, row0, nvalid);
    {
      double q = 0.0, m = 0.0;
#pragma unroll 8
      for (int k = 0; k < MP; k += 4) {
        const double v = rowp[k];
        q = fma(v, v, q);
        m = fma(sm.beta[spart + k], v, m);
      }
      q = fold4(q); m = fold4(m);
      if (spart == 0) { sm.q1[b][srow] = q; sm.mu[b][srow] = m; }
    }
    RT_TICKW(2, 2);
    if (a.Tsave) bulk_wait_read();
    bar_arrive(WS_T_DONE + b, WS_N_PF);
    RT_TICKW(2, 3);
    // ---- u is in the buffer: |u|^2 per row, mean / variance of the tile's rows, bulk store of u; buffer released ----
    bar_sync(WS_U_READY + b, WS_N_PF);
    RT_TICKW(2, 4);
    if (a.Usave) bulk_rows_out(a.Usave, Ks, row0, nvalid);
    {
      double q = 0.0;
#pragma unroll 8
      for (int k = 0; k < MP; k += 4) { const double v = rowp[k]; q = fma(v, v, q); }
      q = fold4(q);
      if (spart == 0 && srow < nvalid) {
        const double c = sm.kxx[i & 3][srow] - sm.q1[b][srow];
        const double v = (a.training ? fmax(c, 0.0) : c) + q;
        a.mu[row0 + srow] = sm.mu[b][srow];
        a.var[row0 + srow] = v;
        if (a.craw) a.craw[row0 + srow] = c;
        if (a.training && c < 0.0 && a.clamp_count) atomicAdd(a.clamp_count, 1u);
      }
    }
    RT_TICKW(2, 5);
    if (a.Usave) bulk_wait_read();
    if (i + 2 < n) bar_arrive(WS_BUF_FREE + b, WS_N_FB);
    RT_TICKW(2, 6);
  }
  RT_FLUSH(2);
}

// Backward through the covariance function for one tile: Ks holds dk = d loss / d K(z_j, row r).  Same thread mapping
// as build_k_tile (warp <-> RPW rows, lane <-> inducing point).  Accumulator conventions (undone at the final flush):
//   th[0] = sum gk a1 E1 gg  (d/da1 = th[0] / a1)     th[1] = sum gk a1 E1 f f'   (d/dv)
//   th[2] = sum gk a1 E1 af Ef (d/daf = th[2] / af)   th[3] = sum gk a1 E1 af Ef (f-f')^2  (d/dlf = th[3] / lf^3)
//   th[4] = sum gk a2 E2     (d/da2 = th[4] / a2)     tl1[c], tl2[c] = sum g D_c^2  (d/dl_c = tl / l_c^3)
// dk reaches the warp through a private 3-chunk cp.async ring (kg_ring, [chunk % 3][row][lane]): a lane copies the
// RPW values it will use two chunks ahead of their use (the synchronous loads were 21 % of the kernel's stall samples,
// profiles/r01r_*); rows past the end and padded inducing points are zero-filled by the copy.
constexpr int KG_NST = 3;
__device__ __forceinline__ void kg_issue(const double* __restrict__ Ks, int ldb, int rbase, int nvalid, int M, int ch,
                                         int nch, double* ring, int lane) {
  if (ch < nch) {
    const int j = 32 * ch + lane;
#pragma unroll
    for (int i = 0; i < RPW; ++i) {
      const bool ok = j < M && rbase + i < nvalid;
      const unsigned sa = (unsigned)__cvta_generic_to_shared(ring + ((ch % KG_NST) * RPW + i) * 32 + lane);
      const int sz = ok ? 8 : 0;
      asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(sa),
                   "l"(ok ? Ks + (size_t)(rbase + i) * ldb + j : Ks), "r"(sz) : "memory");
    }
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
}

template <int KIND, int D, bool PARAM, bool XGRAD, bool SHX, class SM>
__device__ __forceinline__ void kgrad_tile(const RowArgs& a, SM& sm, const double* __restrict__ Ks, int ldb,
                                           long long row0, int nvalid, int warp, int lane, double* ring) {
  const KernFast& kf = sm.kf;
  const double* tab = sm.e2tab;
  const int M = a.M, nch = a.MP / 32;
  const int rbase = warp * RPW;
  kg_issue(Ks, ldb, rbase, nvalid, M, 0, nch, ring, lane);
  kg_issue(Ks, ldb, rbase, nvalid, M, 1, nch, ring, lane);
  // register budget: the accumulators below stay in registers for the whole tile, so the per-dimension coefficients
  // and the rows' coordinates are re-read from shared memory (broadcast loads) instead of being cached
  const double la1 = kf.la1, la2 = kf.la2, laf = kf.laf, cf = kf.cf, vlin = kf.vlin, ilf = kf.ilf;
  double th[5], tl1[D], tl2[D], rdf[RPW], rdx[XGRAD ? RPW : 1][D];
#pragma unroll
  for (int q = 0; q < 5; ++q) th[q] = 0.0;
#pragma unroll
  for (int c = 0; c < D; ++c) { tl1[c] = 0.0; tl2[c] = 0.0; }
#pragma unroll
  for (int i = 0; i < RPW; ++i) rdf[i] = 0.0;
#pragma unroll
  for (int i = 0; i < (XGRAD ? RPW : 1); ++i)
#pragma unroll
    for (int c = 0; c < D; ++c) rdx[i][c] = 0.0;

  for (int ch = 0; ch < nch; ++ch) {
    const int j = 32 * ch + lane;
    kg_issue(Ks, ldb, rbase, nvalid, M, ch + 2, nch, ring, lane);
    asm volatile("cp.async.wait_group 2;" ::: "memory");
    const double* gring = ring + (ch % KG_NST) * RPW * 32 + lane;     // this lane's dk of the chunk: gring[32 i]
    double z[D];
#pragma unroll
    for (int c = 0; c < D; ++c) z[c] = sm.zsT[c][j];
    const double zf = sm.zfs[j], vz = vlin * zf;
    double azf = 0.0;
    if (SHX && KIND == 1) {
      // the warp's rows share x: distances, a1 E1 and a2 E2 once per inducing point; the lengthscale (and x)
      // gradients take the row-summed weights
      double diff[D], d2[D], D1 = la1, D2 = la2;
#pragma unroll
      for (int c = 0; c < D; ++c) {
        const double2 cc = kf.cc[c];
        diff[c] = sm.xs[rbase][c] - z[c];
        d2[c] = diff[c] * diff[c];
        D1 = fma(d2[c], cc.x, D1);
        D2 = fma(d2[c], cc.y, D2);
      }
      const double s1 = exp2_tab(D1, tab), s2 = exp2_tab(D2, tab);
      double G1 = 0.0, G2 = 0.0;
#pragma unroll
      for (int i = 0; i < RPW; ++i) {
        const double gk = gring[32 * i];
        const double fi = sm.fs[rbase + i];
        const double dff = fi - zf, dff2 = dff * dff;
        const double Efp = exp2_tab(fma(dff2, cf, laf), tab);
        const double fz = fi * zf;
        const double gg = fma(vlin, fz, Efp);
        const double gs1 = gk * s1, g2 = gk * s2;
        const double g1 = gs1 * gg, gEf = gs1 * Efp;
        const double q = gEf * (dff * ilf);
        rdf[i] += fma(gs1, vz, -q);
        G1 += g1; G2 += g2;
        if (PARAM) {
          azf += fma(gs1, vlin * fi, q);
          th[1] = fma(gs1, fz, th[1]);
          th[2] += gEf;
          th[3] = fma(gEf, dff2, th[3]);
        }
      }
      if (PARAM) {
        th[0] += G1; th[4] += G2;
#pragma unroll
        for (int c = 0; c < D; ++c) { tl1[c] = fma(G1, d2[c], tl1[c]); tl2[c] = fma(G2, d2[c], tl2[c]); }
      }
      if (XGRAD) {   // d loss / d x of the shared point: booked on the warp's first row, the others stay zero
#pragma unroll
        for (int c = 0; c < D; ++c) rdx[0][c] -= diff[c] * fma(G1, kf.il1[c], G2 * kf.il2[c]);
      }
    } else {
#pragma unroll 2
    for (int i = 0; i < RPW; ++i) {
      const double gk = gring[32 * i];
      const double fi = sm.fs[rbase + i];
      double diff[D], d2[D], D1 = la1, D2 = la2;
#pragma unroll
      for (int c = 0; c < D; ++c) {
        const double2 cc = kf.cc[c];
        diff[c] = sm.xs[rbase + i][c] - z[c];
        d2[c] = diff[c] * diff[c];
        D1 = fma(d2[c], cc.x, D1);
        if (KIND == 1) D2 = fma(d2[c], cc.y, D2);
      }
      if (KIND == 0) {
        const double g1 = gk * exp2_tab(D1, tab);
        if (PARAM) {
          th[0] += g1;
#pragma unroll
          for (int c = 0; c < D; ++c) tl1[c] = fma(g1, d2[c], tl1[c]);
        }
        if (XGRAD) {
#pragma unroll
          for (int c = 0; c < D; ++c) rdx[i][c] = fma(-g1 * diff[c], kf.il1[c], rdx[i][c]);
        }
      } else {
        const double dff = fi - zf, dff2 = dff * dff;
        const double Efp = exp2_tab(fma(dff2, cf, laf), tab);        // af Ef
        const double s1 = exp2_tab(D1, tab), s2 = exp2_tab(D2, tab);  // a1 E1, a2 E2
        const double fz = fi * zf;
        const double gg = fma(vlin, fz, Efp);                         // k_lin + k_f
        const double gs1 = gk * s1, g2 = gk * s2;
        const double g1 = gs1 * gg, gEf = gs1 * Efp;
        const double q = gEf * (dff * ilf);                           // gk a1 E1 af Ef (f - f') / lf^2
        rdf[i] += fma(gs1, vz, -q);
        if (PARAM) {
          azf += fma(gs1, vlin * fi, q);
          th[0] += g1;
          th[1] = fma(gs1, fz, th[1]);
          th[2] += gEf;
          th[3] = fma(gEf, dff2, th[3]);
          th[4] += g2;
#pragma unroll
          for (int c = 0; c < D; ++c) { tl1[c] = fma(g1, d2[c], tl1[c]); tl2[c] = fma(g2, d2[c], tl2[c]); }
        }
        if (XGRAD) {
#pragma unroll
          for (int c = 0; c < D; ++c) rdx[i][c] -= diff[c] * fma(g1, kf.il1[c], g2 * kf.il2[c]);
        }
      }
    }
    }
    if (PARAM && KIND == 1) sm.acc_zf[warp][j] += azf;   // one owner per slot -> deterministic
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  // row-wise sums over the inducing points, and the diag term d k_xx of the variance
#pragma unroll
  for (int i = 0; i < RPW; ++i) {
    const int r = rbase + i;
    const bool rok = r < nvalid;
    const double dvm = sm.dvar[r] * sm.mask[r];
    const double fi = sm.fs[r];
    if (KIND == 1) {
      const double sdf = warp_sum(rdf[i]);
      if (lane == 0 && rok) a.df[row0 + r] = sdf + dvm * 2.0 * kf.a1 * vlin * fi;
    }
    if (XGRAD) {
#pragma unroll
      for (int c = 0; c < D; ++c) {
        const double sx = warp_sum(rdx[i][c]);
        if (lane == 0 && rok) a.dxrow[(size_t)(row0 + r) * D + c] = sx;
      }
    }
    if (PARAM && lane == 0) {
      if (KIND == 0) {
        th[0] += dvm * kf.a1;
      } else {
        th[0] += dvm * kf.a1 * fma(vlin * fi, fi, kf.af);
        th[1] += dvm * kf.a1 * fi * fi;
        th[2] += dvm * kf.a1 * kf.af;
        th[4] += dvm * kf.a2;
      }
    }
  }
  if (PARAM) {
#pragma unroll
    for (int q = 0; q < 5; ++q) {
      const double red = warp_sum(th[q]);
      if (lane == 0) sm.acc_th[warp][q] += red;
    }
#pragma unroll
    for (int c = 0; c < D; ++c) {
      double red = warp_sum(tl1[c]);
      if (lane == 0) sm.acc_th[warp][5 + c] += red;
      if (KIND == 1) {
        red = warp_sum(tl2[c]);
        if (lane == 0) sm.acc_th[warp][5 + kMaxD + c] += red;
      }
    }
  }
}

template <int KIND, bool PARAM, bool XGRAD, bool SHX, class SM>
__device__ __forceinline__ void kgrad_tile_d(const RowArgs& a, SM& sm, const double* Ks, int ldb, long long row0,
                                             int nvalid, int warp, int lane, double* ring) {
  switch (sm.kf.d) {
    case 1: kgrad_tile<KIND, 1, PARAM, XGRAD, SHX>(a, sm, Ks, ldb, row0, nvalid, warp, lane, ring); break;
    case 2: kgrad_tile<KIND, 2, PARAM, XGRAD, SHX>(a, sm, Ks, ldb, row0, nvalid, warp, lane, ring); break;
    case 3: kgrad_tile<KIND, 3, PARAM, XGRAD, SHX>(a, sm, Ks, ldb, row0, nvalid, warp, lane, ring); break;
    case 4: kgrad_tile<KIND, 4, PARAM, XGRAD, SHX>(a, sm, Ks, ldb, row0, nvalid, warp, lane, ring); break;
    case 5: kgrad_tile<KIND, 5, PARAM, XGRAD, SHX>(a, sm, Ks, ldb, row0, nvalid, warp, lane, ring); break;
    case 6: kgrad_tile<KIND, 6, PARAM, XGRAD, SHX>(a, sm, Ks, ldb, row0, nvalid, warp, lane, ring); break;
    case 7: kgrad_tile<KIND, 7, PARAM, XGRAD, SHX>(a, sm, Ks, ldb, row0, nvalid, warp, lane, ring); break;
    default: kgrad_tile<KIND, 8, PARAM, XGRAD, SHX>(a, sm, Ks, ldb, row0, nvalid, warp, lane, ring); break;
  }
}

// ---------------------------------------------------------------------------------------------------
// backward of the row pass: given d loss/d mu_r, d loss/d var_r
//   dt = dmu beta - 2 dvar (mask t - H u);  dk = W^T dt                    (row_bwd_gemm_kernel, DMMA)
//   then through the covariance function: d theta, d zf, d f_r, d x_r      (kgrad_kernel, DFMA)
// The two halves are separate kernels: fused, the covariance gradient's accumulators pushed the products'
// accumulators into local memory (ncu: 16 of 32 spilled and reloaded every k-step, profiles/r01j_*); apart, the
// product kernel is the forward kernel's shape and the gradient kernel gets its own register budget and occupancy.
// dk travels through HBM ([R][MP], written and read once, coalesced).
// The whitened second-order statistics  A2 = sum_r dvar_r t t^T  and  b = sum_r dmu_r t  (t = W k)
// are accumulated by syrk_kernel from the saved T and consumed by the operator backward (matrix_ops.cu).
// ---------------------------------------------------------------------------------------------------
struct BwdSmem {
  double dmu[2][TR], dvar[2][TR], mask[2][TR];      // per-row scalars, double-buffered by the producer warp
  unsigned long long bar;     // mbarrier: the staged u / t rows (and the row scalars) of the next tile have landed
};
constexpr int BWD_THREADS = ROW_THREADS + 32;       // 8 product warps + the producer warp
__device__ __forceinline__ void bar_sync_bwd() { asm volatile("bar.sync 1, %0;" ::"n"(ROW_THREADS) : "memory"); }
constexpr size_t BWD_HEAD = 2048;
// [BwdSmem | X tile | U stage | T stage | A-fragment rings]; tiles are [TR][MP + 4]
__host__ __device__ inline size_t bwd_smem_bytes(int MP) {
  return BWD_HEAD + 3 * tile_bytes(MP) + (size_t)ROW_WARPS * BWD_NST * 32 * sizeof(double2);
}

__device__ __forceinline__ void mbar_init(unsigned long long* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(bar)),
               "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  const unsigned addr = (unsigned)__cvta_generic_to_shared(bar);
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(addr), "r"(parity) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
}
// bulk (TMA engine) global -> shared copy of `bytes` (multiple of 16, both sides 16-byte aligned), completion on `bar`
__device__ __forceinline__ void bulk_g2s(void* smem, const void* gmem, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   (unsigned)__cvta_generic_to_shared(smem)), "l"(gmem), "r"(bytes),
               "r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
}

// One persistent CTA per SM.  The saved u and t rows of tile i+1 are staged into shared memory by the bulk-copy engine
// while tile i's second product runs, and dk leaves straight from the accumulators, so no warp ever waits on HBM
// (with the synchronous loads of the first version the memory phases cost 13 us of every 32 us tile and two CTAs per
// SM did not hide them: profiles/r01z_*).  Per tile: y = H u (B operand read in place from the u stage), dt from y and
// the t stage into the X tile, barrier, dk = W^T dt.  A ninth warp is the PRODUCER: it issues the bulk copies and
// loads the row scalars of the next tile.  (When warp 0 did that on top of its products, the 64 bulk-copy instructions
// cost it 5.5k cycles per tile, it finished its second product that much later, and the other seven warps waited for
// it at the next tile's barrier: 12 % of the kernel, tools/row_bench -DROW_TIMING.)
__global__ void __launch_bounds__(BWD_THREADS, 1) row_bwd_gemm_kernel(const __grid_constant__ RowArgs a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  BwdSmem& sm = *reinterpret_cast<BwdSmem*>(smem_raw);
  static_assert(sizeof(BwdSmem) <= BWD_HEAD, "BwdSmem");
  const int MP = a.MP, ldb = MP + 4;
  double* X = reinterpret_cast<double*>(smem_raw + BWD_HEAD);
  double* BU = reinterpret_cast<double*>(smem_raw + BWD_HEAD + tile_bytes(MP));
  double* BT = reinterpret_cast<double*>(smem_raw + BWD_HEAD + 2 * tile_bytes(MP));
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool producer = warp == ROW_WARPS;
  double2* ring = reinterpret_cast<double2*>(smem_raw + BWD_HEAD + 3 * tile_bytes(MP)) + (producer ? 0 : warp) * BWD_NST * 32;
  const int half = warp % NHALF, p = warp / NHALF;
  const int npairs = MP / 32, ns = MP / 16;
  const bool active = !producer && p < npairs;
  const int sA = p, sB = ns - 1 - p;
  const int g = lane >> 2, t = lane & 3;
  const double* WT = a.ops + ops_block(MP, OPS_WTF);
  const double* H = a.ops + ops_block(MP, OPS_HF);
  const double* beta = a.ops + ops_beta(MP);
  const long long ntiles = (a.R + TR - 1) / TR;
  const unsigned row_bytes = (unsigned)MP * sizeof(double);

  RT_DECL
  if (tid == 0) {
    mbar_init(&sm.bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  if (producer) {
    // row scalars of tile number `it` of this CTA into buffer it & 1, then one bulk copy per row and array; invalid
    // rows of a ragged last tile keep stale (finite or not, never stored: every column of the products depends on its
    // own row only) data.  The mbarrier arrive (release) after the generic writes makes them visible to the waiters.
    auto stage_tile = [&](long long tile, int buf) {
      const long long row0 = tile * TR;
      const int nvalid = (int)min((long long)TR, a.R - row0);
      const long long row = row0 + lane;
      const bool ok = row < a.R;
      sm.dmu[buf][lane] = ok ? a.dmu[row] : 0.0;
      sm.dvar[buf][lane] = ok ? a.dvar[row] : 0.0;
      sm.mask[buf][lane] = (ok && a.training && a.craw) ? (a.craw[row] >= 0.0 ? 1.0 : 0.0) : 1.0;
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic reads of the stages -> async writes
      __syncwarp();
      if (lane == 0) mbar_expect_tx(&sm.bar, 2u * (unsigned)nvalid * row_bytes);
      __syncwarp();
      if (lane < nvalid) {
        bulk_g2s(BU + (size_t)lane * ldb, a.Usave + (size_t)(row0 + lane) * MP, row_bytes, &sm.bar);
        bulk_g2s(BT + (size_t)lane * ldb, a.Tsave + (size_t)(row0 + lane) * MP, row_bytes, &sm.bar);
      }
    };
    long long tile = blockIdx.x;
    if (tile < ntiles) stage_tile(tile, 0);
    int it = 0;
    for (; tile < ntiles; tile += gridDim.x, ++it) {
      __syncthreads();   // this tile's dt is complete: the u / t stages are free
      const long long next = tile + gridDim.x;
      if (next < ntiles) stage_tile(next, (it + 1) & 1);
    }
    return;
  }

  // A-fragment stream as in the forward kernel (frag_segment): four segments per tile (H slab A, H slab B, W^T slab A,
  // W^T slab B), each priming the ring for the next, so that no segment starts with an L2 round trip (4 per tile in the
  // first version, ~6 % of a tile), and the half-zero diagonal blocks skip their zero DMMAs
  if (active) {
    const double2* first = frag_start(H, MP, sA, false, lane);
#pragma unroll
    for (int j = 0; j < 3; ++j) { cp_async16_cg(ring + lane + j * 32, first + j * 32); cp_async_commit_group(); }
  }
  unsigned parity = 0;
  int it = 0;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
    const long long row0 = tile * TR;
    const int nvalid = (int)min((long long)TR, a.R - row0);
    const int sb = it & 1;
    RT_TICKW(1, 0);
    mbar_wait(&sm.bar, parity);
    parity ^= 1u;
    bar_sync_bwd();    // every product warp is done with the previous tile's X
    RT_TICKW(1, 1);
    double acc[2][2][4][2];
    if (active) {
      // ---- y = H u ----
      zero_acc(acc);
      frag_segment<false>(acc[0], H, MP, BU, ldb, sA, half, lane, ring, frag_start(H, MP, sB, false, lane));
      frag_segment<false>(acc[1], H, MP, BU, ldb, sB, half, lane, ring, frag_start(WT, MP, sA, true, lane));
      RT_TICKW(1, 2);
      // ---- dt = dmu beta - 2 dvar (mask t - y) ----
#pragma unroll
      for (int sl = 0; sl < 2; ++sl)
#pragma unroll
        for (int ib = 0; ib < 2; ++ib) {
          const int i = 16 * (sl == 0 ? sA : sB) + 8 * ib + g;
          const double bi = __ldg(beta + i);
#pragma unroll
          for (int ct = 0; ct < 4; ++ct)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const int r = 32 * half + 8 * ct + 2 * t + e;
              const double tv = BT[(size_t)r * ldb + i];
              acc[sl][ib][ct][e] = sm.dmu[sb][r] * bi - 2.0 * sm.dvar[sb][r] * (sm.mask[sb][r] * tv - acc[sl][ib][ct][e]);
            }
        }
      store_acc_to_tile(acc, X, ldb, sA, sB, half, lane);
    }
    RT_TICKW(1, 3);
    __syncthreads();   // dt complete in X; the producer may refill the u / t stages
    RT_TICKW(1, 4);
    // ---- dk = W^T dt, straight from the accumulators to HBM ----
    if (active) {
      zero_acc(acc);
      frag_segment<true>(acc[0], WT, MP, X, ldb, sA, half, lane, ring, frag_start(WT, MP, sB, true, lane));
      frag_segment<true>(acc[1], WT, MP, X, ldb, sB, half, lane, ring, frag_start(H, MP, sA, false, lane));
      RT_TICKW(1, 6);
      store_acc_rows(acc, a.dk, row0, nvalid, MP, sA, sB, half, lane);
    }
  }
  RT_TICKW(1, 7);
  cp_async_wait_group<0>();     // the chained look-ahead of the last segment
  RT_FLUSH(1);
}

// ---- through the covariance function: 4 warps x RPW rows per tile, 3 CTAs per SM ----
constexpr int KG_WARPS = 4, KG_THREADS = KG_WARPS * 32, KG_ROWS = KG_WARPS * RPW, KG_CTAS_PER_SM = 3;
using KgSmem = CovSmem<KG_WARPS, true>;
__host__ __device__ inline size_t kg_smem_bytes() {
  return ((sizeof(KgSmem) + 127) / 128) * 128 + (size_t)KG_WARPS * 3 * RPW * 32 * sizeof(double);
}

template <bool PARAM, bool XGRAD>
__global__ void __launch_bounds__(KG_THREADS, KG_CTAS_PER_SM) kgrad_kernel(const __grid_constant__ RowArgs a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  KgSmem& sm = *reinterpret_cast<KgSmem*>(smem_raw);
  const int MP = a.MP, d = a.d;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  load_inducing(a, sm);
  for (int j = lane; j < MAX_MP; j += 32) sm.acc_zf[warp][j] = 0.0;
  if (lane < kMaxTheta) sm.acc_th[warp][lane] = 0.0;
  __syncthreads();

  // every warp walks its own groups of RPW rows: the rows' state lives in the warp's slice of the shared arrays and
  // nothing is exchanged between warps until the final flush, so there is no CTA barrier in the loop (the per-tile
  // barriers of the first version were 14 % of the stall samples)
  double* ring = reinterpret_cast<double*>(smem_raw + ((sizeof(KgSmem) + 127) / 128) * 128) + warp * KG_NST * RPW * 32;
  const int rbase = warp * RPW;
  const long long ngroups = (a.R + RPW - 1) / RPW;
  for (long long grp = (long long)blockIdx.x * KG_WARPS + warp; grp < ngroups; grp += (long long)gridDim.x * KG_WARPS) {
    const long long rw0 = grp * RPW;                         // first row of the group (>= rbase)
    const int nv = (int)min((long long)RPW, a.R - rw0);
    __syncwarp();
    for (int idx = lane; idx < RPW * d; idx += 32) {
      const int r = idx / d, c = idx - r * d;
      sm.xs[rbase + r][c] = r < nv ? a.x[(size_t)((rw0 + r) / a.xrep) * d + c] : 0.0;
    }
    if (lane < RPW) {
      const bool ok = lane < nv;
      const long long row = rw0 + lane;
      double f = 0.0;
      if (ok && a.kind == 1) {
        if (a.f_direct) {
          f = a.f_direct[row];
        } else {
          const long long pr = row / a.prep;
          f = a.mu_prev[pr] + sqrt(fmax(a.var_prev[pr], kMinVariance)) * a.eps[row % a.eps_mod];
        }
      }
      sm.fs[rbase + lane] = f;
      sm.dvar[rbase + lane] = ok ? a.dvar[row] : 0.0;
      sm.mask[rbase + lane] = (ok && a.training && a.craw) ? (a.craw[row] >= 0.0 ? 1.0 : 0.0) : 1.0;
    }
    __syncwarp();
    // kgrad_tile addresses rows as (tile row0) + rbase + i with validity rbase + i < nvalid
    const long long row0 = rw0 - rbase;
    const int nvalid = rbase + nv;
    const double* dk = a.dk + (size_t)row0 * MP;
    if (a.kind == 0) kgrad_tile_d<0, PARAM, XGRAD, false>(a, sm, dk, MP, row0, nvalid, warp, lane, ring);
    else if (warp_rows_share_x(a, row0, warp)) kgrad_tile_d<1, PARAM, XGRAD, true>(a, sm, dk, MP, row0, nvalid, warp, lane, ring);
    else kgrad_tile_d<1, PARAM, XGRAD, false>(a, sm, dk, MP, row0, nvalid, warp, lane, ring);
  }
  if (PARAM) {
    // ---- flush the per-CTA partials (fixed summation order -> deterministic) ----
    __syncthreads();
    for (int j = tid; j < MP; j += KG_THREADS) {
      double s = 0.0;
      for (int w = 0; w < KG_WARPS; ++w) s += sm.acc_zf[w][j];
      a.part_zf[(size_t)blockIdx.x * MP + j] = s;
    }
    if (tid < kMaxTheta) {
      double s = 0.0;
      for (int w = 0; w < KG_WARPS; ++w) s += sm.acc_th[w][tid];
      // map (scalars | l1 | l2) accumulators to the theta layout and undo the accumulator scalings (see kgrad_tile)
      const KernFast& kf = sm.kf;
      double out = 0.0;
      int slot = -1;
      if (kf.kind == 0) {
        if (tid == 0) { slot = 0; out = kf.a1 > 0.0 ? s / kf.a1 : 0.0; }
        else if (tid >= 5 && tid < 5 + d) { slot = 1 + (tid - 5); out = s * kf.il1[tid - 5] * sqrt(kf.il1[tid - 5]); }
      } else {
        if (tid < 5) {
          slot = tid;
          if (tid == 0) out = kf.a1 > 0.0 ? s / kf.a1 : 0.0;
          else if (tid == 1) out = s;
          else if (tid == 2) out = kf.af > 0.0 ? s / kf.af : 0.0;
          else if (tid == 3) out = s * kf.ilf / kf.lf;
          else out = kf.a2 > 0.0 ? s / kf.a2 : 0.0;
        }
        else if (tid < 5 + d) { slot = tid; out = s * kf.il1[tid - 5] * sqrt(kf.il1[tid - 5]); }
        else if (tid >= 5 + kMaxD && tid < 5 + kMaxD + d) {
          const int c = tid - 5 - kMaxD;
          slot = 5 + d + c;
          out = s * kf.il2[c] * sqrt(kf.il2[c]);
        }
      }
      if (slot >= 0) a.part_theta[(size_t)blockIdx.x * kMaxTheta + slot] = out;
    }
  }
}

// sums the per-CTA partials in a fixed order: out[i] = sum_b part[b][i].  One warp per output element: lanes stride
// over the partials, then a butterfly (the order depends only on nblocks -> deterministic).
__global__ void reduce_partials_kernel(const double* __restrict__ part, int nblocks, int n, int stride,
                                       double* __restrict__ out, int accumulate) {
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (i >= n) return;
  double s = 0.0;
  for (int b = lane; b < nblocks; b += 32) s += part[(size_t)b * stride + i];
  s = warp_sum(s);
  if (lane == 0) out[i] = accumulate ? out[i] + s : s;
}

// ---------------------------------------------------------------------------------------------------
// A2 = sum_r w_r t_r t_r^T from the saved whitened rows T [R][MP] (the SYRK of the backward).
// The lower triangle is cut into 32 x 32 blocks (36 at MP = 256), one block per warp, 12 warps per CTA, so every
// DMMA is useful work and every warp carries the same load.  A CTA streams ALL MP columns of its chunk of rows
// through a 3-stage bulk-copy (TMA engine) + mbarrier pipeline (32 rows per stage, one 2 KB copy per row) and each
// warp reads its two column panels from there.  A thirteenth warp is the producer: it refills a slot as soon as the
// twelve consumer warps have released it (one "empty" mbarrier per slot), so the consumers drift up to two stages
// apart instead of meeting at a CTA barrier every 8 k-steps.
// Partial blocks per row chunk are folded in chunk order by syrk_reduce_kernel, which also mirrors the result to
// the full symmetric matrix.  One launch computes both weight sets, which = blockIdx.z: w_r = dvar_r (which = 0, into
// part_in) or dvar_r * [clamped row] (which = 1, into part_clamped; its CTAs exit at once unless some row was clamped,
// so the rarely needed set costs no launch of its own).  Set 0 also accumulates b = sum_r dmu_r t_r.
// ---------------------------------------------------------------------------------------------------
constexpr int SY_KB = 32, SY_WARPS = 12, SY_STAGES = 3;     // SY_WARPS consumer warps (one 32 x 32 block each)
constexpr int SY_CONS_THREADS = SY_WARPS * 32, SY_THREADS = SY_CONS_THREADS + 32;      // + one producer warp

__host__ __device__ inline size_t syrk_stage_doubles(int MP) { return (size_t)SY_KB * (MP + 4) + 3 * SY_KB; }
// b = sum_r dmu_r t_r rides along: every group of CTAs takes an equal share of the MP columns, a thread one column and
// one of SY_ALPHA_PARTS slices of a stage's rows.  (First version: the first MP threads of group 0 only, 32 FMAs per
// stage each.  Next to warps that stream DMMAs an FP64 instruction of another warp waits ~80 cycles for its turn, so
// those 8 warps fell 2.5k cycles per 6k-cycle stage behind and their CTAs - a third of the grid - set the kernel time.)
constexpr int SY_ALPHA_PARTS = 4;
__host__ __device__ inline size_t syrk_alpha_doubles(int MP, int nchunk) { return (size_t)nchunk * SY_ALPHA_PARTS * MP; }
__host__ __device__ inline int syrk_nblocks(int MP) { const int nb = MP / 32; return nb * (nb + 1) / 2; }

__global__ void __launch_bounds__(SY_THREADS, 1)
syrk_kernel(const double* __restrict__ T, const double* __restrict__ dvar, const double* __restrict__ craw,
            int MP, long long R, int nchunk, double* __restrict__ part_in, const unsigned int* __restrict__ clamp_count,
            const double* __restrict__ dmu_in, double* __restrict__ part_alpha_in, double* __restrict__ part_clamped) {
  const int which = (int)blockIdx.z;
  double* __restrict__ part = which == 1 ? part_clamped : part_in;
  const double* __restrict__ dmu = which == 0 ? dmu_in : nullptr;
  double* __restrict__ part_alpha = which == 0 ? part_alpha_in : nullptr;
  if (which == 1 && (clamp_count == nullptr || *clamp_count == 0u)) return;
  extern __shared__ __align__(16) double sy_sh[];
  __shared__ unsigned long long full[SY_STAGES];     // mbarriers: stage s % SY_STAGES has landed
  __shared__ unsigned long long empty[SY_STAGES];    // mbarriers: every consumer warp is done with the slot
  const int ld = MP + 4;
  const size_t stage = syrk_stage_doubles(MP);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int nblk = syrk_nblocks(MP);
  const int group = blockIdx.x, chunk = blockIdx.y;
  const bool producer = warp == SY_WARPS;
  const int q = group * SY_WARPS + warp;
  const bool active = !producer && q < nblk;
  int bi = 0, bj = 0;
  if (active) { int rem = q; while (rem > bi) { rem -= bi + 1; ++bi; } bj = rem; }
  const long long rows_per = ((R + nchunk - 1) / nchunk + SY_KB - 1) / SY_KB * SY_KB;
  const long long rbeg = (long long)chunk * rows_per;
  const long long rend = min(R, rbeg + rows_per);
  const int nst = rend > rbeg ? (int)((rend - rbeg + SY_KB - 1) / SY_KB) : 0;
  const bool do_alpha = which == 0 && part_alpha != nullptr && dmu != nullptr;
  const int acols = (MP + (int)gridDim.x - 1) / (int)gridDim.x;                 // columns of b per group
  const int aparts = acols * 4 <= SY_CONS_THREADS ? 4 : (acols * 2 <= SY_CONS_THREADS ? 2 : 1);
  const int apart = tid / acols, acol = group * acols + tid % acols;
  const bool alpha_thread = do_alpha && !producer && apart < aparts && acol < MP;
  const int ak0 = apart * (SY_KB / aparts), ak1 = ak0 + SY_KB / aparts;
  const unsigned row_bytes = (unsigned)MP * sizeof(double);
  // the three per-row arrays travel as 256-byte bulk copies when they are 16-byte aligned (always, for fresh
  // allocations); otherwise, and for the ragged last stage, warp 0 loads them itself
  const bool vec_ok = ((((uintptr_t)dvar) | ((uintptr_t)dmu) | ((uintptr_t)craw)) & 15) == 0;

  if (tid == 0) {
    for (int s = 0; s < SY_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], SY_WARPS); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  // the producer warp fills a stage: one 2 KB bulk copy per row of T (the TMA engine computes no per-element addresses: the
  // per-thread 16-byte cp.async loop of the first version spent 14 % of the kernel's samples on index arithmetic,
  // profiles/r01r_*), completion on the stage's mbarrier
  auto issue = [&](int s) {
    const int slot = s % SY_STAGES;
    double* Ts = sy_sh + (size_t)slot * stage;
    double* ws = Ts + (size_t)SY_KB * ld;
    const long long r0 = rbeg + (long long)s * SY_KB;
    const int nrow = (int)min((long long)SY_KB, rend - r0);
    const bool bulk_small = vec_ok && nrow == SY_KB;
    if (lane >= nrow)                                            // ragged last stage: zero rows (their weight is 0)
      for (int j = 0; j < MP; ++j) Ts[(size_t)lane * ld + j] = 0.0;
    if (!bulk_small) {
      const bool ok = lane < nrow;
      ws[lane] = (ok && dvar) ? dvar[r0 + lane] : 0.0;
      ws[SY_KB + lane] = (ok && dmu) ? dmu[r0 + lane] : 0.0;
      ws[2 * SY_KB + lane] = (ok && craw) ? craw[r0 + lane] : 0.0;
    } else {
      if (!dmu) ws[SY_KB + lane] = 0.0;
      if (!craw) ws[2 * SY_KB + lane] = 0.0;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic accesses to the slot -> async writes
    __syncwarp();
    if (lane == 0) {
      unsigned bytes = (unsigned)nrow * row_bytes;
      if (bulk_small) bytes += (unsigned)SY_KB * 8u * (1u + (dmu ? 1u : 0u) + (craw ? 1u : 0u));
      mbar_expect_tx(&full[slot], bytes);                        // release: the generic writes above are visible
      if (bulk_small) {
        bulk_g2s(ws, dvar + r0, SY_KB * 8u, &full[slot]);
        if (dmu) bulk_g2s(ws + SY_KB, dmu + r0, SY_KB * 8u, &full[slot]);
        if (craw) bulk_g2s(ws + 2 * SY_KB, craw + r0, SY_KB * 8u, &full[slot]);
      }
    }
    __syncwarp();
    if (lane < nrow) bulk_g2s(Ts + (size_t)lane * ld, T + (size_t)(r0 + lane) * MP, row_bytes, &full[slot]);
  };

  double acc[4][4][2];
#pragma unroll
  for (int x = 0; x < 4; ++x)
#pragma unroll
    for (int y = 0; y < 4; ++y) { acc[x][y][0] = 0.0; acc[x][y][1] = 0.0; }
  double al[4] = {0.0, 0.0, 0.0, 0.0};

  if (producer) {
    for (int s = 0; s < nst; ++s) {
      if (s >= SY_STAGES) mbar_wait(&empty[s % SY_STAGES], (unsigned)(s / SY_STAGES - 1) & 1u);
      issue(s);
    }
    return;
  }
  for (int it = 0; it < nst; ++it) {
    const int slot = it % SY_STAGES;
    mbar_wait(&full[slot], (unsigned)(it / SY_STAGES) & 1u);
    const double* Ts = sy_sh + (size_t)slot * stage;
    const double* ws = Ts + (size_t)SY_KB * ld;
    if (active) {
      const double* Ap = Ts + 32 * bi + g;
      const double* Bp = Ts + 32 * bj + g;
#pragma unroll 2
      for (int k0 = 0; k0 < SY_KB; k0 += 4) {
        const int k = k0 + t;
        double w = ws[k];
        if (which == 1) w = ws[2 * SY_KB + k] < 0.0 ? w : 0.0;
        double af[4], bf[4];
#pragma unroll
        for (int x = 0; x < 4; ++x) af[x] = Ap[(size_t)k * ld + 8 * x] * w;
#pragma unroll
        for (int y = 0; y < 4; ++y) bf[y] = Bp[(size_t)k * ld + 8 * y];
#pragma unroll
        for (int x = 0; x < 4; ++x)
#pragma unroll
          for (int y = 0; y < 4; ++y) dmma884(acc[x][y][0], acc[x][y][1], af[x], bf[y]);
      }
    }
    if (alpha_thread) {
      for (int k = ak0; k < ak1; k += 4)
#pragma unroll
        for (int c = 0; c < 4; ++c) al[c] = fma(ws[SY_KB + k + c], Ts[(size_t)(k + c) * ld + acol], al[c]);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty[slot]);      // this warp is done with the slot
  }
  if (active) {
    double* out = part + ((size_t)chunk * nblk + q) * 1024;
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
      for (int y = 0; y < 4; ++y)
#pragma unroll
        for (int e = 0; e < 2; ++e) out[(8 * x + g) * 32 + 8 * y + 2 * t + e] = acc[x][y][e];
  }
  if (do_alpha) {       // slices a thread count does not reach stay zero
    if (alpha_thread) part_alpha[((size_t)chunk * SY_ALPHA_PARTS + apart) * MP + acol] = (al[0] + al[1]) + (al[2] + al[3]);
    for (int idx = tid; idx < (SY_ALPHA_PARTS - aparts) * acols; idx += SY_CONS_THREADS) {
      const int pz = aparts + idx / acols, cz = group * acols + idx % acols;
      if (cz < MP) part_alpha[((size_t)chunk * SY_ALPHA_PARTS + pz) * MP + cz] = 0.0;
    }
  }
}

__global__ void syrk_reduce_kernel(const double* __restrict__ part, int nchunk, int MP, double* __restrict__ A,
                                   int which, const unsigned int* __restrict__ clamp_count,
                                   double* __restrict__ clamp_flag_out) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx == 0 && which == 1 && clamp_flag_out) *clamp_flag_out = clamp_count ? (double)(*clamp_count) : 0.0;
  if (idx >= MP * MP) return;
  if (which == 1 && (clamp_count == nullptr || *clamp_count == 0u)) { A[idx] = 0.0; return; }
  int i = idx / MP, j = idx - (idx / MP) * MP;
  if (j > i) { const int tmp = i; i = j; j = tmp; }      // lower triangle (also inside diagonal blocks) -> symmetric
  const int bi = i >> 5, bj = j >> 5;
  const int q = bi * (bi + 1) / 2 + bj;
  const int nblk = syrk_nblocks(MP);
  const size_t off = (size_t)q * 1024 + (size_t)(i & 31) * 32 + (j & 31);
  double s = 0.0;
  for (int c = 0; c < nchunk; ++c) s += part[(size_t)c * nblk * 1024 + off];
  A[idx] = s;
}

// ---------------------------------------------------------------------------------------------------
// host launchers
// ---------------------------------------------------------------------------------------------------
// per-device state (a process normally drives one GPU, but nothing here may assume it)
constexpr int kMaxDevices = 64;
static int current_device() {
  int dev = 0;
  cudaGetDevice(&dev);
  return dev & (kMaxDevices - 1);
}
static int num_sms() {
  static int sms[kMaxDevices] = {0};
  const int dev = current_device();
  if (sms[dev] == 0) {
    cudaDeviceGetAttribute(&sms[dev], cudaDevAttrMultiProcessorCount, dev);
    if (sms[dev] <= 0) sms[dev] = 148;
  }
  return sms[dev];
}
// true the first time it is called with this flag array on the current device (dynamic shared-memory opt-in is a
// per-device function attribute)
static bool first_on_device(bool (&done)[kMaxDevices]) {
  const int dev = current_device();
  if (done[dev]) return false;
  done[dev] = true;
  return true;
}

int row_grid(long long R) {
  const long long ntiles = (R + TR - 1) / TR;
  const long long cap = (long long)num_sms() * ROW_CTAS_PER_SM;
  return (int)(ntiles < cap ? (ntiles > 0 ? ntiles : 1) : cap);
}

// 32-bit row indices in the kernels; callers chunk (MFDGP.ACQ_CHUNK, MFDGP.ACQ_GRAD_CHUNK)
constexpr long long kMaxRows = (1ll << 31) - TR;

int launch_row_fwd(const RowArgs& a, cudaStream_t st) {
  if (a.MP % 32 != 0 || a.MP > MAX_MP || a.d > kMaxD || a.M > a.MP) return -2;
  if (a.R >= kMaxRows) return -2;
  const size_t smem = row_smem_bytes(a.MP);
  static bool attr_done[kMaxDevices] = {false};
  if (first_on_device(attr_done))
    cudaFuncSetAttribute(row_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)row_smem_bytes(MAX_MP));
  static bool attr_done_ws[kMaxDevices] = {false};
  if (first_on_device(attr_done_ws))
    cudaFuncSetAttribute(row_fwd_ws_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ws_smem_bytes(MAX_MP));
  if (a.R <= 0) return 0;
  if (a.kind == 1 && a.xrep >= XSHARE_MIN_REP) {
    // rows are MC samples of few points (S-sample training, acquisition): the warp-specialised kernel, one CTA per SM
    if ((a.Tsave && ((uintptr_t)a.Tsave & 15)) || (a.Usave && ((uintptr_t)a.Usave & 15))) return -2;   // bulk copies
    const long long ntiles = (a.R + TR - 1) / TR;
    const long long grid = ntiles < num_sms() ? ntiles : num_sms();
    MOBO_LAUNCH("row_fwd_ws_kernel", st,
                row_fwd_ws_kernel<<<(int)grid, WS_THREADS, ws_smem_bytes(a.MP), st>>>(a));
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
  }
  MOBO_LAUNCH("row_fwd_kernel", st, row_fwd_kernel<<<row_grid(a.R), ROW_THREADS, smem, st>>>(a));
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

int kgrad_grid(long long R) {
  const long long ntiles = (R + KG_ROWS - 1) / KG_ROWS;
  const long long cap = (long long)num_sms() * KG_CTAS_PER_SM;
  return (int)(ntiles < cap ? (ntiles > 0 ? ntiles : 1) : cap);
}

// product kernel (dk into a.dk) followed by the covariance-gradient kernel; per-CTA partials of the latter are
// indexed by ITS grid (kgrad_grid)
// grid of the backward product kernel: one persistent CTA per SM, minus `reserve` SMs; then the smallest grid that
// needs the same number of tile rounds (the freed SMs run the concurrent side-stream kernels of the fused step: with
// every SM's registers and shared memory taken by this kernel they would otherwise wait for it to finish)
int row_bwd_grid(long long R, int reserve) {
  const long long ntiles = (R + TR - 1) / TR;
  long long cap = num_sms() - reserve;
  if (cap < 1) cap = 1;
  if (ntiles <= cap) return (int)(ntiles > 0 ? ntiles : 1);
  const long long rounds = (ntiles + cap - 1) / cap;
  return (int)((ntiles + rounds - 1) / rounds);
}

int launch_row_bwd(const RowArgs& a, cudaStream_t st) {
  if (a.MP % 32 != 0 || a.MP > MAX_MP || a.d > kMaxD || a.M > a.MP) return -2;
  static bool attr_done[kMaxDevices] = {false};
  if (first_on_device(attr_done)) {
    cudaFuncSetAttribute(row_bwd_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bwd_smem_bytes(MAX_MP));
    cudaFuncSetAttribute(kgrad_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kg_smem_bytes());
    cudaFuncSetAttribute(kgrad_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kg_smem_bytes());
    cudaFuncSetAttribute(kgrad_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kg_smem_bytes());
  }
  if (a.R <= 0) return 0;
  if (((uintptr_t)a.Tsave | (uintptr_t)a.Usave) & 15) return -2;   // bulk copies need 16-byte aligned rows
  const int grid_b = row_bwd_grid(a.R, a.sm_reserve);
  MOBO_LAUNCH("row_bwd_gemm_kernel", st,
              row_bwd_gemm_kernel<<<grid_b, BWD_THREADS, bwd_smem_bytes(a.MP), st>>>(a));
  const int grid = kgrad_grid(a.R);
  const size_t smem = kg_smem_bytes();
  if (a.want_param_grads && a.want_x_grads) {
    MOBO_LAUNCH("kgrad_kernel<param,x>", st, kgrad_kernel<true, true><<<grid, KG_THREADS, smem, st>>>(a));
  } else if (a.want_x_grads) {
    MOBO_LAUNCH("kgrad_kernel<x>", st, kgrad_kernel<false, true><<<grid, KG_THREADS, smem, st>>>(a));
  } else {
    MOBO_LAUNCH("kgrad_kernel<param>", st, kgrad_kernel<true, false><<<grid, KG_THREADS, smem, st>>>(a));
  }
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

int launch_reduce_partials(const double* part, int nblocks, int n, int stride, double* out, int accumulate,
                           cudaStream_t st) {
  MOBO_LAUNCH("reduce_partials_kernel", st, reduce_partials_kernel<<<(n + 3) / 4, 128, 0, st>>>(part, nblocks, n, stride, out, accumulate));
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

int syrk_ngroups(int MP) { return (syrk_nblocks(MP) + SY_WARPS - 1) / SY_WARPS; }

int syrk_nchunk(int MP, long long R) {
  long long want = num_sms() / syrk_ngroups(MP);           // one CTA per SM (the pipeline takes most of its smem)
  const long long maxc = (R + 2 * SY_KB - 1) / (2 * SY_KB);
  if (want > maxc) want = maxc;
  if (want < 1) want = 1;
  return (int)want;
}

size_t syrk_part_doubles(int MP, long long R) { return (size_t)syrk_nblocks(MP) * syrk_nchunk(MP, R) * 1024; }

// the SYRK proper (DMMA-bound), both weight sets (all rows -> part, clamped rows only -> part_clamped) in ONE launch:
// per-chunk partial blocks, syrk_part_doubles(MP, R) doubles each, and partial b into part_alpha,
// syrk_alpha_doubles(MP, syrk_nchunk(MP, R)) doubles
int launch_syrk_both(const double* K, const double* dvar, const double* craw, int MP, long long R, double* part,
                     double* part_clamped, const unsigned int* clamp_count, const double* dmu, double* part_alpha,
                     cudaStream_t st) {
  const int nc = syrk_nchunk(MP, R);
  const size_t smem = SY_STAGES * syrk_stage_doubles(MP) * sizeof(double);
  static bool attr_done[kMaxDevices] = {false};
  if (first_on_device(attr_done))
    cudaFuncSetAttribute(syrk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         (int)(SY_STAGES * syrk_stage_doubles(MAX_MP) * sizeof(double)));
  dim3 grid(syrk_ngroups(MP), nc, 2);
  MOBO_LAUNCH("syrk_kernel", st, syrk_kernel<<<grid, SY_THREADS, smem, st>>>(K, dvar, craw, MP, R, nc, part, clamp_count, dmu,
                                           part_alpha, part_clamped));
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

// fixed-order fold of the partials into the symmetric matrix A (and b), latency-bound: may run on another stream
int launch_syrk_reduce(int which, int MP, long long R, const double* part, double* A,
                       const unsigned int* clamp_count, const double* part_alpha, double* dalpha,
                       double* clamp_flag_out, cudaStream_t st) {
  const int nc = syrk_nchunk(MP, R);
  MOBO_LAUNCH("syrk_reduce_kernel", st, syrk_reduce_kernel<<<(MP * MP + 255) / 256, 256, 0, st>>>(part, nc, MP, A, which, clamp_count, clamp_flag_out));
  if (which == 0 && part_alpha && dalpha)
    MOBO_LAUNCH("reduce_partials_kernel", st, reduce_partials_kernel<<<(MP + 3) / 4, 128, 0, st>>>(part_alpha, nc * SY_ALPHA_PARTS, MP, MP, dalpha, 0));
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

}  // namespace mobo
