// Shared device helpers for the mobocmf_b200 sm_100a kernels.
//
// FP64 matrix work uses the DMMA pipe: on sm_100a every f64 mma.sync shape lowers to DMMA.8x8x4 (checked with
// cuobjdump), which peaks at 37.1 TFLOP/s on B200 (profiles/r01_fp64_probe.log) against 35.4 TFLOP/s for cuBLAS
// DGEMM.  tcgen05/UMMA has no f64 kind, so mma.sync.m8n8k4.f64 is the tensor instruction for this path.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

namespace mobo {

// ---- launch accounting / optional per-launch CUDA-event timing (mobo_profile_* in the C ABI) ----
struct ProfRec { const char* name; cudaEvent_t e0, e1; };
struct ProfState {
  bool on = false;
  long long launches = 0;
  std::vector<ProfRec> recs;
  std::vector<cudaEvent_t> pool;
};
inline ProfState& prof_state() { static ProfState s; return s; }
inline cudaEvent_t prof_event() {
  ProfState& s = prof_state();
  if (!s.pool.empty()) { cudaEvent_t e = s.pool.back(); s.pool.pop_back(); return e; }
  cudaEvent_t e; cudaEventCreate(&e); return e;
}
inline void prof_begin(const char* name, cudaStream_t st) {
  ProfState& s = prof_state();
  ++s.launches;
  if (s.on) { ProfRec r{name, prof_event(), prof_event()}; cudaEventRecord(r.e0, st); s.recs.push_back(r); }
}
inline void prof_end(cudaStream_t st) {
  ProfState& s = prof_state();
  if (s.on) cudaEventRecord(s.recs.back().e1, st);
}
// every kernel launch of the library goes through this macro
#define MOBO_LAUNCH(name, st, ...) do { mobo::prof_begin(name, st); __VA_ARGS__; mobo::prof_end(st); } while (0)

constexpr int kMaxD = 8;               // max number of x columns (ARD dims) handled by the kernels
constexpr int kMaxLayers = 8;          // max number of layers of a model (MOBO_MAX_LAYERS in the C header)
constexpr int kMaxTheta = 5 + 2 * kMaxD;   // hyper-parameter slots of a layer (theta_size(1, kMaxD); MOBO_MAX_THETA)
constexpr double kMinVariance = 1e-10; // gpytorch settings.min_variance (fp64), quirk Q9

// ---- operator buffer layout (doubles), one per (model, layer); MP = M rounded up to a multiple of 32 ----
// [L | W | WT | H | HT | P | LQ | WF | HTF | HF | WTF]  eleven MP x MP blocks, then beta[MP], alpha[MP], scal[16],
// rowstat[4 MP], flags[128]
//   L = chol(K_zz + jitter I), W = L^-1, WT = W^T, H = W tril(L_q), HT = H^T, P = K_zz + jitter I, LQ = tril(L_q)
//   (row-major), and WF / HTF / HF / WTF = W / HT / H / WT again in DMMA A-fragment order (frag_offset below), the
//   form the row kernels stream them in: one 16-byte load per lane and k-step, 512 contiguous bytes per warp.
//   Only the 32 x 32 blocks of the populated triangle (diagonal blocks included) of the fragment copies are written.
// The GRADIENT buffer of an operator buffer has the same layout and carries, by convention of this library,
//   block OPS_W: A2 = sum_r dvar_r t_r t_r^T (t = W k),  block OPS_H: Ac = same over clamped rows only,
//   alpha slot: b = sum_r dmu_r t_r,  scal[SC_KL]: d loss / d KL, scal[SC_CLAMP]: #clamped rows;  rest ignored.
enum OpsBlock { OPS_L = 0, OPS_W = 1, OPS_WT = 2, OPS_H = 3, OPS_HT = 4, OPS_P = 5, OPS_LQ = 6,
                OPS_WF = 7, OPS_HTF = 8, OPS_HF = 9, OPS_WTF = 10, OPS_NBLOCKS = 11 };
// A-fragment order of mma.sync.m8n8k4.f64 for 16-row slabs: element (i, k) of an MP x MP operator lives at
//   ((i / 16) * (MP / 4) + k / 4) * 64 + 2 * lane + (i / 8) % 2,   lane = 4 * (i % 8) + k % 4
// so lane `lane` of a warp working on slab s reads the double2 {A[16 s + g][k0 + t], A[16 s + 8 + g][k0 + t]}.
__host__ __device__ inline size_t frag_offset(int MP, int i, int k) {
  return ((size_t)(i >> 4) * (MP >> 2) + (k >> 2)) * 64 + 2 * (4 * (i & 7) + (k & 3)) + ((i >> 3) & 1);
}
// scal[SC_CLAMP] is meaningful in the GRADIENT buffer: number of clamped rows behind block OPS_H (0 -> Ac == 0)
// scal[SC_RETRIES]: number of psd_safe_cholesky retries the operator chain needed (0 .. 3); SC_STATUS = 1: all failed
enum OpsScal { SC_KL = 0, SC_LOGDET_P = 1, SC_LOGDET_Q = 2, SC_BETA2 = 3, SC_H2 = 4, SC_STATUS = 5, SC_CLAMP = 6,
               SC_RETRIES = 7 };
__host__ __device__ inline size_t ops_block(int MP, int b) { return (size_t)b * MP * MP; }
__host__ __device__ inline size_t ops_beta(int MP) { return (size_t)OPS_NBLOCKS * MP * MP; }
__host__ __device__ inline size_t ops_alpha(int MP) { return (size_t)OPS_NBLOCKS * MP * MP + MP; }
__host__ __device__ inline size_t ops_scal(int MP) { return (size_t)OPS_NBLOCKS * MP * MP + 2 * MP; }
__host__ __device__ inline size_t ops_rowstat(int MP) { return (size_t)OPS_NBLOCKS * MP * MP + 2 * MP + 16; }
// 256 ints of block-to-block flags of the cooperative operator-chain kernel (opchain.cu)
__host__ __device__ inline size_t ops_flags(int MP) { return (size_t)OPS_NBLOCKS * MP * MP + 6 * MP + 16; }
__host__ __device__ inline size_t ops_size(int MP) { return (size_t)OPS_NBLOCKS * MP * MP + 6 * MP + 16 + 128; }

// D(8x8) += A(8x4, row) * B(4x8, col).  lane = 4*g + t:  A[g][t], B[t][g], C[g][2t..2t+1].
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---- layer covariance function --------------------------------------------------------------------
// kind 0 (layer 0,  layers/mfdgp_hidden_layer.py:43-47):   k = a * exp(-1/2 sum_c ((x_c-z_c)/l_c)^2)
// kind 1 (layer>=1, layers/mfdgp_hidden_layer.py:70-88,115): k = a1*E1*(v*f*f' + af*Ef) + a2*E2
// theta (constrained values): kind 0: [a, l_0..l_{d-1}];  kind 1: [a1, v, af, lf, a2, l1_0.., l2_0..]
struct KernParams {
  int kind, d;
  double a1, vlin, af, ilf, a2;
  double il1[kMaxD], il2[kMaxD];  // 1 / l^2
};

__device__ inline void load_kern_params(KernParams& kp, int kind, int d, const double* __restrict__ theta) {
  kp.kind = kind;
  kp.d = d;
  for (int c = 0; c < kMaxD; ++c) { kp.il1[c] = 0.0; kp.il2[c] = 0.0; }
  if (kind == 0) {
    kp.a1 = theta[0];
    kp.vlin = 0.0; kp.af = 0.0; kp.ilf = 0.0; kp.a2 = 0.0;
    for (int c = 0; c < d; ++c) { double l = theta[1 + c]; kp.il1[c] = 1.0 / (l * l); kp.il2[c] = 0.0; }
  } else {
    kp.a1 = theta[0]; kp.vlin = theta[1]; kp.af = theta[2];
    double lf = theta[3];
    kp.ilf = 1.0 / (lf * lf);
    kp.a2 = theta[4];
    for (int c = 0; c < d; ++c) {
      double l1 = theta[5 + c], l2 = theta[5 + d + c];
      kp.il1[c] = 1.0 / (l1 * l1);
      kp.il2[c] = 1.0 / (l2 * l2);
    }
  }
}

__host__ __device__ inline int theta_size(int kind, int d) { return kind == 0 ? 1 + d : 5 + 2 * d; }

// diag k(x,x) for a row with propagated input f
__device__ __forceinline__ double kern_diag(const KernParams& kp, double f) {
  if (kp.kind == 0) return kp.a1;
  return kp.a1 * (kp.vlin * f * f + kp.af) + kp.a2;
}

// k((xa, fa), (xb, fb)) off the diagonal (fa, fb unused for kind 0)
__device__ __forceinline__ double kern_entry(const KernParams& kp, int d, const double* xa, double fa, const double* xb,
                                             double fb) {
  double D1 = 0.0, D2 = 0.0;
  for (int c = 0; c < d; ++c) {
    const double df = xa[c] - xb[c];
    D1 = fma(df * df, kp.il1[c], D1);
    D2 = fma(df * df, kp.il2[c], D2);
  }
  const double E1 = exp(-0.5 * D1);
  if (kp.kind == 0) return kp.a1 * E1;
  const double dff = fa - fb;
  return kp.a1 * E1 * (kp.vlin * fa * fb + kp.af * exp(-0.5 * dff * dff * kp.ilf)) + kp.a2 * exp(-0.5 * D2);
}

// accumulators of g * dk / dtheta: s[0..4] = d / d (a1, v, af, lf-term, a2), l1 / l2 = sum g (a1 E1 gg | a2 E2) D_c^2;
// kern_theta_slot maps them to the theta layout
struct KernAcc {
  double s[5], l1[kMaxD], l2[kMaxD];
  __device__ __forceinline__ void zero() {
#pragma unroll
    for (int q = 0; q < 5; ++q) s[q] = 0.0;
#pragma unroll
    for (int c = 0; c < kMaxD; ++c) { l1[c] = 0.0; l2[c] = 0.0; }
  }
};

// g * dk((xa, fa), (xb, fb)) / dtheta into acc (off the diagonal); ca, cb = dk / dfa, dk / dfb WITHOUT the weight g
// (0 for kind 0), so that each caller keeps its own accumulation order
__device__ __forceinline__ void kern_entry_bwd(const KernParams& kp, int d, const double* xa, double fa,
                                               const double* xb, double fb, double g, KernAcc& acc, double& ca,
                                               double& cb) {
  double d2[kMaxD], D1 = 0.0, D2 = 0.0;
#pragma unroll
  for (int c = 0; c < kMaxD; ++c) {
    const double df = c < d ? xa[c] - xb[c] : 0.0;
    d2[c] = df * df;
    D1 = fma(d2[c], kp.il1[c], D1);
    D2 = fma(d2[c], kp.il2[c], D2);
  }
  const double E1 = exp(-0.5 * D1);
  if (kp.kind == 0) {
    const double gkk = g * kp.a1 * E1;
    acc.s[0] = fma(g, E1, acc.s[0]);
#pragma unroll
    for (int c = 0; c < kMaxD; ++c) acc.l1[c] = fma(gkk, d2[c], acc.l1[c]);
    ca = 0.0; cb = 0.0;
    return;
  }
  const double dff = fa - fb;
  const double Ef = exp(-0.5 * dff * dff * kp.ilf), E2 = exp(-0.5 * D2);
  const double gg = kp.vlin * fa * fb + kp.af * Ef;
  const double s1 = kp.a1 * E1, s2 = kp.a2 * E2;
  const double dEf = s1 * kp.af * Ef * dff * kp.ilf;
  ca = s1 * kp.vlin * fb - dEf;
  cb = s1 * kp.vlin * fa + dEf;
  acc.s[0] = fma(g, E1 * gg, acc.s[0]);
  acc.s[1] = fma(g, s1 * fa * fb, acc.s[1]);
  acc.s[2] = fma(g, s1 * Ef, acc.s[2]);
  acc.s[3] = fma(g, dEf * dff, acc.s[3]);
  acc.s[4] = fma(g, E2, acc.s[4]);
  const double g1 = g * s1 * gg, g2 = g * s2;
#pragma unroll
  for (int c = 0; c < kMaxD; ++c) { acc.l1[c] = fma(g1, d2[c], acc.l1[c]); acc.l2[c] = fma(g2, d2[c], acc.l2[c]); }
}

// g * d kern_diag(f) / dtheta into acc; returns g a1 v, so that g * d kern_diag / df = 2 (g a1 v) f (0 for kind 0)
__device__ __forceinline__ double kern_diag_bwd(const KernParams& kp, double f, double g, KernAcc& acc) {
  if (kp.kind == 0) { acc.s[0] += g; return 0.0; }
  acc.s[0] += g * (kp.vlin * f * f + kp.af);
  acc.s[1] += g * kp.a1 * f * f;
  acc.s[2] += g * kp.a1;
  acc.s[4] += g;
  return g * kp.a1 * kp.vlin;
}

// accumulator q (s[0..4], then l1[0..kMaxD), then l2[0..kMaxD)) summed to s -> its theta slot (return value, -1:
// none) and the value there: a length-scale sum times il^(3/2) is d / d l, s[3] (one il_f inside) times sqrt(il_f)
__device__ __forceinline__ int kern_theta_slot(const KernParams& kp, int q, double s, double& out) {
  if (q < 5) {
    out = q == 3 ? s * sqrt(kp.ilf) : s;
    return kp.kind == 1 ? q : (q == 0 ? 0 : -1);
  }
  const bool first = q < 5 + kMaxD;          // l1 (kind 0: its only length scales) or l2
  const int c = first ? q - 5 : q - 5 - kMaxD;
  const double il = first ? kp.il1[c] : kp.il2[c];
  out = s * il * sqrt(il);
  if (c >= kp.d) return -1;
  if (kp.kind == 0) return first ? 1 + c : -1;
  return first ? q : 5 + kp.d + c;
}

}  // namespace mobo
