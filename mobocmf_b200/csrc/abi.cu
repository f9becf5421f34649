// extern "C" entry points of libmobocmf_b200.so (declared in include/mobocmf_b200.h) and the host-side kernel
// sequences behind them.
#include <string.h>
#include <mutex>
#include "../../include/mobocmf_b200.h"
#include "matrix_ops.cu"
#include "opchain.cu"
#include "row_pass.cu"
#include "step.cu"
#include "small_step.cu"
#include "rff.cu"

using namespace mobo;

static_assert(kMaxLayers == MOBO_MAX_LAYERS && kMaxTheta == MOBO_MAX_THETA, "the kernels' limits are the header's");

static inline int padded(int M) { return ((M + 31) / 32) * 32; }
#define MOBO_TRY(x) do { int _e = (x); if (_e) return _e; } while (0)

extern "C" {

int mobo_abi_version(void) { return 103; }

long long mobo_launch_count(void) { return prof_state().launches; }

void mobo_profile_enable(int on) { prof_state().on = on != 0; }

int mobo_profile_collect(char* names, size_t names_bytes, float* ms, int max_records) {
  ProfState& s = prof_state();
  int n = 0;
  size_t off = 0;
  for (ProfRec& r : s.recs) {
    cudaEventSynchronize(r.e1);
    float t = 0.f;
    cudaEventElapsedTime(&t, r.e0, r.e1);
    if (n < max_records) {
      const size_t len = strlen(r.name) + 1;
      if (off + len <= names_bytes) {
        memcpy(names + off, r.name, len);
        off += len;
        ms[n++] = t;
      }
    }
    s.pool.push_back(r.e0);
    s.pool.push_back(r.e1);
  }
  s.recs.clear();
  return n;
}
int mobo_padded_m(int M) { return padded(M); }
size_t mobo_ops_doubles(int M) { return ops_size(padded(M)); }

size_t mobo_rows_save_doubles(int M, long long R) {
  const long long ntiles = (R + TR - 1) / TR;
  return (size_t)ntiles * TR * padded(M);
}

size_t mobo_rows_bwd_work_doubles(int M, long long R) {
  const int MP = padded(M);
  return (size_t)256 * KG_CTAS_PER_SM * (kMaxTheta + MP) + 2 * syrk_part_doubles(MP, R) +
         syrk_alpha_doubles(MP, syrk_nchunk(MP, R)) + 64 + mobo_rows_save_doubles(M, R);   // + the dk scratch [R][MP]
}

size_t mobo_precompute_bwd_work_doubles(int M) {
  const int MP = padded(M);
  return (size_t)8 * MP * MP + (size_t)((M + KZB_WARPS - 1) / KZB_WARPS) * kMaxTheta + 64;
}

// The operator chains of nl layers in one cooperative launch: a CTA per 32 x 32 block of the lower triangle of every
// layer (opchain.cu).  reset_flags = false: the caller has already zeroed the flags region of every operator buffer
// on this stream.
static int model_precompute(int nl, const int* kinds, int d, int M, const double* const* Zx, const double* const* zf,
                            const double* const* theta, const double* const* m, const double* const* Lq,
                            double jitter, double* const* ops, cudaStream_t st, bool reset_flags) {
  const int MP = padded(M);
  if (nl < 1 || nl > kMaxLayers || d > kMaxD || MP > MAX_MP) return -2;
  LayerBatch b = {};
  b.n = nl; b.d = d; b.M = M; b.MP = MP;
  for (int i = 0; i < nl; ++i) {
    b.kind[i] = kinds[i]; b.Zx[i] = Zx[i]; b.zf[i] = zf[i]; b.theta[i] = theta[i];
    b.m[i] = m[i]; b.Lq[i] = Lq[i]; b.ops[i] = ops[i];
  }
  const int nb = MP / 32, nblk = nb * (nb + 1) / 2;
  if (reset_flags) MOBO_LAUNCH("opchain_reset_kernel", st, opchain_reset_kernel<<<nl, 128, 0, st>>>(b));
  void* args[] = {(void*)&b, (void*)&jitter};
  prof_begin("opchain_kernel", st);
  const cudaError_t e = cudaLaunchCooperativeKernel((const void*)opchain_kernel, dim3(nl * nblk), dim3(OC_THREADS), args,
                                                    0, st);
  prof_end(st);
  if (e != cudaSuccess) return -1;
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

int mobo_layer_precompute(int kind, int d, int M, const double* Zx, const double* zf, const double* theta,
                          const double* m, const double* Lq, double jitter, double* ops, void* stream) {
  return model_precompute(1, &kind, d, M, &Zx, &zf, &theta, &m, &Lq, jitter, &ops, (cudaStream_t)stream, true);
}

// m and Lq reach the backward through the operators built from them (beta, H, LQ)
int mobo_layer_precompute_bwd(int kind, int d, int M, const double* Zx, const double* zf, const double* theta,
                              const double* m, const double* Lq, const double* ops, const double* gops,
                              double* work, double* dtheta, double* dzf, double* dm, double* dLq, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  const int MP = padded(M);
  if (d > kMaxD || MP > MAX_MP) return -2;
  const size_t MP2 = (size_t)MP * MP;
  // work: eight MP x MP blocks, then the per-CTA partials of kzz_bwd_kernel
  double* G2 = work;
  double* V = G2 + MP2;
  double* N = V + MP2;
  double* F = N + MP2;
  double* X1 = F + MP2;
  double* dP = X1 + MP2;
  double* X2 = dP + MP2;
  double* Y2 = X2 + MP2;
  double* part = Y2 + MP2;
  const double* W = ops + ops_block(MP, OPS_W);
  const double* WT = ops + ops_block(MP, OPS_WT);
  const double* H = ops + ops_block(MP, OPS_H);
  const double* beta = ops + ops_beta(MP);
  const double* A2 = gops + ops_block(MP, OPS_W);
  const double* b = gops + ops_alpha(MP);
  const double* dkl = gops + ops_scal(MP) + SC_KL;
  // G2 = H H^T
  MOBO_TRY(gemm(MP, {H, false, 1}, {H, true, 2}, G2, st));
  // V = A2 G2
  MOBO_TRY(gemm(MP, {A2, false, 0}, {G2, false, 0}, V, st));
  // whitened core N and F = 2 A2 + g I
  MOBO_LAUNCH("combine_kernel", st,
              combine_kernel<<<(unsigned)((MP2 + 255) / 256), 256, 0, st>>>(
                  A2, gops + ops_block(MP, OPS_H), V, G2, b, beta, dkl, gops + ops_scal(MP) + SC_CLAMP, N, F, MP));
  // dP = W^T N W
  MOBO_TRY(gemm(MP, {WT, false, 2}, {N, false, 0}, X1, st));
  MOBO_TRY(gemm(MP, {X1, false, 0}, {W, false, 1}, dP, st));
  // dLq = tril(W^T F H) - g diag(1 / Lq_ii)
  MOBO_TRY(gemm(MP, {F, false, 0}, {H, false, 1}, X2, st));
  MOBO_TRY(gemm(MP, {WT, false, 2}, {X2, false, 0}, Y2, st));
  MOBO_LAUNCH("dlq_extract_kernel", st,
              dlq_extract_kernel<<<(M * M + 255) / 256, 256, 0, st>>>(Y2, ops + ops_block(MP, OPS_LQ), dkl, dLq, M, MP));
  // dm = W^T (b + g beta)
  MOBO_LAUNCH("white_vec_kernel", st, white_vec_kernel<<<(M + 7) / 8, 256, 0, st>>>(WT, b, beta, dkl, dm, M, MP));
  // through K(Z, Z)
  const int nblk = (M + KZB_WARPS - 1) / KZB_WARPS;
  MOBO_LAUNCH("kzz_bwd_kernel", st,
              kzz_bwd_kernel<<<nblk, KZB_WARPS * 32, 0, st>>>(kind, d, M, MP, Zx, zf, theta, dP, part, dzf));
  MOBO_LAUNCH("reduce_batch_kernel", st,
              reduce_batch_kernel<<<1, 32, 0, st>>>(part, nblk, kMaxTheta, theta_size(kind, d), dtheta));
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

static void fill_row_args(RowArgs& a, int kind, int d, int M, const double* Zx, const double* zf,
                          const double* theta, const double* ops, const double* x, int xrep, const double* mu_prev,
                          const double* var_prev, int prep, const double* eps, long long eps_mod,
                          const double* f_direct, long long R, int training) {
  a.kind = kind; a.d = d; a.M = M; a.MP = padded(M);
  a.Zx = Zx; a.zf = zf; a.theta = theta; a.ops = ops; a.x = x; a.xrep = xrep < 1 ? 1 : xrep;
  a.mu_prev = mu_prev; a.var_prev = var_prev; a.prep = prep < 1 ? 1 : prep;
  a.eps = eps; a.eps_mod = eps_mod < 1 ? 1 : eps_mod; a.f_direct = f_direct; a.R = R; a.training = training;
  a.mu = nullptr; a.var = nullptr; a.craw = nullptr; a.clamp_count = nullptr;
  a.Tsave = nullptr; a.Usave = nullptr;
  a.dmu = nullptr; a.dvar = nullptr; a.dk = nullptr; a.df = nullptr; a.dxrow = nullptr; a.part_theta = nullptr; a.part_zf = nullptr;
  a.want_param_grads = 0; a.want_x_grads = 0; a.sm_reserve = 0;
}

int mobo_layer_rows_fwd(int kind, int d, int M, const double* Zx, const double* zf, const double* theta,
                        const double* ops, const double* x, int xrep, const double* mu_prev, const double* var_prev,
                        int prep, const double* eps, long long eps_mod, const double* f_direct, long long R,
                        int training, double* mu, double* var, double* craw, unsigned int* clamp_count,
                        double* Tsave, double* Usave, void* stream) {
  RowArgs a;
  fill_row_args(a, kind, d, M, Zx, zf, theta, ops, x, xrep, mu_prev, var_prev, prep, eps, eps_mod, f_direct, R,
                training);
  a.mu = mu; a.var = var; a.craw = craw; a.clamp_count = clamp_count;
  a.Tsave = Tsave; a.Usave = Usave;
  return launch_row_fwd(a, (cudaStream_t)stream);
}

// the whitened statistics of one layer's backward (SYRK): A2, Ac, b into the operator-gradient buffer.  One launch
// for both weight sets (all rows -> part, clamped rows -> part_clamped; clamp_count NULL: none clamped), then the
// fixed-order fold of the partials (latency-bound), which may run on another stream `rs` once `ev` (recorded on `st`
// behind the SYRK) has fired
static int rows_bwd_stats(int MP, long long R, const double* Tsave, const double* dmu, const double* dvar,
                          const double* craw, const unsigned int* clamp_count, double* part, double* part_clamped,
                          double* part_alpha, double* gops, cudaStream_t st, cudaStream_t rs = nullptr,
                          cudaEvent_t ev = nullptr) {
  MOBO_TRY(launch_syrk_both(Tsave, dvar, craw, MP, R, part, part_clamped, clamp_count, dmu, part_alpha, st));
  cudaStream_t r = st;
  if (rs && ev) {
    if (cudaEventRecord(ev, st) != cudaSuccess || cudaStreamWaitEvent(rs, ev, 0) != cudaSuccess) return -1;
    r = rs;
  }
  MOBO_TRY(launch_syrk_reduce(0, MP, R, part, gops + ops_block(MP, OPS_W), clamp_count, part_alpha,
                              gops + ops_alpha(MP), nullptr, r));
  MOBO_TRY(launch_syrk_reduce(1, MP, R, part_clamped, gops + ops_block(MP, OPS_H), clamp_count, nullptr, nullptr,
                              gops + ops_scal(MP) + SC_CLAMP, r));
  return 0;
}

// product kernel + covariance-gradient kernel + the fixed-order reduction of the latter's per-CTA partials
// the fold of the covariance-gradient kernel's per-CTA partials (latency-bound: a few hundred dependent loads per
// output) may run on another stream `rs` once `ev` (recorded on `st` behind the kernel) has fired
static int rows_bwd_main(RowArgs& a, int kind, int d, int M, long long R, double* dk, double* part, double* dtheta,
                         double* dzf, cudaStream_t st, cudaStream_t rs = nullptr, cudaEvent_t ev = nullptr) {
  const int MP = a.MP;
  const int grid = kgrad_grid(R);
  a.dk = dk;
  a.part_theta = part;
  a.part_zf = part + (size_t)grid * kMaxTheta;
  MOBO_TRY(launch_row_bwd(a, st));
  if (a.want_param_grads && dtheta) {
    cudaStream_t r = st;
    if (rs && ev) {
      if (cudaEventRecord(ev, st) != cudaSuccess || cudaStreamWaitEvent(rs, ev, 0) != cudaSuccess) return -1;
      r = rs;
    }
    MOBO_TRY(launch_reduce_partials(a.part_theta, grid, theta_size(kind, d), kMaxTheta, dtheta, 0, r));
    if (kind == 1 && dzf) MOBO_TRY(launch_reduce_partials(a.part_zf, grid, M, MP, dzf, 0, r));
  }
  return 0;
}

static void fill_row_bwd_args(RowArgs& a, const double* dmu, const double* dvar, const double* craw,
                              const double* Tsave, const double* Usave, int want_param_grads, double* df,
                              double* dxrow) {
  a.dmu = dmu; a.dvar = dvar; a.craw = const_cast<double*>(craw);
  a.Tsave = const_cast<double*>(Tsave); a.Usave = const_cast<double*>(Usave);
  a.df = df; a.dxrow = dxrow;
  a.want_param_grads = want_param_grads; a.want_x_grads = dxrow != nullptr;
  if (!a.want_param_grads && !a.want_x_grads) a.want_param_grads = 1;
}

int mobo_layer_rows_bwd(int kind, int d, int M, const double* Zx, const double* zf, const double* theta,
                        const double* ops, const double* x, int xrep, const double* mu_prev, const double* var_prev,
                        int prep, const double* eps, long long eps_mod, const double* f_direct, long long R,
                        int training, const double* dmu, const double* dvar, const double* craw,
                        const unsigned int* clamp_count, const double* Tsave,
                        const double* Usave, int want_param_grads, double* df, double* dxrow, double* dtheta,
                        double* dzf, double* gops, double* work, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  RowArgs a;
  fill_row_args(a, kind, d, M, Zx, zf, theta, ops, x, xrep, mu_prev, var_prev, prep, eps, eps_mod, f_direct, R,
                training);
  fill_row_bwd_args(a, dmu, dvar, craw, Tsave, Usave, want_param_grads, df, dxrow);
  const int MP = a.MP;
  const int grid = kgrad_grid(R);
  double* dk = work;                                             // [R][MP] scratch, first so that it stays aligned
  double* part = work + mobo_rows_save_doubles(M, R);
  double* part_syrk = part + (size_t)grid * (kMaxTheta + MP);
  double* part_clamped = part_syrk + syrk_part_doubles(MP, R);
  double* part_alpha = part_clamped + syrk_part_doubles(MP, R);
  MOBO_TRY(rows_bwd_main(a, kind, d, M, R, dk, part, dtheta, dzf, st));
  if (gops)
    MOBO_TRY(rows_bwd_stats(MP, R, Tsave, dmu, dvar, craw, training ? clamp_count : nullptr, part_syrk, part_clamped,
                            part_alpha, gops, st));
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

// ---------------------------------------------------------------------------------------------------------------
// fused ELBO step
// ---------------------------------------------------------------------------------------------------------------
namespace {

struct StepLayout {
  size_t theta[kMaxLayers], ops[kMaxLayers], gops[kMaxLayers], mu[kMaxLayers], var[kMaxLayers],
      craw[kMaxLayers], dmu[kMaxLayers], dvar[kMaxLayers], df[kMaxLayers], Ts[kMaxLayers],
      Us[kMaxLayers], dtheta_rows[kMaxLayers], dtheta_pre[kMaxLayers], dzf_rows[kMaxLayers],
      dzf_pre[kMaxLayers], dm_pre[kMaxLayers], dLq_tmp[kMaxLayers], pre_work[kMaxLayers],
      ell_part[kMaxLayers], stats0[kMaxLayers], stats1[kMaxLayers], stats_alpha[kMaxLayers],
      kg_part[kMaxLayers];
  long long R[kMaxLayers];
  int ell_blocks[kMaxLayers];
  size_t noise, clamp, rows_work, total;
};

StepLayout step_layout(int L, int d, int M, int S, long long B) {
  StepLayout y;
  size_t off = 0;
  auto take = [&](size_t n) { const size_t o = off; off += (n + 15) / 16 * 16; return o; };
  const int MP = padded(M);
  y.noise = take(kMaxLayers);
  y.clamp = take(kMaxLayers);
  size_t rows_work = 0;
  for (int l = 0; l < L; ++l) {
    const long long R = l == 0 ? B : B * (long long)S;
    y.R[l] = R;
    y.ell_blocks[l] = (int)((R + ELL_THREADS - 1) / ELL_THREADS);
    y.theta[l] = take(kMaxTheta);
    y.ops[l] = take(ops_size(MP));
    y.gops[l] = take(ops_size(MP));
    y.mu[l] = take(R); y.var[l] = take(R); y.craw[l] = take(R);
    y.dmu[l] = take(R); y.dvar[l] = take(R); y.df[l] = take(R);
    y.Ts[l] = take(mobo_rows_save_doubles(M, R));
    y.Us[l] = take(mobo_rows_save_doubles(M, R));
    y.dtheta_rows[l] = take(kMaxTheta); y.dtheta_pre[l] = take(kMaxTheta);
    y.dzf_rows[l] = take(MP); y.dzf_pre[l] = take(MP); y.dm_pre[l] = take(MP);
    y.dLq_tmp[l] = take((size_t)M * M);
    y.pre_work[l] = take(mobo_precompute_bwd_work_doubles(M));
    y.ell_part[l] = take(2 * (size_t)y.ell_blocks[l]);
    const size_t w = mobo_rows_save_doubles(M, R) + (size_t)256 * KG_CTAS_PER_SM * (kMaxTheta + MP) + 64;
    rows_work = w > rows_work ? w : rows_work;
    // SYRK partials per layer and per weight set: their fold runs on the side stream while the main stream is already
    // in the next layer's SYRK
    y.stats0[l] = take(syrk_part_doubles(MP, R));
    y.stats1[l] = take(syrk_part_doubles(MP, R));
    y.stats_alpha[l] = take(syrk_alpha_doubles(MP, syrk_nchunk(MP, R)) + 64);
    // per-CTA partials of the covariance-gradient kernel, per layer: their fold runs on the side stream too
    y.kg_part[l] = take((size_t)256 * KG_CTAS_PER_SM * (kMaxTheta + MP) + 64);
  }
  y.rows_work = take(rows_work);
  y.total = off;
  (void)d;
  return y;
}

}  // namespace

// Side stream of the fused step: the fold of the SYRK partials and the operator-chain backward of layer l run there
// while the main stream already works on layer l - 1's row kernels; forked and joined with events inside
// mobo_elbo_step, so the pattern is also valid under CUDA-graph capture.  The stream and its events belong to a step
// context the caller creates (mobo_step_ctx_create: one per concurrently trained model, so that independent models do
// not serialise on each other's side stream); a step without a context uses one per-device default, created under a
// lock on first use - the only state this library keeps.
namespace {
struct SideCtx {
  int device = -1; cudaStream_t s = nullptr; cudaEvent_t fork[kMaxLayers]; cudaEvent_t join = nullptr;
  cudaEvent_t done[kMaxLayers];      // layer l's operator-chain backward (its d L_q, d m, d theta shares) is complete
  cudaEvent_t kg[kMaxLayers];        // layer l's covariance-gradient kernel is complete (its partials may be folded)
};
bool side_ctx_init(SideCtx& c) {
  if (cudaGetDevice(&c.device) != cudaSuccess) return false;
  if (cudaStreamCreateWithFlags(&c.s, cudaStreamNonBlocking) != cudaSuccess) return false;
  for (int i = 0; i < kMaxLayers; ++i)
    if (cudaEventCreateWithFlags(&c.fork[i], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&c.done[i], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&c.kg[i], cudaEventDisableTiming) != cudaSuccess) return false;
  return cudaEventCreateWithFlags(&c.join, cudaEventDisableTiming) == cudaSuccess;
}
SideCtx* default_side_ctx() {
  static SideCtx ctx[64];
  static std::mutex mu;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
  std::lock_guard<std::mutex> lock(mu);
  SideCtx& c = ctx[dev & 63];
  if (c.device < 0 && !side_ctx_init(c)) return nullptr;
  return &c;
}
}  // namespace

void* mobo_step_ctx_create(void) {
  SideCtx* c = new SideCtx();
  if (!side_ctx_init(*c)) { delete c; return nullptr; }
  return c;
}
int mobo_step_ctx_wait_layer(void* ctx, int layer, void* stream) {
  SideCtx* c = static_cast<SideCtx*>(ctx);
  if (!c || layer < 0 || layer >= kMaxLayers) return -2;
  return cudaStreamWaitEvent((cudaStream_t)stream, c->done[layer], 0) == cudaSuccess ? 0 : -1;
}
void mobo_step_ctx_destroy(void* ctx) {
  SideCtx* c = static_cast<SideCtx*>(ctx);
  if (!c) return;
  if (c->s) cudaStreamDestroy(c->s);
  for (int i = 0; i < kMaxLayers; ++i) { if (c->fork[i]) cudaEventDestroy(c->fork[i]); if (c->done[i]) cudaEventDestroy(c->done[i]); if (c->kg[i]) cudaEventDestroy(c->kg[i]); }
  if (c->join) cudaEventDestroy(c->join);
  delete c;
}

static bool g_side_stream_on = true;
// SMs the backward product kernel (one persistent CTA per SM, all of its registers and shared memory) leaves to the
// side stream's operator-chain backward; measured on C4 (ms / step): round 1: 0 -> 2.84, 4 -> 2.72, 8 -> 2.71, 16 -> 2.75;
// round-2 kernels: 0 -> 2.51, 4 -> 2.41, 8 -> 2.44, 12 -> 2.45, 16 -> 2.45
constexpr int kSideStreamSMs = 4;
void mobo_step_side_stream(int on) { g_side_stream_on = on != 0; }

size_t mobo_elbo_step_workspace_doubles(int L, int d, int M, int S, long long B) {
  if (L < 1 || L > kMaxLayers) return 0;
  return step_layout(L, d, M, S, B).total;
}

int mobo_elbo_step(const mobo_step_desc* D, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  const int L = D->L, d = D->d, M = D->M, S = D->S < 1 ? 1 : D->S;
  if (L < 1 || L > kMaxLayers || d > kMaxD || padded(M) > MAX_MP || D->B < 1) return -2;
  const int MP = padded(M);
  const StepLayout y = step_layout(L, d, M, S, D->B);
  double* ws = D->workspace;
  const double kl_scale = (double)D->B / (double)D->num_data;
  unsigned int* clamp = reinterpret_cast<unsigned int*>(ws + y.clamp);

  int kinds[kMaxLayers];
  const double* Zx[kMaxLayers]; const double* zf[kMaxLayers]; const double* theta[kMaxLayers];
  const double* m[kMaxLayers]; const double* Lq[kMaxLayers];
  double* ops[kMaxLayers]; double* dLq[kMaxLayers];
  // the rows of each layer, which its forward and backward row passes both read: x itself at layer 0, above it x
  // tiled S times, each row propagated from its sample of layer l - 1's q(f)
  RowArgs rows[kMaxLayers];
  for (int l = 0; l < L; ++l) {
    const mobo_layer_desc& ld = D->layer[l];
    kinds[l] = l == 0 ? 0 : 1;
    Zx[l] = ld.Zx; zf[l] = l == 0 ? nullptr : D->layer[l - 1].m; theta[l] = ws + y.theta[l];
    m[l] = ld.m; Lq[l] = ld.Lq;
    ops[l] = ws + y.ops[l];
    dLq[l] = (ld.g_Lq && !D->accumulate) ? ld.g_Lq : ws + y.dLq_tmp[l];
    fill_row_args(rows[l], kinds[l], d, M, Zx[l], zf[l], theta[l], ops[l], D->x, l == 0 ? 1 : S,
                  l == 0 ? nullptr : ws + y.mu[l - 1], l == 0 ? nullptr : ws + y.var[l - 1],
                  l == 0 ? 1 : (int)(y.R[l] / y.R[l - 1]), ld.eps, y.R[l], nullptr, y.R[l], 1);
  }
  // 1. raw -> constrained
  {
    PrepArgs a;
    a.L = L; a.d = d; a.noise = ws + y.noise; a.clamp_count = clamp; a.dkl = kl_scale;
    for (int l = 0; l < kMaxLayers; ++l) {
      const bool ok = l < L;
      for (int i = 0; i < kMaxTheta; ++i) a.raw_theta[l][i] = ok ? D->layer[l].raw_theta[i] : nullptr;
      a.raw_noise[l] = ok ? D->layer[l].raw_noise : nullptr;
      a.noise_lo[l] = ok ? D->layer[l].noise_lower : 0.0; a.noise_hi[l] = ok ? D->layer[l].noise_upper : 0.0;
      a.theta[l] = ok ? ws + y.theta[l] : nullptr;
      a.gops_scal[l] = ok ? ws + y.gops[l] + ops_scal(MP) : nullptr;
      a.ops_scal[l] = ok ? ws + y.ops[l] + ops_scal(MP) : nullptr;
      a.oc_flags[l] = ok ? reinterpret_cast<int*>(ws + y.ops[l] + ops_flags(MP)) : nullptr;
    }
    MOBO_LAUNCH("step_prep_kernel", st, step_prep_kernel<<<L, 96, 0, st>>>(a));
  }
  // 2. operator chain of every layer
  MOBO_TRY(model_precompute(L, kinds, d, M, Zx, zf, theta, m, Lq, D->jitter, ops, st, false));
  // 3. forward row passes, low -> high fidelity
  for (int l = 0; l < L; ++l) {
    RowArgs a = rows[l];
    a.mu = ws + y.mu[l]; a.var = ws + y.var[l]; a.craw = ws + y.craw[l]; a.clamp_count = clamp + l;
    a.Tsave = ws + y.Ts[l]; a.Usave = ws + y.Us[l];
    MOBO_TRY(launch_row_fwd(a, st));
  }
  // 4. ELBO terms and backward row passes, high -> low fidelity.  Per layer the main stream runs the SYRK statistics,
  //    the product and the covariance-gradient kernels; that layer's operator-chain backward (a dozen latency-bound
  //    M x M launches) runs on the side stream, hidden behind the row kernels.
  SideCtx* scp = D->ctx ? static_cast<SideCtx*>(D->ctx) : (g_side_stream_on ? default_side_ctx() : nullptr);
  const bool fork = g_side_stream_on && scp != nullptr;
  SideCtx dummy;
  SideCtx& sc = scp ? *scp : dummy;
  cudaStream_t ss = fork ? sc.s : st;
  for (int l = L - 1; l >= 0; --l) {
    const long long R = y.R[l];
    EllArgs e;
    e.layer = l; e.R = R; e.S = l == 0 ? 1 : S; e.y = D->y; e.fid = D->fid;
    e.mu = ws + y.mu[l]; e.var = ws + y.var[l]; e.noise = ws + y.noise;
    e.df_next = l + 1 < L ? ws + y.df[l + 1] : nullptr;
    e.eps_next = l + 1 < L ? D->layer[l + 1].eps : nullptr;
    e.prep_next = l + 1 < L ? (int)(y.R[l + 1] / R) : 1;
    e.dmu = ws + y.dmu[l]; e.dvar = ws + y.dvar[l]; e.part = ws + y.ell_part[l];
    MOBO_LAUNCH("ell_kernel", st, ell_kernel<<<y.ell_blocks[l], ELL_THREADS, 0, st>>>(e));
    // SYRK proper on the main stream (DMMA-bound like the row kernels: running them side by side only made both
    // slower); the fold of its partials and the latency-bound operator-chain backward of this layer go to the side
    // stream
    double* gl = ws + y.gops[l];
    MOBO_TRY(rows_bwd_stats(MP, R, ws + y.Ts[l], ws + y.dmu[l], ws + y.dvar[l], ws + y.craw[l], clamp + l,
                            ws + y.stats0[l], ws + y.stats1[l], ws + y.stats_alpha[l], gl, st, fork ? ss : nullptr,
                            fork ? sc.fork[l] : nullptr));
    MOBO_TRY(mobo_layer_precompute_bwd(kinds[l], d, M, Zx[l], zf[l], theta[l], m[l], Lq[l], ops[l], gl,
                                       ws + y.pre_work[l], ws + y.dtheta_pre[l], ws + y.dzf_pre[l], ws + y.dm_pre[l],
                                       dLq[l], (void*)ss));
    // d L_q of this layer is final (it is written straight into the caller's gradient): a multi-GPU caller may start
    // its all-reduce now, behind the lower layers' row kernels (mobo_step_ctx_wait_layer)
    if (scp && !D->accumulate && cudaEventRecord(sc.done[l], ss) != cudaSuccess) return -1;
    // main stream: dk = W^T dt and the covariance gradient
    RowArgs a = rows[l];
    fill_row_bwd_args(a, ws + y.dmu[l], ws + y.dvar[l], ws + y.craw[l], ws + y.Ts[l], ws + y.Us[l], 1, ws + y.df[l],
                      nullptr);
    a.clamp_count = clamp + l;
    a.sm_reserve = fork ? kSideStreamSMs : 0;
    MOBO_TRY(rows_bwd_main(a, kinds[l], d, M, R, ws + y.rows_work, ws + y.kg_part[l], ws + y.dtheta_rows[l],
                           l == 0 ? nullptr : ws + y.dzf_rows[l], st, fork ? ss : nullptr, fork ? sc.kg[l] : nullptr));
  }
  // 5. join: the gradient assembly needs both streams' results
  if (fork && (cudaEventRecord(sc.join, ss) != cudaSuccess || cudaStreamWaitEvent(st, sc.join, 0) != cudaSuccess)) return -1;
  // 6. gradient assembly
  {
    FinishArgs a;
    a.L = L; a.d = d; a.M = M; a.MP = MP; a.kl_scale = kl_scale; a.out = D->out; a.accumulate = D->accumulate;
    for (int l = 0; l < kMaxLayers; ++l) {
      const bool ok = l < L;
      for (int i = 0; i < kMaxTheta; ++i) {
        a.raw_theta[l][i] = ok ? D->layer[l].raw_theta[i] : nullptr;
        a.g_raw_theta[l][i] = ok ? D->layer[l].g_raw_theta[i] : nullptr;
      }
      a.dtheta_rows[l] = ok ? ws + y.dtheta_rows[l] : nullptr;
      a.dtheta_pre[l] = ok ? ws + y.dtheta_pre[l] : nullptr;
      a.dzf_rows[l] = (ok && l > 0) ? ws + y.dzf_rows[l] : nullptr;
      a.dzf_pre[l] = (ok && l > 0) ? ws + y.dzf_pre[l] : nullptr;
      a.dm_pre[l] = ok ? ws + y.dm_pre[l] : nullptr;
      a.g_m[l] = ok ? D->layer[l].g_m : nullptr;
      a.raw_noise[l] = ok ? D->layer[l].raw_noise : nullptr;
      a.noise_lo[l] = ok ? D->layer[l].noise_lower : 0.0; a.noise_hi[l] = ok ? D->layer[l].noise_upper : 0.0;
      a.g_raw_noise[l] = ok ? D->layer[l].g_raw_noise : nullptr;
      a.ell_part[l] = ok ? ws + y.ell_part[l] : nullptr;
      a.ell_blocks[l] = ok ? y.ell_blocks[l] : 0;
      a.ops_scal[l] = ok ? ws + y.ops[l] + ops_scal(MP) : nullptr;
    }
    MOBO_LAUNCH("step_finish_kernel", st, step_finish_kernel<<<1, 256, 0, st>>>(a));
  }
  if (D->accumulate)
    for (int l = 0; l < L; ++l)
      if (D->layer[l].g_Lq) {
        const long long n = (long long)M * M;
        MOBO_LAUNCH("add_matrix_kernel", st,
                    add_matrix_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(D->layer[l].g_Lq, dLq[l], n));
      }
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

static bool small_shape_ok(int L, int d, int M, long long B) {
  return L >= 1 && L <= kMaxLayers && d >= 1 && d <= kMaxD && M >= 1 && M <= SS_MAX_M && B >= 1;
}

size_t mobo_elbo_step_small_workspace_doubles(int L, int d, int M, int S, long long B) {
  if (!small_shape_ok(L, d, M, B)) return 0;
  return ss_workspace_doubles(L, M, S < 1 ? 1 : S, B);
}

// SS_PER_LAUNCH descriptors per launch (they travel as the kernel's parameter, no host-to-device copy), one CTA each
int mobo_elbo_step_small(const mobo_step_desc* descs, int n_models, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (n_models < 1 || !descs) return -2;
  for (int i = 0; i < n_models; ++i)
    if (!small_shape_ok(descs[i].L, descs[i].d, descs[i].M, descs[i].B)) return -2;
  static bool attr_done[kMaxDevices] = {false};
  if (first_on_device(attr_done))
    cudaFuncSetAttribute(small_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         (int)ss_smem_bytes(SS_MAX_M));
  for (int i0 = 0; i0 < n_models; i0 += SS_PER_LAUNCH) {
    SmallBatch b;
    memset(&b, 0, sizeof(b));
    b.n = n_models - i0 < SS_PER_LAUNCH ? n_models - i0 : SS_PER_LAUNCH;
    int maxM = 1;
    for (int i = 0; i < b.n; ++i) {
      b.desc[i] = descs[i0 + i];
      if (b.desc[i].M > maxM) maxM = b.desc[i].M;
    }
    MOBO_LAUNCH("small_step_kernel", st, small_step_kernel<<<b.n, SS_THREADS, ss_smem_bytes(maxM), st>>>(b));
    if (cudaGetLastError() != cudaSuccess) return -1;
  }
  return 0;
}

int mobo_adam(int nt, const mobo_adam_tensor* tensors, double lr, double beta1, double beta2, double eps,
              long long step, long long* step_dev, const double* skip_flag, void* stream) {
  if (nt < 1 || nt > ADAM_MAX_TENSORS || (step < 1 && !step_dev)) return -2;
  cudaStream_t st = (cudaStream_t)stream;
  AdamArgs a;
  a.nt = nt; a.lr = lr; a.beta1 = beta1; a.beta2 = beta2; a.eps = eps; a.step_dev = step_dev; a.skip = skip_flag;
  a.bc1 = step_dev ? 1.0 : 1.0 - pow(beta1, (double)step);
  a.bc2_sqrt = step_dev ? 1.0 : sqrt(1.0 - pow(beta2, (double)step));
  long long mx = 1;
  for (int i = 0; i < ADAM_MAX_TENSORS; ++i) {
    const bool ok = i < nt;
    a.p[i] = ok ? tensors[i].p : nullptr; a.g[i] = ok ? tensors[i].g : nullptr;
    a.m[i] = ok ? tensors[i].exp_avg : nullptr; a.v[i] = ok ? tensors[i].exp_avg_sq : nullptr;
    a.n[i] = ok ? tensors[i].n : 0;
    if (ok && tensors[i].n > mx) mx = tensors[i].n;
  }
  long long gx = (mx + 255) / 256;
  if (gx > 64) gx = 64;
  MOBO_LAUNCH("adam_kernel", st, adam_kernel<<<dim3((unsigned)gx, nt), 256, 0, st>>>(a));
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

int mobo_adam_tick(long long* step_dev, const double* skip_flag, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  MOBO_LAUNCH("adam_tick_kernel", st, adam_tick_kernel<<<1, 1, 0, st>>>(step_dev, skip_flag));
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

// the rows of layer l of the acquisition chain, which mobo_acq_moments and the forward recomputed by
// mobo_acq_moments_bwd both read: the n candidates at layer 0, above it row i*S+s = (candidate i, sample s), its
// propagated input from row i (layer 1) or row i*S+s (layers >= 2) of the layer below, eval mode
static void fill_acq_row_args(RowArgs& a, int l, int d, int M, int S, long long n, const double* Zx,
                              const double* const* zf, const double* const* theta, const double* const* ops,
                              const double* const* samples, const double* X, const double* mu_prev,
                              const double* var_prev) {
  const long long R = l == 0 ? n : n * (long long)S;
  fill_row_args(a, l == 0 ? 0 : 1, d, M, Zx, l == 0 ? nullptr : zf[l], theta[l], ops[l], X, l == 0 ? 1 : S,
                l == 0 ? nullptr : mu_prev, l == 0 ? nullptr : var_prev, l == 1 ? S : 1,
                l == 0 ? nullptr : samples[l], S, nullptr, R, 0);
}

int mobo_acq_moments(int fidelity, int d, int M, int S, long long n, const double* Zx, const double* const* zf,
                     const double* const* theta, const double* const* ops, const double* const* samples,
                     const double* raw_noise, double noise_lower, double noise_upper, const double* X,
                     double* out_mu, double* out_var, double* scratch, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (fidelity < 0 || fidelity >= kMaxLayers || n < 1 || S < 1) return -2;
  const long long RS = n * (long long)S;
  double* mu[2] = {scratch, scratch + 2 * RS};
  double* var[2] = {scratch + RS, scratch + 3 * RS};
  for (int l = 0; l <= fidelity; ++l) {
    const int cur = l & 1, prv = cur ^ 1;
    RowArgs a;
    fill_acq_row_args(a, l, d, M, S, n, Zx, zf, theta, ops, samples, X, mu[prv], var[prv]);
    a.mu = mu[cur]; a.var = var[cur];
    MOBO_TRY(launch_row_fwd(a, st));
  }
  MomentArgs a;
  a.n = n; a.S = S; a.tiled = fidelity >= 1 ? 1 : 0;
  a.mu = mu[fidelity & 1]; a.var = var[fidelity & 1];
  a.noise_lo = noise_lower; a.noise_hi = noise_upper; a.raw_noise = raw_noise;
  a.out_mu = out_mu; a.out_var = out_var;
  MOBO_LAUNCH("moment_kernel", st, moment_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(a));
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

// ---------------------------------------------------------------------------------------------------------------
// backward of the acquisition chain: recompute the chunk's forward with t and u saved, then the row backward of
// every layer, high -> low, and the fold of d / dX
// ---------------------------------------------------------------------------------------------------------------
namespace {

struct AcqBwdLayout {
  size_t mu[kMaxLayers], var[kMaxLayers], Ts[kMaxLayers], Us[kMaxLayers], dxrow[kMaxLayers];
  size_t dmu, dvar, df, dk, noise_part, total;
  int noise_blocks;
};

bool acq_bwd_shape_ok(int fidelity, int d, int M, int S, long long n) {
  return fidelity >= 0 && fidelity < kMaxLayers && d >= 1 && d <= kMaxD && M >= 1 && padded(M) <= MAX_MP && S >= 1 &&
         n >= 1 && n < kMaxRows && n * (long long)S < kMaxRows;
}

// every region starts at a multiple of 16 doubles (the bulk copies of the row kernels need 16-byte aligned T / U
// rows); the order is the one include/mobocmf_b200.h documents
AcqBwdLayout acq_bwd_layout(int fidelity, int d, int M, int S, long long n) {
  AcqBwdLayout y;
  size_t off = 0;
  auto take = [&](size_t k) { const size_t o = off; off += (k + 15) / 16 * 16; return o; };
  const long long RF = fidelity == 0 ? n : n * (long long)S;
  for (int l = 0; l <= fidelity; ++l) {
    const long long R = l == 0 ? n : n * (long long)S;
    y.mu[l] = take(R); y.var[l] = take(R);
    y.Ts[l] = take(mobo_rows_save_doubles(M, R)); y.Us[l] = take(mobo_rows_save_doubles(M, R));
    y.dxrow[l] = take((size_t)R * d);
  }
  y.dmu = take(RF); y.dvar = take(RF); y.df = take(RF);
  y.dk = take(mobo_rows_save_doubles(M, RF));
  y.noise_blocks = (int)((n + ACQ_THREADS - 1) / ACQ_THREADS);
  y.noise_part = take(y.noise_blocks);
  y.total = off;
  return y;
}

}  // namespace

size_t mobo_acq_bwd_work_doubles(int fidelity, int d, int M, int S, long long n) {
  if (!acq_bwd_shape_ok(fidelity, d, M, S, n)) return 0;
  return acq_bwd_layout(fidelity, d, M, S, n).total;
}

int mobo_acq_moments_bwd(int fidelity, int d, int M, int S, long long n, const double* Zx,
                         const double* const* zf, const double* const* theta, const double* const* ops,
                         const double* const* samples, const double* raw_noise, double noise_lower,
                         double noise_upper, const double* X, const double* d_mu, const double* d_var,
                         int accumulate, double* dX, double* d_raw_noise, double* work, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!acq_bwd_shape_ok(fidelity, d, M, S, n)) return -2;
  const AcqBwdLayout y = acq_bwd_layout(fidelity, d, M, S, n);
  double* w = work;
  // 1. the forward of mobo_acq_moments, every layer's moments and t / u kept
  RowArgs rows[kMaxLayers];
  for (int l = 0; l <= fidelity; ++l) {
    fill_acq_row_args(rows[l], l, d, M, S, n, Zx, zf, theta, ops, samples, X, l == 0 ? nullptr : w + y.mu[l - 1],
                      l == 0 ? nullptr : w + y.var[l - 1]);
    RowArgs a = rows[l];
    a.mu = w + y.mu[l]; a.var = w + y.var[l]; a.Tsave = w + y.Ts[l]; a.Usave = w + y.Us[l];
    MOBO_TRY(launch_row_fwd(a, st));
  }
  // 2. moment matching -> d mu, d var of the top layer's rows (and the partials of d / d raw_noise)
  {
    AcqMomentBwdArgs a;
    a.n = n; a.S = S; a.tiled = fidelity >= 1 ? 1 : 0;
    a.mu = w + y.mu[fidelity]; a.var = w + y.var[fidelity];
    a.noise_lo = noise_lower; a.noise_hi = noise_upper; a.raw_noise = raw_noise;
    a.d_mu = d_mu; a.d_var = d_var; a.dmu = w + y.dmu; a.dvar = w + y.dvar;
    a.part = d_raw_noise ? w + y.noise_part : nullptr;
    MOBO_LAUNCH("acq_moment_bwd_kernel", st,
                acq_moment_bwd_kernel<<<y.noise_blocks, ACQ_THREADS, 0, st>>>(a));
    if (d_raw_noise) MOBO_TRY(launch_reduce_partials(w + y.noise_part, y.noise_blocks, 1, 1, d_raw_noise, accumulate, st));
  }
  // 3. row backward of every layer (d / dx of its rows, d / df of its propagated input), and through the propagation
  //    into the moments of the layer below
  for (int l = fidelity; l >= 0; --l) {
    RowArgs a = rows[l];
    fill_row_bwd_args(a, w + y.dmu, w + y.dvar, nullptr, w + y.Ts[l], w + y.Us[l], 0, l == 0 ? nullptr : w + y.df,
                      w + y.dxrow[l]);
    a.dk = w + y.dk;
    MOBO_TRY(launch_row_bwd(a, st));
    if (l >= 1) {
      const long long Rp = rows[l - 1].R;
      MOBO_LAUNCH("acq_prop_bwd_kernel", st,
                  acq_prop_bwd_kernel<<<(unsigned)((Rp + ACQ_THREADS - 1) / ACQ_THREADS), ACQ_THREADS, 0, st>>>(
                      w + y.df, w + y.var[l - 1], samples[l], Rp, l == 1 ? S : 1, S, w + y.dmu, w + y.dvar));
    }
  }
  // 4. d / dX
  {
    AcqDxFoldArgs a;
    a.n = n; a.d = d; a.S = S; a.nl = fidelity + 1; a.dX = dX; a.accumulate = accumulate;
    for (int l = 0; l < kMaxLayers; ++l) a.dxrow[l] = l <= fidelity ? w + y.dxrow[l] : nullptr;
    MOBO_LAUNCH("acq_dx_fold_kernel", st,
                acq_dx_fold_kernel<<<(unsigned)((n * d + ACQ_THREADS - 1) / ACQ_THREADS), ACQ_THREADS, 0, st>>>(a));
  }
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

int mobo_jes(const double* var_uncond, const double* var_cond, long long n, int accumulate, double* out,
             void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (n < 1) return 0;
  MOBO_LAUNCH("jes_kernel", st,
              jes_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(var_uncond, var_cond, out, n, accumulate));
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

int mobo_rff_eval(int L, int d, int F, const double* const* params, const double* scales, const double* x, long long n,
                  double* f, double* grad, void* stream) {
  if (L < 1 || L > RFF_MAX_LAYERS) return -2;
  RffArgs a;
  a.L = L; a.d = d; a.F = F; a.want_grad = grad != nullptr;
  for (int l = 0; l < RFF_MAX_LAYERS; ++l) {
    a.params[l] = l < L ? params[l] : nullptr;
    for (int q = 0; q < 3; ++q) a.scale[l][q] = l < L ? scales[3 * l + q] : 0.0;
  }
  a.x = x; a.n = n; a.f = f; a.grad = grad;
  return launch_rff_eval(a, (cudaStream_t)stream);
}

int mobo_pareto_mask(const double* pts, long long n, int k, unsigned char* mask, void* stream) {
  return launch_pareto_mask(pts, n, k, mask, (cudaStream_t)stream);
}

}  // extern "C"
