// ELBO steps of several small MFDGPs in ONE launch: one CTA runs one model's complete step (mobo_elbo_step_small).
//
// At the reference's own sizes (M = N = 16 - 75, SURVEY.md section 8 C1 - C3) a step of mobo_elbo_step is ~45 kernels
// whose arithmetic is a few microseconds: the step is launch and barrier latency.  Here every stage of that step runs
// inside one CTA, separated by CTA barriers instead of kernel boundaries:
//   constraint transforms (softplus, Interval sigmoid; mobocmf/models/mfdgp.py:116)
//   per layer: P = K(Z_l, Z_l) + jitter I with psd_safe_cholesky's retries, L = chol(P), W = L^-1, H = W tril(L_q),
//              beta = W m, KL (opchain.cu);  the row pass of its B (layer 0) or B S rows (row_pass.cu)
//   ELBO terms (ell_kernel), row backward (dt, dk = W^T dt, through the covariance function), whitened statistics
//   A2 / A1 / b, operator-chain backward (matrix_ops.cu), through K(Z, Z) (kzz_bwd_kernel), gradient assembly
//   (step_finish_kernel).
// The formulation is the one of those kernels, and so is the code of every per-entry and per-row formula: the
// covariance entry and its derivatives (common.cuh), the constraint transforms, ELBO row term, propagation backward,
// raw-gradient store and result flags (step.cu); only the schedule differs.  M <= 64 keeps the six working M x M
// matrices of a layer in shared memory (6 x 33 KB at M = 64); per-row t = W k and u = H^T t go to the model's
// workspace (L2-resident at these sizes).  Plain FP64 FMA: at M <= 64 a product is a few thousand FMAs per thread.
// Every sum has a fixed order and there are no atomics: a model's result does not depend on the other models of the
// launch, and two launches are bit-identical.
#include "common.cuh"

namespace mobo {

constexpr int SS_THREADS = 256, SS_WARPS = SS_THREADS / 32, SS_MAX_M = 64;
// descriptors per launch: they travel as one __grid_constant__ parameter (at most 32 764 bytes)
constexpr int SS_PER_LAUNCH = 8;

struct SmallBatch {
  int n;
  mobo_step_desc desc[SS_PER_LAUNCH];
};
static_assert(sizeof(SmallBatch) <= 32764, "kernel parameter limit");

__host__ __device__ inline int ss_ld(int M) { return M | 1; }          // odd stride: conflict-free column walks
__host__ __device__ inline long long ss_rows(int l, int S, long long B) { return l == 0 ? B : B * (long long)S; }
// per layer: W, H (M x M), beta (M), theta, mu, var, craw, f, dmu, dvar, df (R each), T, U (R x M each)
__host__ __device__ inline size_t ss_layer_doubles(int M, long long R) {
  return 2 * (size_t)M * M + M + kMaxTheta + 7 * (size_t)R + 2 * (size_t)R * M;
}
__host__ __device__ inline size_t ss_workspace_doubles(int L, int M, int S, long long B) {
  size_t n = 0;
  for (int l = 0; l < L; ++l) n += ss_layer_doubles(M, ss_rows(l, S, B));
  return n;
}
// dynamic shared memory: six M x ld matrices, then three 64-vectors per warp
__host__ __device__ inline size_t ss_smem_bytes(int M) {
  return (6 * (size_t)M * ss_ld(M) + (size_t)SS_WARPS * 3 * SS_MAX_M) * sizeof(double);
}

struct SsLayer {
  double *W, *H, *beta, *theta, *mu, *var, *craw, *f, *dmu, *dvar, *df, *T, *U;
  long long R;
};
// layer l's regions; off = sum of ss_layer_doubles of the layers below, R = its rows
__device__ inline SsLayer ss_layer(double* ws, size_t off, long long R, int M) {
  SsLayer y;
  double* p = ws + off;
  y.R = R;
  y.W = p; p += (size_t)M * M;
  y.H = p; p += (size_t)M * M;
  y.beta = p; p += M;
  y.theta = p; p += kMaxTheta;
  y.mu = p; p += R; y.var = p; p += R; y.craw = p; p += R; y.f = p; p += R;
  y.dmu = p; p += R; y.dvar = p; p += R; y.df = p; p += R;
  y.T = p; p += (size_t)R * M;
  y.U = p;
  return y;
}

// sum over the CTA in a fixed order (butterfly within warps, then warps in order); every thread gets the result
__device__ __forceinline__ double ss_block_sum(double v, double* red) {
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  double s = 0.0;
#pragma unroll
  for (int w = 0; w < SS_WARPS; ++w) s += red[w];
  return s;
}

// the CTA's accumulators -> d loss / d theta in the theta layout, into out[kMaxTheta]
__device__ void ss_reduce_acc(const KernAcc& acc, const KernParams& kp, double (*red)[kMaxTheta], double* out) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, tid = threadIdx.x;
  double v[kMaxTheta];
#pragma unroll
  for (int q = 0; q < 5; ++q) v[q] = acc.s[q];
#pragma unroll
  for (int c = 0; c < kMaxD; ++c) { v[5 + c] = acc.l1[c]; v[5 + kMaxD + c] = acc.l2[c]; }
  __syncthreads();
#pragma unroll
  for (int q = 0; q < kMaxTheta; ++q) {
    const double s = warp_sum(v[q]);
    if (lane == 0) red[warp][q] = s;
  }
  __syncthreads();
  if (tid < kMaxTheta) {
    double s = 0.0;
    for (int w = 0; w < SS_WARPS; ++w) s += red[w][tid];
    double o;
    const int slot = kern_theta_slot(kp, tid, s, o);
    if (slot >= 0) out[slot] = o;
  }
  __syncthreads();
}

// whitened statistics of a layer's rows: A2 = sum dvar t t^T -> mA2, A1 = the same over unclamped rows -> mA1 (both
// full symmetric), b = sum dmu t -> vb.  Each thread owns up to 9 entries of the lower triangle, rows ascending; the
// rows are staged through stg (2 M x ld doubles) in chunks of 2 M.  Out of line: its accumulators would otherwise
// share the register budget of the rest of the step.
__device__ __noinline__ void ss_stats(const double* __restrict__ T, const double* __restrict__ dvar,
                                      const double* __restrict__ dmu, const double* __restrict__ craw, long long R,
                                      int M, int ld, double* stg, double* mA1, double* mA2, double* vb,
                                      double* rowsc) {
  const int tid = threadIdx.x;
  double* sdv = rowsc;                   // the chunk's dvar, dmu, mask
  double* sdm = rowsc + 2 * SS_MAX_M;
  double* smk = rowsc + 4 * SS_MAX_M;
  const int nE = M * (M + 1) / 2;
  int ei[9], ej[9];
  double a2[9], a1[9];
#pragma unroll
  for (int q = 0; q < 9; ++q) {
    const int e = tid + SS_THREADS * q;
    int i = (int)((sqrt(8.0 * e + 1.0) - 1.0) * 0.5);
    while (i * (i + 1) / 2 > e) --i;
    while ((i + 1) * (i + 2) / 2 <= e) ++i;
    ei[q] = e < nE ? i : 0;
    ej[q] = e < nE ? e - i * (i + 1) / 2 : 0;
    a2[q] = 0.0; a1[q] = 0.0;
  }
  double bsum = 0.0;
  const int nc = 2 * M;
  for (long long r0 = 0; r0 < R; r0 += nc) {
    const int n = (int)min((long long)nc, R - r0);
    for (int idx = tid; idx < n * M; idx += SS_THREADS) {
      const int rr = idx / M, i = idx - rr * M;
      stg[rr * ld + i] = T[(size_t)(r0 + rr) * M + i];
    }
    for (int rr = tid; rr < n; rr += SS_THREADS) {
      sdv[rr] = dvar[r0 + rr];
      sdm[rr] = dmu[r0 + rr];
      smk[rr] = craw[r0 + rr] >= 0.0 ? 1.0 : 0.0;
    }
    __syncthreads();
    for (int rr = 0; rr < n; ++rr) {
      const double w = sdv[rr], mk = smk[rr];
      const double* trow = stg + rr * ld;
#pragma unroll
      for (int q = 0; q < 9; ++q) {
        const double p = w * trow[ei[q]] * trow[ej[q]];
        a2[q] += p;
        a1[q] += mk * p;
      }
      if (tid < M) bsum = fma(sdm[rr], trow[tid], bsum);
    }
    __syncthreads();
  }
#pragma unroll
  for (int q = 0; q < 9; ++q) {
    if (tid + SS_THREADS * q < nE) {
      const int i = ei[q], j = ej[q];
      mA2[i * ld + j] = a2[q]; mA2[j * ld + i] = a2[q];
      mA1[i * ld + j] = a1[q]; mA1[j * ld + i] = a1[q];
    }
  }
  if (tid < M) vb[tid] = bsum;
  __syncthreads();
}

// named barrier over the first n threads (n = 32: warp 0 alone)
__device__ __forceinline__ void ss_team_sync(int n) { asm volatile("bar.sync 1, %0;" ::"r"(n) : "memory"); }

__global__ void __launch_bounds__(SS_THREADS, 1) small_step_kernel(const __grid_constant__ SmallBatch batch) {
  extern __shared__ double sm[];
  __shared__ KernParams kp;
  __shared__ double red[SS_WARPS][kMaxTheta];
  __shared__ double vbeta[SS_MAX_M], vb[SS_MAX_M], vm[SS_MAX_M], rinv[SS_MAX_M], lqd[SS_MAX_M];
  __shared__ double dzr[SS_MAX_M], dzp[SS_MAX_M];            // d loss / d m_{l-1} of layer l: rows, K(Z, Z)
  __shared__ double azf[SS_WARPS][SS_MAX_M];                 // per-warp row shares of dzr
  __shared__ double th_rows[kMaxTheta], th_pre[kMaxTheta];
  __shared__ double rowsc[3 * 2 * SS_MAX_M];
  __shared__ double noise_s[kMaxLayers], kl_s[kMaxLayers], data_s[kMaxLayers], ds2_s[kMaxLayers];
  __shared__ int status_s[kMaxLayers], retries_s[kMaxLayers];
  __shared__ int failed_s;
  __shared__ size_t lay_off[kMaxLayers];       // workspace offset and rows of each layer
  __shared__ long long lay_rows[kMaxLayers];

  const mobo_step_desc& D = batch.desc[blockIdx.x];
  const int L = D.L, d = D.d, M = D.M, S = D.S < 1 ? 1 : D.S;
  const long long B = D.B;
  const int ld = ss_ld(M);
  const int MM = M * ld;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // slots: W, H, then C and E adjacent (the staging area of the statistics pass), D, F
  double* mW = sm;
  double* mH = mW + MM;
  double* mC = mH + MM;
  double* mE = mC + MM;
  double* mD = mE + MM;
  double* mF = mD + MM;
  double* wbuf = mF + MM + (size_t)warp * 3 * SS_MAX_M;     // this warp's three row vectors
  double* va = wbuf;
  double* vt = wbuf + SS_MAX_M;
  double* vu = wbuf + 2 * SS_MAX_M;
  double* ws = D.workspace;
  // B / N: the KL's weight in the loss, so also d loss / d KL of every layer (kept in shared memory: a register
  // held across the whole step is what the allocator spilled)
  __shared__ double kl_scale;
  if (tid == 0) kl_scale = (double)B / (double)D.num_data;

  if (tid == 0) {
    size_t off = 0;
    for (int l = 0; l < L; ++l) {
      lay_off[l] = off;
      lay_rows[l] = ss_rows(l, S, B);
      off += ss_layer_doubles(M, lay_rows[l]);
    }
  }
  __syncthreads();

  // ---- constraint transforms ----
  for (int l = 0; l < L; ++l) {
    const SsLayer y = ss_layer(ws, lay_off[l], lay_rows[l], M);
    const int nth = theta_size(l == 0 ? 0 : 1, d);
    if (tid < nth) y.theta[tid] = softplus_fwd(*D.layer[l].raw_theta[tid]);
    if (tid == 32) {
      const mobo_layer_desc& ldsc = D.layer[l];
      noise_s[l] = interval_fwd(ldsc.noise_lower, ldsc.noise_upper, *ldsc.raw_noise);
    }
  }
  __syncthreads();

  // ---- forward, low -> high fidelity: operators of layer l, then its rows ----
  for (int l = 0; l < L; ++l) {
    const int kind = l == 0 ? 0 : 1;
    const SsLayer y = ss_layer(ws, lay_off[l], lay_rows[l], M);
    const double* Zx = D.layer[l].Zx;
    const double* zf = l == 0 ? nullptr : D.layer[l - 1].m;
    const double* Lq = D.layer[l].Lq;
    if (tid == 0) load_kern_params(kp, kind, d, y.theta);
    for (int i = tid; i < M; i += SS_THREADS) vm[i] = D.layer[l].m[i];
    __syncthreads();
    // P, its factor (psd_safe_cholesky: retried with 1e-8, 1e-7, 1e-6 more on the diagonal, as opchain_kernel does)
    int attempt = 0;
    for (;;) {
      for (int idx = tid; idx < M * M; idx += SS_THREADS) {
        const int i = idx / M, j = idx - i * M;
        if (j <= i) mC[i * ld + j] = oc_kernel_entry(kp, kind, d, Zx, zf, M, i, j, D.jitter, attempt);
      }
      __syncthreads();
      // right-looking, the arithmetic of chol32_inwarp: L_jj = p rsqrt(p), L_ij = A_ij rsqrt(p),
      // A_ic -= L_ij L_cj; the factor goes to mD, A is updated in mC.  M <= 32: warp 0 alone
      const int team = M <= 32 ? 32 : SS_THREADS;
      if (tid < team) {
        int fail = 0;
        for (int j = 0; j < M; ++j) {
          const double djj = mC[j * ld + j];
          if (!(djj > 0.0)) fail = 1;
          const double r = rsqrt(djj);
          const int n1 = M - 1 - j;
          for (int q = tid; q < n1 * n1 + 1; q += team) {
            if (q == n1 * n1) {
              mD[j * ld + j] = djj * r;
              rinv[j] = r;
              continue;
            }
            const int i = j + 1 + q / n1, c = j + 1 + q % n1;
            const double lij = mC[i * ld + j] * r;
            if (c == j + 1) mD[i * ld + j] = lij;
            if (c <= i) mC[i * ld + c] = fma(-lij, mC[c * ld + j] * r, mC[i * ld + c]);
          }
          ss_team_sync(team);
        }
        if (tid == 0) failed_s = fail;
      }
      __syncthreads();
      if (!failed_s || attempt >= 3) break;
      ++attempt;
    }
    if (tid == 0) { status_s[l] = failed_s; retries_s[l] = attempt; }
    // W = L^-1: 4 threads per column j, right-looking (opchain_kernel's order: x_k *= 1 / L_kk, x_i -= L_ik x_k)
    for (int idx = tid; idx < M * M; idx += SS_THREADS) {
      const int i = idx / M, j = idx - i * M;
      mW[i * ld + j] = i == j ? 1.0 : 0.0;
    }
    __syncthreads();
    {
      const int j = tid >> 2, p = tid & 3;
      const bool own = j < M;
      for (int k = 0; k < M; ++k) {
        const double xk = own ? mW[k * ld + j] * rinv[k] : 0.0;
        __syncwarp();
        if (own) {
          if (p == 0) mW[k * ld + j] = xk;
          for (int i = k + 1 + p; i < M; i += 4) mW[i * ld + j] = fma(-mD[i * ld + k], xk, mW[i * ld + j]);
        }
        __syncwarp();
      }
    }
    // tril(L_q) into mE
    for (int idx = tid; idx < M * M; idx += SS_THREADS) {
      const int i = idx / M, j = idx - i * M;
      mE[i * ld + j] = j <= i ? Lq[idx] : 0.0;
    }
    __syncthreads();
    // H = W tril(L_q), beta = W m, and the KL pieces
    double h2 = 0.0, b2 = 0.0, ldp = 0.0, ldq = 0.0;
    for (int idx = tid; idx < M * M; idx += SS_THREADS) {
      const int i = idx / M, j = idx - i * M;
      double s = 0.0;
      for (int k = j; k <= i; ++k) s = fma(mW[i * ld + k], mE[k * ld + j], s);
      mH[i * ld + j] = s;
      y.H[idx] = s;
      y.W[idx] = mW[i * ld + j];
      h2 = fma(s, s, h2);
    }
    for (int i = tid; i < M; i += SS_THREADS) {
      double s = 0.0;
      for (int k = 0; k <= i; ++k) s = fma(mW[i * ld + k], vm[k], s);
      vbeta[i] = s;
      y.beta[i] = s;
      b2 = fma(s, s, b2);
      ldp += 2.0 * log(mD[i * ld + i]);
      const double qii = mE[i * ld + i];
      ldq += log(qii * qii);
    }
    h2 = ss_block_sum(h2, red[0]);
    b2 = ss_block_sum(b2, red[1]);
    ldp = ss_block_sum(ldp, red[2]);
    ldq = ss_block_sum(ldq, red[3]);
    if (tid == 0) kl_s[l] = 0.5 * (ldp - ldq + b2 + h2 - (double)M);
    __syncthreads();

    // ---- rows of this layer: one warp per row; lane <-> inducing points lane, lane + 32 ----
    const int xrep = l == 0 ? 1 : S;
    const long long prep = l == 0 ? 1 : y.R / lay_rows[l - 1];
    const SsLayer yp = ss_layer(ws, lay_off[l > 0 ? l - 1 : 0], lay_rows[l > 0 ? l - 1 : 0], M);
    const double* eps = D.layer[l].eps;
    for (long long r = warp; r < y.R; r += SS_WARPS) {
      const double* xr = D.x + (size_t)(r / xrep) * d;
      double f = 0.0;
      if (kind == 1) {
        const long long pr = r / prep;
        f = yp.mu[pr] + sqrt(fmax(yp.var[pr], kMinVariance)) * eps[r];
      }
      for (int j = lane; j < M; j += 32) va[j] = kern_entry(kp, d, xr, f, Zx + (size_t)j * d, kind ? zf[j] : 0.0);
      __syncwarp();
      double q1 = 0.0, mu = 0.0, q2 = 0.0;
      for (int i = lane; i < M; i += 32) {
        double s = 0.0;
        for (int j = 0; j <= i; ++j) s = fma(mW[i * ld + j], va[j], s);
        vt[i] = s;
        y.T[(size_t)r * M + i] = s;
        q1 = fma(s, s, q1);
        mu = fma(vbeta[i], s, mu);
      }
      __syncwarp();
      for (int i = lane; i < M; i += 32) {
        double s = 0.0;
        for (int j = i; j < M; ++j) s = fma(mH[j * ld + i], vt[j], s);
        y.U[(size_t)r * M + i] = s;
        q2 = fma(s, s, q2);
      }
      q1 = warp_sum(q1); mu = warp_sum(mu); q2 = warp_sum(q2);
      if (lane == 0) {
        const double c = kern_diag(kp, f) - q1;
        y.mu[r] = mu;
        y.var[r] = fmax(c, 0.0) + q2;
        y.craw[r] = c;
        y.f[r] = f;
      }
      __syncwarp();
    }
    __syncthreads();
  }

  // ---- ELBO terms and backward, high -> low fidelity ----
  for (int l = L - 1; l >= 0; --l) {
    const int kind = l == 0 ? 0 : 1;
    const SsLayer y = ss_layer(ws, lay_off[l], lay_rows[l], M);
    const mobo_layer_desc& ldsc = D.layer[l];
    const double* Zx = ldsc.Zx;
    const long long R = y.R;
    // expected log-likelihood of the rows and the seed of their backward (ell_kernel)
    {
      const int Sl = l == 0 ? 1 : S;
      const double s2 = noise_s[l];
      const bool has_next = l + 1 < L;
      const int prep_next = l == 0 ? S : 1;           // rows of layer l + 1 per row of layer l
      const double* df_next = has_next ? ss_layer(ws, lay_off[l + 1], lay_rows[l + 1], M).df : nullptr;
      const double* eps_next = has_next ? D.layer[l + 1].eps : nullptr;
      double data = 0.0, ds2 = 0.0;
      for (long long r = tid; r < R; r += SS_THREADS) {
        const long long b = r / Sl;
        const double v = y.var[r];
        double ds2r, dmu, dv;
        data += ell_row(D.y[b], D.fid[b], l, Sl, y.mu[r], v, s2, ds2r, dmu, dv);
        ds2 += ds2r;
        if (has_next) {
          double gmu, gv;
          prop_bwd(df_next, eps_next, r * prep_next, prep_next, 0, v, gmu, gv);
          dmu += gmu;
          dv += gv;
        }
        y.dmu[r] = dmu;
        y.dvar[r] = dv;
      }
      data = ss_block_sum(data, red[0]);
      ds2 = ss_block_sum(ds2, red[1]);
      if (tid == 0) { data_s[l] = data; ds2_s[l] = ds2; }
    }
    // this layer's operators back into shared memory
    if (tid == 0) load_kern_params(kp, kind, d, y.theta);
    for (int idx = tid; idx < M * M; idx += SS_THREADS) {
      const int i = idx / M, j = idx - i * M;
      mW[i * ld + j] = y.W[idx];
      mH[i * ld + j] = y.H[idx];
    }
    for (int i = tid; i < M; i += SS_THREADS) { vbeta[i] = y.beta[i]; lqd[i] = ldsc.Lq[(size_t)i * M + i]; }
    __syncthreads();
    // row backward: dt = dmu beta - 2 dvar (mask t - H u), dk = W^T dt, then through the covariance function
    {
      KernAcc acc;
      acc.zero();
      double az0 = 0.0, az1 = 0.0;
      for (long long r = warp; r < R; r += SS_WARPS) {
        const double dmu = y.dmu[r], dvar = y.dvar[r];
        const double mask = y.craw[r] >= 0.0 ? 1.0 : 0.0;
        const double f = y.f[r];
        const double* xr = D.x + (size_t)(r / (l == 0 ? 1 : S)) * d;
        for (int i = lane; i < M; i += 32) { vt[i] = y.T[(size_t)r * M + i]; vu[i] = y.U[(size_t)r * M + i]; }
        __syncwarp();
        for (int i = lane; i < M; i += 32) {
          double s = 0.0;
          for (int j = 0; j <= i; ++j) s = fma(mH[i * ld + j], vu[j], s);
          va[i] = dmu * vbeta[i] - 2.0 * dvar * (mask * vt[i] - s);
        }
        __syncwarp();
        double gf = 0.0;
        for (int jj = 0; jj < 2; ++jj) {
          const int j = lane + 32 * jj;
          if (j >= M) break;
          double gk = 0.0;
          for (int i = j; i < M; ++i) gk = fma(mW[i * ld + j], va[i], gk);
          double ca, cb;
          kern_entry_bwd(kp, d, xr, f, Zx + (size_t)j * d, kind ? D.layer[l - 1].m[j] : 0.0, gk, acc, ca, cb);
          // the weighted f-derivatives are rounded before they are summed (__dmul_rn: never fused into the sums)
          const double gfa = __dmul_rn(gk, ca), gfb = __dmul_rn(gk, cb);
          gf += gfa;
          if (jj == 0) az0 += gfb; else az1 += gfb;
        }
        const double dvm = dvar * mask;
        if (lane == 0) gf += __dmul_rn(2.0 * kern_diag_bwd(kp, f, dvm, acc), f);
        gf = warp_sum(gf);
        if (kind == 1 && lane == 0) y.df[r] = gf;
        __syncwarp();
      }
      if (lane < M) azf[warp][lane] = az0;
      if (lane + 32 < M) azf[warp][lane + 32] = az1;
      ss_reduce_acc(acc, kp, red, th_rows);
    }
    // whitened statistics A2 = sum dvar t t^T -> mF, A1 = the same over unclamped rows -> mD, b = sum dmu t -> vb
    ss_stats(y.T, y.dvar, y.dmu, y.craw, R, M, ld, mC, mD, mF, vb, rowsc);
    // operator-chain backward (mobo_layer_precompute_bwd): G2 = H H^T -> mC, V = A2 G2 -> mE
    for (int idx = tid; idx < M * M; idx += SS_THREADS) {
      const int i = idx / M, j = idx - i * M;
      double s = 0.0;
      const int kmax = min(i, j);
      for (int k = 0; k <= kmax; ++k) s = fma(mH[i * ld + k], mH[j * ld + k], s);
      mC[i * ld + j] = s;
    }
    __syncthreads();
    for (int idx = tid; idx < M * M; idx += SS_THREADS) {
      const int i = idx / M, j = idx - i * M;
      double s = 0.0;
      for (int k = 0; k < M; ++k) s = fma(mF[i * ld + k], mC[k * ld + j], s);
      mE[i * ld + j] = s;
    }
    __syncthreads();
    // N = A1 - V - V^T - 1/2 (beta b^T + b beta^T) + g/2 (I - beta beta^T - G2), in place of A1
    for (int idx = tid; idx < M * M; idx += SS_THREADS) {
      const int i = idx / M, j = idx - i * M;
      const double eye = i == j ? 1.0 : 0.0;
      mD[i * ld + j] = mD[i * ld + j] - mE[i * ld + j] - mE[j * ld + i] -
                       0.5 * (vbeta[i] * vb[j] + vb[i] * vbeta[j]) +
                       0.5 * kl_scale * (eye - vbeta[i] * vbeta[j] - mC[i * ld + j]);
    }
    // dm = W^T (b + g beta); the gradient of m_l is complete with layer l + 1's shares through Z_{l+1} = [Zx, m_l]
    for (int j = tid; j < M; j += SS_THREADS) {
      double s = 0.0;
      for (int i = j; i < M; ++i) s = fma(mW[i * ld + j], vb[i] + kl_scale * vbeta[i], s);
      if (ldsc.g_m) {
        double g = s;
        if (l + 1 < L) g += dzr[j] + dzp[j];
        store_grad(ldsc.g_m + j, g, D.accumulate);
      }
    }
    __syncthreads();
    // X2 = F H with F = 2 A2 + g I -> mC;  X1 = W^T N -> mE
    for (int idx = tid; idx < M * M; idx += SS_THREADS) {
      const int i = idx / M, j = idx - i * M;
      double s = 0.0;
      for (int k = j; k < M; ++k) s = fma(2.0 * mF[i * ld + k] + (k == i ? kl_scale : 0.0), mH[k * ld + j], s);
      mC[i * ld + j] = s;
      double t = 0.0;
      for (int k = i; k < M; ++k) t = fma(mW[k * ld + i], mD[k * ld + j], t);
      mE[i * ld + j] = t;
    }
    __syncthreads();
    // dLq = tril(W^T X2) - g diag(1 / Lq_ii): straight into the caller's gradient, zeros above the diagonal
    if (ldsc.g_Lq) {
      for (int idx = tid; idx < M * M; idx += SS_THREADS) {
        const int i = idx / M, j = idx - i * M;
        double v = 0.0;
        if (j <= i) {
          for (int k = i; k < M; ++k) v = fma(mW[k * ld + i], mC[k * ld + j], v);
          if (i == j) v -= kl_scale / lqd[i];
        }
        store_grad(ldsc.g_Lq + idx, v, D.accumulate);
      }
    }
    // dP = X1 W -> mF (A2 is no longer needed)
    for (int idx = tid; idx < M * M; idx += SS_THREADS) {
      const int i = idx / M, j = idx - i * M;
      double s = 0.0;
      for (int k = j; k < M; ++k) s = fma(mE[i * ld + k], mW[k * ld + j], s);
      mF[i * ld + j] = s;
    }
    // the rows' shares of d loss / d m_{l-1}, fixed warp order
    for (int j = tid; j < M; j += SS_THREADS) {
      double s = 0.0;
      for (int w = 0; w < SS_WARPS; ++w) s += azf[w][j];
      dzr[j] = s;
    }
    __syncthreads();
    // through K(Z, Z) (kzz_bwd_kernel): one warp per inducing point i, lanes over j
    {
      KernAcc acc;
      acc.zero();
      for (int i = warp; i < M; i += SS_WARPS) {
        const double* zf = kind ? D.layer[l - 1].m : nullptr;
        const double fi = kind ? zf[i] : 0.0;
        double dzi = 0.0;
        for (int j = lane; j < M; j += 32) {
          const double gk = mF[i * ld + j];
          if (i == j) {
            dzi += __dmul_rn(2.0 * kern_diag_bwd(kp, fi, gk, acc), fi);
          } else {
            double ca, cb;
            kern_entry_bwd(kp, d, Zx + (size_t)i * d, fi, Zx + (size_t)j * d, kind ? zf[j] : 0.0, gk, acc, ca, cb);
            dzi += 2.0 * __dmul_rn(gk, ca);
          }
        }
        dzi = warp_sum(dzi);
        if (lane == 0) dzp[i] = dzi;
      }
      ss_reduce_acc(acc, kp, red, th_pre);
    }
    // d loss / d raw theta and d loss / d raw noise of this layer
    store_raw_grads(tid, theta_size(kind, d), ldsc.raw_theta, ldsc.g_raw_theta, th_rows, th_pre, ldsc.raw_noise,
                    ldsc.g_raw_noise, ldsc.noise_lower, ldsc.noise_upper, ds2_s[l], D.accumulate);
    __syncthreads();
  }

  // ---- results (step_finish_kernel's out[8]) ----
  if (tid == 0) {
    double data = 0.0, kl = 0.0, status = 0.0, retries = 0.0;
    for (int l = 0; l < L; ++l) {
      data += data_s[l];
      kl += kl_s[l];
      if (status_s[l] && status == 0.0) status = (double)(l + 1);
      retries = fmax(retries, (double)retries_s[l]);
    }
    write_step_result(D.out, data, kl, kl_scale, status, retries);
  }
}

}  // namespace mobo
