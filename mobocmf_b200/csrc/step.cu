// Fused ELBO step and acquisition chains: the small kernels that glue the operator chain and the row passes into ONE
// host-sync-free enqueue per step (CUDA-graph capturable), plus the Adam update.
//
// Replaces the body of BlackBoxMFDGPFitter._update_model (mobocmf/util/blackbox_mfdgp_fitter.py:161-171):
//   output = model(x_batch); res = elbo(output, y_batch.T, fidelities); loss = -res[0]; loss.backward(); optimizer.step()
// i.e. MFDGP.forward (mobocmf/models/mfdgp.py:174-196), VariationalELBOMF.forward
// (mobocmf/mlls/variational_elbo_mf.py:24-51), GaussianLikelihood.expected_log_prob [upstream gpytorch], the
// constraint transforms (Positive = softplus, Interval = sigmoid; models/mfdgp.py:116) and torch.optim.Adam
// (fitter.py:126,132).
#include "common.cuh"

namespace mobo {

constexpr double kLog2Pi = 1.8378770664093454835606594728112;

__device__ __forceinline__ double softplus_fwd(double x) { return x > 20.0 ? x : log1p(exp(x)); }   // torch softplus
__device__ __forceinline__ double softplus_grad(double x) {
  if (x > 20.0) return 1.0;
  const double z = exp(x);
  return z / (z + 1.0);
}
__device__ __forceinline__ double sigmoid_fwd(double x) { return 1.0 / (1.0 + exp(-x)); }

// ---- raw -> constrained parameters -----------------------------------------------------------------
struct PrepArgs {
  int L, d;
  const double* raw_theta[kMaxLayers][kMaxTheta];         // address of every raw hyper-parameter, theta order
  const double* raw_noise[kMaxLayers];
  double noise_lo[kMaxLayers], noise_hi[kMaxLayers];
  double* theta[kMaxLayers];          // out: constrained, kernels' layout
  double* noise;                      // out: [L]
  double* gops_scal[kMaxLayers];      // scal block of each operator-gradient buffer
  double* ops_scal[kMaxLayers];       // scal block of each operator buffer (zeroed here)
  unsigned int* clamp_count;          // [L]
  double dkl;                         // d loss / d KL = B / N
  int* oc_flags[kMaxLayers];          // block-to-block flags of the operator-chain kernel (256 ints), zeroed here
};

__global__ void step_prep_kernel(const __grid_constant__ PrepArgs a) {
  const int l = blockIdx.x, tid = threadIdx.x;
  const int nth = theta_size(l == 0 ? 0 : 1, a.d);
  if (tid < nth) a.theta[l][tid] = softplus_fwd(*a.raw_theta[l][tid]);
  if (tid == 32) a.noise[l] = a.noise_lo[l] + (a.noise_hi[l] - a.noise_lo[l]) * sigmoid_fwd(*a.raw_noise[l]);
  if (tid == 33) a.clamp_count[l] = 0u;
  if (tid >= 64 && tid < 80) {
    a.gops_scal[l][tid - 64] = (tid - 64 == SC_KL) ? a.dkl : 0.0;
    a.ops_scal[l][tid - 64] = 0.0;    // the workspace is caller memory: never assume it is zeroed
  }
  // what opchain_reset_kernel does for the stand-alone entry point: one launch less on the step's critical path
  for (int i = tid; i < 256; i += blockDim.x) a.oc_flags[l][i] = 0;
}

// ---- expected log-likelihood of one layer's rows + the seed of its backward -------------------------
//   row r of layer l belongs to minibatch point b = r / S_l; weight w = [fid_b == l] / S_l
//   data  += w * -1/2 [ ((y - mu)^2 + max(v, 1e-10)) / s2 + log s2 + log 2 pi ]
//   dmu    = d(-data)/dmu  + sum over the next layer's rows fed by this row of df
//   dvar   = d(-data)/dv   + sum df * eps / (2 sqrt(max(v, 1e-10)))        (both v-paths gated by v >= 1e-10)
// per-block partials (data, d(-data)/d s2) are folded in block order by step_finish_kernel.
struct EllArgs {
  int layer;
  long long R;            // rows of this layer
  int S;                  // rows per minibatch point (1 for layer 0)
  const double* y; const double* fid;
  const double* mu; const double* var;
  const double* noise;    // [L]
  const double* df_next;  // next layer's d loss / d f per row (or NULL)
  const double* eps_next; // next layer's normals
  int prep_next;          // next-layer rows per row of this layer
  double* dmu; double* dvar;
  double* part;           // [gridDim.x][2]
};

constexpr int ELL_THREADS = 256;

__global__ void __launch_bounds__(ELL_THREADS) ell_kernel(const __grid_constant__ EllArgs a) {
  __shared__ double red[2][ELL_THREADS / 32];
  const long long r = (long long)blockIdx.x * ELL_THREADS + threadIdx.x;
  double data = 0.0, ds2 = 0.0;
  if (r < a.R) {
    const long long b = r / a.S;
    const double s2 = a.noise[a.layer];
    const double w = (a.fid[b] == (double)a.layer) ? 1.0 / (double)a.S : 0.0;
    const double mu = a.mu[r], v = a.var[r];
    const bool live = v >= kMinVariance;
    const double vu = live ? v : kMinVariance;
    const double res = a.y[b] - mu;
    const double q = res * res + vu;
    data = w * -0.5 * (q / s2 + log(s2) + kLog2Pi);
    ds2 = w * 0.5 * (1.0 / s2 - q / (s2 * s2));
    double dmu = -w * res / s2;
    double dv = live ? w * 0.5 / s2 : 0.0;
    if (a.df_next) {
      double s0 = 0.0, s1 = 0.0;
      const long long base = r * a.prep_next;
      for (int k = 0; k < a.prep_next; ++k) {
        const double g = a.df_next[base + k];
        s0 += g;
        s1 = fma(g, a.eps_next[base + k], s1);
      }
      dmu += s0;
      if (live) dv += s1 / (2.0 * sqrt(vu));
    }
    a.dmu[r] = dmu;
    a.dvar[r] = dv;
  }
  data = warp_sum(data);
  ds2 = warp_sum(ds2);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { red[0][warp] = data; red[1][warp] = ds2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double s0 = 0.0, s1 = 0.0;
    for (int w = 0; w < ELL_THREADS / 32; ++w) { s0 += red[0][w]; s1 += red[1][w]; }
    a.part[2 * blockIdx.x] = s0;
    a.part[2 * blockIdx.x + 1] = s1;
  }
}

// ---- gradient assembly ------------------------------------------------------------------------------
struct FinishArgs {
  int L, d, M, MP;
  double kl_scale;                       // B / N
  const double* raw_theta[kMaxLayers][kMaxTheta];
  double* g_raw_theta[kMaxLayers][kMaxTheta];
  const double* dtheta_rows[kMaxLayers];
  const double* dtheta_pre[kMaxLayers];
  const double* dzf_rows[kMaxLayers];      // layer l's d loss / d zf (zf_l = m_{l-1}); NULL for l = 0
  const double* dzf_pre[kMaxLayers];
  const double* dm_pre[kMaxLayers];
  double* g_m[kMaxLayers];
  const double* raw_noise[kMaxLayers];
  double noise_lo[kMaxLayers], noise_hi[kMaxLayers];
  double* g_raw_noise[kMaxLayers];
  const double* ell_part[kMaxLayers];
  int ell_blocks[kMaxLayers];
  const double* ops_scal[kMaxLayers];
  double* out;                           // [0] loss, [1] KL * B / N, [2] data term, [3] status, [4] sticky status,
                                         // [5] sticky "loss not finite", [6] this step is bad (Adam skips), [7] retries
  int accumulate;
};

__global__ void __launch_bounds__(256) step_finish_kernel(const __grid_constant__ FinishArgs a) {
  __shared__ double sdata[kMaxLayers], sds2[kMaxLayers];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // fold the per-block ELBO partials, one warp per layer, fixed order (lane-strided then butterfly)
  for (int l = warp; l < a.L; l += 8) {
    double s0 = 0.0, s1 = 0.0;
    for (int b = lane; b < a.ell_blocks[l]; b += 32) { s0 += a.ell_part[l][2 * b]; s1 += a.ell_part[l][2 * b + 1]; }
    s0 = warp_sum(s0);
    s1 = warp_sum(s1);
    if (lane == 0) { sdata[l] = s0; sds2[l] = s1; }
  }
  __syncthreads();
  if (tid == 0) {
    double data = 0.0, kl = 0.0, status = 0.0, retries = 0.0;
    for (int l = 0; l < a.L; ++l) {
      data += sdata[l];
      kl += a.ops_scal[l][SC_KL];
      if (a.ops_scal[l][SC_STATUS] != 0.0 && status == 0.0) status = (double)(l + 1);
      retries = fmax(retries, a.ops_scal[l][SC_RETRIES]);
    }
    const double loss = -(data - kl * a.kl_scale);
    a.out[0] = loss;
    a.out[1] = kl * a.kl_scale;
    a.out[2] = data;
    a.out[3] = status;
    // the host reads these at its own pace (no per-step synchronisation): the first failure sticks, and the optimiser
    // update of a bad step is skipped on the device (mobo_adam's skip flag)
    const bool finite = isfinite(loss);
    if (status != 0.0 && a.out[4] == 0.0) a.out[4] = status;
    if (!finite && status == 0.0) a.out[5] = 1.0;
    a.out[6] = (status != 0.0 || !finite) ? 1.0 : 0.0;
    a.out[7] = retries;
  }
  for (int l = 0; l < a.L; ++l) {
    const int nth = theta_size(l == 0 ? 0 : 1, a.d);
    if (tid < nth && a.g_raw_theta[l][tid]) {
      const double g = (a.dtheta_rows[l][tid] + a.dtheta_pre[l][tid]) * softplus_grad(*a.raw_theta[l][tid]);
      double* dst = a.g_raw_theta[l][tid];
      *dst = a.accumulate ? *dst + g : g;
    }
    if (tid == 64 && a.g_raw_noise[l]) {
      const double s = sigmoid_fwd(*a.raw_noise[l]);
      const double g = sds2[l] * (a.noise_hi[l] - a.noise_lo[l]) * s * (1.0 - s);
      *a.g_raw_noise[l] = a.accumulate ? *a.g_raw_noise[l] + g : g;
    }
    if (a.g_m[l]) {
      for (int j = tid; j < a.M; j += 256) {
        double g = a.dm_pre[l][j];
        if (l + 1 < a.L) g += a.dzf_rows[l + 1][j] + a.dzf_pre[l + 1][j];
        a.g_m[l][j] = a.accumulate ? a.g_m[l][j] + g : g;
      }
    }
  }
}

// dst (M x M) (+)= src (M x M): used only when gradients are accumulated
__global__ void add_matrix_kernel(double* __restrict__ dst, const double* __restrict__ src, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] += src[i];
}

// ---- Adam (torch.optim.Adam defaults: no weight decay, no amsgrad) -----------------------------------
constexpr int ADAM_MAX_TENSORS = 64;
struct AdamArgs {
  int nt;
  double* p[ADAM_MAX_TENSORS];
  const double* g[ADAM_MAX_TENSORS];
  double* m[ADAM_MAX_TENSORS];
  double* v[ADAM_MAX_TENSORS];
  long long n[ADAM_MAX_TENSORS];
  double lr, beta1, beta2, eps, bc1, bc2_sqrt;
  const long long* step_dev;     // optional device-resident step count (CUDA-graph replays): overrides bc1 / bc2_sqrt
  const double* skip;            // optional device flag: != 0 -> leave parameters and moments untouched
};

__global__ void adam_tick_kernel(long long* step_dev, const double* skip) {
  if (skip && *skip != 0.0) return;
  *step_dev += 1;
}

__global__ void __launch_bounds__(256) adam_kernel(const __grid_constant__ AdamArgs a) {
  if (a.skip && *a.skip != 0.0) return;
  const int t = blockIdx.y;
  const long long n = a.n[t];
  double* __restrict__ p = a.p[t];
  const double* __restrict__ g = a.g[t];
  double* __restrict__ m = a.m[t];
  double* __restrict__ v = a.v[t];
  double bc1 = a.bc1, bc2_sqrt = a.bc2_sqrt;
  if (a.step_dev) {
    const double st = (double)(*a.step_dev);
    bc1 = 1.0 - pow(a.beta1, st);
    bc2_sqrt = sqrt(1.0 - pow(a.beta2, st));
  }
  const double step_size = a.lr / bc1;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    const double gi = g[i];
    const double mi = a.beta1 * m[i] + (1.0 - a.beta1) * gi;          // exp_avg.lerp_(grad, 1 - beta1)
    const double vi = a.beta2 * v[i] + (1.0 - a.beta2) * gi * gi;     // exp_avg_sq.mul_(b2).addcmul_(g, g, 1 - b2)
    m[i] = mi;
    v[i] = vi;
    const double denom = sqrt(vi) / bc2_sqrt + a.eps;
    p[i] -= step_size * (mi / denom);                                 // param.addcdiv_(exp_avg, denom, -step_size)
  }
}

// ---- acquisition epilogue: moment matching over the S samples and the JES term ---------------------------------
//   mus = mean_s mu~;  v = mean_s (max(v~ + noise, 1e-10) + mu~^2) - mus^2        (models/mfdgp.py:256-260)
//   jes = 1/2 max(0, log v_u - log v_c)                                          (acquisition_functions/...py:52)
struct MomentArgs {
  long long n; int S;     // samples per candidate
  int tiled;              // 1: row i*S+s holds (candidate i, sample s); 0: one row per candidate (fidelity 0: the S
                          // copies of a candidate coincide, models/mfdgp.py:248)
  const double* mu; const double* var; double noise_lo, noise_hi; const double* raw_noise;
  double* out_mu; double* out_var;
};
__global__ void moment_kernel(const __grid_constant__ MomentArgs a) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  const double noise = a.noise_lo + (a.noise_hi - a.noise_lo) * sigmoid_fwd(*a.raw_noise);
  double s1 = 0.0, s2 = 0.0;
  for (int s = 0; s < a.S; ++s) {
    const long long r = a.tiled ? i * a.S + s : i;
    const double m = a.mu[r];
    double v = a.var[r] + noise;
    v = v < kMinVariance ? kMinVariance : v;
    s1 += m;
    s2 += v + m * m;
  }
  const double mean = s1 / (double)a.S;
  a.out_mu[i] = mean;
  a.out_var[i] = s2 / (double)a.S - mean * mean;
}

// ---- backward of the acquisition chain (mobo_acq_moments_bwd) ---------------------------------------------------
// moment matching, per candidate i (tiled: rows i*S+s; untiled, fidelity 0: the S copies of row i coincide):
//   dmu_s = d_mu / S + d_var 2 (mu_s - out_mu) / S,   dv_s = d_var / S [v_s + noise >= 1e-10]
//   untiled: dmu = d_mu, dv = d_var [v + noise >= 1e-10]
// and, when `part` is set, the per-block partials of d / d raw_noise:
//   sum_i d_var[i] (1/S) sum_s [v_s + noise >= 1e-10] (hi - lo) sigmoid'(raw)
// (folded in a fixed order by reduce_partials_kernel).  d_mu / d_var NULL: zero.
struct AcqMomentBwdArgs {
  long long n; int S; int tiled;
  const double* mu; const double* var; double noise_lo, noise_hi; const double* raw_noise;
  const double* d_mu; const double* d_var;
  double* dmu; double* dvar;  // [R] of the top layer
  double* part;               // [gridDim.x] or NULL
};
constexpr int ACQ_THREADS = 256;
__global__ void __launch_bounds__(ACQ_THREADS) acq_moment_bwd_kernel(const __grid_constant__ AcqMomentBwdArgs a) {
  __shared__ double red[ACQ_THREADS / 32];
  const long long i = (long long)blockIdx.x * ACQ_THREADS + threadIdx.x;
  const double sg = sigmoid_fwd(*a.raw_noise);
  const double noise = a.noise_lo + (a.noise_hi - a.noise_lo) * sg;
  double dn = 0.0;
  if (i < a.n) {
    const double gm = a.d_mu ? a.d_mu[i] : 0.0, gv = a.d_var ? a.d_var[i] : 0.0;
    if (a.tiled) {
      double s1 = 0.0;      // out_mu exactly as moment_kernel sums it
      for (int s = 0; s < a.S; ++s) s1 += a.mu[i * a.S + s];
      const double mean = s1 / (double)a.S, inv = 1.0 / (double)a.S;
      int live = 0;
      for (int s = 0; s < a.S; ++s) {
        const long long r = i * a.S + s;
        const bool ok = a.var[r] + noise >= kMinVariance;
        a.dmu[r] = gm * inv + gv * 2.0 * (a.mu[r] - mean) * inv;
        a.dvar[r] = ok ? gv * inv : 0.0;
        live += ok;
      }
      dn = gv * (double)live / (double)a.S;
    } else {
      const bool ok = a.var[i] + noise >= kMinVariance;
      a.dmu[i] = gm;
      a.dvar[i] = ok ? gv : 0.0;
      dn = ok ? gv : 0.0;
    }
  }
  if (!a.part) return;
  dn = warp_sum(dn);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = dn;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < ACQ_THREADS / 32; ++w) s += red[w];
    a.part[blockIdx.x] = s * (a.noise_hi - a.noise_lo) * sg * (1.0 - sg);
  }
}

// through the sample propagation f = mu_prev + sqrt(max(var_prev, 1e-10)) eps of the layer above, per row i of the
// layer below (the rows i*prep .. i*prep+prep-1 above read it, row r reads eps[r % S]):
//   dmu_prev[i] = sum_s df[i*prep+s],   dvar_prev[i] = [var_prev >= 1e-10] sum_s df eps / (2 sqrt(max(var_prev, 1e-10)))
__global__ void __launch_bounds__(ACQ_THREADS) acq_prop_bwd_kernel(const double* __restrict__ df,
                                                                   const double* __restrict__ var_prev,
                                                                   const double* __restrict__ eps, long long R_prev,
                                                                   int prep, int S, double* __restrict__ dmu_prev,
                                                                   double* __restrict__ dvar_prev) {
  const long long i = (long long)blockIdx.x * ACQ_THREADS + threadIdx.x;
  if (i >= R_prev) return;
  const long long base = i * prep;
  double s0 = 0.0, s1 = 0.0;
  for (int s = 0; s < prep; ++s) {
    const double g = df[base + s];
    s0 += g;
    s1 = fma(g, eps[(base + s) % S], s1);
  }
  const double v = var_prev[i];
  dmu_prev[i] = s0;
  dvar_prev[i] = v >= kMinVariance ? s1 / (2.0 * sqrt(v)) : 0.0;
}

// dX[i][c] (+)= sum_l sum_{s < xrep_l} dxrow_l[i*xrep_l+s][c]: layer 0 first (xrep 1), then the layers above
// (xrep S), s ascending
struct AcqDxFoldArgs {
  long long n; int d, S, nl;
  const double* dxrow[kMaxLayers];
  double* dX; int accumulate;
};
__global__ void __launch_bounds__(ACQ_THREADS) acq_dx_fold_kernel(const __grid_constant__ AcqDxFoldArgs a) {
  const long long k = (long long)blockIdx.x * ACQ_THREADS + threadIdx.x;
  if (k >= a.n * a.d) return;
  const long long i = k / a.d;
  const int c = (int)(k - i * a.d);
  double s = a.dxrow[0][k];
  for (int l = 1; l < a.nl; ++l)
    for (int j = 0; j < a.S; ++j) s += a.dxrow[l][(i * a.S + j) * a.d + c];
  a.dX[k] = a.accumulate ? a.dX[k] + s : s;
}

__global__ void jes_kernel(const double* __restrict__ vu, const double* __restrict__ vc, double* __restrict__ out,
                           long long n, int accumulate) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double t = 0.5 * (log(vu[i]) - log(vc[i]));
  const double j = t > 0.0 ? t : 0.0;
  out[i] = accumulate ? out[i] + j : j;
}

}  // namespace mobo
