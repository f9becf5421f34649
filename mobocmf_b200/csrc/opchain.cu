// Per-step operator chain of all layers in ONE cooperative launch: one CTA per 32 x 32 block of the lower triangle of
// each layer's M x M matrices (36 CTAs per layer at M = 256), synchronised block-to-block through release/acquire
// flags in global memory (data-flow, no grid-wide barrier).
//
//   P = K(Z_l, Z_l) + jitter I  ->  L = chol(P)  ->  W = L^-1  ->  H = W tril(L_q),  beta = W m,  KL
//
// replaces the K_zz + jitter, psd_safe_cholesky, triangular solves and kl_mvn_mvn that the reference reaches through
// UnwhitenedVariationalStrategy [upstream gpytorch] (mobocmf/layers/mfdgp_hidden_layer.py:17-20,141,145,286;
// mobocmf/mlls/variational_elbo_mf.py:40).  A single-CTA blocked factorisation of a 256 x 256 fp64 matrix is
// latency-bound (0.53 ms measured); here the critical path is 8 diagonal blocks (factor + invert in one warp,
// ~6 us each) with panels, trailing updates, the inverse and H overlapping it on other SMs.
//
//   factorisation (right-looking, owner computes): A_ij -= L_ik L_jk^T (k < j);  L_jj = chol(A_jj), D_j = L_jj^-1;
//                                                  L_ij = A_ij D_j^T
//   inverse:   W_jj = D_j;  W_ij = -D_i sum_{k=j}^{i-1} L_ik W_kj
//   H_ij = sum_{k=j}^{i} W_ik LQ_kj;   beta_i = sum_{k<=i} W_ik m_k   (diagonal CTAs)
// All CTAs of the launch must be co-resident (they wait on one another): launched with cudaLaunchCooperativeKernel.
#include "common.cuh"

namespace mobo {

constexpr int OC_THREADS = 128, OC_LD = 36, OC_MAXBLK = 64;

// flags region of an operator buffer, as ints: [0, 64) L-block done, [64, 128) W-block done (value = attempt that
// produced the block, 1-based), [128] arrival counter, [129 + a] attempt a hit a non-positive pivot (a = 0 .. 3)
constexpr int OC_FAIL = 129, OC_MAX_RETRIES = 3;
__device__ __forceinline__ int* oc_flags(double* ops, int MP) { return reinterpret_cast<int*>(ops + ops_flags(MP)); }

__device__ __forceinline__ int ld_acquire(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release(int* p, int v) {
  asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// Flags carry the number of the factorisation attempt that produced the block (1-based, see the retry loop of
// opchain_kernel): every thread of the CTA may read the producer's data of attempt `want` after this returns
__device__ __forceinline__ void oc_wait(const int* flag, int want) {
  if (threadIdx.x == 0) {
    while (ld_acquire(flag) < want) __nanosleep(40);
  }
  __syncthreads();
}
// call after the CTA's global writes; makes them visible before the flag(s)
__device__ __forceinline__ void oc_signal(int want, int* flag, int* flag2 = nullptr) {
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    st_release(flag, want);
    if (flag2) st_release(flag2, want);
  }
}

// 32 x 32 block (row-major, leading dimension ld) from global (L2: written by other SMs) into shared [32][OC_LD]
__device__ __forceinline__ void oc_load(double* __restrict__ dst, const double* __restrict__ src, int ld) {
  const int r = threadIdx.x >> 2, c0 = (threadIdx.x & 3) * 8;
  const double2* p = reinterpret_cast<const double2*>(src + (size_t)r * ld + c0);
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const double2 v = __ldcg(p + q);
    dst[r * OC_LD + c0 + 2 * q] = v.x;
    dst[r * OC_LD + c0 + 2 * q + 1] = v.y;
  }
}
// shared [32][OC_LD] -> global block, optionally transposed
__device__ __forceinline__ void oc_store(double* __restrict__ dst, int ld, const double* __restrict__ src, bool transpose) {
  const int r = threadIdx.x >> 2, c0 = (threadIdx.x & 3) * 8;
#pragma unroll
  for (int q = 0; q < 8; ++q) dst[(size_t)r * ld + c0 + q] = transpose ? src[(c0 + q) * OC_LD + r] : src[r * OC_LD + c0 + q];
}
// shared [32][OC_LD] (optionally read transposed) -> block (rb, cb) of a fragment-order operator copy (common.cuh
// frag_offset): the block is 2 slabs x 8 k-steps of 64 contiguous doubles
__device__ __forceinline__ void oc_store_frag(double* __restrict__ frag, int MP, int rb, int cb,
                                              const double* __restrict__ src, bool transpose) {
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const int e = threadIdx.x + OC_THREADS * q;
    const int ib = e & 1, lane = (e >> 1) & 31, kq = (e >> 6) & 7, sl = e >> 9;
    const int r = 16 * sl + 8 * ib + (lane >> 2), c = 4 * kq + (lane & 3);
    frag[((size_t)(2 * rb + sl) * (MP >> 2) + 8 * cb + kq) * 64 + (e & 63)] =
        transpose ? src[c * OC_LD + r] : src[r * OC_LD + c];
  }
}
__device__ __forceinline__ void oc_zero_block(double* __restrict__ dst, int ld) {
  const int r = threadIdx.x >> 2, c0 = (threadIdx.x & 3) * 8;
#pragma unroll
  for (int q = 0; q < 8; ++q) dst[(size_t)r * ld + c0 + q] = 0.0;
}

// acc (this warp's 16 x 16 quadrant of a 32 x 32 product) += sgn * A[r][k] * B,  B given as Bs[n][k] (BT) or Bs[k][n]
template <bool BT>
__device__ __forceinline__ void oc_mma(double (&acc)[2][2][2], const double* __restrict__ As,
                                       const double* __restrict__ Bs, double sgn, int wr, int wc, int g, int t) {
#pragma unroll
  for (int kk = 0; kk < 32; kk += 4) {
    double af[2], bf[2];
#pragma unroll
    for (int x = 0; x < 2; ++x) af[x] = sgn * As[(16 * wr + 8 * x + g) * OC_LD + kk + t];
#pragma unroll
    for (int y = 0; y < 2; ++y)
      bf[y] = BT ? Bs[(16 * wc + 8 * y + g) * OC_LD + kk + t] : Bs[(kk + t) * OC_LD + 16 * wc + 8 * y + g];
#pragma unroll
    for (int x = 0; x < 2; ++x)
#pragma unroll
      for (int y = 0; y < 2; ++y) dmma884(acc[x][y][0], acc[x][y][1], af[x], bf[y]);
  }
}
__device__ __forceinline__ void oc_acc_to_smem(const double (&acc)[2][2][2], double* __restrict__ dst, int wr, int wc,
                                               int g, int t) {
#pragma unroll
  for (int x = 0; x < 2; ++x)
#pragma unroll
    for (int y = 0; y < 2; ++y)
#pragma unroll
      for (int e = 0; e < 2; ++e) dst[(16 * wr + 8 * x + g) * OC_LD + 16 * wc + 8 * y + 2 * t + e] = acc[x][y][e];
}
__device__ __forceinline__ void oc_zero_acc(double (&acc)[2][2][2]) {
#pragma unroll
  for (int x = 0; x < 2; ++x)
#pragma unroll
    for (int y = 0; y < 2; ++y) { acc[x][y][0] = 0.0; acc[x][y][1] = 0.0; }
}

#ifdef OC_TIMING
__device__ unsigned long long oc_times[64][8];
__device__ __forceinline__ unsigned long long oc_now() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#define OC_TICK(k) do { if (threadIdx.x == 0 && blockIdx.x < 64) oc_times[blockIdx.x][k] = oc_now(); } while (0)
#else
#define OC_TICK(k)
#endif

__global__ void opchain_reset_kernel(LayerBatch b) {
  int* fl = oc_flags(b.ops[blockIdx.x], b.MP);
  for (int i = threadIdx.x; i < 256; i += blockDim.x) fl[i] = 0;
}

// attempt > 0: upstream psd_safe_cholesky's retries (linear_operator, reached through UnwhitenedVariationalStrategy):
// Aprime.diagonal().add_(1e-8 * 10^i - previous) for i = 0 .. attempt - 1, the same sequence of fp64 additions
__device__ inline double oc_kernel_entry(const KernParams& kp, int kind, int d, const double* __restrict__ Zx,
                                         const double* __restrict__ zf, int M, int i, int j, double jitter,
                                         int attempt) {
  if (i >= M || j >= M) return i == j ? 1.0 : 0.0;
  if (i == j) {
    double v = kern_diag(kp, kind == 1 ? zf[i] : 0.0) + jitter;
    double prev = 0.0, p10 = 1.0;
    for (int a = 0; a < attempt; ++a) {
      const double jn = 1e-8 * p10;
      v += jn - prev;
      prev = jn;
      p10 *= 10.0;
    }
    return v;
  }
  return kern_entry(kp, d, Zx + (size_t)i * d, kind == 1 ? zf[i] : 0.0, Zx + (size_t)j * d, kind == 1 ? zf[j] : 0.0);
}

__global__ void __launch_bounds__(OC_THREADS) opchain_kernel(LayerBatch b, double jitter) {
  __shared__ __align__(16) double Abuf[32 * OC_LD], Bbuf[32 * OC_LD], Cbuf[32 * OC_LD], Dbuf[32 * OC_LD];
  __shared__ KernParams kp;
  __shared__ bool retry;
  __shared__ double part[4][4];     // [warp][h2, beta2, logdetP, logdetQ]
  __shared__ double rdiag[32];
  __shared__ bool last;
  const int MP = b.MP, M = b.M, d = b.d;
  const int nb = MP / 32, nblk = nb * (nb + 1) / 2;
  const int layer = blockIdx.x / nblk, q = blockIdx.x - layer * nblk;
  int bi = 0, bj = 0;
  { int rem = q; while (rem > bi) { rem -= bi + 1; ++bi; } bj = rem; }
  const bool diag = bi == bj;
  const int kind = b.kind[layer];
  double* ops = b.ops[layer];
  double* Lg = ops + ops_block(MP, OPS_L);
  double* Wg = ops + ops_block(MP, OPS_W);
  double* WTg = ops + ops_block(MP, OPS_WT);
  double* Hg = ops + ops_block(MP, OPS_H);
  double* HTg = ops + ops_block(MP, OPS_HT);
  double* Pg = ops + ops_block(MP, OPS_P);
  double* LQg = ops + ops_block(MP, OPS_LQ);
  int* flags = oc_flags(ops, MP);
  auto Lflag = [&](int i, int j) { return flags + i * (i + 1) / 2 + j; };
  auto Wflag = [&](int i, int j) { return flags + OC_MAXBLK + i * (i + 1) / 2 + j; };
  auto blk = [&](double* base, int i, int j) { return base + (size_t)(32 * i) * MP + 32 * j; };
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3, wr = warp >> 1, wc = warp & 1;
  const double* Zx = b.Zx[layer];
  const double* zf = b.zf[layer];
  const double* Lq = b.Lq[layer];
  const double* mvec = b.m[layer];
  double* rowstat = ops + ops_rowstat(MP);     // [nblk][4] per-CTA partials

  OC_TICK(0);
  if (tid == 0) load_kern_params(kp, kind, d, b.theta[layer]);
  __syncthreads();

  // Upstream factors P with psd_safe_cholesky: when a pivot is not positive the factorisation is retried with
  // 1e-8, 1e-7, 1e-6 more on the diagonal (SURVEY.md quirk Q5).  Here every CTA runs the attempt to its end (a failed
  // attempt only produces garbage that nobody keeps; the flags still advance, so nothing dead-locks), learns the
  // outcome from the last diagonal block's flag + the attempt's failure flag, and all CTAs repeat together.  Flags
  // hold the attempt number, so a block of attempt a is never taken for one of attempt a + 1; the success path pays
  // one acquire load.  The attempt is a lambda instantiated twice: attempt 0 as straight-line code (wrapped in a loop
  // the compiler kept the unrolled 32 x 32 factorisation of the diagonal CTAs in local memory: 0.22 -> 0.35 ms), the
  // retries in a loop whose code quality does not matter.
  auto run_attempt = [&](const int attempt) -> bool {
  const int want = attempt + 1;
  double acc[2][2][2];
  // ---- own block of P = K(Z, Z) + jitter I (identity padded) ----
#pragma unroll
  for (int x = 0; x < 2; ++x)
#pragma unroll
    for (int y = 0; y < 2; ++y)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int r = 16 * wr + 8 * x + g, c = 16 * wc + 8 * y + 2 * t + e;
        acc[x][y][e] = oc_kernel_entry(kp, kind, d, Zx, zf, M, 32 * bi + r, 32 * bj + c, jitter, attempt);
      }
  oc_acc_to_smem(acc, Cbuf, wr, wc, g, t);
  __syncthreads();
  oc_store(blk(Pg, bi, bj), MP, Cbuf, false);
  if (!diag) oc_store(blk(Pg, bj, bi), MP, Cbuf, true);

  OC_TICK(1);
  // ---- factorisation ----
  for (int k = 0; k < bj; ++k) {
    oc_wait(Lflag(bi, k), want);
    if (!diag) oc_wait(Lflag(bj, k), want);
    oc_load(Abuf, blk(Lg, bi, k), MP);
    if (!diag) oc_load(Bbuf, blk(Lg, bj, k), MP);
    __syncthreads();
    oc_mma<true>(acc, Abuf, diag ? Abuf : Bbuf, -1.0, wr, wc, g, t);
    __syncthreads();
  }
  OC_TICK(2);
  if (diag) {
    oc_acc_to_smem(acc, Cbuf, wr, wc, g, t);
    __syncthreads();
    if (warp == 0) {
      double row[32], rinv = 1.0;
#pragma unroll
      for (int c = 0; c < 32; ++c) row[c] = Cbuf[lane * OC_LD + c];
      int fail = 0;
      chol32_inwarp(row, rinv, lane, fail);
      if (fail && lane == 0) atomicExch(flags + OC_FAIL + attempt, 1);   // ordered before the block's flags below
#pragma unroll
      for (int c = 0; c < 32; ++c) Abuf[lane * OC_LD + c] = c <= lane ? row[c] : 0.0;   // L_jj
      rdiag[lane] = rinv;
      __syncwarp();
      // D_j = L_jj^-1, lane = column, right-looking forward substitution: the dependent chain is one multiply and
      // one fma per row; the updates of the rows below are independent
      double x[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) x[i] = (i == lane) ? 1.0 : 0.0;
#pragma unroll
      for (int k = 0; k < 32; ++k) {
        x[k] *= rdiag[k];
#pragma unroll
        for (int i = k + 1; i < 32; ++i) x[i] = fma(-Abuf[i * OC_LD + k], x[k], x[i]);
      }
#pragma unroll
      for (int i = 0; i < 32; ++i) Dbuf[i * OC_LD + lane] = x[i];                        // D_j = W_jj
    }
    __syncthreads();
    OC_TICK(3);
    oc_store(blk(Lg, bi, bi), MP, Abuf, false);
    oc_store(blk(Wg, bi, bi), MP, Dbuf, false);
    oc_store(blk(WTg, bi, bi), MP, Dbuf, true);
    oc_signal(want, Lflag(bi, bi), Wflag(bi, bi));
    OC_TICK(4);
  } else {
    oc_acc_to_smem(acc, Abuf, wr, wc, g, t);
    oc_wait(Lflag(bj, bj), want);
    oc_load(Bbuf, blk(Wg, bj, bj), MP);
    __syncthreads();
    oc_zero_acc(acc);
    oc_mma<true>(acc, Abuf, Bbuf, 1.0, wr, wc, g, t);                                   // L_ij = A D_j^T
    __syncthreads();
    oc_acc_to_smem(acc, Cbuf, wr, wc, g, t);
    __syncthreads();
    oc_store(blk(Lg, bi, bj), MP, Cbuf, false);
    oc_zero_block(blk(Lg, bj, bi), MP);
    oc_signal(want, Lflag(bi, bj));
    OC_TICK(3);
    // ---- inverse: W_ij = -D_i sum_{k=j}^{i-1} L_ik W_kj ----
    oc_zero_acc(acc);
    for (int k = bj; k < bi; ++k) {
      if (k != bj) oc_wait(Lflag(bi, k), want);
      oc_wait(Wflag(k, bj), want);
      if (k != bj) oc_load(Abuf, blk(Lg, bi, k), MP);
      else for (int idx = tid; idx < 32 * OC_LD; idx += OC_THREADS) Abuf[idx] = Cbuf[idx];   // own L_ij
      oc_load(Bbuf, blk(Wg, k, bj), MP);
      __syncthreads();
      oc_mma<false>(acc, Abuf, Bbuf, 1.0, wr, wc, g, t);
      __syncthreads();
    }
    oc_acc_to_smem(acc, Bbuf, wr, wc, g, t);                                            // S
    oc_wait(Lflag(bi, bi), want);
    oc_load(Abuf, blk(Wg, bi, bi), MP);                                                 // D_i
    __syncthreads();
    oc_zero_acc(acc);
    oc_mma<false>(acc, Abuf, Bbuf, -1.0, wr, wc, g, t);
    __syncthreads();
    oc_acc_to_smem(acc, Dbuf, wr, wc, g, t);                                            // W_ij
    __syncthreads();
    oc_store(blk(Wg, bi, bj), MP, Dbuf, false);
    oc_store(blk(WTg, bj, bi), MP, Dbuf, true);
    oc_zero_block(blk(Wg, bj, bi), MP);
    oc_zero_block(blk(WTg, bi, bj), MP);
    oc_signal(want, Wflag(bi, bj));
    OC_TICK(4);
  }
  // here Dbuf = own W_ij (diag: D_j)

  // ---- H_ij = sum_{k=j}^{i} W_ik LQ_kj,  LQ = tril(L_q) zero padded ----
  oc_zero_acc(acc);
  for (int k = bj; k <= bi; ++k) {
    const double* Asrc = Dbuf;
    if (k != bj) {
      if (k == bi) oc_wait(Lflag(bi, bi), want); else oc_wait(Wflag(bi, k), want);
      oc_load(Abuf, blk(Wg, bi, k), MP);
      Asrc = Abuf;
    }
    {
      const int r = tid >> 2, c0 = (tid & 3) * 8;
      const int row = 32 * k + r;
#pragma unroll
      for (int qq = 0; qq < 8; ++qq) {
        const int col = 32 * bj + c0 + qq;
        Bbuf[r * OC_LD + c0 + qq] = (row < M && col <= row) ? Lq[(size_t)row * M + col] : 0.0;
      }
    }
    __syncthreads();
    if (k == bi) {   // LQ_ij is this CTA's block of the padded tril(L_q)
      oc_store(blk(LQg, bi, bj), MP, Bbuf, false);
      if (!diag) oc_zero_block(blk(LQg, bj, bi), MP);
    }
    oc_mma<false>(acc, Asrc, Bbuf, 1.0, wr, wc, g, t);
    __syncthreads();
  }
  oc_acc_to_smem(acc, Cbuf, wr, wc, g, t);
  __syncthreads();
  oc_store(blk(Hg, bi, bj), MP, Cbuf, false);
  oc_store(blk(HTg, bj, bi), MP, Cbuf, true);
  if (!diag) { oc_zero_block(blk(Hg, bj, bi), MP); oc_zero_block(blk(HTg, bi, bj), MP); }
  // fragment-order copies for the row kernels (nobody in this launch waits for them): Dbuf = W_ij, Cbuf = H_ij
  oc_store_frag(ops + ops_block(MP, OPS_WF), MP, bi, bj, Dbuf, false);
  oc_store_frag(ops + ops_block(MP, OPS_WTF), MP, bj, bi, Dbuf, true);
  oc_store_frag(ops + ops_block(MP, OPS_HF), MP, bi, bj, Cbuf, false);
  oc_store_frag(ops + ops_block(MP, OPS_HTF), MP, bj, bi, Cbuf, true);

  OC_TICK(5);
  // ---- per-CTA pieces of the KL: |H_ij|_F^2; diagonal CTAs add beta_i, |beta_i|^2 and the log-determinants ----
  double h2 = 0.0;
#pragma unroll
  for (int x = 0; x < 2; ++x)
#pragma unroll
    for (int y = 0; y < 2; ++y)
#pragma unroll
      for (int e = 0; e < 2; ++e) h2 = fma(acc[x][y][e], acc[x][y][e], h2);
  h2 = warp_sum(h2);
  if (lane == 0) { part[warp][0] = h2; part[warp][1] = 0.0; part[warp][2] = 0.0; part[warp][3] = 0.0; }
  if (diag) {
    // beta_i = sum_{k <= i} W_ik m_k : 4 threads per row, each over a quarter of every 32-block
    const int r = tid >> 2, part4 = tid & 3;
    double s = 0.0;
    for (int k = 0; k <= bi; ++k) {
      const double* Ws = Dbuf;
      if (k != bi) {
        oc_wait(Wflag(bi, k), want);
        oc_load(Abuf, blk(Wg, bi, k), MP);
        __syncthreads();
        Ws = Abuf;
      }
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const int col = 32 * k + 8 * part4 + c;
        s = fma(Ws[r * OC_LD + 8 * part4 + c], col < M ? mvec[col] : 0.0, s);
      }
      __syncthreads();
    }
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    const int row = 32 * bi + r;
    if (row >= M) s = 0.0;
    if (part4 == 0) (ops + ops_beta(MP))[row] = s;
    // row statistics: beta_r^2, 2 log L_rr, log Lq_rr^2  (identity padding contributes nothing)
    double b2 = part4 == 0 ? s * s : 0.0, ldp = 0.0, ldq = 0.0;
    if (part4 == 0 && row < M) {
      const double lrr = __ldcg(blk(Lg, bi, bi) + (size_t)r * MP + r);
      const double qrr = Lq[(size_t)row * M + row];
      ldp = 2.0 * log(lrr);
      ldq = log(qrr * qrr);
    }
    b2 = warp_sum(b2); ldp = warp_sum(ldp); ldq = warp_sum(ldq);
    if (lane == 0) { part[warp][1] = b2; part[warp][2] = ldp; part[warp][3] = ldq; }
  }
  __syncthreads();
  if (tid < 4) rowstat[4 * q + tid] = (part[0][tid] + part[1][tid]) + (part[2][tid] + part[3][tid]);
  // ---- did this attempt factor P?  The last diagonal block is factored after every other one ----
  oc_wait(Lflag(nb - 1, nb - 1), want);
  if (tid == 0) retry = ld_acquire(flags + OC_FAIL + attempt) != 0 && attempt < OC_MAX_RETRIES;
  __syncthreads();
  return retry;
  };  // run_attempt
  int attempt = 0;
  if (run_attempt(0)) {
    do { ++attempt; } while (run_attempt(attempt));
  }
  __threadfence();
  __syncthreads();
  OC_TICK(6);
  if (tid == 0) last = atomicAdd(flags + 128, 1) == nblk - 1;
  __syncthreads();
  if (last && warp == 0) {
    __threadfence();
    double v[4];
#pragma unroll
    for (int s4 = 0; s4 < 4; ++s4) {
      double s = 0.0;
      for (int c = lane; c < nblk; c += 32) s += __ldcg(rowstat + 4 * c + s4);
      v[s4] = warp_sum(s);
    }
    if (lane == 0) {
      double* scal = ops + ops_scal(MP);
      scal[SC_H2] = v[0]; scal[SC_BETA2] = v[1]; scal[SC_LOGDET_P] = v[2]; scal[SC_LOGDET_Q] = v[3];
      scal[SC_KL] = 0.5 * (v[2] - v[3] + v[1] + v[0] - (double)M);
      scal[SC_STATUS] = ld_acquire(flags + OC_FAIL + attempt) ? 1.0 : 0.0;
      scal[SC_RETRIES] = (double)attempt;
    }
  }
}

}  // namespace mobo
