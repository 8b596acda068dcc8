// Greedy Fisher-information selection for multi-class models over the last FC layer or the last two (block form, sm_100a).
//
// Last-layer FI of a sample with posteriors pi (c classes) and feature vector u (d):  F_i = A(pi_i) (x) ut_i ut_i^T,
// A(pi) = diag pi - pi pi^T (NN.LLFC_hess, NN.py:891-901), ut = [u;1], D = c(d+1).  A(pi) = L L^T with the closed-form
// c x (c-1) factor (a_j, b_j: tail sums of pi from j and from j+1)
//     L[j,j] = sqrt(pi_j b_j / a_j),   L[i,j] = -pi_i sqrt(pi_j / (a_j b_j))  (i > j),   column j = 0 if pi_j = 0 or b_j = 0,
// so sample i owns r = c-1 columns G_i = L_i (x) ut_i and the block kernel is K_ij = (L_i^T L_j) s_ij, s_ij = u_i.u_j + 1.
// Greedy step (|S| = t, alpha = (t+1) delta, C = (alpha I + K_SS)^-1, k_j = [K_ij]_{i in S}, Y_j = C k_j):
//     Sigma_j = alpha I + K_jj - k_j^T Y_j,  E_j = Y_j^T Y_j,  loss_j = tr(Sigma_j^-1 (I + E_j)),
// pick argmin (ties: lowest candidate index); reduced objective after the pick  red = (t+1)(tr C + loss_w).
// Y_j is formed through Z = C Lblk^T (tr x tc, once per step, Lblk = blockdiag of the winners' L):
//     Y_j = (sum_a s_{w_a j} Z[:, a-block]) L_j
// so a candidate costs ~t^2 r c multiply-adds per step.  All algebra after the u.u dot is float64.  Kernels per step:
//     append (block row of K_SS) -> build (alpha I + K_SS, identity-padded to a multiple of 64) -> nnal_gj64_invert ->
//     Z + tr C -> eval (per-candidate loss, block arg-min, last-CTA global arg-min) -> column (s_{., w} for the winner).
// The host only enqueues; results are read once at the end.
//
// Two layers (n_layers = 2: the last FC (W3, b3) and the one before it (W2, b2)).  a = input of the feature layer's FC
// (d_p = prev_dim), at = [a;1], m = 1[u > 0], M = diag m.  The score of class y is
//     g_y = [(e_y - pi) (x) ut ; (M W3^T (e_y - pi)) (x) at],   D = c(d+1) + d(d_p+1),
// so F_i = sum_y pi_y g_y g_y^T = G_i G_i^T with the same L_i, and the block kernel keeps its shape:
//     K_ij = L_i^T N_ij L_j,   N_ij = s_ij I_c + s'_ij Q_ij,
//     s_ij = u_i.u_j + 1,  s'_ij = a_i.a_j + 1,  Q_ij = W3 diag(m_i o m_j) W3^T   (c x c, symmetric).
// At c = 2 this is sqrt(w_i w_j) [2 s_ij + (delta2_i.delta2_j) s'_ij], the binary two-layer kernel of fi.cu.  The greedy step
// is unchanged; only k_j changes, and with it
//     Y_j = C k_j = (sum_a Z[:, a-block] N_{w_a j}) L_j
// (~t^2 r c^2 multiply-adds per candidate and step).  A column of winner w holds, per candidate j, cw = c(c+1)/2 + 2
// doubles [s_wj, s'_wj, Q_wj (upper triangle, row-major)].  Q_{., w} = Mask P_w is a GEMM with an exact 0/1 A operand
// (Mask[j,k] = m_j[k]) and P_w[k,(y,z)] = m_w[k] W3[y,k] W3[z,k] (exact in float64: a product of two floats), accumulated
// in float64 in a fixed order.  Set-up runs the same GEMM with P = P_1 (m_w = 1) for Q_jj.
//
// Kept classes (one layer).  Every candidate carries an ascending list of q class ids and the float32 posteriors of those
// classes: without a class cap the identity 0..c-1 (q = c <= 32), with a cap r the r-hat = min(r, c) most probable classes
// (ties: lower class index, topc_kernel), renormalised over the kept ones.  L_i is then q x (q-1) in kept order, and every
// sum over classes above runs over the classes two candidates share, in ascending class order:
//     K_ij = s_ij sum_{cls_i[x] = cls_j[x']} L_i[x,:]^T L_j[x',:],   Z = C Lblk^T keeps q columns per winner,
//     W_j[rho, x'] = sum_a s_{w_a j} Z[rho, (a, x)] over the x with cls_{w_a}[x] = cls_j[x'],   Y_j = W_j L_j.
// With the identity list these are the dense sums in the same order, so an uncapped run is the dense block form bit for bit.
// The two-layer kernels run on the identity list only (q = c).
#include "nnal_common.cuh"
#include "dots.cuh"
#include "../../include/nnal_b200.h"
#include <algorithm>
#include <climits>
#include <cmath>

namespace fib {

constexpr int MAX_C = 32;              // the fused head's class limit; the most classes kept per candidate
constexpr int64_t MAX_KR = 4096;       // k (q-1): order of the largest system inverted per step
constexpr int RT = 8;                  // rows of Z per eval tile
constexpr int EVAL_THREADS = 256;
constexpr size_t EVAL_SMEM_MAX = 200 * 1024;
constexpr size_t EVAL2_SMEM_MAX = 110 * 1024;

struct State {
  int64_t n = 0;
  int c = 0, q = 0, r = 0, d = 0;       // classes, classes kept per candidate, r = q-1
  const float* post = nullptr;           // [c][ldp] posteriors (null: kept classes given by the host)
  int64_t ldp = 0;
  const float* U = nullptr;              // [.][d] feature rows
  int64_t* rows = nullptr;               // candidate i -> row of post / U (null: identity)
  bool use_rows = false;
  bool have = false;                     // candidates set
  float *ownP = nullptr, *ownU = nullptr;
  int64_t cap_p = 0, cap_u = 0, cap_rows = 0;
  int* cls = nullptr;                    // [n][q] kept class ids, ascending
  float* pk = nullptr;                   // [n][q] their posteriors
  int64_t cap_cls = 0, cap_pk = 0;
  double *Lall = nullptr, *Kd = nullptr; // [n][q][r], [n][r][r]
  int64_t cap_L = 0, cap_K = 0;
  unsigned char* avail = nullptr;
  int64_t cap_avail = 0;
  // greedy
  double *Scols = nullptr;               // [k][n]  s_{i, w_t}
  int64_t cap_scols = 0;
  double *Kss = nullptr, *M = nullptr, *Z = nullptr, *Lsel = nullptr, *red = nullptr, *trC = nullptr;
  int64_t cap_kss = 0, cap_m = 0, cap_z = 0, cap_lsel = 0, cap_red = 0;
  long long* sel = nullptr;
  int64_t cap_sel = 0;
  int* Csel = nullptr;                   // [k][q] the winners' class ids
  int64_t cap_csel = 0;
  double* blk_loss = nullptr;
  long long* blk_idx = nullptr;
  int64_t cap_blk = 0, cap_blk_idx = 0;
  unsigned int* ticket = nullptr;
  // two layers
  int nl = 1, dp = 0, nq = 0, cw = 1;    // layers covered, prev dim, c(c+1)/2, doubles per candidate in a column
  const float* A = nullptr;              // [.][dp] inputs of the feature layer's FC (rows as U)
  const float* W3 = nullptr;             // [c][d] last FC weights
  float *ownA = nullptr, *ownW = nullptr;
  int64_t cap_a = 0, cap_w = 0;
  double *Cd = nullptr, *Pw = nullptr;   // [n][cw] candidates' own columns (set-up), [d][nq] P_w of the current winner
  int64_t cap_cd = 0, cap_pw = 0;
  // nnal_pool_top_classes
  int64_t* tc_rows = nullptr;
  int* tc_cls = nullptr;
  float* tc_p = nullptr;
  int64_t cap_tc_rows = 0, cap_tc_cls = 0, cap_tc_p = 0;
};

static State* get(nnal_ctx* ctx) {
  if (!ctx->fi_block_state) ctx->fi_block_state = new State();
  return (State*)ctx->fi_block_state;
}

// grow-only device buffer
template <typename T>
static int grow(nnal_ctx* ctx, T*& p, int64_t& cap, int64_t want) {
  if (p && cap >= want) return NNAL_OK;
  if (p) { CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream)); CUDA_TRY(ctx, cudaFree(p)); p = nullptr; cap = 0; }
  CUDA_TRY(ctx, cudaMalloc(&p, (size_t)std::max<int64_t>(want, 1) * sizeof(T)));
  cap = want;
  return NNAL_OK;
}

// ---- kept classes: the q largest of c posteriors per candidate (ties: lower class index), written in ascending class order ----
// One warp per candidate.  Lane l < q holds one kept entry; the classes stream past in chunks of 32 (one per lane), and a
// chunk entry that beats the worst kept entry replaces it.  Requires q <= c (every placeholder gets replaced).
__device__ inline void worst_kept(float kv, int ki, int q, float& wv, int& wi, int& wl) {
  const int lane = threadIdx.x & 31;
  wv = lane < q ? kv : INFINITY;                              // lanes >= q never hold the worst
  wi = lane < q ? ki : -1;
  wl = lane;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, wv, o);
    const int oi = __shfl_xor_sync(0xffffffffu, wi, o), ol = __shfl_xor_sync(0xffffffffu, wl, o);
    // worst: smallest value, then largest class, then lowest lane (placeholders tie: every lane must agree on one)
    if (ov < wv || (ov == wv && (oi > wi || (oi == wi && ol < wl)))) { wv = ov; wi = oi; wl = ol; }
  }
}

__global__ void __launch_bounds__(256) topc_kernel(const float* __restrict__ post, int64_t ldp, const int64_t* __restrict__ rows,
                                                   int64_t n, int c, int q, int* __restrict__ cls, float* __restrict__ pk) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t i = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < n; i += nw) {
    const int64_t row = rows ? rows[i] : i;
    float kv = -INFINITY, wv;
    int ki = INT_MAX, wi, wl;
    worst_kept(kv, ki, q, wv, wi, wl);
    for (int x0 = 0; x0 < c; x0 += 32) {
      const int x = x0 + lane;
      bool live = x < c;
      const float v = live ? post[(int64_t)x * ldp + row] : 0.f;
      while (true) {
        const unsigned m = __ballot_sync(0xffffffffu, live && (v > wv || (v == wv && x < wi)));
        if (!m) break;
        const int src = __ffs(m) - 1;
        const float nv = __shfl_sync(0xffffffffu, v, src);
        const int nx = __shfl_sync(0xffffffffu, x, src);
        if (lane == wl) { kv = nv; ki = nx; }
        if (lane == src) live = false;
        worst_kept(kv, ki, q, wv, wi, wl);
      }
    }
    int rank = 0;
    for (int l = 0; l < q; ++l) rank += __shfl_sync(0xffffffffu, ki, l) < ki;
    if (lane < q) {
      cls[i * q + rank] = ki;
      pk[i * q + rank] = kv;
    }
  }
}

// ---- setup: per candidate L_i (q x r) from the kept posteriors renormalised in float64, K_ii = L_i^T L_i (|u_i|^2 + 1) -------
__global__ void __launch_bounds__(256) setup_kernel(const float* __restrict__ pk, const float* __restrict__ U,
                                                    const int64_t* __restrict__ rows, int64_t n, int q, int d,
                                                    double* __restrict__ Lall, double* __restrict__ Kd,
                                                    unsigned char* __restrict__ avail) {
  __shared__ double ps[8][MAX_C], tail[8][MAX_C + 1];
  const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
  const int r = q - 1;
  double* p = ps[wp];
  double* tl = tail[wp];
  const int64_t nw = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t i = (int64_t)blockIdx.x * (blockDim.x >> 5) + wp; i < n; i += nw) {
    const int64_t row = rows ? rows[i] : i;
    const float* u = U + row * (int64_t)d;
    double uu = 0.0;
    for (int k = lane; k < d; k += 32) { const double v = (double)u[k]; uu = fma(v, v, uu); }
    uu = warp_sum(uu);
    if (lane < q) p[lane] = (double)pk[i * q + lane];
    __syncwarp();
    if (lane == 0) {                                          // ascending class order: the sums of the dense form
      double sum = 0.0;
      for (int j = 0; j < q; ++j) sum += p[j];
      for (int j = 0; j < q; ++j) p[j] = sum > 0.0 ? p[j] / sum : 0.0;
      tl[q] = 0.0;
      for (int j = q - 1; j >= 0; --j) tl[j] = tl[j + 1] + p[j];
      avail[i] = 1;
    }
    __syncwarp();
    double* L = Lall + i * (int64_t)q * r;
    if (lane < r) {
      const int j = lane;
      const double a = tl[j], b = tl[j + 1];
      const bool zero = !(p[j] > 0.0) || !(b > 0.0);
      const double dj = zero ? 0.0 : sqrt(p[j] * b / a);
      const double off = zero ? 0.0 : sqrt(p[j] / (a * b));
      for (int i2 = 0; i2 < q; ++i2) L[i2 * r + j] = i2 < j ? 0.0 : (i2 == j ? dj : -p[i2] * off);
    }
    __syncwarp();
    const double sq = uu + 1.0;
    double* K = Kd + i * (int64_t)r * r;
    for (int e = lane; e < r * r; e += 32) {
      const int y = e / r, z = e - y * r;
      double acc = 0.0;
      for (int x = 0; x < q; ++x) acc = fma(L[x * r + y], L[x * r + z], acc);
      K[e] = acc * sq;
    }
    __syncwarp();                                             // p and tl are reused by the warp's next candidate
  }
}

// ---- column: s_{i,w} = u_i.u_w + 1 for every candidate, w = sel[t] (read on the device) --------------------------------------
__global__ void __launch_bounds__(256) column_kernel(const float* __restrict__ U, const int64_t* __restrict__ rows, int64_t n, int d,
                                                     const long long* __restrict__ sel, int t, double* __restrict__ col) {
  const int lane = threadIdx.x & 31;
  const long long w = sel[t];
  const float* uw = U + (rows ? rows[w] : w) * (int64_t)d;
  const int64_t nw = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t i = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < n; i += nw) {
    const float* u = U + (rows ? rows[i] : i) * (int64_t)d;
    double acc = 0.0;
    for (int k = lane; k < d; k += 32) acc = fma((double)u[k], (double)uw[k], acc);
    acc = warp_sum(acc);
    if (lane == 0) col[i] = acc + 1.0;
  }
}

// ---- two layers ----------------------------------------------------------------------------------------------------------
// packed index of Q[y][z] = Q[z][y]: upper triangle, row-major
__host__ __device__ inline int qidx(int y, int z, int c) {
  if (y > z) { const int tmp = y; y = z; z = tmp; }
  return y * c - (y * (y - 1)) / 2 + (z - y);
}

// (La^T N Lb)[y, z] with N = col[0] I + col[1] Q, Q packed at col + 2.  L[x, y] = 0 for x < y.
__device__ inline double lnl(const double* __restrict__ La, const double* __restrict__ Lb, const double* __restrict__ col, int c,
                             int r, int y, int z) {
  double ll = 0.0, lq = 0.0;
  for (int x = y; x < c; ++x) {
    const double lay = La[x * r + y];
    double qz = 0.0;
    for (int x2 = z; x2 < c; ++x2) qz = fma(col[2 + qidx(x, x2, c)], Lb[x2 * r + z], qz);
    ll = fma(lay, Lb[x * r + z], ll);
    lq = fma(lay, qz, lq);
  }
  return col[0] * ll + col[1] * lq;
}

// s_{i,w} = u_i.u_w + 1 and s'_{i,w} = a_i.a_w + 1 into col[i][0..1] for every candidate; w = sel[t] (sel = null: w = i)
__global__ void __launch_bounds__(256) dots2_kernel(const float* __restrict__ U, const float* __restrict__ A,
                                                    const int64_t* __restrict__ rows, int64_t n, int d, int dp,
                                                    const long long* __restrict__ sel, int t, double* __restrict__ col, int cw) {
  const int lane = threadIdx.x & 31;
  const int64_t rw = sel ? (rows ? rows[sel[t]] : sel[t]) : -1;
  const int64_t nw = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t i = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < n; i += nw) {
    const int64_t ri = rows ? rows[i] : i;
    const int64_t rj = sel ? rw : ri;
    const float *u = U + ri * d, *uw = U + rj * d, *a = A + ri * dp, *aw = A + rj * dp;
    double su = 0.0, sa = 0.0;
    for (int k = lane; k < d; k += 32) su = fma((double)u[k], (double)uw[k], su);
    for (int k = lane; k < dp; k += 32) sa = fma((double)a[k], (double)aw[k], sa);
    su = warp_sum(su);
    sa = warp_sum(sa);
    if (lane == 0) { col[i * cw] = su + 1.0; col[i * cw + 1] = sa + 1.0; }
  }
}

// P[k][(y,z)] = m_w[k] W3[y][k] W3[z][k], w = sel[t] (sel = null: m_w = 1)
__global__ void __launch_bounds__(256) pw_kernel(const float* __restrict__ W3, const float* __restrict__ U,
                                                 const int64_t* __restrict__ rows, int d, int c, int nq,
                                                 const long long* __restrict__ sel, int t, double* __restrict__ P) {
  const float* uw = sel ? U + (rows ? rows[sel[t]] : sel[t]) * (int64_t)d : nullptr;
  const int64_t total = (int64_t)d * nq;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int k = (int)(e / nq);
    int q = (int)(e - (int64_t)k * nq), y = 0;
    while (q >= c - y) { q -= c - y; ++y; }
    const int z = y + q;
    const bool on = !uw || uw[k] > 0.f;
    P[e] = on ? (double)W3[(int64_t)y * d + k] * (double)W3[(int64_t)z * d + k] : 0.0;
  }
}

// col[j][2 + q] = sum_k 1[u_j[k] > 0] P[k][q]: 64 candidates x 64 entries per CTA, 4 x 4 per thread, k in steps of 16,
// float64 in ascending k (deterministic)
constexpr int MG_J = 64, MG_Q = 64, MG_K = 16;
__global__ void __launch_bounds__(256) maskgemm_kernel(const float* __restrict__ U, const int64_t* __restrict__ rows, int64_t n,
                                                       int d, int nq, const double* __restrict__ P, double* __restrict__ col,
                                                       int cw) {
  __shared__ double Ms[MG_K][MG_J + 1];
  __shared__ double Ps[MG_K][MG_Q];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int64_t j0 = (int64_t)blockIdx.x * MG_J;
  const int q0 = blockIdx.y * MG_Q;
  double acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int q = 0; q < 4; ++q) acc[i][q] = 0.0;
  for (int k0 = 0; k0 < d; k0 += MG_K) {
    for (int e = threadIdx.x; e < MG_J * MG_K; e += 256) {
      const int jl = e / MG_K, kk = e - jl * MG_K;
      const int64_t j = j0 + jl;
      const int k = k0 + kk;
      const float v = (j < n && k < d) ? U[(rows ? rows[j] : j) * (int64_t)d + k] : 0.f;
      Ms[kk][jl] = v > 0.f ? 1.0 : 0.0;
    }
    for (int e = threadIdx.x; e < MG_K * MG_Q; e += 256) {
      const int kk = e / MG_Q, ql = e - kk * MG_Q;
      Ps[kk][ql] = (k0 + kk < d && q0 + ql < nq) ? P[(int64_t)(k0 + kk) * nq + q0 + ql] : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < MG_K; ++kk) {
      double m[4], p[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { m[i] = Ms[kk][ty + 16 * i]; p[i] = Ps[kk][tx + 16 * i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int q = 0; q < 4; ++q) acc[i][q] = fma(m[i], p[q], acc[i][q]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t j = j0 + ty + 16 * i;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int qq = q0 + tx + 16 * q;
      if (j < n && qq < nq) col[j * cw + 2 + qq] = acc[i][q];
    }
  }
}

// K_jj = L_j^T N_jj L_j from the candidates' own columns
__global__ void __launch_bounds__(256) kd2_kernel(const double* __restrict__ Lall, const double* __restrict__ Cd, int64_t n, int c,
                                                  int r, int cw, double* __restrict__ Kd) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t i = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < n; i += nw) {
    const double* L = Lall + i * (int64_t)c * r;
    for (int e = lane; e < r * r; e += 32) {
      const int y = e / r, z = e - y * r;
      Kd[i * (int64_t)r * r + e] = lnl(L, L, Cd + i * cw, c, r, y, z);
    }
  }
}

// block row a = t-1 of K_SS and its transpose: K[(a,y),(b,z)] = (L_{w_a}^T N_{w_a w_b} L_{w_b})[y,z].  lnl(y,z) and lnl(z,y)
// round differently, so in the diagonal block only y <= z computes and writes both entries (one writer per entry).
__global__ void __launch_bounds__(256) append2_kernel(const double* __restrict__ Lsel, const double* __restrict__ Scols, int64_t lds,
                                                      int cw, const long long* __restrict__ sel, int a, int c, int r,
                                                      double* __restrict__ Kss, int64_t ldk) {
  const int64_t total = (int64_t)(a + 1) * r * r;
  const double* La = Lsel + (int64_t)a * c * r;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(e / (r * r));
    const int yz = (int)(e - (int64_t)b * r * r);
    const int y = yz / r, z = yz - (yz / r) * r;
    if (b == a && y > z) continue;
    const double v = lnl(La, Lsel + (int64_t)b * c * r, Scols + (int64_t)a * lds + sel[b] * cw, c, r, y, z);
    Kss[(int64_t)(a * r + y) * ldk + b * r + z] = v;
    Kss[(int64_t)(b * r + z) * ldk + a * r + y] = v;
  }
}

// ---- system: block row a = t-1 of K_SS (and its transpose): K[(a,y),(b,z)] = (L_{w_a}^T L_{w_b})[y,z] s_{w_a w_b} -------------
// (sum over the classes both winners kept, ascending)
__global__ void __launch_bounds__(256) append_kernel(const double* __restrict__ Lsel, const int* __restrict__ Csel,
                                                     const double* __restrict__ Scols, int64_t lds,
                                                     const long long* __restrict__ sel, int a, int q, int r,
                                                     double* __restrict__ Kss, int64_t ldk) {
  const int64_t total = (int64_t)(a + 1) * r * r;
  const double* La = Lsel + (int64_t)a * q * r;
  const int* Ca = Csel + (int64_t)a * q;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(e / (r * r));
    const int yz = (int)(e - (int64_t)b * r * r);
    const int y = yz / r, z = yz - (yz / r) * r;
    const double* Lb = Lsel + (int64_t)b * q * r;
    const int* Cb = Csel + (int64_t)b * q;
    double acc = 0.0;
    for (int xa = 0, xb = 0; xa < q && xb < q;) {
      const int ga = Ca[xa], gb = Cb[xb];
      if (ga == gb) acc = fma(La[xa * r + y], Lb[xb * r + z], acc);
      xa += ga <= gb;
      xb += gb <= ga;
    }
    const double v = acc * Scols[(int64_t)a * lds + sel[b]];
    Kss[(int64_t)(a * r + y) * ldk + b * r + z] = v;
    Kss[(int64_t)(b * r + z) * ldk + a * r + y] = v;
  }
}

__global__ void __launch_bounds__(256) build_kernel(const double* __restrict__ Kss, int64_t ldk, int m, int np, double alpha,
                                                    double* __restrict__ M) {
  const int64_t total = (int64_t)np * np;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)(e / np), j = (int)(e - (int64_t)i * np);
    M[e] = (i < m && j < m) ? Kss[(int64_t)i * ldk + j] + (i == j ? alpha : 0.0) : (i == j ? 1.0 : 0.0);
  }
}

// Z[rho, (a,x)] = sum_y C[rho, (a,y)] L_{w_a}[x,y]   (x: winner a's kept classes)
__global__ void __launch_bounds__(256) z_kernel(const double* __restrict__ Cm, int np, const double* __restrict__ Lsel, int t, int q,
                                                int r, double* __restrict__ Z, int64_t ldz) {
  const int m = t * r;
  const int64_t total = (int64_t)m * t * q;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int rho = (int)(e / ((int64_t)t * q));
    const int col = (int)(e - (int64_t)rho * t * q);
    const int a = col / q, x = col - (col / q) * q;
    const double* Crow = Cm + (int64_t)rho * np + a * r;
    const double* La = Lsel + (int64_t)a * q * r + x * r;
    double acc = 0.0;
    for (int y = 0; y < r; ++y) acc = fma(Crow[y], La[y], acc);
    Z[(int64_t)rho * ldz + col] = acc;
  }
}

// tr C over the first m diagonal entries, fixed summation order (one CTA)
__global__ void __launch_bounds__(256) trace_kernel(const double* __restrict__ Cm, int np, int m, double* __restrict__ out) {
  __shared__ double part[256];
  double acc = 0.0;
  for (int i = threadIdx.x; i < m; i += 256) acc += Cm[(int64_t)i * np + i];
  part[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) part[threadIdx.x] += part[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) *out = part[0];
}

// ---- eval: per-candidate loss, block arg-min, last-CTA global arg-min ----------------------------------------------------
struct EvalArgs {
  const double* Lall; const double* Kd; const double* Z; int64_t ldz;
  const double* Scols; int64_t lds;
  const int* cls; int* Csel;
  double* Lsel; unsigned char* avail;
  int64_t n; int q, r, t, JC, AT, cw; double alpha;
  const double* trC;
  double* blk_loss; long long* blk_idx; unsigned int* ticket;
  long long* sel; double* red;
};

struct EvalLayout {
  int Ls, E, G, Zs, Ss, Ws, Ys, Ks, loss, Cj, Ct, total;     // offsets in doubles (Cj, Ct: int arrays)
};

__host__ __device__ inline EvalLayout eval_layout(int JC, int AT, int q, int r, int cw) {
  EvalLayout l;
  int o = 0;
  l.Ls = o; o += JC * q * r;
  l.E = o; o += JC * r * r;
  l.G = o; o += JC * r * r;
  l.Zs = o; o += RT * AT * q;
  l.Ss = o; o += AT * JC * cw;
  l.Ws = o; o += JC * RT * q;
  l.Ys = o; o += JC * RT * r;
  l.Ks = o; o += JC * RT * r;
  l.loss = o; o += JC;
  l.Cj = o; o += (JC * q + 1) / 2;
  l.Ct = o; o += (AT * q + 1) / 2;
  l.total = o;
  return l;
}

// loss = tr(Sigma^-1 (I + E)) by Cholesky of Sigma (in place, r x r), columnwise forward substitution; +inf if not SPD
__device__ double block_loss(double* __restrict__ Sg, const double* __restrict__ E, int r, double* __restrict__ v,
                             double* __restrict__ w) {
  for (int j = 0; j < r; ++j) {
    double s = Sg[j * r + j];
    for (int k = 0; k < j; ++k) s -= Sg[j * r + k] * Sg[j * r + k];
    if (!(s > 0.0)) return INFINITY;
    const double l = sqrt(s);
    Sg[j * r + j] = l;
    for (int i = j + 1; i < r; ++i) {
      double q = Sg[i * r + j];
      for (int k = 0; k < j; ++k) q -= Sg[i * r + k] * Sg[j * r + k];
      Sg[i * r + j] = q / l;
    }
  }
  // tr(Sigma^-1 M) = sum_i (L^-1 e_i) . (L^-1 m_i),  M = I + E
  double tr = 0.0;
  for (int i = 0; i < r; ++i) {
    for (int y = 0; y < r; ++y) {
      double a = (y == i ? 1.0 : 0.0), b = E[y * r + i] + (y == i ? 1.0 : 0.0);
      for (int k = 0; k < y; ++k) { a -= Sg[y * r + k] * v[k]; b -= Sg[y * r + k] * w[k]; }
      v[y] = a / Sg[y * r + y];
      w[y] = b / Sg[y * r + y];
    }
    for (int y = i; y < r; ++y) tr = fma(v[y], w[y], tr);      // (L^-1 e_i) vanishes above i
  }
  return tr;
}

// position of class g in the ascending list C[0..q-1], -1 if absent: first try `hint` (exact for the identity list), else bisect
__device__ inline int find_class(const int* C, int q, int g, int hint) {
  if (C[hint] == g) return hint;
  int lo = 0, hi = q;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (C[mid] < g) lo = mid + 1;
    else hi = mid;
  }
  return lo < q && C[lo] == g ? lo : -1;
}

// NL = 2: Ss holds the winners' whole columns [AT][JC][cw], W_j sums Z[:, a-block] N_{w_a j}, and k_j = L^T N L (q = c).
// ALL: every candidate keeps every class (q = c), so each id list is 0..c-1 and every class lookup is its hint.
template <int NL, bool ALL>
__global__ void __launch_bounds__(EVAL_THREADS) eval_kernel(EvalArgs ea) {
  extern __shared__ __align__(16) double sm[];
  const int q = ea.q, r = ea.r, t = ea.t, JC = ea.JC, AT = ea.AT, cw = NL == 2 ? ea.cw : 1;
  const EvalLayout lay = eval_layout(JC, AT, q, r, cw);
  double* Ls = sm + lay.Ls;
  double* E = sm + lay.E;
  double* G = sm + lay.G;
  double* Zs = sm + lay.Zs;
  double* Ss = sm + lay.Ss;
  double* Ws = sm + lay.Ws;
  double* Ys = sm + lay.Ys;
  double* Ks = sm + lay.Ks;
  double* lossv = sm + lay.loss;
  int* Cj = (int*)(sm + lay.Cj);                  // [JC][q] the candidates' class ids
  int* Ct = (int*)(sm + lay.Ct);                  // [AT][q] class ids of the winners in the Z tile
  const int tid = threadIdx.x;
  const int64_t j0 = (int64_t)blockIdx.x * JC;
  for (int e = tid; e < JC * q * r; e += blockDim.x) {
    const int64_t j = j0 + e / (q * r);
    Ls[e] = j < ea.n ? ea.Lall[j0 * q * r + e] : 0.0;
  }
  for (int e = tid; e < JC * q; e += blockDim.x) Cj[e] = j0 + e / q < ea.n ? ea.cls[j0 * q + e] : -1;
  for (int e = tid; e < 2 * JC * r * r; e += blockDim.x) E[e] = 0.0;      // E and G are adjacent
  const int m = t * r;
  const int ZW = AT * q;
  for (int rho0 = 0; rho0 < m; rho0 += RT) {
    // W_j[rho, x'] = sum_a s_{w_a j} Z[rho, (a,x)],  cls_{w_a}[x] = cls_j[x']
    const bool wt = tid < JC * q;
    const int wj = wt ? tid / q : 0, wx = wt ? tid - (tid / q) * q : 0;
    double acc[RT];
#pragma unroll
    for (int qq = 0; qq < RT; ++qq) acc[qq] = 0.0;
    for (int a0 = 0; a0 < t; a0 += AT) {
      __syncthreads();
      for (int e = tid; e < RT * ZW; e += blockDim.x) {
        const int qq = e / ZW, col = e - qq * ZW;
        const int a = a0 + col / q;
        Zs[e] = (rho0 + qq < m && a < t) ? ea.Z[(int64_t)(rho0 + qq) * ea.ldz + (int64_t)a0 * q + col] : 0.0;
      }
      if constexpr (NL == 1) {
        for (int e = tid; e < AT * JC; e += blockDim.x) {
          const int a = e / JC, jj = e - a * JC;
          Ss[e] = (a0 + a < t && j0 + jj < ea.n) ? ea.Scols[(int64_t)(a0 + a) * ea.lds + j0 + jj] : 0.0;
        }
        for (int e = tid; e < AT * q; e += blockDim.x) Ct[e] = a0 + e / q < t ? ea.Csel[(int64_t)a0 * q + e] : -1;
      } else {
        for (int e = tid; e < AT * JC * cw; e += blockDim.x) {
          const int a = e / (JC * cw), jf = e - a * JC * cw;
          Ss[e] = (a0 + a < t && j0 + jf / cw < ea.n) ? ea.Scols[(int64_t)(a0 + a) * ea.lds + j0 * cw + jf] : 0.0;
        }
      }
      __syncthreads();
      if (wt) {
        const int na = min(AT, t - a0);
        for (int a = 0; a < na; ++a) {
          if constexpr (NL == 1) {
            const int x = ALL ? wx : find_class(Ct + a * q, q, Cj[wj * q + wx], wx);
            if (x >= 0) {
              const double sa = Ss[a * JC + wj];
#pragma unroll
              for (int qq = 0; qq < RT; ++qq) acc[qq] = fma(sa, Zs[qq * ZW + a * q + x], acc[qq]);
            }
          } else {
            const double* col = Ss + (a * JC + wj) * cw;           // N[x, wx] = s [x == wx] + s' Q[x, wx]
            for (int x = 0; x < q; ++x) {
              const double nx = fma(col[1], col[2 + qidx(x, wx, q)], x == wx ? col[0] : 0.0);
#pragma unroll
              for (int qq = 0; qq < RT; ++qq) acc[qq] = fma(nx, Zs[qq * ZW + a * q + x], acc[qq]);
            }
          }
        }
      }
    }
    if (wt) {
#pragma unroll
      for (int qq = 0; qq < RT; ++qq) Ws[(wj * RT + qq) * q + wx] = acc[qq];
    }
    __syncthreads();
    // Y_j[rho, y] = W_j[rho, :] L_j[:, y];   k_j[rho, y] = s_{w_a' j} (L_{w_a'}^T L_j)[x', y] over shared classes,  rho = (a', x')
    if (tid < JC * r) {
      const int jj = tid / r, y = tid - (tid / r) * r;
      const int64_t j = j0 + jj;
      const double* Lj = Ls + jj * q * r;
      for (int qq = 0; qq < RT; ++qq) {
        const int row = rho0 + qq;
        double yv = 0.0, kv = 0.0;
        if (row < m && j < ea.n) {
          const int ap = row / r, xp = row - (row / r) * r;
          const double* Wq = Ws + (jj * RT + qq) * q;
          if constexpr (NL == 1) {
            const double* La = ea.Lsel + (int64_t)ap * q * r + xp;
            const int* Ca = ea.Csel + (int64_t)ap * q;
            const int* Cjj = Cj + jj * q;
            for (int x = 0; x < q; ++x) {                      // j's classes ascending: the shared ones in class order
              const double lj = Lj[x * r + y];
              yv = fma(Wq[x], lj, yv);
              const int xa = ALL ? x : find_class(Ca, q, Cjj[x], x);
              if (xa >= 0) kv = fma(La[xa * r], lj, kv);
            }
            kv *= ea.Scols[(int64_t)ap * ea.lds + j];
          } else {
            for (int x = 0; x < q; ++x) yv = fma(Wq[x], Lj[x * r + y], yv);
            kv = lnl(ea.Lsel + (int64_t)ap * q * r, Lj, ea.Scols + (int64_t)ap * ea.lds + j * cw, q, r, xp, y);
          }
        }
        Ys[(jj * RT + qq) * r + y] = yv;
        Ks[(jj * RT + qq) * r + y] = kv;
      }
    }
    __syncthreads();
    // E_j += Y^T Y,  G_j += k^T Y  (row y of each, owned by thread (j, y))
    if (tid < JC * r) {
      const int jj = tid / r, y = tid - (tid / r) * r;
      const double* Yj = Ys + jj * RT * r;
      const double* Kj = Ks + jj * RT * r;
      double* Ej = E + (jj * r + y) * r;
      double* Gj = G + (jj * r + y) * r;
      for (int z = 0; z < r; ++z) {
        double e = Ej[z], g = Gj[z];
#pragma unroll
        for (int qq = 0; qq < RT; ++qq) {
          e = fma(Yj[qq * r + y], Yj[qq * r + z], e);
          g = fma(Kj[qq * r + y], Yj[qq * r + z], g);
        }
        Ej[z] = e;
        Gj[z] = g;
      }
    }
  }
  __syncthreads();
  if (tid < JC) {
    const int64_t j = j0 + tid;
    double loss = INFINITY;
    if (j < ea.n && ea.avail[j]) {
      double* Sg = G + tid * r * r;
      const double* Kj = ea.Kd + j * r * r;
      for (int e = 0; e < r * r; ++e) Sg[e] = Kj[e] - Sg[e] + ((e / r) == (e - (e / r) * r) ? ea.alpha : 0.0);
      double* scratch = Ys + tid * RT * r;        // RT >= 2: room for two r-vectors
      loss = block_loss(Sg, E + tid * r * r, r, scratch, scratch + r);
    }
    lossv[tid] = loss;
  }
  __syncthreads();
  __shared__ bool last;
  __shared__ long long win;
  if (tid == 0) {
    double bl = INFINITY;
    long long bi = -1;
    for (int jj = 0; jj < JC; ++jj)                 // first minimum: ties go to the lowest candidate index
      if (lossv[jj] < bl) { bl = lossv[jj]; bi = j0 + jj; }
    ea.blk_loss[blockIdx.x] = bl;
    ea.blk_idx[blockIdx.x] = bi;
    __threadfence();
    last = atomicAdd(ea.ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!last) return;
  if (tid == 0) {
    __threadfence();
    double bl = INFINITY;
    long long bi = -1;
    for (unsigned b = 0; b < gridDim.x; ++b) {
      const double l = ((volatile double*)ea.blk_loss)[b];
      const long long i = ((volatile long long*)ea.blk_idx)[b];
      if (l < bl) { bl = l; bi = i; }          // blocks are in candidate order
    }
    if (bi < 0) bi = 0;                        // unreachable: k <= n candidates
    ea.sel[t] = bi;
    ea.red[t] = (double)(t + 1) * (*ea.trC + bl);
    ea.avail[bi] = 0;
    *ea.ticket = 0;
    win = bi;
  }
  __syncthreads();
  for (int e = tid; e < q * r; e += blockDim.x) ea.Lsel[(int64_t)t * q * r + e] = ea.Lall[win * q * r + e];
  for (int e = tid; e < q; e += blockDim.x) ea.Csel[(int64_t)t * q + e] = ea.cls[win * q + e];
}

static int warp_grid(nnal_ctx* ctx, int64_t n) {
  const int64_t blocks = (n + 7) / 8;
  return (int)std::max<int64_t>(1, std::min<int64_t>(blocks, (int64_t)ctx->sm_count * 16));
}

static int flat_grid(nnal_ctx* ctx, int64_t total) {
  return (int)std::max<int64_t>(1, std::min<int64_t>((total + 255) / 256, (int64_t)ctx->sm_count * 32));
}

// candidates per eval CTA and winners per Z tile: as many candidates as 256 threads cover, fewer where shared memory runs out
// (two layers: at most EVAL2_SMEM_MAX, so that two CTAs share an SM)
static void eval_plan(int q, int r, int cw, int* JC, int* AT, size_t* smem) {
  const size_t cap = cw == 1 ? EVAL_SMEM_MAX : EVAL2_SMEM_MAX;
  int jc = std::max(1, std::min(64, EVAL_THREADS / q)), at = 32;
  while (true) {
    const size_t bytes = (size_t)eval_layout(jc, at, q, r, cw).total * sizeof(double);
    if (bytes <= cap || (jc == 1 && at == 1)) { *JC = jc; *AT = at; *smem = bytes; return; }
    if (at > (cw == 1 ? 8 : 1)) at /= 2;
    else if (jc > 1) --jc;
    else at = std::max(1, at / 2);
  }
}

// Two-layer columns grow with k n c^2: a size the device cannot hold is refused here instead of failing inside cudaMalloc.
// `held`: bytes of the buffer being grown, freed before the new allocation.
static int check_fits(nnal_ctx* ctx, double want, double held, const char* what) {
  size_t free_b = 0, total_b = 0;
  CUDA_TRY(ctx, cudaMemGetInfo(&free_b, &total_b));
  if (want > (double)free_b + held) {
    char msg[256];
    snprintf(msg, sizeof(msg), "two-layer block FI: %s need %.3g GB, %.3g GB of device memory free", what, want * 1e-9,
             ((double)free_b + held) * 1e-9);
    NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, msg);
  }
  return NNAL_OK;
}

// kept classes of n candidates (rows: positions in post, null = identity) into cls / pk [n][q]
static void launch_topc(nnal_ctx* ctx, const float* post, int64_t ldp, const int64_t* rows, int64_t n, int c, int q, int* cls,
                        float* pk) {
  topc_kernel<<<warp_grid(ctx, n), 256, 0, ctx->stream>>>(post, ldp, rows, n, c, q, cls, pk);
  ctx->launches++;
}

// s->post set: kept classes are selected from it first; null: s->cls / s->pk already hold them
static int setup(nnal_ctx* ctx, State* s) {
  const int64_t n = s->n;
  const int c = s->c, q = s->q, r = s->r;
  NNAL_TRY(grow(ctx, s->cls, s->cap_cls, n * q));
  NNAL_TRY(grow(ctx, s->pk, s->cap_pk, n * q));
  NNAL_TRY(grow(ctx, s->Lall, s->cap_L, n * q * r));
  NNAL_TRY(grow(ctx, s->Kd, s->cap_K, n * r * r));
  NNAL_TRY(grow(ctx, s->avail, s->cap_avail, n));
  if (s->nl == 2) {
    NNAL_TRY(check_fits(ctx, 8.0 * n * s->cw, 8.0 * s->cap_cd, "the candidates' own columns"));
    NNAL_TRY(grow(ctx, s->Cd, s->cap_cd, n * s->cw));
    NNAL_TRY(grow(ctx, s->Pw, s->cap_pw, (int64_t)s->d * s->nq));
  }
  if (n == 0) return NNAL_OK;
  const int64_t* rows = s->use_rows ? s->rows : nullptr;
  if (s->post) launch_topc(ctx, s->post, s->ldp, rows, n, c, q, s->cls, s->pk);
  setup_kernel<<<warp_grid(ctx, n), 256, 0, ctx->stream>>>(s->pk, s->U, rows, n, q, s->d, s->Lall, s->Kd, s->avail);
  ctx->launches++;
  if (s->nl == 2) {
    dots2_kernel<<<warp_grid(ctx, n), 256, 0, ctx->stream>>>(s->U, s->A, rows, n, s->d, s->dp, nullptr, 0, s->Cd, s->cw);
    pw_kernel<<<flat_grid(ctx, (int64_t)s->d * s->nq), 256, 0, ctx->stream>>>(s->W3, s->U, rows, s->d, c, s->nq, nullptr, 0, s->Pw);
    maskgemm_kernel<<<dim3((unsigned)((n + MG_J - 1) / MG_J), (unsigned)((s->nq + MG_Q - 1) / MG_Q)), 256, 0, ctx->stream>>>(
        s->U, rows, n, s->d, s->nq, s->Pw, s->Cd, s->cw);
    kd2_kernel<<<warp_grid(ctx, n), 256, 0, ctx->stream>>>(s->Lall, s->Cd, n, c, r, s->cw, s->Kd);
    ctx->launches += 4;
  }
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}

static void set_layers(State* s, int nl, int c, int dp, const float* A, const float* W3) {
  s->nl = nl;
  s->dp = nl == 2 ? dp : 0;
  s->A = nl == 2 ? A : nullptr;
  s->W3 = nl == 2 ? W3 : nullptr;
  s->nq = nl == 2 ? c * (c + 1) / 2 : 0;
  s->cw = nl == 2 ? s->nq + 2 : 1;
}

// cap = 0: every class (c <= MAX_C); else the min(cap, c) most probable, 2 <= cap <= MAX_C (one layer)
static int set_candidates(nnal_ctx* ctx, const int64_t* cand, int64_t n_cand, int n_layers, int cap) {
  if (!ctx || n_cand < 0) return NNAL_ERR_INVALID;
  if (n_layers != 1 && n_layers != 2) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "block FI covers the last 1 or 2 fully-connected layers");
  if (!ctx->pool_post || !ctx->pool_feat || ctx->keep < 1) NNAL_FAIL(ctx, NNAL_ERR_STATE, "pool pass did not keep the feature layer");
  if (n_layers == 2 && (!ctx->pool_prev || ctx->keep < 2)) NNAL_FAIL(ctx, NNAL_ERR_STATE, "pool pass did not keep the previous FC output");
  if (ctx->n_class < 2 || (!cap && ctx->n_class > MAX_C)) NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "block FI supports 2 <= c <= 32");
  if (ctx->feature_layer != (int)ctx->layers.size() - 2) NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "feature layer must feed the last FC layer");
  if (n_layers == 2 && (ctx->feature_layer < 1 || ctx->layers[ctx->feature_layer - 1].type != NNAL_LAYER_FC))
    NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "two-layer block FI needs an FC layer before the feature layer");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const int64_t n = cand ? n_cand : ctx->pool_n;
  if (cand)
    for (int64_t i = 0; i < n; ++i)
      if (cand[i] < 0 || cand[i] >= ctx->pool_n) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "candidate position outside the pool");
  State* s = get(ctx);
  s->have = false;
  s->n = n; s->c = ctx->n_class; s->q = cap ? std::min(cap, s->c) : s->c; s->r = s->q - 1; s->d = ctx->feat_dim;
  s->post = ctx->pool_post; s->ldp = ctx->pool_n; s->U = ctx->pool_feat;
  set_layers(s, n_layers, s->c, ctx->prev_dim, ctx->pool_prev, ctx->layers.back().W);
  s->use_rows = cand != nullptr;
  if (cand && n) {
    NNAL_TRY(grow(ctx, s->rows, s->cap_rows, n));
    CUDA_TRY(ctx, cudaMemcpyAsync(s->rows, cand, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
  }
  NNAL_TRY(setup(ctx, s));
  NNAL_SYNC_CHECKED(ctx);                                 // `cand` is caller-owned host memory; fp16 range flag of the pool pass
  s->have = true;
  return NNAL_OK;
}

}  // namespace fib

int nnal_fi_block_release(nnal_ctx* ctx) {
  if (!ctx->fi_block_state) return NNAL_OK;
  fib::State* s = (fib::State*)ctx->fi_block_state;
  void* ptrs[] = {s->ownP, s->ownU, s->rows, s->cls, s->pk, s->Lall, s->Kd, s->avail, s->Scols, s->Kss, s->M, s->Z, s->Lsel,
                  s->Csel, s->red, s->trC, s->sel, s->blk_loss, s->blk_idx, s->ticket, s->ownA, s->ownW, s->Cd, s->Pw,
                  s->tc_rows, s->tc_cls, s->tc_p};
  for (void* p : ptrs) if (p) cudaFree(p);
  delete s;
  ctx->fi_block_state = nullptr;
  return NNAL_OK;
}

extern "C" int nnal_fi_block_set_candidates_nl(nnal_ctx* ctx, const int64_t* cand, int64_t n_cand, int n_layers) {
  return fib::set_candidates(ctx, cand, n_cand, n_layers, 0);
}

extern "C" int nnal_fi_block_set_candidates(nnal_ctx* ctx, const int64_t* cand, int64_t n_cand) {
  return fib::set_candidates(ctx, cand, n_cand, 1, 0);
}

extern "C" int nnal_fi_block_set_candidates_cls(nnal_ctx* ctx, const int64_t* cand, int64_t n_cand, int r) {
  if (ctx && (r < 2 || r > fib::MAX_C)) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "block FI keeps 2 to 32 classes per candidate");
  return fib::set_candidates(ctx, cand, n_cand, 1, r);
}

extern "C" int nnal_fi_block_set_factors_nl(nnal_ctx* ctx, int64_t n, int c, int d, int d_prev, const float* post, const float* U,
                                            const float* A_prev, const float* w_last) {
  if (!ctx || n < 0 || d <= 0 || (n > 0 && (!post || !U))) return NNAL_ERR_INVALID;
  if ((A_prev != nullptr) != (w_last != nullptr) || (A_prev && d_prev <= 0))
    NNAL_FAIL(ctx, NNAL_ERR_INVALID, "two-layer block FI needs both the previous activations and the last-layer weights");
  if (c < 2 || c > fib::MAX_C) NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "block FI supports 2 <= c <= 32");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  fib::State* s = fib::get(ctx);
  s->have = false;
  s->n = n; s->c = c; s->q = c; s->r = c - 1; s->d = d;
  NNAL_TRY(fib::grow(ctx, s->ownP, s->cap_p, n * c));
  NNAL_TRY(fib::grow(ctx, s->ownU, s->cap_u, n * d));
  if (n) {
    CUDA_TRY(ctx, cudaMemcpyAsync(s->ownP, post, (size_t)n * c * 4, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(s->ownU, U, (size_t)n * d * 4, cudaMemcpyHostToDevice, ctx->stream));
  }
  if (A_prev) {
    NNAL_TRY(fib::grow(ctx, s->ownA, s->cap_a, n * d_prev));
    NNAL_TRY(fib::grow(ctx, s->ownW, s->cap_w, (int64_t)c * d));
    if (n) CUDA_TRY(ctx, cudaMemcpyAsync(s->ownA, A_prev, (size_t)n * d_prev * 4, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(s->ownW, w_last, (size_t)c * d * 4, cudaMemcpyHostToDevice, ctx->stream));
  }
  s->post = s->ownP; s->ldp = n; s->U = s->ownU; s->use_rows = false;
  fib::set_layers(s, A_prev ? 2 : 1, c, d_prev, s->ownA, s->ownW);
  NNAL_TRY(fib::setup(ctx, s));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  s->have = true;
  return NNAL_OK;
}

extern "C" int nnal_fi_block_set_factors(nnal_ctx* ctx, int64_t n, int c, int d, const float* post, const float* U) {
  return nnal_fi_block_set_factors_nl(ctx, n, c, d, 0, post, U, nullptr, nullptr);
}

extern "C" int nnal_fi_block_set_factors_cls(nnal_ctx* ctx, int64_t n, int c, int r, int d, const int32_t* cls, const float* p,
                                             const float* U) {
  if (!ctx || n < 0 || d <= 0 || (n > 0 && (!cls || !p || !U))) return NNAL_ERR_INVALID;
  if (c < 2) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "block FI needs c >= 2 classes");
  if (r < 2 || r > fib::MAX_C || r > c) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "block FI keeps 2 to min(32, c) classes per candidate");
  for (int64_t i = 0; i < n; ++i)
    for (int x = 0; x < r; ++x) {
      const int32_t g = cls[i * r + x];
      if (g < 0 || g >= c) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "kept class id outside 0..c-1");
      if (x > 0 && !(g > cls[i * r + x - 1])) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "kept class ids must be strictly ascending");
    }
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  fib::State* s = fib::get(ctx);
  s->have = false;
  s->n = n; s->c = c; s->q = r; s->r = r - 1; s->d = d;
  NNAL_TRY(fib::grow(ctx, s->cls, s->cap_cls, n * r));
  NNAL_TRY(fib::grow(ctx, s->pk, s->cap_pk, n * r));
  NNAL_TRY(fib::grow(ctx, s->ownU, s->cap_u, n * d));
  if (n) {
    CUDA_TRY(ctx, cudaMemcpyAsync(s->cls, cls, (size_t)n * r * 4, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(s->pk, p, (size_t)n * r * 4, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(s->ownU, U, (size_t)n * d * 4, cudaMemcpyHostToDevice, ctx->stream));
  }
  s->post = nullptr; s->ldp = 0; s->U = s->ownU; s->use_rows = false;
  fib::set_layers(s, 1, c, 0, nullptr, nullptr);
  NNAL_TRY(fib::setup(ctx, s));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  s->have = true;
  return NNAL_OK;
}

extern "C" int nnal_pool_top_classes(nnal_ctx* ctx, const int64_t* rows, int64_t n, int r, int32_t* cls_out, float* p_out) {
  if (!ctx || n < 0 || (n > 0 && (!cls_out || !p_out))) return NNAL_ERR_INVALID;
  if (r < 2 || r > fib::MAX_C) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "block FI keeps 2 to 32 classes per candidate");
  if (!ctx->pool_post) NNAL_FAIL(ctx, NNAL_ERR_STATE, "no pool pass");
  if (!rows && n > ctx->pool_n) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "more rows than the pool holds");
  if (rows)
    for (int64_t i = 0; i < n; ++i)
      if (rows[i] < 0 || rows[i] >= ctx->pool_n) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "row outside the pool");
  if (n == 0) return NNAL_OK;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  fib::State* s = fib::get(ctx);
  const int c = ctx->n_class, q = std::min(r, c);
  NNAL_TRY(fib::grow(ctx, s->tc_cls, s->cap_tc_cls, n * q));
  NNAL_TRY(fib::grow(ctx, s->tc_p, s->cap_tc_p, n * q));
  if (rows) {
    NNAL_TRY(fib::grow(ctx, s->tc_rows, s->cap_tc_rows, n));
    CUDA_TRY(ctx, cudaMemcpyAsync(s->tc_rows, rows, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
  }
  fib::launch_topc(ctx, ctx->pool_post, ctx->pool_n, rows ? s->tc_rows : nullptr, n, c, q, s->tc_cls, s->tc_p);
  CUDA_TRY(ctx, cudaGetLastError());
  CUDA_TRY(ctx, cudaMemcpyAsync(cls_out, s->tc_cls, (size_t)n * q * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(p_out, s->tc_p, (size_t)n * q * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return NNAL_OK;
}

extern "C" int nnal_fi_block_greedy(nnal_ctx* ctx, int64_t k, double delta, int64_t* sel_out, double* obj_out, double* red_out) {
  if (!ctx || k < 0 || !(delta > 0) || (k > 0 && !sel_out)) return NNAL_ERR_INVALID;
  if (!ctx->fi_block_state || !((fib::State*)ctx->fi_block_state)->have) NNAL_FAIL(ctx, NNAL_ERR_STATE, "block FI candidates not set");
  fib::State* s = (fib::State*)ctx->fi_block_state;
  const int64_t n = s->n;
  const int c = s->c, q = s->q, r = s->r, cw = s->cw;
  if (k > n) k = n;
  if (k * r > fib::MAX_KR)
    NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "block FI greedy supports k (q-1) <= 4096, q = classes kept per candidate (c without a cap)");
  if (k == 0) return NNAL_OK;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const int64_t mmax = k * r;
  const int npmax = (int)((mmax + 63) / 64 * 64);
  const int64_t ldk = mmax, ldz = k * q, lds = n * cw;    // column t of candidate j, entry e: Scols[t lds + j cw + e]
  int JC, AT;
  size_t smem;
  fib::eval_plan(q, r, cw, &JC, &AT, &smem);
  const int nblk = (int)((n + JC - 1) / JC);
  if (s->nl == 2) NNAL_TRY(fib::check_fits(ctx, 8.0 * k * lds, 8.0 * s->cap_scols, "the winners' columns"));
  NNAL_TRY(fib::grow(ctx, s->Scols, s->cap_scols, k * lds));
  NNAL_TRY(fib::grow(ctx, s->Kss, s->cap_kss, mmax * mmax));
  NNAL_TRY(fib::grow(ctx, s->M, s->cap_m, (int64_t)npmax * npmax));
  NNAL_TRY(fib::grow(ctx, s->Z, s->cap_z, mmax * ldz));
  NNAL_TRY(fib::grow(ctx, s->Lsel, s->cap_lsel, k * q * r));
  NNAL_TRY(fib::grow(ctx, s->Csel, s->cap_csel, k * q));
  NNAL_TRY(fib::grow(ctx, s->red, s->cap_red, k));
  NNAL_TRY(fib::grow(ctx, s->sel, s->cap_sel, k));
  NNAL_TRY(fib::grow(ctx, s->blk_loss, s->cap_blk, (int64_t)nblk));
  NNAL_TRY(fib::grow(ctx, s->blk_idx, s->cap_blk_idx, (int64_t)nblk));
  if (!s->trC) { CUDA_TRY(ctx, cudaMalloc(&s->trC, sizeof(double))); }
  if (!s->ticket) {
    CUDA_TRY(ctx, cudaMalloc(&s->ticket, 64));
    CUDA_TRY(ctx, cudaMemsetAsync(s->ticket, 0, 64, ctx->stream));
  }
  static bool attr = false;
  if (!attr) {
    CUDA_TRY(ctx, cudaFuncSetAttribute(fib::eval_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fib::EVAL_SMEM_MAX));
    CUDA_TRY(ctx, cudaFuncSetAttribute(fib::eval_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fib::EVAL_SMEM_MAX));
    CUDA_TRY(ctx, cudaFuncSetAttribute(fib::eval_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fib::EVAL_SMEM_MAX));
    attr = true;
  }
  CUDA_TRY(ctx, cudaMemsetAsync(s->avail, 1, (size_t)n, ctx->stream));
  CUDA_TRY(ctx, cudaMemsetAsync(s->trC, 0, sizeof(double), ctx->stream));
  const int64_t* rows = s->use_rows ? s->rows : nullptr;
  fib::EvalArgs ea;
  ea.Lall = s->Lall; ea.Kd = s->Kd; ea.Z = s->Z; ea.ldz = ldz; ea.Scols = s->Scols; ea.lds = lds; ea.cls = s->cls; ea.Csel = s->Csel;
  ea.Lsel = s->Lsel; ea.avail = s->avail; ea.n = n; ea.q = q; ea.r = r; ea.JC = JC; ea.AT = AT; ea.cw = cw;
  ea.trC = s->trC; ea.blk_loss = s->blk_loss; ea.blk_idx = s->blk_idx; ea.ticket = s->ticket; ea.sel = s->sel; ea.red = s->red;
  for (int t = 0; t < (int)k; ++t) {
    const double alpha = (double)(t + 1) * delta;
    if (t > 0) {
      prof_begin(ctx, NNAL_PROF_FIB_SYSTEM);
      const int m = t * r;
      const int np = (m + 63) / 64 * 64;
      if (s->nl == 2)
        fib::append2_kernel<<<fib::flat_grid(ctx, (int64_t)t * r * r), 256, 0, ctx->stream>>>(s->Lsel, s->Scols, lds, cw, s->sel,
                                                                                                t - 1, c, r, s->Kss, ldk);
      else
        fib::append_kernel<<<fib::flat_grid(ctx, (int64_t)t * r * r), 256, 0, ctx->stream>>>(s->Lsel, s->Csel, s->Scols, lds, s->sel,
                                                                                               t - 1, q, r, s->Kss, ldk);
      fib::build_kernel<<<fib::flat_grid(ctx, (int64_t)np * np), 256, 0, ctx->stream>>>(s->Kss, ldk, m, np, alpha, s->M);
      ctx->launches += 2;
      NNAL_TRY(nnal_gj64_invert(ctx, s->M, np));
      fib::z_kernel<<<fib::flat_grid(ctx, (int64_t)m * t * q), 256, 0, ctx->stream>>>(s->M, np, s->Lsel, t, q, r, s->Z, ldz);
      fib::trace_kernel<<<1, 256, 0, ctx->stream>>>(s->M, np, m, s->trC);
      ctx->launches += 2;
      prof_end(ctx);
    }
    prof_begin(ctx, NNAL_PROF_FIB_EVAL);
    ea.t = t;
    ea.alpha = alpha;
    if (s->nl == 2) fib::eval_kernel<2, true><<<nblk, fib::EVAL_THREADS, smem, ctx->stream>>>(ea);
    else if (q == c) fib::eval_kernel<1, true><<<nblk, fib::EVAL_THREADS, smem, ctx->stream>>>(ea);
    else fib::eval_kernel<1, false><<<nblk, fib::EVAL_THREADS, smem, ctx->stream>>>(ea);
    ctx->launches++;
    prof_end(ctx);
    if (t + 1 < (int)k) {
      prof_begin(ctx, NNAL_PROF_FIB_COLUMN);
      double* col = s->Scols + (int64_t)t * lds;
      if (s->nl == 2) {
        fib::dots2_kernel<<<fib::warp_grid(ctx, n), 256, 0, ctx->stream>>>(s->U, s->A, rows, n, s->d, s->dp, s->sel, t, col, cw);
        fib::pw_kernel<<<fib::flat_grid(ctx, (int64_t)s->d * s->nq), 256, 0, ctx->stream>>>(s->W3, s->U, rows, s->d, c, s->nq,
                                                                                              s->sel, t, s->Pw);
        fib::maskgemm_kernel<<<dim3((unsigned)((n + fib::MG_J - 1) / fib::MG_J), (unsigned)((s->nq + fib::MG_Q - 1) / fib::MG_Q)),
                               256, 0, ctx->stream>>>(s->U, rows, n, s->d, s->nq, s->Pw, col, cw);
        ctx->launches += 3;
      } else {
        fib::column_kernel<<<fib::warp_grid(ctx, n), 256, 0, ctx->stream>>>(s->U, rows, n, s->d, s->sel, t, col);
        ctx->launches++;
      }
      prof_end(ctx);
    }
    CUDA_TRY(ctx, cudaGetLastError());
  }
  std::vector<double> red((size_t)k);
  static_assert(sizeof(long long) == sizeof(int64_t), "");
  CUDA_TRY(ctx, cudaMemcpyAsync(sel_out, s->sel, (size_t)k * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(red.data(), s->red, (size_t)k * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  const double D = (double)c * (s->d + 1.0) + (s->nl == 2 ? (double)s->d * (s->dp + 1.0) : 0.0);
  for (int64_t t = 0; t < k; ++t) {
    if (red_out) red_out[t] = red[t];
    if (obj_out) obj_out[t] = (D - (double)(t + 1) * r) / delta + red[t];
  }
  return NNAL_OK;
}
