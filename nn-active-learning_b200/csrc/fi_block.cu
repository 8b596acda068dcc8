// Greedy Fisher-information selection for multi-class models over the last FC layer (block form, sm_100a).
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
#include "nnal_common.cuh"
#include "dots.cuh"
#include "../../include/nnal_b200.h"
#include <algorithm>
#include <cmath>

namespace fib {

constexpr int MAX_C = 32;              // the fused head's class limit
constexpr int64_t MAX_KR = 4096;       // k (c-1): order of the largest system inverted per step
constexpr int RT = 8;                  // rows of Z per eval tile
constexpr int EVAL_THREADS = 256;
constexpr size_t EVAL_SMEM_MAX = 200 * 1024;

struct State {
  int64_t n = 0;
  int c = 0, r = 0, d = 0;
  const float* post = nullptr;           // [c][ldp] posteriors
  int64_t ldp = 0;
  const float* U = nullptr;              // [.][d] feature rows
  int64_t* rows = nullptr;               // candidate i -> row of post / U (null: identity)
  bool use_rows = false;
  bool have = false;                     // candidates set
  float *ownP = nullptr, *ownU = nullptr;
  int64_t cap_p = 0, cap_u = 0, cap_rows = 0;
  double *Lall = nullptr, *Kd = nullptr; // [n][c][r], [n][r][r]
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
  double* blk_loss = nullptr;
  long long* blk_idx = nullptr;
  int64_t cap_blk = 0, cap_blk_idx = 0;
  unsigned int* ticket = nullptr;
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

// ---- setup: per candidate L_i (c x r) from the renormalised float64 posteriors and K_ii = L_i^T L_i (|u_i|^2 + 1) ----------
__global__ void __launch_bounds__(256) setup_kernel(const float* __restrict__ post, int64_t ldp, const float* __restrict__ U,
                                                    const int64_t* __restrict__ rows, int64_t n, int c, int d,
                                                    double* __restrict__ Lall, double* __restrict__ Kd,
                                                    unsigned char* __restrict__ avail) {
  const int lane = threadIdx.x & 31;
  const int r = c - 1;
  const int64_t nw = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t i = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < n; i += nw) {
    const int64_t row = rows ? rows[i] : i;
    const float* u = U + row * (int64_t)d;
    double uu = 0.0;
    for (int k = lane; k < d; k += 32) { const double v = (double)u[k]; uu = fma(v, v, uu); }
    uu = warp_sum(uu);
    double* L = Lall + i * (int64_t)c * r;
    if (lane == 0) {
      double p[MAX_C], tail[MAX_C + 1];
      double sum = 0.0;
      for (int j = 0; j < c; ++j) { p[j] = (double)post[(int64_t)j * ldp + row]; sum += p[j]; }
      for (int j = 0; j < c; ++j) p[j] = sum > 0.0 ? p[j] / sum : 0.0;
      tail[c] = 0.0;
      for (int j = c - 1; j >= 0; --j) tail[j] = tail[j + 1] + p[j];
      for (int j = 0; j < r; ++j) {
        const double a = tail[j], b = tail[j + 1];
        const bool zero = !(p[j] > 0.0) || !(b > 0.0);
        const double dj = zero ? 0.0 : sqrt(p[j] * b / a);
        const double off = zero ? 0.0 : sqrt(p[j] / (a * b));
        for (int i2 = 0; i2 < c; ++i2) L[i2 * r + j] = i2 < j ? 0.0 : (i2 == j ? dj : -p[i2] * off);
      }
      avail[i] = 1;
    }
    __syncwarp();
    const double sq = uu + 1.0;
    double* K = Kd + i * (int64_t)r * r;
    for (int e = lane; e < r * r; e += 32) {
      const int y = e / r, z = e - y * r;
      double acc = 0.0;
      for (int x = 0; x < c; ++x) acc = fma(L[x * r + y], L[x * r + z], acc);
      K[e] = acc * sq;
    }
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

// ---- system: block row a = t-1 of K_SS (and its transpose): K[(a,y),(b,z)] = (L_{w_a}^T L_{w_b})[y,z] s_{w_a w_b} -------------
__global__ void __launch_bounds__(256) append_kernel(const double* __restrict__ Lsel, const double* __restrict__ Scols, int64_t lds,
                                                     const long long* __restrict__ sel, int a, int c, int r,
                                                     double* __restrict__ Kss, int64_t ldk) {
  const int64_t total = (int64_t)(a + 1) * r * r;
  const double* La = Lsel + (int64_t)a * c * r;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(e / (r * r));
    const int yz = (int)(e - (int64_t)b * r * r);
    const int y = yz / r, z = yz - (yz / r) * r;
    const double* Lb = Lsel + (int64_t)b * c * r;
    double acc = 0.0;
    for (int x = 0; x < c; ++x) acc = fma(La[x * r + y], Lb[x * r + z], acc);
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

// Z[rho, (a,x)] = sum_y C[rho, (a,y)] L_{w_a}[x,y]
__global__ void __launch_bounds__(256) z_kernel(const double* __restrict__ Cm, int np, const double* __restrict__ Lsel, int t, int c,
                                                int r, double* __restrict__ Z, int64_t ldz) {
  const int m = t * r;
  const int64_t total = (int64_t)m * t * c;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int rho = (int)(e / ((int64_t)t * c));
    const int col = (int)(e - (int64_t)rho * t * c);
    const int a = col / c, x = col - (col / c) * c;
    const double* Crow = Cm + (int64_t)rho * np + a * r;
    const double* La = Lsel + (int64_t)a * c * r + x * r;
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
  double* Lsel; unsigned char* avail;
  int64_t n; int c, r, t, JC, AT; double alpha;
  const double* trC;
  double* blk_loss; long long* blk_idx; unsigned int* ticket;
  long long* sel; double* red;
};

struct EvalLayout {
  int Ls, E, G, Zs, Ss, Ws, Ys, Ks, loss, total;     // offsets in doubles
};

__host__ __device__ inline EvalLayout eval_layout(int JC, int AT, int c, int r) {
  EvalLayout l;
  int o = 0;
  l.Ls = o; o += JC * c * r;
  l.E = o; o += JC * r * r;
  l.G = o; o += JC * r * r;
  l.Zs = o; o += RT * AT * c;
  l.Ss = o; o += AT * JC;
  l.Ws = o; o += JC * RT * c;
  l.Ys = o; o += JC * RT * r;
  l.Ks = o; o += JC * RT * r;
  l.loss = o; o += JC;
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

__global__ void __launch_bounds__(EVAL_THREADS) eval_kernel(EvalArgs ea) {
  extern __shared__ __align__(16) double sm[];
  const int c = ea.c, r = ea.r, t = ea.t, JC = ea.JC, AT = ea.AT;
  const EvalLayout lay = eval_layout(JC, AT, c, r);
  double* Ls = sm + lay.Ls;
  double* E = sm + lay.E;
  double* G = sm + lay.G;
  double* Zs = sm + lay.Zs;
  double* Ss = sm + lay.Ss;
  double* Ws = sm + lay.Ws;
  double* Ys = sm + lay.Ys;
  double* Ks = sm + lay.Ks;
  double* lossv = sm + lay.loss;
  const int tid = threadIdx.x;
  const int64_t j0 = (int64_t)blockIdx.x * JC;
  for (int e = tid; e < JC * c * r; e += blockDim.x) {
    const int64_t j = j0 + e / (c * r);
    Ls[e] = j < ea.n ? ea.Lall[j0 * c * r + e] : 0.0;
  }
  for (int e = tid; e < 2 * JC * r * r; e += blockDim.x) E[e] = 0.0;      // E and G are adjacent
  const int m = t * r;
  const int ZW = AT * c;
  for (int rho0 = 0; rho0 < m; rho0 += RT) {
    // W_j[rho, x] = sum_a s_{w_a j} Z[rho, (a,x)]
    const bool wt = tid < JC * c;
    const int wj = wt ? tid / c : 0, wx = wt ? tid - (tid / c) * c : 0;
    double acc[RT];
#pragma unroll
    for (int q = 0; q < RT; ++q) acc[q] = 0.0;
    for (int a0 = 0; a0 < t; a0 += AT) {
      __syncthreads();
      for (int e = tid; e < RT * ZW; e += blockDim.x) {
        const int q = e / ZW, col = e - q * ZW;
        const int a = a0 + col / c;
        Zs[e] = (rho0 + q < m && a < t) ? ea.Z[(int64_t)(rho0 + q) * ea.ldz + (int64_t)a0 * c + col] : 0.0;
      }
      for (int e = tid; e < AT * JC; e += blockDim.x) {
        const int a = e / JC, jj = e - a * JC;
        Ss[e] = (a0 + a < t && j0 + jj < ea.n) ? ea.Scols[(int64_t)(a0 + a) * ea.lds + j0 + jj] : 0.0;
      }
      __syncthreads();
      if (wt) {
        const int na = min(AT, t - a0);
        for (int a = 0; a < na; ++a) {
          const double sa = Ss[a * JC + wj];
#pragma unroll
          for (int q = 0; q < RT; ++q) acc[q] = fma(sa, Zs[q * ZW + a * c + wx], acc[q]);
        }
      }
    }
    if (wt) {
#pragma unroll
      for (int q = 0; q < RT; ++q) Ws[(wj * RT + q) * c + wx] = acc[q];
    }
    __syncthreads();
    // Y_j[rho, y] = W_j[rho, :] L_j[:, y];   k_j[rho, y] = s_{w_a' j} (L_{w_a'}^T L_j)[x', y],  rho = (a', x')
    if (tid < JC * r) {
      const int jj = tid / r, y = tid - (tid / r) * r;
      const int64_t j = j0 + jj;
      const double* Lj = Ls + jj * c * r;
      for (int q = 0; q < RT; ++q) {
        const int row = rho0 + q;
        double yv = 0.0, kv = 0.0;
        if (row < m && j < ea.n) {
          const int ap = row / r, xp = row - (row / r) * r;
          const double* Wq = Ws + (jj * RT + q) * c;
          const double* La = ea.Lsel + (int64_t)ap * c * r + xp;
          for (int x = 0; x < c; ++x) {
            yv = fma(Wq[x], Lj[x * r + y], yv);
            kv = fma(La[x * r], Lj[x * r + y], kv);
          }
          kv *= ea.Scols[(int64_t)ap * ea.lds + j];
        }
        Ys[(jj * RT + q) * r + y] = yv;
        Ks[(jj * RT + q) * r + y] = kv;
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
        for (int q = 0; q < RT; ++q) {
          e = fma(Yj[q * r + y], Yj[q * r + z], e);
          g = fma(Kj[q * r + y], Yj[q * r + z], g);
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
  for (int e = tid; e < c * r; e += blockDim.x) ea.Lsel[(int64_t)t * c * r + e] = ea.Lall[win * c * r + e];
}

static int warp_grid(nnal_ctx* ctx, int64_t n) {
  const int64_t blocks = (n + 7) / 8;
  return (int)std::max<int64_t>(1, std::min<int64_t>(blocks, (int64_t)ctx->sm_count * 16));
}

static int flat_grid(nnal_ctx* ctx, int64_t total) {
  return (int)std::max<int64_t>(1, std::min<int64_t>((total + 255) / 256, (int64_t)ctx->sm_count * 32));
}

// candidates per eval CTA and winners per Z tile: as many candidates as 256 threads cover, fewer where shared memory runs out
static void eval_plan(int c, int r, int* JC, int* AT, size_t* smem) {
  int jc = std::max(1, std::min(64, EVAL_THREADS / c)), at = 32;
  while (true) {
    const size_t bytes = (size_t)eval_layout(jc, at, c, r).total * sizeof(double);
    if (bytes <= EVAL_SMEM_MAX || (jc == 1 && at == 1)) { *JC = jc; *AT = at; *smem = bytes; return; }
    if (at > 8) at /= 2;
    else if (jc > 1) --jc;
    else at = std::max(1, at / 2);
  }
}

static int setup(nnal_ctx* ctx, State* s) {
  const int64_t n = s->n;
  const int c = s->c, r = s->r;
  NNAL_TRY(grow(ctx, s->Lall, s->cap_L, n * c * r));
  NNAL_TRY(grow(ctx, s->Kd, s->cap_K, n * r * r));
  NNAL_TRY(grow(ctx, s->avail, s->cap_avail, n));
  if (n == 0) return NNAL_OK;
  setup_kernel<<<warp_grid(ctx, n), 256, 0, ctx->stream>>>(s->post, s->ldp, s->U, s->use_rows ? s->rows : nullptr, n, c, s->d,
                                                           s->Lall, s->Kd, s->avail);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}

}  // namespace fib

int nnal_fi_block_release(nnal_ctx* ctx) {
  if (!ctx->fi_block_state) return NNAL_OK;
  fib::State* s = (fib::State*)ctx->fi_block_state;
  void* ptrs[] = {s->ownP, s->ownU, s->rows, s->Lall, s->Kd, s->avail, s->Scols, s->Kss, s->M, s->Z, s->Lsel, s->red, s->trC,
                  s->sel, s->blk_loss, s->blk_idx, s->ticket};
  for (void* p : ptrs) if (p) cudaFree(p);
  delete s;
  ctx->fi_block_state = nullptr;
  return NNAL_OK;
}

extern "C" int nnal_fi_block_set_candidates(nnal_ctx* ctx, const int64_t* cand, int64_t n_cand) {
  if (!ctx || n_cand < 0) return NNAL_ERR_INVALID;
  if (!ctx->pool_post || !ctx->pool_feat || ctx->keep < 1) NNAL_FAIL(ctx, NNAL_ERR_STATE, "pool pass did not keep the feature layer");
  if (ctx->n_class < 2 || ctx->n_class > fib::MAX_C) NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "block FI supports 2 <= c <= 32");
  if (ctx->feature_layer != (int)ctx->layers.size() - 2) NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "feature layer must feed the last FC layer");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const int64_t n = cand ? n_cand : ctx->pool_n;
  if (cand)
    for (int64_t i = 0; i < n; ++i)
      if (cand[i] < 0 || cand[i] >= ctx->pool_n) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "candidate position outside the pool");
  fib::State* s = fib::get(ctx);
  s->have = false;
  s->n = n; s->c = ctx->n_class; s->r = ctx->n_class - 1; s->d = ctx->feat_dim;
  s->post = ctx->pool_post; s->ldp = ctx->pool_n; s->U = ctx->pool_feat;
  s->use_rows = cand != nullptr;
  if (cand && n) {
    NNAL_TRY(fib::grow(ctx, s->rows, s->cap_rows, n));
    CUDA_TRY(ctx, cudaMemcpyAsync(s->rows, cand, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
  }
  NNAL_TRY(fib::setup(ctx, s));
  NNAL_SYNC_CHECKED(ctx);                                 // `cand` is caller-owned host memory; fp16 range flag of the pool pass
  s->have = true;
  return NNAL_OK;
}

extern "C" int nnal_fi_block_set_factors(nnal_ctx* ctx, int64_t n, int c, int d, const float* post, const float* U) {
  if (!ctx || n < 0 || d <= 0 || (n > 0 && (!post || !U))) return NNAL_ERR_INVALID;
  if (c < 2 || c > fib::MAX_C) NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "block FI supports 2 <= c <= 32");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  fib::State* s = fib::get(ctx);
  s->have = false;
  s->n = n; s->c = c; s->r = c - 1; s->d = d;
  NNAL_TRY(fib::grow(ctx, s->ownP, s->cap_p, n * c));
  NNAL_TRY(fib::grow(ctx, s->ownU, s->cap_u, n * d));
  if (n) {
    CUDA_TRY(ctx, cudaMemcpyAsync(s->ownP, post, (size_t)n * c * 4, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(s->ownU, U, (size_t)n * d * 4, cudaMemcpyHostToDevice, ctx->stream));
  }
  s->post = s->ownP; s->ldp = n; s->U = s->ownU; s->use_rows = false;
  NNAL_TRY(fib::setup(ctx, s));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  s->have = true;
  return NNAL_OK;
}

extern "C" int nnal_fi_block_greedy(nnal_ctx* ctx, int64_t k, double delta, int64_t* sel_out, double* obj_out, double* red_out) {
  if (!ctx || k < 0 || !(delta > 0) || (k > 0 && !sel_out)) return NNAL_ERR_INVALID;
  if (!ctx->fi_block_state || !((fib::State*)ctx->fi_block_state)->have) NNAL_FAIL(ctx, NNAL_ERR_STATE, "block FI candidates not set");
  fib::State* s = (fib::State*)ctx->fi_block_state;
  const int64_t n = s->n;
  const int c = s->c, r = s->r;
  if (k > n) k = n;
  if (k * r > fib::MAX_KR) NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "block FI greedy supports k (c-1) <= 4096");
  if (k == 0) return NNAL_OK;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const int64_t mmax = k * r;
  const int npmax = (int)((mmax + 63) / 64 * 64);
  const int64_t ldk = mmax, ldz = k * c, lds = n;
  int JC, AT;
  size_t smem;
  fib::eval_plan(c, r, &JC, &AT, &smem);
  const int nblk = (int)((n + JC - 1) / JC);
  NNAL_TRY(fib::grow(ctx, s->Scols, s->cap_scols, k * n));
  NNAL_TRY(fib::grow(ctx, s->Kss, s->cap_kss, mmax * mmax));
  NNAL_TRY(fib::grow(ctx, s->M, s->cap_m, (int64_t)npmax * npmax));
  NNAL_TRY(fib::grow(ctx, s->Z, s->cap_z, mmax * ldz));
  NNAL_TRY(fib::grow(ctx, s->Lsel, s->cap_lsel, k * c * r));
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
    CUDA_TRY(ctx, cudaFuncSetAttribute(fib::eval_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fib::EVAL_SMEM_MAX));
    attr = true;
  }
  CUDA_TRY(ctx, cudaMemsetAsync(s->avail, 1, (size_t)n, ctx->stream));
  CUDA_TRY(ctx, cudaMemsetAsync(s->trC, 0, sizeof(double), ctx->stream));
  const int64_t* rows = s->use_rows ? s->rows : nullptr;
  fib::EvalArgs ea;
  ea.Lall = s->Lall; ea.Kd = s->Kd; ea.Z = s->Z; ea.ldz = ldz; ea.Scols = s->Scols; ea.lds = lds;
  ea.Lsel = s->Lsel; ea.avail = s->avail; ea.n = n; ea.c = c; ea.r = r; ea.JC = JC; ea.AT = AT;
  ea.trC = s->trC; ea.blk_loss = s->blk_loss; ea.blk_idx = s->blk_idx; ea.ticket = s->ticket; ea.sel = s->sel; ea.red = s->red;
  for (int t = 0; t < (int)k; ++t) {
    const double alpha = (double)(t + 1) * delta;
    if (t > 0) {
      prof_begin(ctx, NNAL_PROF_FIB_SYSTEM);
      const int m = t * r;
      const int np = (m + 63) / 64 * 64;
      fib::append_kernel<<<fib::flat_grid(ctx, (int64_t)t * r * r), 256, 0, ctx->stream>>>(s->Lsel, s->Scols, lds, s->sel, t - 1, c,
                                                                                             r, s->Kss, ldk);
      fib::build_kernel<<<fib::flat_grid(ctx, (int64_t)np * np), 256, 0, ctx->stream>>>(s->Kss, ldk, m, np, alpha, s->M);
      ctx->launches += 2;
      NNAL_TRY(nnal_gj64_invert(ctx, s->M, np));
      fib::z_kernel<<<fib::flat_grid(ctx, (int64_t)m * t * c), 256, 0, ctx->stream>>>(s->M, np, s->Lsel, t, c, r, s->Z, ldz);
      fib::trace_kernel<<<1, 256, 0, ctx->stream>>>(s->M, np, m, s->trC);
      ctx->launches += 2;
      prof_end(ctx);
    }
    prof_begin(ctx, NNAL_PROF_FIB_EVAL);
    ea.t = t;
    ea.alpha = alpha;
    fib::eval_kernel<<<nblk, fib::EVAL_THREADS, smem, ctx->stream>>>(ea);
    ctx->launches++;
    prof_end(ctx);
    if (t + 1 < (int)k) {
      prof_begin(ctx, NNAL_PROF_FIB_COLUMN);
      fib::column_kernel<<<fib::warp_grid(ctx, n), 256, 0, ctx->stream>>>(s->U, rows, n, s->d, s->sel, t, s->Scols + (int64_t)t * lds);
      ctx->launches++;
      prof_end(ctx);
    }
    CUDA_TRY(ctx, cudaGetLastError());
  }
  std::vector<double> red((size_t)k);
  static_assert(sizeof(long long) == sizeof(int64_t), "");
  CUDA_TRY(ctx, cudaMemcpyAsync(sel_out, s->sel, (size_t)k * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(red.data(), s->red, (size_t)k * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  const double D = (double)c * (s->d + 1.0);
  for (int64_t t = 0; t < k; ++t) {
    if (red_out) red_out[t] = red[t];
    if (obj_out) obj_out[t] = (D - (double)(t + 1) * r) / delta + red[t];
  }
  return NNAL_OK;
}
