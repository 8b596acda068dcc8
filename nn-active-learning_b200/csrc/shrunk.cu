// Shrunk class-score gradients (the reference's FI coordinates, SURVEY.md 8a rows 8-10).
//
// The reference's `fi` query calls, for each of the B pre-filtered samples and each class y, sess.run(model.grad_posts[y])
// = tf.gradients(log posteriors[y,0], all trainable variables) (NN.get_gradients NN.py:621-645, PW_NNAL.gen_A_matrices
// PW_NNAL.py:773-807) -- 2B single-sample backprops over 36 M parameters -- and then keeps ONE number per parameterised
// layer: NNAL_tools.shrink_gradient(grad,'sum') = (sum gW_t + sum gb_t) / (size W_t + size b_t) (NNAL_tools.py:784-796).
// The per-layer sums factor through the pre-activation gradients dz_t, so no parameter gradient is ever formed:
//   fc   : sum gW = (sum_o dz_o)(sum_i a_i),            sum gb = sum_o dz_o
//   conv : sum gW = sum_p (sum_co dz[p,co]) box[p],     sum gb = sum_p sum_co dz[p,co],
//          box[p] = sum over the kh x kw window at p of sum_ci x_padded[.,ci]
// What remains is a batched DATA-gradient backward pass: forward keeping every activation as fp32 (tcgen05 conv / fc
// kernels where the forward pass has them, unfused), then dz walks back through fc (dz W: the forward's split-plane
// tcgen05 GEMM on power-of-two scaled gradients, fp32 CUDA cores for small layers), ReLU masks, max-pool (gradient to
// the first maximum of each window, as tf.nn.max_pool's gradient) and conv (correlation of dz with the flipped filter,
// fp32 CUDA cores).  For the binary model both class gradients are multiples of one
// pass, d log p_0 = p_1 h, d log p_1 = -p_0 h with h = d(z_0 - z_1), and shrink_gradient is linear, so one pass serves both.
#include "nnal_common.cuh"
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

bool nnal_layer_on_tc(const nnal_ctx* ctx, int i);

namespace {

// transposed fp16 hi/lo planes [in][Kp(out)] of an fc weight: the B operand of the tensor-core data-gradient GEMM
struct TWeight {
  nnal_h* h = nullptr;
  nnal_h* l = nullptr;
  int Kp = 0;
};

struct BwState {
  DevBuf acts, g[2], post, gout, sred, amax;
  std::vector<TWeight> wt;
  std::vector<void*> cw;          // conv layers: flipped, transposed filter packed for the tensor-core data-gradient convolution
  unsigned long long wt_version = ~0ull;
};

BwState* bw_state(nnal_ctx* ctx) {
  if (!ctx->bw_state) ctx->bw_state = new BwState();
  return (BwState*)ctx->bw_state;
}

int64_t bw_chunk(const nnal_ctx* ctx) { return ctx->dbg.bw_chunk > 0 ? ctx->dbg.bw_chunk : 2048; }

inline int grid_for(const nnal_ctx* ctx, int64_t total, int per_sm) {
  int64_t b = (total + 255) / 256, cap = (int64_t)ctx->sm_count * per_sm;
  return (int)std::max<int64_t>(1, std::min(b, cap));
}

// ---- dz at the logits: e_y - pi (tf.gradients of log softmax), or h = e_0 - e_1 for the binary single pass ----------
__global__ void dlogits_kernel(const float* __restrict__ post, float* __restrict__ dz, int64_t n, int c, int y) {
  const int64_t total = n * c;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t s = e / c;
    const int j = (int)(e - s * c);
    dz[e] = y < 0 ? (j == 0 ? 1.f : -1.f) : ((j == y ? 1.f : 0.f) - post[(int64_t)j * n + s]);
  }
}

// ---- ReLU: dz = d where the layer's output is positive (tf.nn.relu's gradient) -------------------------------------
__global__ void relu_mask_kernel(float* __restrict__ d, const float* __restrict__ a, int64_t count) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < count; e += (int64_t)gridDim.x * blockDim.x)
    if (!(a[e] > 0.f)) d[e] = 0.f;
}

// ---- max-pool SAME, window == stride: every input cell asks whether it is the FIRST maximum of its window ----------
// (window (yo, xo) starts at (yo*s - pt, xo*s - pl): TF's SAME padding before, as in forward_simt.cu)
__global__ void pool_bwd_kernel(const float* __restrict__ d_out, const float* __restrict__ in, float* __restrict__ d_in,
                                int64_t total_in, int H, int Wd, int C, int Ho, int Wo, int s, int pt, int pl) {
  const int per = H * Wd * C;                      // one sample: 32-bit index arithmetic below
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total_in; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t smp = e / per;
    const int r = (int)(e - smp * per);
    const int c = r % C;
    const int t = r / C;
    const int x = t % Wd, y = t / Wd;
    const int yo = (y + pt) / s, xo = (x + pl) / s;
    const float* base = in + smp * per;
    float m = -INFINITY;
    int wy = -1, wx = -1;
    const int y0 = yo * s - pt, x0 = xo * s - pl;
    const int y1 = min(y0 + s, H), x1 = min(x0 + s, Wd);
    for (int y2 = max(y0, 0); y2 < y1; ++y2) {
      for (int x2 = max(x0, 0); x2 < x1; ++x2) {
        const float v = base[(y2 * Wd + x2) * C + c];
        if (v > m) { m = v; wy = y2; wx = x2; }
      }
    }
    d_in[e] = (wy == y && wx == x) ? d_out[((smp * Ho + yo) * Wo + xo) * (int64_t)C + c] : 0.f;
  }
}

// four channels per thread (C % 4 == 0): 16-byte loads, four independent comparisons in flight
__global__ void pool_bwd_vec4_kernel(const float* __restrict__ d_out, const float* __restrict__ in, float* __restrict__ d_in,
                                     int64_t total4, int H, int Wd, int C, int Ho, int Wo, int s, int pt, int pl) {
  const int C4 = C / 4, per4 = H * Wd * C4;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total4; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t smp = e / per4;
    const int r = (int)(e - smp * per4);
    const int c4 = r % C4;
    const int t = r / C4;
    const int x = t % Wd, y = t / Wd;
    const int yo = (y + pt) / s, xo = (x + pl) / s;
    const float* base = in + smp * (int64_t)per4 * 4 + 4 * c4;
    float m[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
    int win[4] = {-1, -1, -1, -1};
    const int y0 = yo * s - pt, x0 = xo * s - pl;
    const int y1 = min(y0 + s, H), x1 = min(x0 + s, Wd);
    for (int y2 = max(y0, 0); y2 < y1; ++y2) {
      for (int x2 = max(x0, 0); x2 < x1; ++x2) {
        const float4 v = *reinterpret_cast<const float4*>(base + (int64_t)(y2 * Wd + x2) * C);
        const float vv[4] = {v.x, v.y, v.z, v.w};
        const int id = y2 * Wd + x2;
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (vv[k] > m[k]) { m[k] = vv[k]; win[k] = id; }
      }
    }
    const float4 g = *reinterpret_cast<const float4*>(d_out + ((smp * Ho + yo) * Wo + xo) * (int64_t)C + 4 * c4);
    const int me = y * Wd + x;
    float4 o;
    o.x = win[0] == me ? g.x : 0.f;
    o.y = win[1] == me ? g.y : 0.f;
    o.z = win[2] == me ? g.z : 0.f;
    o.w = win[3] == me ? g.w : 0.f;
    *reinterpret_cast<float4*>(d_in + e * 4) = o;
  }
}

// ---- conv data gradient: d_in[y][x][ci] = sum_{dy,dx,co} dz[y-dy+ph][x-dx+pw][co] W[dy][dx][ci][co] ------------------
// One CTA per sample; dz is staged zero-padded in shared memory so that the flipped tap (dy',dx') = (kh-1-dy, kw-1-dx)
// reads padded position (y+dy', x+dx').  A thread owns TC input channels x TP positions and walks co four at a time.
// WS: the whole filter is staged in shared memory behind the tile (once per CTA); otherwise it is read through L2.
// Shared-memory layout against bank conflicts (the first version spent 5x more cycles in the LSU than in the FMA pipe):
//  * threads of a warp share the channel group and own CONSECUTIVE positions, so a filter load is one broadcast;
//  * a tile position holds CP = Cout (+4 when Cout/4 is even) floats, so the eight 16-byte loads of a quarter-warp
//    (consecutive positions) fall into eight different bank groups.
__host__ __device__ inline int conv_bwd_cp(int Cout) { return (Cout % 4 == 0 && (Cout / 4) % 2 == 0) ? Cout + 4 : Cout; }

template <int TP, int TC, bool WS, int NT>
__global__ void __launch_bounds__(NT) conv_bwd_data_kernel(const float* __restrict__ dz, const float* __restrict__ Wt,
                                                             float* __restrict__ d_in, int64_t n, int H, int Wd, int Cin,
                                                             int Cout, int kh, int kw) {
  extern __shared__ float s_dz[];
  const int Hp = H + kh - 1, Wp = Wd + kw - 1;
  const int ph = kh / 2, pw = kw / 2;
  const int CP = conv_bwd_cp(Cout);
  const int ci_groups = (Cin + TC - 1) / TC;
  const int PG = blockDim.x / ci_groups;
  const int tid = threadIdx.x;
  const int cg = tid / PG, pg = tid % PG;
  const bool active = cg < ci_groups;
  const int ci0 = cg * TC;
  const int HW = H * Wd;
  const bool vec = (Cout % 4) == 0;
  float* s_w = s_dz + (Hp * Wp * CP + 3) / 4 * 4;
  if (WS) {
    for (int e = tid; e < kh * kw * Cin * Cout; e += blockDim.x) s_w[e] = Wt[e];
  }
  const float* wbase = WS ? s_w : Wt;
  for (int64_t s = blockIdx.x; s < n; s += gridDim.x) {
    const float* src = dz + s * (int64_t)HW * Cout;
    if (vec) {
      const int C4 = Cout / 4;
      for (int e = tid; e < Hp * Wp * C4; e += blockDim.x) {
        const int c4 = e % C4;
        const int t = e / C4;
        const int xx = t % Wp - pw, yy = t / Wp - ph;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (xx >= 0 && xx < Wd && yy >= 0 && yy < H) v = *reinterpret_cast<const float4*>(src + ((int64_t)yy * Wd + xx) * Cout + 4 * c4);
        *reinterpret_cast<float4*>(&s_dz[t * CP + 4 * c4]) = v;
      }
    } else {
      for (int e = tid; e < Hp * Wp * Cout; e += blockDim.x) {
        const int co = e % Cout;
        const int t = e / Cout;
        const int xx = t % Wp - pw, yy = t / Wp - ph;
        s_dz[t * CP + co] = (xx >= 0 && xx < Wd && yy >= 0 && yy < H) ? src[((int64_t)yy * Wd + xx) * Cout + co] : 0.f;
      }
    }
    __syncthreads();
    if (active) {
      for (int p0 = 0; p0 < HW; p0 += PG * TP) {
        float acc[TP][TC];
        int off[TP];
#pragma unroll
        for (int t = 0; t < TP; ++t) {
          const int p = p0 + pg + t * PG;
          const int pc = p < HW ? p : 0;
          off[t] = ((pc / Wd) * Wp + (pc % Wd)) * CP;
#pragma unroll
          for (int c = 0; c < TC; ++c) acc[t][c] = 0.f;
        }
        for (int fy = 0; fy < kh; ++fy)
          for (int fx = 0; fx < kw; ++fx) {
            const int toff = (fy * Wp + fx) * CP;
            const int tap = (kh - 1 - fy) * kw + (kw - 1 - fx);
            const float* wtap = wbase + (int64_t)tap * Cin * Cout;
            if (vec) {
              for (int co = 0; co < Cout; co += 4) {
                float4 w[TC];
#pragma unroll
                for (int c = 0; c < TC; ++c)
                  w[c] = (ci0 + c >= Cin) ? make_float4(0.f, 0.f, 0.f, 0.f)
                         : WS   ? *reinterpret_cast<const float4*>(wtap + (ci0 + c) * Cout + co)
                                : __ldg(reinterpret_cast<const float4*>(wtap + (int64_t)(ci0 + c) * Cout + co));
#pragma unroll
                for (int t = 0; t < TP; ++t) {
                  const float4 a = *reinterpret_cast<const float4*>(&s_dz[off[t] + toff + co]);
#pragma unroll
                  for (int c = 0; c < TC; ++c) {
                    acc[t][c] = fmaf(a.x, w[c].x, acc[t][c]);
                    acc[t][c] = fmaf(a.y, w[c].y, acc[t][c]);
                    acc[t][c] = fmaf(a.z, w[c].z, acc[t][c]);
                    acc[t][c] = fmaf(a.w, w[c].w, acc[t][c]);
                  }
                }
              }
            } else {
              for (int co = 0; co < Cout; ++co) {
                float w[TC];
#pragma unroll
                for (int c = 0; c < TC; ++c) w[c] = (ci0 + c >= Cin) ? 0.f : WS ? wtap[(ci0 + c) * Cout + co] : __ldg(wtap + (int64_t)(ci0 + c) * Cout + co);
#pragma unroll
                for (int t = 0; t < TP; ++t) {
                  const float a = s_dz[off[t] + toff + co];
#pragma unroll
                  for (int c = 0; c < TC; ++c) acc[t][c] = fmaf(a, w[c], acc[t][c]);
                }
              }
            }
          }
#pragma unroll
        for (int t = 0; t < TP; ++t) {
          const int p = p0 + pg + t * PG;
          if (p < HW) {
#pragma unroll
            for (int c = 0; c < TC; ++c)
              if (ci0 + c < Cin) d_in[(s * HW + p) * (int64_t)Cin + ci0 + c] = acc[t][c];
          }
        }
      }
    }
    __syncthreads();
  }
}

template <int TP, int TC, bool WS, int NT = 256>
int conv_bwd_launch(nnal_ctx* ctx, const Layer& L, const float* dz, float* d_in, int64_t n, size_t smem) {
  auto k = conv_bwd_data_kernel<TP, TC, WS, NT>;
  CUDA_TRY(ctx, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 1;
  CUDA_TRY(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, NT, smem));
  // persistent CTAs: the staged filter (WS) is amortised over the CTA's samples
  const int grid = (int)std::min<int64_t>(n, (int64_t)ctx->sm_count * std::max(1, per_sm));
  k<<<grid, NT, smem, ctx->stream>>>(dz, L.W, d_in, n, L.in_h, L.in_w, L.in_c, L.out_c, L.kh, L.kw);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}

// Register tile: TC input channels x TP positions per thread; one step (tap, 4 output channels) issues TC + TP 16-byte
// shared-memory loads for 4 TC TP multiply-adds.  Large rasters with Cin % 8 == 0 (PW1 conv2: 625 positions, 24
// channels; tile + filter = 198 KB, one CTA per SM) take 8 channels x 4 positions in a 512-thread CTA (3 groups x 170
// position groups x 4 = 680 slots, 10.7 FMAs per load; the 8 x 8 tile in 256 threads left the schedulers idle 57 % of the
// time with two warps each -- profiles/r1_conv_bwd_full.md); 13 x 13 rasters take
// TC = 4 and the TP that covers the raster in one pass (conv3: 32 groups x 6 = 192 slots for 169 positions, filter in
// shared memory; conv4: 21 x 9 = 189, filter 166 KB + tile 90 KB do not fit together: filter through L2, one
// warp-uniform load per TP x 16 multiply-adds).
template <int TC>
int conv_bwd_pick(nnal_ctx* ctx, const Layer& L, const float* dz, float* d_in, int64_t n) {
  const int groups = (L.in_c + TC - 1) / TC, PG = 256 / groups;
  const int need = (L.in_h * L.in_w + PG - 1) / PG;         // (TC = 8 runs 512 threads: twice the position groups)
  const size_t tile = ((size_t)(L.in_h + L.kh - 1) * (L.in_w + L.kw - 1) * conv_bwd_cp(L.out_c) + 3) / 4 * 4 * sizeof(float);
  const size_t wbytes = (size_t)L.kh * L.kw * L.in_c * L.out_c * sizeof(float);
  if (tile > 200 * 1024) NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "conv gradient tile exceeds shared memory");
  const bool no_ws = ctx->dbg.bw_no_ws != 0;
  const bool ws = !no_ws && tile + wbytes <= 220 * 1024;
  if constexpr (TC == 8) {
    if (ws) return conv_bwd_launch<4, TC, true, 512>(ctx, L, dz, d_in, n, tile + wbytes);
    return conv_bwd_launch<4, TC, false, 512>(ctx, L, dz, d_in, n, tile);
  } else {
  if (ws) {
    if (need <= 4) return conv_bwd_launch<4, TC, true>(ctx, L, dz, d_in, n, tile + wbytes);
    if (need <= 6) return conv_bwd_launch<6, TC, true>(ctx, L, dz, d_in, n, tile + wbytes);
    return conv_bwd_launch<9, TC, true>(ctx, L, dz, d_in, n, tile + wbytes);
  }
  if (need <= 4) return conv_bwd_launch<4, TC, false>(ctx, L, dz, d_in, n, tile);
  if (need <= 6) return conv_bwd_launch<6, TC, false>(ctx, L, dz, d_in, n, tile);
  if (need <= 9) return conv_bwd_launch<9, TC, false>(ctx, L, dz, d_in, n, tile);
  return conv_bwd_launch<12, TC, false>(ctx, L, dz, d_in, n, tile);
  }
}

int conv_bwd_data(nnal_ctx* ctx, const Layer& L, const float* dz, float* d_in, int64_t n) {
  if (n == 0) return NNAL_OK;
  if (L.in_c > 256) NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "conv gradient: more than 256 input channels");
  const bool no_tc8 = ctx->dbg.bw_no_tc8 != 0;
  if (!no_tc8 && L.in_c % 8 == 0 && L.in_h * L.in_w >= 400) return conv_bwd_pick<8>(ctx, L, dz, d_in, n);
  if (L.in_c % 4 == 0) return conv_bwd_pick<4>(ctx, L, dz, d_in, n);
  return conv_bwd_pick<1>(ctx, L, dz, d_in, n);
}

// ---- fc data gradient: d[M][N] = dz[M][K] . W[K][N]  (W = the layer's [out][in] weight, read as stored) -------------
// 128x128x16 tiles, 256 threads, 8x8 register micro-tiles; fp32 throughout.  Used where the tensor-core path below
// does not apply (layers narrower than 64 or not a multiple of 8, nnal_set_tensor_cores(0)).
#define BW_BM 128
#define BW_BN 128
#define BW_BK 16
__global__ void __launch_bounds__(256) fc_bwd_kernel(const float* __restrict__ A, const float* __restrict__ B,
                                                      float* __restrict__ C, int64_t M, int N, int K) {
  __shared__ float As[BW_BK][BW_BM + 4];
  __shared__ float Bs[BW_BK][BW_BN + 4];
  const int tid = threadIdx.x;
  const int64_t m0 = (int64_t)blockIdx.y * BW_BM;
  const int n0 = blockIdx.x * BW_BN;
  const int tx = tid % 16, ty = tid / 16;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  const bool vecA = (K % 4) == 0, vecB = (N % 4) == 0;
  for (int k0 = 0; k0 < K; k0 += BW_BK) {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      // A tile: 128 rows x 16 k, a thread loads 4 consecutive k of one row
      const int row = tid / 4 + 64 * i, kq = (tid % 4) * 4;
      float va[4] = {0.f, 0.f, 0.f, 0.f};
      const int64_t gm = m0 + row;
      if (gm < M) {
        if (vecA && k0 + kq + 3 < K) {
          const float4 t = *reinterpret_cast<const float4*>(A + gm * K + k0 + kq);
          va[0] = t.x; va[1] = t.y; va[2] = t.z; va[3] = t.w;
        } else {
#pragma unroll
          for (int c = 0; c < 4; ++c)
            if (k0 + kq + c < K) va[c] = A[gm * K + k0 + kq + c];
        }
      }
#pragma unroll
      for (int c = 0; c < 4; ++c) As[kq + c][row] = va[c];
      // B tile: 16 k x 128 columns, a thread loads 4 consecutive columns of one k
      const int kr = tid / 32 + 8 * i, cq = (tid % 32) * 4;
      float vb[4] = {0.f, 0.f, 0.f, 0.f};
      if (k0 + kr < K) {
        const float* bp = B + (int64_t)(k0 + kr) * N + n0 + cq;
        if (vecB && n0 + cq + 3 < N) {
          const float4 t = __ldg(reinterpret_cast<const float4*>(bp));
          vb[0] = t.x; vb[1] = t.y; vb[2] = t.z; vb[3] = t.w;
        } else {
#pragma unroll
          for (int c = 0; c < 4; ++c)
            if (n0 + cq + c < N) vb[c] = __ldg(bp + c);
        }
      }
      *reinterpret_cast<float4*>(&Bs[kr][cq]) = make_float4(vb[0], vb[1], vb[2], vb[3]);
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < BW_BK; ++k) {
      float a[8], b[8];
      float4 t;
      t = *reinterpret_cast<const float4*>(&As[k][ty * 4]);       a[0] = t.x; a[1] = t.y; a[2] = t.z; a[3] = t.w;
      t = *reinterpret_cast<const float4*>(&As[k][64 + ty * 4]);  a[4] = t.x; a[5] = t.y; a[6] = t.z; a[7] = t.w;
      t = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);       b[0] = t.x; b[1] = t.y; b[2] = t.z; b[3] = t.w;
      t = *reinterpret_cast<const float4*>(&Bs[k][64 + tx * 4]);  b[4] = t.x; b[5] = t.y; b[6] = t.z; b[7] = t.w;
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int64_t gm = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + i - 4);
    if (gm >= M) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int gn = n0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + j - 4);
      if (gn < N) C[gm * N + gn] = acc[i][j];
    }
  }
}

int fc_bwd_data(nnal_ctx* ctx, const Layer& L, const float* dz, float* d_in, int64_t n) {
  if (n == 0) return NNAL_OK;
  dim3 grid(cdiv(L.in_dim, BW_BN), cdiv(n, BW_BM));
  fc_bwd_kernel<<<grid, 256, 0, ctx->stream>>>(dz, L.W, d_in, n, L.in_dim, L.out_dim);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}

// ---- fc data gradient on the tensor cores -----------------------------------------------------------------------
// d = dz . W as the split-plane GEMM of the forward pass (gemm_tc.cu): A = dz in fp16 hi/lo planes, B = W^T planes
// (built once per weight set).  Gradients are small and span many binades, so dz is first multiplied by the power of
// two that lifts its largest magnitude to [2^13, 2^14): every entry then carries an absolute error below 2^-39 of the
// largest one, and entries within 2^-17 of it keep 22 significant bits -- the same footing as the weights.
__global__ void absmax_kernel(const float* __restrict__ x, int64_t count, unsigned int* __restrict__ out) {
  unsigned int m = 0;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < count; e += (int64_t)gridDim.x * blockDim.x) {
    const unsigned int b = __float_as_uint(x[e]) & 0x7fffffffu;      // |x| as an order-preserving integer
    if (b < 0x7f800000u && b > m) m = b;                              // finite values only
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_down_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}

// fp32 [rows][K] * scale -> fp16 hi/lo planes [rows][Kp] (zero-padded columns)
__global__ void __launch_bounds__(256) bw_split_kernel(const float* __restrict__ in, nnal_h* __restrict__ hi,
                                                        nnal_h* __restrict__ lo, int64_t rows, int K, int Kp, float scale) {
  const int64_t total = rows * (int64_t)(Kp / 2);
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = e / (Kp / 2);
    const int c = (int)(e - r * (Kp / 2)) * 2;
    const float x0 = c < K ? in[r * K + c] * scale : 0.f;
    const float x1 = c + 1 < K ? in[r * K + c + 1] * scale : 0.f;
    nnal_h h0, h1, l0, l1;
    nnal_split(x0, h0, l0);
    nnal_split(x1, h1, l1);
    *reinterpret_cast<uint32_t*>(hi + r * Kp + c) = nnal_pack2(h0, h1);
    *reinterpret_cast<uint32_t*>(lo + r * Kp + c) = nnal_pack2(l0, l1);
  }
}

// W fp32 [out][in] * scale -> planes of W^T: [in][Kp], Kp >= out (one-off per weight set)
__global__ void __launch_bounds__(256) bw_split_transposed_kernel(const float* __restrict__ W, nnal_h* __restrict__ hi,
                                                                   nnal_h* __restrict__ lo, int out_dim, int in_dim, int Kp,
                                                                   float scale) {
  const int64_t total = (int64_t)in_dim * Kp;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = e / Kp;
    const int o = (int)(e - i * Kp);
    const float x = o < out_dim ? W[(int64_t)o * in_dim + i] * scale : 0.f;
    nnal_h h, l;
    nnal_split(x, h, l);
    hi[e] = h;
    lo[e] = l;
  }
}

bool fc_bwd_tc_eligible(const nnal_ctx* ctx, const Layer& L) {
  const bool off = ctx->dbg.bw_no_tc != 0;
  return !off && L.type == NNAL_LAYER_FC && L.out_dim >= 64 && L.in_dim >= 64 && L.out_dim % 8 == 0 &&
         L.in_dim % 8 == 0;
}

void free_transposed(BwState* st) {
  for (auto& t : st->wt) { if (t.h) cudaFree(t.h); if (t.l) cudaFree(t.l); }
  st->wt.clear();
  for (void* p : st->cw) if (p) cudaFree(p);
  st->cw.clear();
}

int ensure_transposed(nnal_ctx* ctx, BwState* st) {
  if (st->wt_version == ctx->weights_version && st->wt.size() == ctx->layers.size()) return NNAL_OK;
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  free_transposed(st);
  st->wt.resize(ctx->layers.size());
  st->cw.assign(ctx->layers.size(), nullptr);
  for (size_t i = 1; i < ctx->layers.size(); ++i) {        // layer 0 needs no data gradient
    const Layer& L = ctx->layers[i];
    if (L.type == NNAL_LAYER_CONV && L.has_weights && nnal_tc_conv_bwd_supported(ctx, L)) {      // (bw_no_tc is tested at use)
      NNAL_TRY(nnal_tc_conv_bwd_prepare(ctx, L, &st->cw[i]));
      continue;
    }
    if (!fc_bwd_tc_eligible(ctx, L) || !L.has_weights) continue;
    TWeight& t = st->wt[i];
    t.Kp = (L.out_dim + 63) / 64 * 64;
    const size_t bytes = (size_t)L.in_dim * t.Kp * sizeof(nnal_h);
    CUDA_TRY(ctx, cudaMalloc(&t.h, bytes));
    CUDA_TRY(ctx, cudaMalloc(&t.l, bytes));
    const int64_t total = (int64_t)L.in_dim * t.Kp;
    bw_split_transposed_kernel<<<grid_for(ctx, total, 16), 256, 0, ctx->stream>>>(L.W, t.h, t.l, L.out_dim, L.in_dim, t.Kp,
                                                                                  L.w_scale);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
  }
  st->wt_version = ctx->weights_version;
  return NNAL_OK;
}

// exponent e of the power of two that lifts the largest |dz| of the chunk to [2^13, 2^14); *zero: every entry is zero
int gradient_exponent(nnal_ctx* ctx, BwState* st, const float* dz, int64_t cnt, int* e_out, bool* zero) {
  NNAL_TRY(devbuf_reserve(ctx, st->amax, 256));
  unsigned int* d_max = (unsigned int*)st->amax.p;
  CUDA_TRY(ctx, cudaMemsetAsync(d_max, 0, 4, ctx->stream));
  absmax_kernel<<<grid_for(ctx, cnt, 8), 256, 0, ctx->stream>>>(dz, cnt, d_max);
  ctx->launches++;
  unsigned int bits = 0;
  CUDA_TRY(ctx, cudaMemcpyAsync(&bits, d_max, 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  float mx;
  memcpy(&mx, &bits, 4);
  *zero = !(mx > 0.f);
  int ex = 0;
  if (!*zero) frexpf(mx, &ex);                              // mx = f 2^ex, f in [0.5, 1)
  *e_out = std::max(-100, std::min(100, 14 - ex));
  return NNAL_OK;
}

int fc_bwd_data_tc(nnal_ctx* ctx, BwState* st, const Layer& L, const TWeight& t, const float* dz, float* d_in, int64_t n) {
  int e;
  bool zero;
  NNAL_TRY(gradient_exponent(ctx, st, dz, n * L.out_dim, &e, &zero));
  if (zero) {                                               // all-zero gradient (every unit masked): so is the result
    CUDA_TRY(ctx, cudaMemsetAsync(d_in, 0, (size_t)n * L.in_dim * sizeof(float), ctx->stream));
    return NNAL_OK;
  }
  const float s = ldexpf(1.f, e);
  const size_t plane = (size_t)n * t.Kp * sizeof(nnal_h);
  NNAL_TRY(devbuf_reserve(ctx, ctx->splitA[0], plane));
  NNAL_TRY(devbuf_reserve(ctx, ctx->splitA[1], plane));
  nnal_h* Ah = (nnal_h*)ctx->splitA[0].p;
  nnal_h* Al = (nnal_h*)ctx->splitA[1].p;
  bw_split_kernel<<<grid_for(ctx, n * (int64_t)(t.Kp / 2), 16), 256, 0, ctx->stream>>>(dz, Ah, Al, n, L.out_dim, t.Kp, s);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  // out[n][in] = (1 / (s w_scale)) A[n][out] . B[in][out]^T
  return nnal_tc_gemm_planes(ctx, Ah, Al, t.Kp, n, t.h, t.l, t.Kp, L.in_dim, L.out_dim, nullptr,
                             ldexpf(1.f, -e) * L.w_scale_inv, 0, 0, d_in, L.in_dim, nullptr, nullptr, 0);
}

// ---- conv data gradient on the tensor cores ------------------------------------------------------------------------
// The forward pass's shift-GEMM kernel (conv_tc.cu) on dz: fp16 hi/lo planes of dz * 2^e (same scaling as the fc gradient),
// the flipped, transposed filter packed once per weight set, float32 output.  Replaces conv_bwd_data_kernel (fp32 CUDA cores,
// 15 of the 23 ms of the backward pass at B = 10,000) for PW1's conv2 / conv3 / conv4.
int conv_bwd_data_tc(nnal_ctx* ctx, BwState* st, const Layer& L, const void* packed, const float* dz, float* d_in, int64_t n) {
  int e;
  bool zero;
  const int64_t rows = n * L.out_h * L.out_w;
  NNAL_TRY(gradient_exponent(ctx, st, dz, rows * L.out_c, &e, &zero));
  if (zero) {
    CUDA_TRY(ctx, cudaMemsetAsync(d_in, 0, (size_t)n * L.in_h * L.in_w * L.in_c * sizeof(float), ctx->stream));
    return NNAL_OK;
  }
  const size_t plane = (size_t)rows * L.out_c * sizeof(nnal_h);       // out_c is a multiple of 8 for every supported shape
  NNAL_TRY(devbuf_reserve(ctx, ctx->splitA[0], plane));
  NNAL_TRY(devbuf_reserve(ctx, ctx->splitA[1], plane));
  nnal_h* Ah = (nnal_h*)ctx->splitA[0].p;
  nnal_h* Al = (nnal_h*)ctx->splitA[1].p;
  bw_split_kernel<<<grid_for(ctx, rows * (int64_t)(L.out_c / 2), 16), 256, 0, ctx->stream>>>(dz, Ah, Al, rows, L.out_c, L.out_c,
                                                                                             ldexpf(1.f, e));
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return nnal_tc_conv_bwd(ctx, L, packed, Ah, Al, d_in, n, ldexpf(1.f, -e) * L.w_scale_inv);
}

// ---- block reduction in float64 ----------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}
__device__ double block_sum(double v, double* s_red) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  v = warp_sum(v);
  __syncthreads();                      // s_red may still be read from the previous call
  if (lane == 0) s_red[w] = v;
  __syncthreads();
  double r = 0.0;
  if (w == 0) {
    r = lane < (int)(blockDim.x >> 5) ? s_red[lane] : 0.0;
    r = warp_sum(r);
  }
  return r;                             // valid in thread 0
}

// ---- shrink_gradient(.,'sum') of an fc layer: (sum dz)(sum a + 1) / (in*out + out) --------------------------------
__global__ void __launch_bounds__(256) shrink_fc_kernel(const float* __restrict__ dz, const float* __restrict__ a,
                                                         int out_dim, int in_dim, double inv_size, double* __restrict__ g,
                                                         int tau, int t) {
  __shared__ double s_red[8];
  const int64_t s = blockIdx.x;
  double sd = 0.0, sa = 0.0;
  for (int j = threadIdx.x; j < out_dim; j += blockDim.x) sd += (double)dz[s * out_dim + j];
  for (int j = threadIdx.x; j < in_dim; j += blockDim.x) sa += (double)a[s * (int64_t)in_dim + j];
  sd = block_sum(sd, s_red);
  sa = block_sum(sa, s_red);
  if (threadIdx.x == 0) g[s * tau + t] = (sd * sa + sd) * inv_size;
}

// ---- shrink_gradient(.,'sum') of a conv layer: sum_p D[p] (box[p] + 1) / (kh*kw*cin*cout + cout) -------------------
__global__ void __launch_bounds__(256) shrink_conv_kernel(const float* __restrict__ dz, const float* __restrict__ in, int H,
                                                           int Wd, int Cin, int Cout, int kh, int kw, double inv_size,
                                                           double* __restrict__ g, int tau, int t) {
  extern __shared__ double s_xs[];      // [Hp][Wp] channel sums of the zero-padded input
  __shared__ double s_red[8];
  const int Hp = H + kh - 1, Wp = Wd + kw - 1, ph = kh / 2, pw = kw / 2;
  const int64_t s = blockIdx.x;
  const float* xin = in + s * (int64_t)H * Wd * Cin;
  const float* dzs = dz + s * (int64_t)H * Wd * Cout;
  for (int e = threadIdx.x; e < Hp * Wp; e += blockDim.x) {
    const int xx = e % Wp - pw, yy = e / Wp - ph;
    double v = 0.0;
    if (xx >= 0 && xx < Wd && yy >= 0 && yy < H) {
      const float* p = xin + ((int64_t)yy * Wd + xx) * Cin;
      if (Cin % 4 == 0) {
        for (int c = 0; c < Cin; c += 4) {
          const float4 q4 = *reinterpret_cast<const float4*>(p + c);
          v += ((double)q4.x + (double)q4.y) + ((double)q4.z + (double)q4.w);
        }
      } else {
        for (int c = 0; c < Cin; ++c) v += (double)p[c];
      }
    }
    s_xs[e] = v;
  }
  __syncthreads();
  double acc = 0.0;
  for (int p = threadIdx.x; p < H * Wd; p += blockDim.x) {
    const int y = p / Wd, x = p % Wd;
    const float* q = dzs + (int64_t)p * Cout;
    double D = 0.0;
    if (Cout % 4 == 0) {
      for (int c = 0; c < Cout; c += 4) {
        const float4 q4 = *reinterpret_cast<const float4*>(q + c);
        D += ((double)q4.x + (double)q4.y) + ((double)q4.z + (double)q4.w);
      }
    } else {
      for (int c = 0; c < Cout; ++c) D += (double)q[c];
    }
    double box = 0.0;
    for (int dy = 0; dy < kh; ++dy)
      for (int dx = 0; dx < kw; ++dx) box += s_xs[(y + dy) * Wp + x + dx];
    acc += D * (box + 1.0);
  }
  acc = block_sum(acc, s_red);
  if (threadIdx.x == 0) g[s * tau + t] = acc * inv_size;
}

// ---- binary model: both class gradients from the single pass  g0 = p1 S, g1 = -p0 S ---------------------------------
__global__ void binary_scale_kernel(const double* __restrict__ S, const float* __restrict__ post, int64_t n, int tau,
                                    double* __restrict__ G) {
  const int64_t total = n * tau;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t s = e / tau;
    const double p0 = (double)post[s], p1 = (double)post[n + s];
    G[e] = p1 * S[e];
    G[total + e] = -p0 * S[e];
  }
}

int count_tau(const nnal_ctx* ctx) {
  int tau = 0;
  for (auto& L : ctx->layers) tau += (L.type != NNAL_LAYER_POOL);
  return tau;
}

// one chunk: inputs are fp32 NHWC in ctx->xin
int shrunk_chunk(nnal_ctx* ctx, BwState* st, int64_t nb, int64_t n_total, int64_t o, float* post_out, double* g_out) {
  const int nl = (int)ctx->layers.size();
  const int c = ctx->n_class, tau = count_tau(ctx);
  // ---- forward, keeping every layer output ----
  std::vector<int64_t> elems(nl), offs(nl);
  int64_t tot = 0, mx = (int64_t)ctx->in_h * ctx->in_w * ctx->in_c;
  for (int i = 0; i < nl; ++i) {
    const Layer& L = ctx->layers[i];
    elems[i] = L.type == NNAL_LAYER_FC ? L.out_dim : (int64_t)L.out_h * L.out_w * L.out_c;
    offs[i] = tot;
    if (L.type == NNAL_LAYER_CONV) mx = std::max(mx, (int64_t)L.in_h * L.in_w * ((L.in_c + 7) / 8 * 8));   // padded operand planes
    tot += (elems[i] * nb + 63) / 64 * 64;          // 256-byte aligned blocks: the fc kernels read rows as float4
    mx = std::max(mx, elems[i]);
  }
  NNAL_TRY(devbuf_reserve(ctx, st->acts, (size_t)tot * sizeof(float)));
  NNAL_TRY(devbuf_reserve(ctx, st->g[0], (size_t)mx * nb * sizeof(float)));
  NNAL_TRY(devbuf_reserve(ctx, st->g[1], (size_t)mx * nb * sizeof(float)));
  NNAL_TRY(devbuf_reserve(ctx, st->post, (size_t)c * nb * sizeof(float)));
  NNAL_TRY(devbuf_reserve(ctx, st->gout, (size_t)c * nb * tau * sizeof(double)));
  NNAL_TRY(devbuf_reserve(ctx, st->sred, (size_t)nb * tau * sizeof(double)));
  float* acts = (float*)st->acts.p;
  auto in_of = [&](int i) -> const float* { return i == 0 ? (const float*)ctx->xin.p : acts + offs[i - 1]; };
  const bool simt_fwd = ctx->dbg.bw_simt_fwd != 0;
  prof_begin(ctx, NNAL_PROF_BW_FORWARD);
  for (int i = 0; i < nl; ++i) {
    const Layer& L = ctx->layers[i];
    if (!L.has_weights && L.type != NNAL_LAYER_POOL) NNAL_FAIL(ctx, NNAL_ERR_STATE, "layer weights not set");
    float* out = acts + offs[i];
    if (i == nl - 1) {
      NNAL_TRY(nnal_k_head(ctx, L, in_of(i), nb, nb, 0, (float*)st->post.p, nullptr));
    } else if (L.type == NNAL_LAYER_CONV) {
      if (!simt_fwd && nnal_layer_on_tc(ctx, i)) {
        // tcgen05 conv kernels (unfused: the pre-pool activations are needed by the backward pass); the gradient
        // buffers are idle during the forward pass and hold the fp16 hi/lo operand planes
        const int cp = (L.in_c + 7) / 8 * 8;
        const int64_t iep = nb * (int64_t)L.in_h * L.in_w * cp, oe = nb * elems[i];
        nnal_h* ih = (nnal_h*)st->g[0].p;
        nnal_h* oh = (nnal_h*)st->g[1].p;
        NNAL_TRY(nnal_k_split_pad(ctx, in_of(i), ih, ih + iep, nb * (int64_t)L.in_h * L.in_w, L.in_c, cp));
        const bool wt = ctx->use_wt >= 3 ? nnal_wt_conv_supported(ctx, L) : ctx->use_wt >= 1 && nnal_wt_conv_preferred(ctx, L);
        if (wt) NNAL_TRY(nnal_wt_conv(ctx, L, ih, ih + iep, oh, oh + oe, nb, 0));
        else NNAL_TRY(nnal_tc_conv(ctx, L, ih, ih + iep, oh, oh + oe, nb));
        NNAL_TRY(nnal_k_merge_flat(ctx, oh, oh + oe, out, oe));
      } else {
        NNAL_TRY(nnal_k_conv_simt(ctx, L, in_of(i), out, nb));
      }
    } else if (L.type == NNAL_LAYER_POOL) {
      NNAL_TRY(nnal_k_pool(ctx, L, in_of(i), out, nb));
    } else if (nnal_layer_on_tc(ctx, i)) {
      NNAL_TRY(nnal_tc_fc(ctx, L, in_of(i), out, nb));
    } else {
      NNAL_TRY(nnal_k_fc_simt(ctx, L, in_of(i), out, nb));
    }
  }
  prof_end(ctx);
  NNAL_TRY(ensure_transposed(ctx, st));
  // ---- backward: one pass of h = e_0 - e_1 (binary) or one pass per class ----
  const bool binary = c == 2;
  const int passes = binary ? 1 : c;
  prof_begin(ctx, NNAL_PROF_BW_BACKWARD);
  double* G = (double*)st->gout.p;
  for (int y = 0; y < passes; ++y) {
    double* S = binary ? (double*)st->sred.p : G + (int64_t)y * nb * tau;
    int pp = 0;
    float* d = (float*)st->g[pp].p;
    dlogits_kernel<<<grid_for(ctx, nb * c, 8), 256, 0, ctx->stream>>>((const float*)st->post.p, d, nb, c, binary ? -1 : y);
    ctx->launches++;
    int t = tau - 1;
    for (int i = nl - 1; i >= 0; --i) {
      const Layer& L = ctx->layers[i];
      float* other = (float*)st->g[pp ^ 1].p;
      if (L.type == NNAL_LAYER_POOL) {
        const int64_t total_in = nb * L.in_h * L.in_w * L.in_c;
        if (L.in_c % 4 == 0)
          pool_bwd_vec4_kernel<<<grid_for(ctx, total_in / 4, 16), 256, 0, ctx->stream>>>(d, in_of(i), other, total_in / 4, L.in_h,
                                                                                         L.in_w, L.in_c, L.out_h, L.out_w, L.kh,
                                                                                         L.pad_t, L.pad_l);
        else
          pool_bwd_kernel<<<grid_for(ctx, total_in, 16), 256, 0, ctx->stream>>>(d, in_of(i), other, total_in, L.in_h, L.in_w,
                                                                                L.in_c, L.out_h, L.out_w, L.kh, L.pad_t, L.pad_l);
        ctx->launches++;
        d = other; pp ^= 1;
        continue;
      }
      if (i != nl - 1) {                 // the last fc has no activation (NN.py:231-241)
        const int64_t cnt = nb * elems[i];
        relu_mask_kernel<<<grid_for(ctx, cnt, 16), 256, 0, ctx->stream>>>(d, acts + offs[i], cnt);
        ctx->launches++;
      }
      if (L.type == NNAL_LAYER_FC) {
        const double inv = 1.0 / ((double)L.in_dim * L.out_dim + L.out_dim);
        shrink_fc_kernel<<<(unsigned)nb, 256, 0, ctx->stream>>>(d, in_of(i), L.out_dim, L.in_dim, inv, S, tau, t);
        ctx->launches++;
        if (i > 0) {
          if (ctx->use_tc && st->wt[i].h) NNAL_TRY(fc_bwd_data_tc(ctx, st, L, st->wt[i], d, other, nb));
          else NNAL_TRY(fc_bwd_data(ctx, L, d, other, nb));
          d = other; pp ^= 1;
        }
      } else {
        const double inv = 1.0 / ((double)L.kh * L.kw * L.in_c * L.out_c + L.out_c);
        const size_t sm = (size_t)(L.in_h + L.kh - 1) * (L.in_w + L.kw - 1) * sizeof(double);
        if (sm > 40 * 1024) NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "conv input plane exceeds shared memory");
        shrink_conv_kernel<<<(unsigned)nb, 256, sm, ctx->stream>>>(d, in_of(i), L.in_h, L.in_w, L.in_c, L.out_c, L.kh, L.kw,
                                                                   inv, S, tau, t);
        ctx->launches++;
        if (i > 0) {
          if (ctx->use_tc && !ctx->dbg.bw_no_tc && st->cw[i]) NNAL_TRY(conv_bwd_data_tc(ctx, st, L, st->cw[i], d, other, nb));
          else NNAL_TRY(conv_bwd_data(ctx, L, d, other, nb));
          d = other; pp ^= 1;
        }
      }
      --t;
    }
    CUDA_TRY(ctx, cudaGetLastError());
  }
  prof_end(ctx);
  if (binary) {
    binary_scale_kernel<<<grid_for(ctx, nb * tau, 8), 256, 0, ctx->stream>>>((const double*)st->sred.p,
                                                                             (const float*)st->post.p, nb, tau, G);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
  }
  for (int y = 0; y < c; ++y) {
    CUDA_TRY(ctx, cudaMemcpyAsync(g_out + ((size_t)y * n_total + o) * tau, G + (size_t)y * nb * tau,
                                  (size_t)nb * tau * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    if (post_out)
      CUDA_TRY(ctx, cudaMemcpyAsync(post_out + (size_t)y * n_total + o, (const float*)st->post.p + (size_t)y * nb,
                                    (size_t)nb * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  }
  NNAL_SYNC_CHECKED(ctx);                                // the workspaces are reused by the next chunk
  return NNAL_OK;
}

int check_model(nnal_ctx* ctx) {
  if (ctx->layers.empty()) NNAL_FAIL(ctx, NNAL_ERR_STATE, "model not set");
  if (ctx->n_class < 2) NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "shrunk gradients need at least two classes");
  return NNAL_OK;
}

}  // namespace

int nnal_bw_release(nnal_ctx* ctx) {
  if (!ctx->bw_state) return NNAL_OK;
  BwState* st = (BwState*)ctx->bw_state;
  DevBuf* bufs[] = {&st->acts, &st->g[0], &st->g[1], &st->post, &st->gout, &st->sred, &st->amax};
  for (DevBuf* b : bufs) { if (b->p) cudaFree(b->p); b->p = nullptr; b->cap = 0; }
  free_transposed(st);
  delete st;
  ctx->bw_state = nullptr;
  return NNAL_OK;
}

extern "C" int nnal_fi_shrunk_tau(nnal_ctx* ctx, int* tau) {
  if (!ctx || !tau) return NNAL_ERR_INVALID;
  NNAL_TRY(check_model(ctx));
  *tau = count_tau(ctx);
  return NNAL_OK;
}

extern "C" int nnal_fi_shrunk_images(nnal_ctx* ctx, const float* x, int64_t n, float* post_out, double* g_out) {
  if (!ctx || n < 0 || (n > 0 && (!x || !g_out))) return NNAL_ERR_INVALID;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  NNAL_TRY(check_model(ctx));
  if (n == 0) return NNAL_OK;
  BwState* st = bw_state(ctx);
  const int64_t chunk = std::min(bw_chunk(ctx), n);
  const size_t per = (size_t)ctx->in_h * ctx->in_w * ctx->in_c;
  NNAL_TRY(devbuf_reserve(ctx, ctx->xin, (size_t)chunk * per * sizeof(float)));
  for (int64_t o = 0; o < n; o += chunk) {
    const int64_t nb = std::min(chunk, n - o);
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->xin.p, x + o * per, (size_t)nb * per * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    NNAL_TRY(shrunk_chunk(ctx, st, nb, n, o, post_out, g_out));
  }
  return NNAL_OK;
}

extern "C" int nnal_fi_shrunk_voxels(nnal_ctx* ctx, int subject, const int64_t* inds, int64_t n, int d1, int d2, int d3,
                                     const double* stats, int norm_mode, float* post_out, double* g_out) {
  if (!ctx || n < 0 || (n > 0 && (!inds || !g_out))) return NNAL_ERR_INVALID;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  NNAL_TRY(check_model(ctx));
  const Volume* v;
  NNAL_TRY(nnal_check_gather_args(ctx, subject, n, d1, d2, d3, &v));
  if (d1 != ctx->in_h || d2 != ctx->in_w || d3 * v->m != ctx->in_c)
    NNAL_FAIL(ctx, NNAL_ERR_INVALID, "patch shape does not match the model input");
  if (n == 0) return NNAL_OK;
  double* d_stats;
  NNAL_TRY(nnal_upload_stats(ctx, stats, v->m, norm_mode, &d_stats));
  BwState* st = bw_state(ctx);
  const int64_t chunk = std::min(bw_chunk(ctx), n);
  const size_t per = (size_t)ctx->in_h * ctx->in_w * ctx->in_c;
  NNAL_TRY(devbuf_reserve(ctx, ctx->xin, (size_t)chunk * per * sizeof(float)));
  NNAL_TRY(devbuf_reserve(ctx, ctx->inds, (size_t)n * 8));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->inds.p, inds, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
  const int64_t* d_inds = (const int64_t*)ctx->inds.p;
  for (int64_t o = 0; o < n; o += chunk) {
    const int64_t nb = std::min(chunk, n - o);
    NNAL_TRY(nnal_k_gather_norm_f32(ctx, *v, d_inds + o, nb, d1, d2, d3, d_stats, norm_mode, (float*)ctx->xin.p));
    NNAL_TRY(shrunk_chunk(ctx, st, nb, n, o, post_out, g_out));
  }
  return NNAL_OK;
}
