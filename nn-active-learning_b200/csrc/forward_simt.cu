// FP32 CUDA-core forward kernels: direct conv (SAME, stride 1, bias, ReLU), max-pool (SAME,
// window == stride), FC (W x + b, optional ReLU).  They restate the TF ops the reference graph is
// built from (NN.py:285-290 conv2d+bias+relu, NN.py:1473-1477 max_pool, NN.py:322-327 matmul+bias)
// for ANY layer dictionary NN.CNN accepts.  The tensor-core kernels (gemm_tc.cu / conv_tc.cu)
// take over the shapes they are specialised for; these kernels cover every other shape and serve
// as the on-device fp32 cross-check of the tensor-core path in tests (NNAL_FORCE_SIMT=1).
#include "nnal_common.cuh"

// ------------------------------------------------------------------------------------------
// direct convolution, one CTA per sample, padded input tile in shared memory
// ------------------------------------------------------------------------------------------
template <int TP, int TC>
__global__ void __launch_bounds__(256) conv_simt_kernel(const float* __restrict__ in, const float* __restrict__ Wt,
                                                         const float* __restrict__ bias, float* __restrict__ out,
                                                         nnal_h* __restrict__ out_hi, nnal_h* __restrict__ out_lo,
                                                         int64_t n, int H, int Wd, int Cin, int Cout, int kh, int kw) {
  extern __shared__ float s_in[];
  const int ph = kh / 2, pw = kw / 2;
  const int Hp = H + kh - 1, Wp = Wd + kw - 1;
  const int co_groups = (Cout + TC - 1) / TC;
  const int PG = blockDim.x / co_groups;
  const int tid = threadIdx.x;
  const int cg = tid % co_groups, pg = tid / co_groups;
  const bool active = pg < PG;
  const int co0 = cg * TC;
  const int HW = H * Wd;
  for (int64_t s = blockIdx.x; s < n; s += gridDim.x) {
    const float* src = in + s * (int64_t)HW * Cin;
    for (int e = tid; e < Hp * Wp * Cin; e += blockDim.x) {
      int ci = e % Cin;
      int t = e / Cin;
      int xx = t % Wp - pw, yy = t / Wp - ph;
      s_in[e] = (xx >= 0 && xx < Wd && yy >= 0 && yy < H) ? src[((int64_t)yy * Wd + xx) * Cin + ci] : 0.f;
    }
    __syncthreads();
    if (active) {
      for (int p0 = 0; p0 < HW; p0 += PG * TP) {
        float acc[TP][TC];
        int off[TP];
#pragma unroll
        for (int t = 0; t < TP; ++t) {
          int p = p0 + pg + t * PG;
          int pc = p < HW ? p : 0;
          off[t] = ((pc / Wd) * Wp + (pc % Wd)) * Cin;
#pragma unroll
          for (int c = 0; c < TC; ++c) acc[t][c] = 0.f;
        }
        for (int dy = 0; dy < kh; ++dy)
          for (int dx = 0; dx < kw; ++dx) {
            const int toff = (dy * Wp + dx) * Cin;
            const float* wrow = Wt + (int64_t)((dy * kw + dx) * Cin) * Cout + co0;
            for (int ci = 0; ci < Cin; ++ci) {
              float w[TC];
              if (TC == 4 && (Cout % 4) == 0) {
                float4 w4 = __ldg(reinterpret_cast<const float4*>(wrow + (int64_t)ci * Cout));
                w[0] = w4.x; w[1 % TC] = w4.y; w[2 % TC] = w4.z; w[3 % TC] = w4.w;
              } else {
#pragma unroll
                for (int c = 0; c < TC; ++c) w[c] = (co0 + c < Cout) ? __ldg(wrow + (int64_t)ci * Cout + c) : 0.f;
              }
#pragma unroll
              for (int t = 0; t < TP; ++t) {
                float a = s_in[off[t] + toff + ci];
#pragma unroll
                for (int c = 0; c < TC; ++c) acc[t][c] = fmaf(a, w[c], acc[t][c]);
              }
            }
          }
#pragma unroll
        for (int t = 0; t < TP; ++t) {
          int p = p0 + pg + t * PG;
          if (p < HW) {
#pragma unroll
            for (int c = 0; c < TC; ++c)
              if (co0 + c < Cout) {
                const float v = fmaxf(acc[t][c] + bias[co0 + c], 0.f);
                const int64_t o = (s * HW + p) * (int64_t)Cout + co0 + c;
                if (out) out[o] = v;
                if (out_hi) {
                  nnal_h h, l;
                  nnal_split(v, h, l);
                  out_hi[o] = h;
                  out_lo[o] = l;
                }
              }
          }
        }
      }
    }
    __syncthreads();
  }
}

static int conv_simt_launch(nnal_ctx* ctx, const Layer& L, const float* in, float* out, nnal_h* out_hi,
                            nnal_h* out_lo, int64_t n) {
  if (n == 0) return NNAL_OK;
  size_t smem = (size_t)(L.in_h + L.kh - 1) * (L.in_w + L.kw - 1) * L.in_c * sizeof(float);
  if (smem > 200 * 1024) NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "conv input tile exceeds shared memory");
  int grid = (int)(n < (int64_t)ctx->sm_count * 8 ? n : (int64_t)ctx->sm_count * 8);
  if (L.out_c % 4 == 0) {
    auto k = conv_simt_kernel<8, 4>;
    CUDA_TRY(ctx, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k<<<grid, 256, smem, ctx->stream>>>(in, L.W, L.b, out, out_hi, out_lo, n, L.in_h, L.in_w, L.in_c, L.out_c, L.kh, L.kw);
  } else {
    auto k = conv_simt_kernel<8, 1>;
    CUDA_TRY(ctx, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k<<<grid, 256, smem, ctx->stream>>>(in, L.W, L.b, out, out_hi, out_lo, n, L.in_h, L.in_w, L.in_c, L.out_c, L.kh, L.kw);
  }
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}

int nnal_k_conv_simt(nnal_ctx* ctx, const Layer& L, const float* in, float* out, int64_t n) {
  return conv_simt_launch(ctx, L, in, out, nullptr, nullptr, n);
}
// same kernel, output written as fp16 hi/lo planes (operand format of the tensor-core layers)
int nnal_k_conv_simt_split(nnal_ctx* ctx, const Layer& L, const float* in, nnal_h* out_hi, nnal_h* out_lo, int64_t n) {
  return conv_simt_launch(ctx, L, in, nullptr, out_hi, out_lo, n);
}

// ------------------------------------------------------------------------------------------
// max-pool SAME, window == stride (NN.py:1473-1477): output ceil(n/s); window (yo, xo) starts at (yo*s - pt, xo*s - pl)
// with TF's padding before (pt, pl; 0 for s = 2), and padded cells never win
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) pool_kernel(const float* __restrict__ in, float* __restrict__ out, int64_t total,
                                                    int H, int Wd, int C, int Ho, int Wo, int s, int pt, int pl) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    int c = e % C;
    int64_t t = e / C;
    int xo = t % Wo; t /= Wo;
    int yo = t % Ho;
    int64_t smp = t / Ho;
    float m = -INFINITY;
    const int y0 = yo * s - pt, x0 = xo * s - pl;
    const int y1 = min(y0 + s, H), x1 = min(x0 + s, Wd);
    for (int y = max(y0, 0); y < y1; ++y) {
      for (int x = max(x0, 0); x < x1; ++x) {
        m = fmaxf(m, in[((smp * H + y) * Wd + x) * (int64_t)C + c]);
      }
    }
    out[e] = m;
  }
}

// max-pool on fp16 hi/lo planes: the max of x = hi + lo is the pair whose sum is largest (exact).
// One thread pools 8 channels (one 16-byte vector of each plane) of one output position.
__device__ __forceinline__ void pool8_update(const uint4& h, const uint4& l, float* m, uint32_t* bh, uint32_t* bl) {
  const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const uint32_t hb = (hw[k >> 1] >> ((k & 1) * 16)) & 0xffffu, lb = (lw[k >> 1] >> ((k & 1) * 16)) & 0xffffu;
    const float v = __half2float(__ushort_as_half((unsigned short)hb)) + __half2float(__ushort_as_half((unsigned short)lb));
    if (v > m[k]) { m[k] = v; bh[k] = hb; bl[k] = lb; }
  }
}
__global__ void __launch_bounds__(256) pool_split_kernel(const nnal_h* __restrict__ in_hi, const nnal_h* __restrict__ in_lo,
                                                          nnal_h* __restrict__ out_hi, nnal_h* __restrict__ out_lo,
                                                          int64_t total8, int H, int Wd, int C, int Ho, int Wo, int s,
                                                          int pt, int pl) {
  const int C8 = C / 8;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total8; e += (int64_t)gridDim.x * blockDim.x) {
    int c8 = e % C8;
    int64_t t = e / C8;
    int xo = t % Wo; t /= Wo;
    int yo = t % Ho;
    int64_t smp = t / Ho;
    float m[8];
    uint32_t bh[8], bl[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) { m[k] = -INFINITY; bh[k] = 0; bl[k] = 0; }
    const int y0 = yo * s - pt, x0 = xo * s - pl;
    const int y1 = min(y0 + s, H), x1 = min(x0 + s, Wd);
    for (int y = max(y0, 0); y < y1; ++y) {
      for (int x = max(x0, 0); x < x1; ++x) {
        int64_t idx = ((smp * H + y) * Wd + x) * (int64_t)C + c8 * 8;
        uint4 h = *reinterpret_cast<const uint4*>(in_hi + idx);
        uint4 l = *reinterpret_cast<const uint4*>(in_lo + idx);
        pool8_update(h, l, m, bh, bl);
      }
    }
    uint4 oh = make_uint4(bh[0] | (bh[1] << 16), bh[2] | (bh[3] << 16), bh[4] | (bh[5] << 16), bh[6] | (bh[7] << 16));
    uint4 ol = make_uint4(bl[0] | (bl[1] << 16), bl[2] | (bl[3] << 16), bl[4] | (bl[5] << 16), bl[6] | (bl[7] << 16));
    *reinterpret_cast<uint4*>(out_hi + e * 8) = oh;
    *reinterpret_cast<uint4*>(out_lo + e * 8) = ol;
  }
}
// scalar variant for channel counts that are not a multiple of 8
__global__ void __launch_bounds__(256) pool_split_scalar_kernel(const nnal_h* __restrict__ in_hi, const nnal_h* __restrict__ in_lo,
                                                                 nnal_h* __restrict__ out_hi, nnal_h* __restrict__ out_lo,
                                                                 int64_t total, int H, int Wd, int C, int Ho, int Wo, int s,
                                                                 int pt, int pl) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    int c = e % C;
    int64_t t = e / C;
    int xo = t % Wo; t /= Wo;
    int yo = t % Ho;
    int64_t smp = t / Ho;
    float m = -INFINITY;
    nnal_h bh = __float2half_rn(0.f), bl = bh;
    const int y0 = yo * s - pt, x0 = xo * s - pl;
    const int y1 = min(y0 + s, H), x1 = min(x0 + s, Wd);
    for (int y = max(y0, 0); y < y1; ++y) {
      for (int x = max(x0, 0); x < x1; ++x) {
        int64_t idx = ((smp * H + y) * Wd + x) * (int64_t)C + c;
        nnal_h h = in_hi[idx], l = in_lo[idx];
        float v = nnal_merge(h, l);
        if (v > m) { m = v; bh = h; bl = l; }
      }
    }
    out_hi[e] = bh;
    out_lo[e] = bl;
  }
}

int nnal_k_pool_split(nnal_ctx* ctx, const Layer& L, const nnal_h* in_hi, const nnal_h* in_lo, nnal_h* out_hi,
                      nnal_h* out_lo, int64_t n) {
  int64_t total = n * L.out_h * L.out_w * L.out_c;
  if (total == 0) return NNAL_OK;
  if (L.out_c % 8 == 0) {
    int64_t total8 = total / 8;
    int grid = (int)((total8 + 255) / 256 < (int64_t)ctx->sm_count * 32 ? (total8 + 255) / 256 : (int64_t)ctx->sm_count * 32);
    pool_split_kernel<<<grid, 256, 0, ctx->stream>>>(in_hi, in_lo, out_hi, out_lo, total8, L.in_h, L.in_w, L.in_c, L.out_h, L.out_w, L.kh,
        L.pad_t, L.pad_l);
  } else {
    int grid = (int)((total + 255) / 256 < (int64_t)ctx->sm_count * 16 ? (total + 255) / 256 : (int64_t)ctx->sm_count * 16);
    pool_split_scalar_kernel<<<grid, 256, 0, ctx->stream>>>(in_hi, in_lo, out_hi, out_lo, total, L.in_h, L.in_w, L.in_c, L.out_h, L.out_w, L.kh,
        L.pad_t, L.pad_l);
  }
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}

int nnal_k_pool(nnal_ctx* ctx, const Layer& L, const float* in, float* out, int64_t n) {
  int64_t total = n * L.out_h * L.out_w * L.out_c;
  if (total == 0) return NNAL_OK;
  int grid = (int)((total + 255) / 256 < (int64_t)ctx->sm_count * 16 ? (total + 255) / 256 : (int64_t)ctx->sm_count * 16);
  pool_kernel<<<grid, 256, 0, ctx->stream>>>(in, out, total, L.in_h, L.in_w, L.in_c, L.out_h, L.out_w, L.kh, L.pad_t, L.pad_l);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}

// ------------------------------------------------------------------------------------------
// FC:  out[n][N] = act(in[n][K] . W[N][K]^T + b)   (sample-major restatement of W@x+b, NN.py:322-327)
// 128x128x16 tiles, 256 threads, 8x8 register micro-tiles.
// ------------------------------------------------------------------------------------------
#define FC_BM 128
#define FC_BN 128
#define FC_BK 16
__global__ void __launch_bounds__(256) fc_simt_kernel(const float* __restrict__ A, const float* __restrict__ Wt,
                                                       const float* __restrict__ bias, float* __restrict__ C, int64_t M,
                                                       int N, int K, int relu) {
  __shared__ float As[FC_BK][FC_BM + 4];
  __shared__ float Bs[FC_BK][FC_BN + 4];
  const int tid = threadIdx.x;
  const int64_t m0 = (int64_t)blockIdx.y * FC_BM;
  const int n0 = blockIdx.x * FC_BN;
  const int tx = tid % 16, ty = tid / 16;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  const bool vec = (K % 4) == 0;
  for (int k0 = 0; k0 < K; k0 += FC_BK) {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      int row = tid / 4 + 64 * i, kq = (tid % 4) * 4;
      float va[4] = {0, 0, 0, 0}, vb[4] = {0, 0, 0, 0};
      int64_t gm = m0 + row;
      int gn = n0 + row;
      if (vec && k0 + kq + 3 < K) {
        if (gm < M) { float4 t = *reinterpret_cast<const float4*>(A + gm * K + k0 + kq); va[0] = t.x; va[1] = t.y; va[2] = t.z; va[3] = t.w; }
        if (gn < N) { float4 t = __ldg(reinterpret_cast<const float4*>(Wt + (int64_t)gn * K + k0 + kq)); vb[0] = t.x; vb[1] = t.y; vb[2] = t.z; vb[3] = t.w; }
      } else {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          if (k0 + kq + c < K) {
            if (gm < M) va[c] = A[gm * K + k0 + kq + c];
            if (gn < N) vb[c] = __ldg(Wt + (int64_t)gn * K + k0 + kq + c);
          }
        }
      }
#pragma unroll
      for (int c = 0; c < 4; ++c) { As[kq + c][row] = va[c]; Bs[kq + c][row] = vb[c]; }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < FC_BK; ++k) {
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
    int64_t gm = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + i - 4);
    if (gm >= M) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int gn = n0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + j - 4);
      if (gn < N) {
        float v = acc[i][j] + bias[gn];
        C[gm * N + gn] = relu ? fmaxf(v, 0.f) : v;
      }
    }
  }
}

int nnal_k_fc_simt(nnal_ctx* ctx, const Layer& L, const float* in, float* out, int64_t n) {
  if (n == 0) return NNAL_OK;
  dim3 grid(cdiv(L.out_dim, FC_BN), cdiv(n, FC_BM));
  fc_simt_kernel<<<grid, 256, 0, ctx->stream>>>(in, L.W, L.b, out, n, L.out_dim, L.in_dim, L.relu);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}

// ------------------------------------------------------------------------------------------
// The reference flattens conv output with reshape(transpose(x)) (NN.py:296-301, 337-340): flat row
// = c*(W*H) + w*H + h.  Activations here stay NHWC, so the first FC weight is re-indexed ONCE:
// Wnative[o][(h*W + w)*C + c] = Wtf[o][c*W*H + w*H + h].
// ------------------------------------------------------------------------------------------
__global__ void permute_fc_weight_kernel(const float* __restrict__ Wtf, float* __restrict__ Wn, int out, int C, int H,
                                         int Wd) {
  int64_t total = (int64_t)out * C * H * Wd;
  int K = C * H * Wd;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    int o = e / K;
    int r = e - (int64_t)o * K;
    int c = r % C;
    int t = r / C;
    int w = t % Wd, h = t / Wd;
    Wn[e] = Wtf[(int64_t)o * K + c * (Wd * H) + w * H + h];
  }
}

int nnal_k_permute_fc_weight(nnal_ctx* ctx, const float* Wtf, float* Wn, int out, int C, int H, int Wd) {
  int64_t total = (int64_t)out * C * H * Wd;
  int grid = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
  permute_fc_weight_kernel<<<grid, 256, 0, ctx->stream>>>(Wtf, Wn, out, C, H, Wd);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}
