// Scoring kernels: fused last-FC + softmax head (2..32 classes), the wide head's softmax (64 classes or more), entropy /
// binary-uncertainty scores, exact top-k.
//
// Reference behaviour replaced:
//   * posteriors = softmax over classes of the last FC output (NN.py:184-188, 322-327)
//   * NNAL_tools.compute_entropy / uncertainty_filtering (NNAL_tools.py:71-85, 22-36)
//   * abs(P(class1) - 0.5) ranking (PW_NNAL.py:64, 109-110, 671-681, 724-730)
//   * np.argsort(score)[:k] (PW_NNAL.py:64,730; NNAL.py:310; NNAL_tools.py:34) with the tie-break
//     this build defines: lowest pool position first (SURVEY H7).
#include "nnal_common.cuh"

// ------------------------------------------------------------------------------------------
// head: one warp per sample; logits = W[c][d] . feat[d] + b ; warp-shuffle reduction; softmax
// ------------------------------------------------------------------------------------------
template <int CMAX>
__global__ void __launch_bounds__(256) head_kernel(const float* __restrict__ feat, const float* __restrict__ Wt,
                                                    const float* __restrict__ bias, int64_t n, int d, int c,
                                                    int64_t pool_n, int64_t offset, float* __restrict__ post,
                                                    float* __restrict__ logits_out, DropSpec drop) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t s = warp; s < n; s += nwarps) {
    float acc[CMAX];
#pragma unroll
    for (int j = 0; j < CMAX; ++j) acc[j] = 0.f;
    const float* f = feat + s * d;
    if ((d & 3) == 0) {
      for (int k = lane * 4; k < d; k += 128) {
        float4 a = *reinterpret_cast<const float4*>(f + k);
#pragma unroll
        for (int j = 0; j < CMAX; ++j)
          if (j < c) {
            float4 w = __ldg(reinterpret_cast<const float4*>(Wt + (int64_t)j * d + k));
            acc[j] = fmaf(a.x, w.x, fmaf(a.y, w.y, fmaf(a.z, w.z, fmaf(a.w, w.w, acc[j]))));
          }
      }
    } else {
      for (int k = lane; k < d; k += 32) {
        float a = f[k];
#pragma unroll
        for (int j = 0; j < CMAX; ++j)
          if (j < c) acc[j] = fmaf(a, __ldg(Wt + (int64_t)j * d + k), acc[j]);
      }
    }
#pragma unroll
    for (int j = 0; j < CMAX; ++j) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], o);
    }
    // every lane holds all logits; lane j finalises class j
    float zmax = -INFINITY;
#pragma unroll
    for (int j = 0; j < CMAX; ++j)
      if (j < c) {
        acc[j] += bias[j];
        if (drop.thresh) {             // PW1 drops out the logits too (dropout layer 8 = fc3, NN.py:1338)
          uint32_t r4[4];
          philox4x32_10((uint32_t)j >> 2, (uint32_t)(drop.row0 + offset + s), drop.pass, drop.site, drop.k0, drop.k1, r4);
          acc[j] = r4[j & 3] < drop.thresh ? acc[j] / drop.keep : 0.f;
        }
        zmax = fmaxf(zmax, acc[j]);
      }
    float sum = 0.f;
    float mine = 0.f, myz = 0.f;
#pragma unroll
    for (int j = 0; j < CMAX; ++j)
      if (j < c) {
        float e = expf(acc[j] - zmax);
        sum += e;
        if (j == lane) { mine = e; myz = acc[j]; }
      }
    if (lane < c) {
      post[(int64_t)lane * pool_n + offset + s] = mine / sum;
      if (logits_out) logits_out[s * c + lane] = myz;
    }
  }
}

// ------------------------------------------------------------------------------------------
// wide head (c >= 64): the logits come from the FC GEMM (tensor cores or CUDA cores) into a [n][ldz] scratch; this kernel
// turns them into post[j][pool_n] at offset + s, exp(z - max) / sum.  Memory-bound: per sample 4c B read twice (the second
// read from L2) and 4c B written.  One CTA per tile of 32 pool positions, aligned to multiples of 32 of the global position
// offset + s, so every warp store of a class row covers the same 32-position group (partial at both ends of the range).
// Pass 1: one warp per sample, max and sum over the row.  Pass 2: 32 x 128 (sample x class) blocks through shared
// memory, read along the logits rows and written along the class rows.  Nothing is sized by c.  Pass 1 reads the row twice
// (max, then the sum of exponentials; the second read hits L1/L2) with four independent loads per lane in flight: an online
// max/sum loop carries a dependency through every element and ran at 13 % of the HBM bound at c = 1,000.
// ------------------------------------------------------------------------------------------
constexpr int WSM_THREADS = 512, WSM_CB = 4;
__global__ void __launch_bounds__(WSM_THREADS) wide_softmax_kernel(const float* __restrict__ z, int64_t ldz, int64_t n, int c,
                                                                    int64_t pool_n, int64_t offset, float* __restrict__ post) {
  constexpr int NW = WSM_THREADS / 32;
  __shared__ float t[WSM_CB][32][33];
  __shared__ float s_max[32], s_sum[32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int64_t g_first = offset & ~(int64_t)31;                 // first tile's global position
  const int64_t ntiles = ((offset + n + 31) >> 5) - (offset >> 5);
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t s0 = g_first + tile * 32 - offset;             // chunk-relative sample of tile row 0 (may be < 0)
    for (int r = wid; r < 32; r += NW) {
      const int64_t s = s0 + r;
      float m = -INFINITY, sum = 0.f;
      if (s >= 0 && s < n) {
        const float* row = z + s * ldz;
        float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
        for (int j = lane; j < c; j += 128) {
#pragma unroll
          for (int u = 0; u < 4; ++u)
            if (j + 32 * u < c) m4[u] = fmaxf(m4[u], row[j + 32 * u]);
        }
        m = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        float e4[4] = {0.f, 0.f, 0.f, 0.f};
        for (int j = lane; j < c; j += 128) {
#pragma unroll
          for (int u = 0; u < 4; ++u)
            if (j + 32 * u < c) e4[u] += expf(row[j + 32 * u] - m);
        }
        sum = (e4[0] + e4[1]) + (e4[2] + e4[3]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
      }
      if (lane == 0) { s_max[r] = m; s_sum[r] = sum; }
    }
    __syncthreads();
    for (int j0 = 0; j0 < c; j0 += 32 * WSM_CB) {              // WSM_CB blocks of 32 classes per barrier pair
      for (int r = wid; r < 32; r += NW) {                       // sample r, class j0 + 32 u + lane
        const int64_t s = s0 + r;
        if (s >= 0 && s < n) {
#pragma unroll
          for (int u = 0; u < WSM_CB; ++u) {
            const int j = j0 + 32 * u + lane;
            if (j < c) t[u][r][lane] = expf(z[s * ldz + j] - s_max[r]) / s_sum[r];
          }
        }
      }
      __syncthreads();
      for (int r = wid; r < 32; r += NW) {                       // class j0 + 32 u + r, sample lane
        const int64_t s = s0 + lane;
        if (s >= 0 && s < n) {
#pragma unroll
          for (int u = 0; u < WSM_CB; ++u) {
            const int j = j0 + 32 * u + r;
            if (j < c) post[(int64_t)j * pool_n + offset + s] = t[u][lane][r];
          }
        }
      }
      __syncthreads();
    }
  }
}

int nnal_k_softmax_wide(nnal_ctx* ctx, const float* logits, int64_t ldz, int64_t n, int c, int64_t pool_n, int64_t offset,
                        float* post) {
  if (n == 0) return NNAL_OK;
  const int64_t ntiles = ((offset + n + 31) >> 5) - (offset >> 5);
  const int grid = (int)(ntiles < (int64_t)ctx->sm_count * 4 ? ntiles : (int64_t)ctx->sm_count * 4);
  wide_softmax_kernel<<<grid, WSM_THREADS, 0, ctx->stream>>>(logits, ldz, n, c, pool_n, offset, post);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}

// c >= 64 from fp32 features: the logits GEMM on the tensor cores (the head's own predicate, nnal_tc_head_supported) or
// the CUDA-core FC kernel, then the softmax.  Dropout on the logits is applied by the tensor-core GEMM's epilogue only:
// MC-dropout needs the hidden FC layers on the tensor cores, so its wide head never takes the CUDA-core path.
static int wide_head_f32(nnal_ctx* ctx, const Layer& L, const float* feat, int64_t n, int64_t pool_n, int64_t offset,
                         float* post, const DropSpec* drop) {
  const int c = L.out_dim;
  if (ctx->use_tc && nnal_tc_head_supported(ctx, L)) {
    const int ldz = nnal_head_ldz(c);
    NNAL_TRY(devbuf_reserve(ctx, ctx->head_logits, (size_t)n * ldz * sizeof(float)));
    NNAL_TRY(nnal_tc_head(ctx, L, feat, (float*)ctx->head_logits.p, n, drop));
    return nnal_k_softmax_wide(ctx, (const float*)ctx->head_logits.p, ldz, n, c, pool_n, offset, post);
  }
  if (drop && drop->thresh)
    NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "MC-dropout on the logits of a head with more than 32 classes needs the tensor-core path");
  NNAL_TRY(devbuf_reserve(ctx, ctx->head_logits, (size_t)n * c * sizeof(float)));
  NNAL_TRY(nnal_k_fc_simt(ctx, L, feat, (float*)ctx->head_logits.p, n));
  return nnal_k_softmax_wide(ctx, (const float*)ctx->head_logits.p, c, n, c, pool_n, offset, post);
}

int nnal_k_head(nnal_ctx* ctx, const Layer& L, const float* feat, int64_t n, int64_t pool_n, int64_t offset,
                float* post, float* logits_out, const DropSpec* dropp) {
  if (n == 0) return NNAL_OK;
  if (L.out_dim >= NNAL_WIDE_HEAD_MIN && !logits_out) return wide_head_f32(ctx, L, feat, n, pool_n, offset, post, dropp);
  const DropSpec drop = dropp ? *dropp : DropSpec();
  int c = L.out_dim, d = L.in_dim;
  int64_t blocks = (n * 32 + 255) / 256;
  int grid = (int)(blocks < (int64_t)ctx->sm_count * 8 ? blocks : (int64_t)ctx->sm_count * 8);
  if (c <= 2)
    head_kernel<2><<<grid, 256, 0, ctx->stream>>>(feat, L.W, L.b, n, d, c, pool_n, offset, post, logits_out, drop);
  else if (c <= 16)
    head_kernel<16><<<grid, 256, 0, ctx->stream>>>(feat, L.W, L.b, n, d, c, pool_n, offset, post, logits_out, drop);
  else if (c <= 32)
    head_kernel<32><<<grid, 256, 0, ctx->stream>>>(feat, L.W, L.b, n, d, c, pool_n, offset, post, logits_out, drop);
  else
    NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "33 to 63 classes are not supported (fused head: 2 to 32, wide head: 64 or more)");
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}

// ------------------------------------------------------------------------------------------
// scores in float64 (the reference ranks float64 copies of the float32 posteriors)
//   kind 0: |p1 - 0.5|  (row 1 of post, PW_NN.py:526-529 keeps P(class 1))
//   kind 1: -H,  H = -sum_c p log p with zeros replaced by eps (1e-7 compute_entropy / 1e-8
//           uncertainty_filtering)
//   kind 2: +H
// Templated on the posterior element type: float (pool path) or double (host API parity).
// ------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) score_kernel(const T* __restrict__ post, int c, int64_t n, int kind, double eps,
                                                     double* __restrict__ score) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    double v;
    if (kind == 0) {
      v = fabs((double)post[n + i] - 0.5);
    } else {
      double h = 0.0;
      for (int j = 0; j < c; ++j) {
        double p = (double)post[(int64_t)j * n + i];
        if (p == 0.0) p += eps;
        h += p * log(p);
      }
      v = (kind == 1) ? h : -h;     // kind 1: -H = sum p log p
    }
    score[i] = v + 0.0;             // canonicalise -0.0
  }
}

template <typename T>
static int launch_scores(nnal_ctx* ctx, const T* post, int c, int64_t n, int kind, double eps, double* score) {
  if (n == 0) return NNAL_OK;
  int64_t blocks = (n + 255) / 256;
  int grid = (int)(blocks < (int64_t)ctx->sm_count * 16 ? blocks : (int64_t)ctx->sm_count * 16);
  score_kernel<T><<<grid, 256, 0, ctx->stream>>>(post, c, n, kind, eps, score);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}
int nnal_k_scores_f32(nnal_ctx* ctx, const float* post, int c, int64_t n, int kind, double eps, double* score) {
  return launch_scores<float>(ctx, post, c, n, kind, eps, score);
}
int nnal_k_scores_f64(nnal_ctx* ctx, const double* post, int c, int64_t n, int kind, double eps, double* score) {
  return launch_scores<double>(ctx, post, c, n, kind, eps, score);
}

// ------------------------------------------------------------------------------------------
// MC-dropout running means (PW_NNAL.py:67-87 MC-entropy, :232-282 BALD), float64 like the reference:
//   av_posts = (posts + i * av_posts) / (i + 1)
//   ents = -p log p - (1-p) log(1-p) with zeros bumped by 1e-6;  av_ents = (ents + i * av_ents) / (i + 1)
// posts = P(class 1) of pass i (float32 from the head kernel, promoted as batch_eval does, PW_NN.py:526-529)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) mc_accum_kernel(const float* __restrict__ post1, int64_t n, int t,
                                                        double* __restrict__ av_post, double* __restrict__ av_ent) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    double p = (double)post1[i];
    av_post[i] = t == 0 ? p : (p + t * av_post[i]) / (t + 1);
    double q = 1.0 - p;
    if (p == 0.0) p += 1e-6;
    if (q == 0.0) q += 1e-6;
    const double e = -p * log(p) - q * log(q);
    av_ent[i] = t == 0 ? e : (e + t * av_ent[i]) / (t + 1);
  }
}
// c > 2: the same recurrences over every class, av_post [c][pool_n] (the layout of the head's posteriors) and
//   ents = -sum_j p_j log p_j with zeros bumped by 1e-6.  Memory-bound: 4c B read, 16c + 16 B read and written per sample.
__global__ void __launch_bounds__(256) mc_class_accum_kernel(const float* __restrict__ post, int c, int64_t stride, int64_t n,
                                                              int t, double* __restrict__ av_post, double* __restrict__ av_ent) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    double e = 0.0;
    for (int j = 0; j < c; ++j) {
      double p = (double)post[(int64_t)j * stride + i];
      double* a = av_post + (int64_t)j * stride + i;
      *a = t == 0 ? p : (p + t * *a) / (t + 1);
      if (p == 0.0) p += 1e-6;
      e -= p * log(p);
    }
    av_ent[i] = t == 0 ? e : (e + t * av_ent[i]) / (t + 1);
  }
}
// c == 2 keeps the binary statistics (av_post = mean P(class 1), [pool_n]); c > 2 keeps every class ([c][pool_n])
int nnal_k_mc_accumulate(nnal_ctx* ctx, const float* post, int c, int64_t pool_n, int64_t offset, int64_t n, int t,
                         double* av_post, double* av_ent) {
  if (n == 0) return NNAL_OK;
  int64_t blocks = (n + 255) / 256;
  int grid = (int)(blocks < (int64_t)ctx->sm_count * 16 ? blocks : (int64_t)ctx->sm_count * 16);
  if (c == 2)
    mc_accum_kernel<<<grid, 256, 0, ctx->stream>>>(post + pool_n + offset, n, t, av_post + offset, av_ent + offset);
  else
    mc_class_accum_kernel<<<grid, 256, 0, ctx->stream>>>(post + offset, c, pool_n, n, t, av_post + offset, av_ent + offset);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}
//   kind 10 (MC-entropy): |av_posts - 0.5|                                           (PW_NNAL.py:84-85, 241)
//   kind 11 (BALD):       -(H(av_posts) - av_ents), H with the same 1e-6 zero bumps   (PW_NNAL.py:270-278; ascending
//                         top-k of the negated score = argsort(-scores)[:k])
//   kind 12:              -H(av_posts), the predictive entropy of kind 10's c-class form (monotone in |av_posts - 0.5|)
//   kind 13:              kind 11
__global__ void __launch_bounds__(256) mc_score_kernel(const double* __restrict__ av_post, const double* __restrict__ av_ent,
                                                        int64_t n, int kind, double* __restrict__ score) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    double p = av_post[i], v;
    if (kind == 10) {
      v = fabs(p - 0.5);
    } else {
      double q = 1.0 - p;
      if (p == 0.0) p += 1e-6;
      if (q == 0.0) q += 1e-6;
      const double h = -p * log(p) - q * log(q);
      v = kind == 12 ? -h : -(h - av_ent[i]);
    }
    score[i] = v + 0.0;
  }
}
// c > 2, av_post [c][n]:  kind 12: -H(av_posts);  kind 13: -(H(av_posts) - av_ents);  zeros bumped by 1e-6
__global__ void __launch_bounds__(256) mc_class_score_kernel(const double* __restrict__ av_post, const double* __restrict__ av_ent,
                                                              int c, int64_t n, int kind, double* __restrict__ score) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    double h = 0.0;
    for (int j = 0; j < c; ++j) {
      double p = av_post[(int64_t)j * n + i];
      if (p == 0.0) p += 1e-6;
      h -= p * log(p);
    }
    const double v = kind == 12 ? -h : -(h - av_ent[i]);
    score[i] = v + 0.0;
  }
}
int nnal_k_scores_mc(nnal_ctx* ctx, const double* av_post, const double* av_ent, int c, int64_t n, int kind, double* score) {
  if (n == 0) return NNAL_OK;
  int64_t blocks = (n + 255) / 256;
  int grid = (int)(blocks < (int64_t)ctx->sm_count * 16 ? blocks : (int64_t)ctx->sm_count * 16);
  if (c == 2) mc_score_kernel<<<grid, 256, 0, ctx->stream>>>(av_post, av_ent, n, kind, score);
  else mc_class_score_kernel<<<grid, 256, 0, ctx->stream>>>(av_post, av_ent, c, n, kind, score);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}

// ------------------------------------------------------------------------------------------
// pixel-wise entropy map in float32 (config 4: posteriors [c][n] float32 -> H [n] float32, the shape of
// eval_utils.full_slice_segment's [c,h,w,z] tensor): -sum_c p log p with the compute_entropy zero guard.
// Memory-bound: (c+1)*4 B per sample; 4 samples per thread, 16-byte loads/stores when n % 4 == 0.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) entropy_f32_kernel(const float* __restrict__ post, int c, int64_t n, float eps,
                                                           float* __restrict__ H) {
  const int64_t nv = n >> 2;
  const bool vec = (n & 3) == 0;
  if (vec) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (int64_t)gridDim.x * blockDim.x) {
      float4 h = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int j = 0; j < c; ++j) {
        float4 p = __ldcs(reinterpret_cast<const float4*>(post + (int64_t)j * n) + i);
        p.x = p.x == 0.f ? eps : p.x; p.y = p.y == 0.f ? eps : p.y; p.z = p.z == 0.f ? eps : p.z; p.w = p.w == 0.f ? eps : p.w;
        h.x = fmaf(-p.x, logf(p.x), h.x); h.y = fmaf(-p.y, logf(p.y), h.y);
        h.z = fmaf(-p.z, logf(p.z), h.z); h.w = fmaf(-p.w, logf(p.w), h.w);
      }
      __stcs(reinterpret_cast<float4*>(H) + i, h);
    }
  } else {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
      float h = 0.f;
      for (int j = 0; j < c; ++j) {
        float p = post[(int64_t)j * n + i];
        p = p == 0.f ? eps : p;
        h = fmaf(-p, logf(p), h);
      }
      H[i] = h;
    }
  }
}

int nnal_k_entropy_f32(nnal_ctx* ctx, const float* post, int c, int64_t n, float eps, float* H) {
  if (n == 0) return NNAL_OK;
  // one 16-byte column group per thread: every load of the map is in flight at once
  int64_t blocks = ((n + 3) / 4 + 255) / 256;
  if ((n & 3) != 0) blocks = (n + 255) / 256;
  int grid = (int)(blocks < (int64_t)0x7fffffff ? blocks : (int64_t)0x7fffffff);
  entropy_f32_kernel<<<grid, 256, 0, ctx->stream>>>(post, c, n, eps, H);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}

// ------------------------------------------------------------------------------------------
// exact top-k (k smallest scores, ties -> lowest position): 8-pass MSB radix select on
// order-preserving 64-bit keys, stable tie compaction, bitonic sort of the k survivors.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long f64_key(double v) {
  unsigned long long b = (unsigned long long)__double_as_longlong(v);
  return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double key_f64(unsigned long long k) {
  unsigned long long b = (k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k;
  return __longlong_as_double((long long)b);
}

struct TopkState {
  unsigned long long prefix;      // selected high bits so far
  unsigned long long remaining;   // rank (1-based count) still to find inside the prefix bucket
  unsigned int hist[256];
  unsigned int count_lt;          // compaction cursor for keys < threshold
  unsigned int pad;
};

__global__ void topk_init_kernel(TopkState* st, unsigned long long k) {
  if (threadIdx.x == 0) { st->prefix = 0; st->remaining = k; st->count_lt = 0; }
  if (threadIdx.x < 256) st->hist[threadIdx.x] = 0;
}

__global__ void __launch_bounds__(256) topk_hist_kernel(const double* __restrict__ score, int64_t n, int shift,
                                                         TopkState* st) {
  __shared__ unsigned int h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  const unsigned long long prefix = st->prefix;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    unsigned long long key = f64_key(score[i]);
    bool match = (shift == 56) || (((key ^ prefix) >> (shift + 8)) == 0);
    if (match) atomicAdd(&h[(key >> shift) & 255], 1u);
  }
  __syncthreads();
  if (h[threadIdx.x]) atomicAdd(&st->hist[threadIdx.x], h[threadIdx.x]);
}

__global__ void topk_pick_kernel(TopkState* st, int shift) {
  // single warp: find the bin containing the remaining-th element
  if (threadIdx.x == 0) {
    unsigned long long rem = st->remaining, cum = 0;
    int b = 0;
    for (; b < 256; ++b) {
      unsigned long long c = st->hist[b];
      if (cum + c >= rem) break;
      cum += c;
    }
    if (b > 255) b = 255;
    st->prefix |= ((unsigned long long)b) << shift;
    st->remaining = rem - cum;
  }
  __syncthreads();
  if (threadIdx.x < 256) st->hist[threadIdx.x] = 0;
}

// keys strictly below the threshold: unordered compaction (they are sorted afterwards)
__global__ void __launch_bounds__(256) topk_compact_lt_kernel(const double* __restrict__ score, int64_t n,
                                                               TopkState* st, unsigned long long* __restrict__ okey,
                                                               unsigned int* __restrict__ oidx) {
  const unsigned long long T = st->prefix;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    unsigned long long key = f64_key(score[i]);
    if (key < T) {
      unsigned int slot = atomicAdd(&st->count_lt, 1u);
      okey[slot] = key;
      oidx[slot] = (unsigned int)i;
    }
  }
}

// ties at the threshold: stable (index-ordered) compaction in three steps
__global__ void __launch_bounds__(256) topk_tie_count_kernel(const double* __restrict__ score, int64_t n, int64_t per_block,
                                                              const TopkState* st, unsigned int* __restrict__ counts) {
  __shared__ unsigned int cnt;
  if (threadIdx.x == 0) cnt = 0;
  __syncthreads();
  const unsigned long long T = st->prefix;
  int64_t lo = (int64_t)blockIdx.x * per_block, hi = lo + per_block < n ? lo + per_block : n;
  unsigned int local = 0;
  for (int64_t i = lo + threadIdx.x; i < hi; i += blockDim.x) local += (f64_key(score[i]) == T);
  if (local) atomicAdd(&cnt, local);
  __syncthreads();
  if (threadIdx.x == 0) counts[blockIdx.x] = cnt;
}

__global__ void topk_tie_scan_kernel(unsigned int* counts, int nblocks) {
  if (threadIdx.x == 0) {
    unsigned int run = 0;
    for (int b = 0; b < nblocks; ++b) { unsigned int c = counts[b]; counts[b] = run; run += c; }
  }
}

__global__ void __launch_bounds__(256) topk_tie_emit_kernel(const double* __restrict__ score, int64_t n, int64_t per_block,
                                                             const TopkState* st, const unsigned int* __restrict__ counts,
                                                             unsigned long long k, unsigned long long* __restrict__ okey,
                                                             unsigned int* __restrict__ oidx) {
  __shared__ unsigned int warp_tot[8];
  __shared__ unsigned int base;
  const unsigned long long T = st->prefix;
  const unsigned long long need = st->remaining;          // number of ties to take
  const unsigned long long L = k - need;                   // keys < T occupy [0, L)
  if (threadIdx.x == 0) base = counts[blockIdx.x];
  __syncthreads();
  if (base >= need) return;
  int64_t lo = (int64_t)blockIdx.x * per_block, hi = lo + per_block < n ? lo + per_block : n;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (int64_t c0 = lo; c0 < hi; c0 += blockDim.x) {
    int64_t i = c0 + threadIdx.x;
    bool tie = (i < hi) && (f64_key(score[i]) == T);
    unsigned int bal = __ballot_sync(0xffffffffu, tie);
    unsigned int wrank = __popc(bal & ((1u << lane) - 1));
    if (lane == 0) warp_tot[wid] = __popc(bal);
    __syncthreads();
    unsigned int before = 0, tot = 0;
    for (int w = 0; w < 8; ++w) { if (w < wid) before += warp_tot[w]; tot += warp_tot[w]; }
    unsigned int b0 = base;
    if (tie) {
      unsigned long long rank = (unsigned long long)b0 + before + wrank;
      if (rank < need) { okey[L + rank] = T; oidx[L + rank] = (unsigned int)i; }
    }
    __syncthreads();
    if (threadIdx.x == 0) base = b0 + tot;
    __syncthreads();
    if (base >= need) return;
  }
}

__device__ __forceinline__ bool kv_less(unsigned long long ka, unsigned int ia, unsigned long long kb, unsigned int ib) {
  return ka < kb || (ka == kb && ia < ib);
}

__global__ void topk_pad_kernel(unsigned long long* key, unsigned int* idx, int64_t k, int64_t kp) {
  for (int64_t i = k + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < kp; i += (int64_t)gridDim.x * blockDim.x) {
    key[i] = ~0ull;
    idx[i] = ~0u;
  }
}

// one global compare-exchange step of the bitonic network
__global__ void __launch_bounds__(256) bitonic_step_kernel(unsigned long long* key, unsigned int* idx, int64_t kp, int64_t jj,
                                                            int64_t kk) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < kp / 2; t += (int64_t)gridDim.x * blockDim.x) {
    int64_t i = 2 * t - (t & (jj - 1));      // index with bit jj cleared
    int64_t l = i + jj;
    bool up = ((i & kk) == 0);
    unsigned long long ka = key[i], kb = key[l];
    unsigned int ia = idx[i], ib = idx[l];
    bool swap = up ? kv_less(kb, ib, ka, ia) : kv_less(ka, ia, kb, ib);
    if (swap) { key[i] = kb; key[l] = ka; idx[i] = ib; idx[l] = ia; }
  }
}

// all steps with partner distance < 2048 inside shared memory (tile of 4096 elements per CTA)
#define BT_TILE 4096
__global__ void __launch_bounds__(1024) bitonic_smem_kernel(unsigned long long* key, unsigned int* idx, int64_t kp,
                                                             int64_t kk_start, int64_t kk_end, int64_t jj_start) {
  __shared__ unsigned long long sk[BT_TILE];
  __shared__ unsigned int si[BT_TILE];
  const int64_t base = (int64_t)blockIdx.x * BT_TILE;
  const int tile = (int)(kp < BT_TILE ? kp : BT_TILE);
  for (int t = threadIdx.x; t < tile; t += blockDim.x) { sk[t] = key[base + t]; si[t] = idx[base + t]; }
  __syncthreads();
  for (int64_t kk = kk_start; kk <= kk_end; kk <<= 1) {
    int64_t j0 = (kk == kk_start) ? jj_start : (kk >> 1);
    if (j0 >= tile) j0 = tile >> 1;
    for (int64_t jj = j0; jj > 0; jj >>= 1) {
      for (int t = threadIdx.x; t < tile / 2; t += blockDim.x) {
        int i = 2 * t - (t & (int)(jj - 1));
        int l = i + (int)jj;
        bool up = (((base + i) & kk) == 0);
        unsigned long long ka = sk[i], kb = sk[l];
        unsigned int ia = si[i], ib = si[l];
        bool swap = up ? kv_less(kb, ib, ka, ia) : kv_less(ka, ia, kb, ib);
        if (swap) { sk[i] = kb; sk[l] = ka; si[i] = ib; si[l] = ia; }
      }
      __syncthreads();
    }
  }
  for (int t = threadIdx.x; t < tile; t += blockDim.x) { key[base + t] = sk[t]; idx[base + t] = si[t]; }
}

__global__ void topk_out_kernel(const unsigned long long* key, const unsigned int* idx, int64_t k, int64_t* oidx,
                                double* oscore) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < k; i += (int64_t)gridDim.x * blockDim.x) {
    oidx[i] = (int64_t)idx[i];
    if (oscore) oscore[i] = key_f64(key[i]);
  }
}

int nnal_k_topk(nnal_ctx* ctx, const double* score, int64_t n, int64_t k, int64_t* d_idx_out, double* d_score_out) {
  if (k > n) k = n;
  if (k <= 0) return NNAL_OK;
  if (n > 0xfffffff0ll) NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "top-k over more than 2^32 scores");
  int64_t kp = 1;
  while (kp < k) kp <<= 1;
  const int TB = 1024;                                       // tie blocks
  size_t need = sizeof(TopkState) + 256 + (size_t)kp * 12 + 256 + TB * 4 + 256;
  NNAL_TRY(devbuf_reserve(ctx, ctx->topk_ws, need));
  char* ws = (char*)ctx->topk_ws.p;
  TopkState* st = (TopkState*)ws;
  unsigned long long* okey = (unsigned long long*)(ws + ((sizeof(TopkState) + 255) / 256) * 256);
  unsigned int* oidx = (unsigned int*)((char*)okey + (size_t)kp * 8);
  unsigned int* counts = (unsigned int*)((char*)oidx + (((size_t)kp * 4 + 255) / 256) * 256);
  cudaStream_t s = ctx->stream;
  int64_t blocks = (n + 255) / 256;
  int grid = (int)(blocks < (int64_t)ctx->sm_count * 8 ? blocks : (int64_t)ctx->sm_count * 8);
  topk_init_kernel<<<1, 256, 0, s>>>(st, (unsigned long long)k);
  for (int shift = 56; shift >= 0; shift -= 8) {
    topk_hist_kernel<<<grid, 256, 0, s>>>(score, n, shift, st);
    topk_pick_kernel<<<1, 256, 0, s>>>(st, shift);
  }
  topk_compact_lt_kernel<<<grid, 256, 0, s>>>(score, n, st, okey, oidx);
  int64_t per_block = (n + TB - 1) / TB;
  per_block = ((per_block + 255) / 256) * 256;
  int nb = (int)((n + per_block - 1) / per_block);
  topk_tie_count_kernel<<<nb, 256, 0, s>>>(score, n, per_block, st, counts);
  topk_tie_scan_kernel<<<1, 32, 0, s>>>(counts, nb);
  topk_tie_emit_kernel<<<nb, 256, 0, s>>>(score, n, per_block, st, counts, (unsigned long long)k, okey, oidx);
  ctx->launches += 21;
  if (kp > k) { topk_pad_kernel<<<cdiv(kp - k, 256) > 1024 ? 1024 : cdiv(kp - k, 256), 256, 0, s>>>(okey, oidx, k, kp); ctx->launches++; }
  // bitonic sort of kp (key, idx) pairs
  if (kp <= BT_TILE) {
    bitonic_smem_kernel<<<1, 1024, 0, s>>>(okey, oidx, kp, 2, kp, 1);
    ctx->launches++;
  } else {
    int ntiles = (int)(kp / BT_TILE);
    bitonic_smem_kernel<<<ntiles, 1024, 0, s>>>(okey, oidx, kp, 2, BT_TILE, 1);
    ctx->launches++;
    for (int64_t kk = BT_TILE * 2; kk <= kp; kk <<= 1) {
      for (int64_t jj = kk >> 1; jj >= BT_TILE; jj >>= 1) {
        int g = (int)((kp / 2 + 255) / 256 < 4096 ? (kp / 2 + 255) / 256 : 4096);
        bitonic_step_kernel<<<g, 256, 0, s>>>(okey, oidx, kp, jj, kk);
        ctx->launches++;
      }
      bitonic_smem_kernel<<<ntiles, 1024, 0, s>>>(okey, oidx, kp, kk, kk, BT_TILE / 2);
      ctx->launches++;
    }
  }
  topk_out_kernel<<<cdiv(k, 256) > 1024 ? 1024 : cdiv(k, 256), 256, 0, s>>>(okey, oidx, k, d_idx_out, d_score_out);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}
