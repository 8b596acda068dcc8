// extern "C" boundary of libnnal_b200 (see include/nnal_b200.h).
#include "nnal_common.cuh"
#include "../../include/nnal_b200.h"
#include <cstdlib>
#include <cmath>
#include <algorithm>
#include <thread>
#include <cstring>

static const int NNAL_VERSION = 100;
static const int64_t DEFAULT_CHUNK = 16384;   // samples per forward chunk (measured: 8192 -> 16384 = +1.5 %, flat beyond)

static int64_t chunk_size(const nnal_ctx* ctx) { return ctx->dbg.chunk > 0 ? ctx->dbg.chunk : DEFAULT_CHUNK; }

// test hook: kernel-selection switches (see DebugOpts).  Unknown names are an error.
extern "C" int nnal_debug_option(nnal_ctx* ctx, const char* name, long value) {
  if (!ctx || !name) return NNAL_ERR_INVALID;
  const std::string n(name);
  DebugOpts& d = ctx->dbg;
  if (n == "chunk") d.chunk = value;
  else if (n == "bw_chunk") d.bw_chunk = value;
  else if (n == "no_fused_gather") d.no_fused_gather = (int)value;
  else if (n == "no_fused_conv1") d.no_fused_conv1 = (int)value;
  else if (n == "wt_flags") d.wt_flags = (int)value;
  else if (n == "sdp_no_coop") d.sdp_no_coop = (int)value;
  else if (n == "bw_no_ws") d.bw_no_ws = (int)value;
  else if (n == "bw_no_tc8") d.bw_no_tc8 = (int)value;
  else if (n == "bw_no_tc") d.bw_no_tc = (int)value;
  else if (n == "bw_simt_fwd") d.bw_simt_fwd = (int)value;
  else if (n == "fi_flags") d.fi_flags = (int)value;
  else if (n == "plain_upload") d.plain_upload = (int)value;
  else if (n == "conv_grid") d.conv_grid = (int)value;
  else if (n == "conv_wt") ctx->use_wt = (int)value;       // 0 conv_tc.cu only, 1 conv_wt.cu where faster, 2 (default) + pool fusion, 3 wherever supported
  else if (n == "conv_x16") ctx->use_x16 = (int)value;     // conv1 on the x-im2col'd input (set BEFORE the weights are uploaded)
  else NNAL_FAIL(ctx, NNAL_ERR_INVALID, "unknown debug option");
  return NNAL_OK;
}

extern "C" int nnal_version(void) { return NNAL_VERSION; }

extern "C" int nnal_device_memory(nnal_ctx* ctx, uint64_t* free_bytes, uint64_t* total_bytes) {
  if (!ctx) return NNAL_ERR_INVALID;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  size_t f = 0, t = 0;
  CUDA_TRY(ctx, cudaMemGetInfo(&f, &t));
  if (free_bytes) *free_bytes = f;
  if (total_bytes) *total_bytes = t;
  return NNAL_OK;
}

// ---- content hash of caller-owned HOST arrays (volumes, weights) -------------------------------------------------
// The host layer skips an upload only when the FULL content of the arrays is unchanged (the reference passes the same
// padded volumes on every query and fine-tunes the weights between queries; a sampled checksum or object identity would
// miss in-place edits).  64-bit multiply-xor hash over 8-byte words, 4 MiB chunks hashed independently on up to 16
// threads and combined in chunk order: the value does not depend on the thread count; ~50 GB/s on the box's host cores.
static uint64_t hash_chunk(const unsigned char* p, size_t n, uint64_t seed) {
  const uint64_t K = 0x9E3779B97F4A7C15ull;
  uint64_t h0 = seed ^ K, h1 = seed + 0xC2B2AE3D27D4EB4Full, h2 = ~seed, h3 = seed * K + 1;
  size_t i = 0;
  for (; i + 32 <= n; i += 32) {
    uint64_t w[4];
    memcpy(w, p + i, 32);
    h0 = (h0 ^ w[0]) * K; h1 = (h1 ^ w[1]) * K; h2 = (h2 ^ w[2]) * K; h3 = (h3 ^ w[3]) * K;
  }
  uint64_t t = 0;
  for (int sh = 0; i < n; ++i, sh = (sh + 8) & 63) t ^= (uint64_t)p[i] << sh;
  uint64_t h = (h0 ^ (h1 >> 29) ^ (h2 << 17) ^ (h3 >> 41) ^ t ^ (uint64_t)n) * K;
  h ^= h >> 32;
  return h * K;
}

extern "C" int nnal_host_hash(const void* data, uint64_t bytes, uint64_t* out) {
  if (!out || (!data && bytes)) return NNAL_ERR_INVALID;
  const size_t CH = (size_t)4 << 20;
  const size_t nch = (size_t)((bytes + CH - 1) / CH);
  std::vector<uint64_t> hs(nch ? nch : 1, 0);
  const unsigned char* p = (const unsigned char*)data;
  auto work = [&](size_t first, size_t step) {
    for (size_t c = first; c < nch; c += step) hs[c] = hash_chunk(p + c * CH, (size_t)std::min<uint64_t>(CH, bytes - c * CH), c + 1);
  };
  unsigned nt = std::thread::hardware_concurrency();
  nt = std::max(1u, std::min(std::min(nt, 16u), (unsigned)std::max<size_t>(nch, 1)));
  if (nt <= 1) work(0, 1);
  else {
    std::vector<std::thread> th;
    for (unsigned t = 0; t < nt; ++t) th.emplace_back(work, (size_t)t, (size_t)nt);
    for (auto& t : th) t.join();
  }
  uint64_t h = 0x1234567ull ^ bytes;
  for (size_t c = 0; c < nch; ++c) h = (h ^ hs[c]) * 0x9E3779B97F4A7C15ull + c;
  *out = h;
  return NNAL_OK;
}

// ---- fp16 range guard (see nnal_common.cuh) ------------------------------------------------------------------
static std::vector<int (*)(unsigned int*)>& ovf_binders() {
  static std::vector<int (*)(unsigned int*)> v;      // function-local: constructed before the first registrar runs
  return v;
}
void nnal_ovf_register(int (*bind)(unsigned int*)) { ovf_binders().push_back(bind); }

static int ovf_bind_device(nnal_ctx* ctx) {
  static unsigned int* words[64] = {nullptr};        // one flag word per device, shared by its contexts, never freed
  if (ctx->device < 0 || ctx->device >= 64) return NNAL_ERR_NO_DEVICE;
  if (!words[ctx->device]) {
    unsigned int* w = nullptr;
    if (cudaMalloc(&w, 256) != cudaSuccess || cudaMemset(w, 0, 256) != cudaSuccess) return NNAL_ERR_CUDA;
    for (auto bind : ovf_binders())
      if (bind(w) != 0) return NNAL_ERR_CUDA;
    words[ctx->device] = w;
  }
  ctx->ovf_word = words[ctx->device];
  if (cudaMallocHost(&ctx->ovf_host, 64) != cudaSuccess) return NNAL_ERR_CUDA;
  *ctx->ovf_host = 0;
  return NNAL_OK;
}

int nnal_ovf_enqueue(nnal_ctx* ctx) {
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->ovf_host, ctx->ovf_word, 4, cudaMemcpyDeviceToHost, ctx->stream));
  return NNAL_OK;
}
int nnal_ovf_test(nnal_ctx* ctx) {
  if (*ctx->ovf_host == 0) return NNAL_OK;
  *ctx->ovf_host = 0;
  CUDA_TRY(ctx, cudaMemsetAsync(ctx->ovf_word, 0, 4, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  NNAL_FAIL(ctx, NNAL_ERR_OVERFLOW, "an input, weight or activation left the fp16 operand range (|x| > 65504 or not finite): the "
                                    "tensor-core path would saturate it; rescale the input or call nnal_set_tensor_cores(ctx, 0)");
}

extern "C" int nnal_ctx_create(int device, nnal_ctx** out) {
  if (!out) return NNAL_ERR_INVALID;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) return NNAL_ERR_NO_DEVICE;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return NNAL_ERR_NO_DEVICE;
  if (prop.major != 10) return NNAL_ERR_NO_DEVICE;     // sm_100a kernels only
  if (cudaSetDevice(device) != cudaSuccess) return NNAL_ERR_NO_DEVICE;
  nnal_ctx* ctx = new nnal_ctx();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return NNAL_ERR_CUDA; }
  if (ovf_bind_device(ctx) != NNAL_OK) { cudaStreamDestroy(ctx->stream); delete ctx; return NNAL_ERR_CUDA; }
  ctx->use_tc = 1;
  ctx->use_wt = 2;                       // conv_wt.cu where it is the faster kernel, with the fused max-pool
  ctx->use_x16 = 0;                      // measured: conv1 4.2 -> 3.2 ms but the gather writes twice the bytes (0.84 -> 1.6 ms): off
  *out = ctx;
  return NNAL_OK;
}

static void free_layers(nnal_ctx* ctx) {
  for (auto& L : ctx->layers) {
    if (L.W) cudaFree(L.W);
    if (L.b) cudaFree(L.b);
    if (L.Wh) cudaFree(L.Wh);
    if (L.Wl) cudaFree(L.Wl);
    if (L.Wt) cudaFree(L.Wt);
    if (L.Wx) cudaFree(L.Wx);
  }
  ctx->layers.clear();
}
static void upload_stage_release(nnal_ctx* ctx);
int nnal_p2p_release(nnal_ctx* ctx);       // p2p.cu
static void free_buf(DevBuf& b) { if (b.p) cudaFree(b.p); b.p = nullptr; b.cap = 0; }
static void free_pool(nnal_ctx* ctx) {
  if (ctx->pool_post) cudaFree(ctx->pool_post);
  if (ctx->pool_score) cudaFree(ctx->pool_score);
  if (ctx->pool_mc_post) cudaFree(ctx->pool_mc_post);
  if (ctx->pool_mc_ent) cudaFree(ctx->pool_mc_ent);
  ctx->pool_mc_post = ctx->pool_mc_ent = nullptr; ctx->pool_cap_mc = 0;
  if (ctx->pool_feat) cudaFree(ctx->pool_feat);
  if (ctx->pool_prev) cudaFree(ctx->pool_prev);
  ctx->pool_post = nullptr; ctx->pool_score = nullptr; ctx->pool_feat = nullptr; ctx->pool_prev = nullptr;
  ctx->pool_n = 0; ctx->pool_cap_n = 0; ctx->pool_cap_score = 0; ctx->pool_cap_nfeat = 0; ctx->pool_cap_nprev = 0;
}

extern "C" int nnal_volume_clear(nnal_ctx* ctx) {
  if (!ctx) return NNAL_ERR_INVALID;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  for (auto& v : ctx->vols) if (v.data) cudaFree(v.data);
  ctx->vols.clear();
  return NNAL_OK;
}

int nnal_fi_release(nnal_ctx* ctx);
int nnal_fi_block_release(nnal_ctx* ctx);
int nnal_sims_release(nnal_ctx* ctx);

extern "C" int nnal_ctx_destroy(nnal_ctx* ctx) {
  if (!ctx) return NNAL_OK;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  nnal_volume_clear(ctx);
  free_layers(ctx);
  free_pool(ctx);
  nnal_fi_release(ctx);
  nnal_fi_block_release(ctx);
  nnal_sims_release(ctx);
  nnal_bw_release(ctx);
  nnal_sdp_release(ctx);
  nnal_tc_release(ctx);
  upload_stage_release(ctx);
  nnal_p2p_release(ctx);
  free_buf(ctx->stage); free_buf(ctx->inds); free_buf(ctx->act[0]); free_buf(ctx->act[1]); free_buf(ctx->xin);
  free_buf(ctx->featbuf); free_buf(ctx->prevbuf); free_buf(ctx->logits); free_buf(ctx->splitA[0]); free_buf(ctx->splitA[1]);
  free_buf(ctx->head_logits);
  free_buf(ctx->topk_ws); free_buf(ctx->fi_ws);
  cudaStreamDestroy(ctx->stream);
  if (ctx->ovf_host) cudaFreeHost(ctx->ovf_host);
  delete ctx;
  return NNAL_OK;
}

extern "C" const char* nnal_last_error(nnal_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }
extern "C" long long nnal_launch_count(nnal_ctx* ctx) { return ctx ? ctx->launches : 0; }
extern "C" int nnal_set_tensor_cores(nnal_ctx* ctx, int enable) { if (!ctx) return NNAL_ERR_INVALID; ctx->use_tc = enable ? 1 : 0; return NNAL_OK; }
extern "C" void* nnal_stream(nnal_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
extern "C" int nnal_synchronize(nnal_ctx* ctx) {
  if (!ctx) return NNAL_ERR_INVALID;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return NNAL_OK;
}

bool nnal_layer_on_tc(const nnal_ctx* ctx, int i);

extern "C" int nnal_profile(nnal_ctx* ctx, int enable) {
  if (!ctx) return NNAL_ERR_INVALID;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  for (auto& r : ctx->prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  ctx->prof.clear();
  ctx->profile = enable ? 1 : 0;
  return NNAL_OK;
}

extern "C" int nnal_profile_read(nnal_ctx* ctx, int cls, double* total_ms, long long* count) {
  if (!ctx || !total_ms || !count) return NNAL_ERR_INVALID;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  double t = 0; long long c = 0;
  for (auto& r : ctx->prof) {
    if (r.cls != cls) continue;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) { t += ms; ++c; }
  }
  *total_ms = t; *count = c;
  return NNAL_OK;
}

extern "C" int nnal_model_layer_info(nnal_ctx* ctx, int layer, int* type, long long* macs_per_sample, int* uses_tc) {
  if (!ctx || layer < 0 || layer >= (int)ctx->layers.size()) return NNAL_ERR_INVALID;
  const Layer& L = ctx->layers[layer];
  if (type) *type = L.type;
  long long macs = 0;
  if (L.type == NNAL_LAYER_CONV) macs = (long long)L.out_h * L.out_w * L.out_c * L.kh * L.kw * L.in_c;
  else if (L.type == NNAL_LAYER_FC) macs = (long long)L.in_dim * L.out_dim;
  if (macs_per_sample) *macs_per_sample = macs;
  if (uses_tc) {
    *uses_tc = nnal_layer_on_tc(ctx, layer) ? 1 : 0;
    // 2: the weight-stationary tcgen05 conv kernel (conv_wt.cu) -- same choice as the forward driver makes
    if (*uses_tc && L.type == NNAL_LAYER_CONV &&
        (ctx->use_wt >= 3 ? nnal_wt_conv_supported(ctx, L) : ctx->use_wt >= 1 && nnal_wt_conv_preferred(ctx, L)))
      *uses_tc = 2;
  }
  return NNAL_OK;
}

// ---------------------------------------------------------------------------------------------
// model
// ---------------------------------------------------------------------------------------------
extern "C" int nnal_model_set(nnal_ctx* ctx, const nnal_layer_spec* specs, int n_layers, int in_h, int in_w, int in_c,
                              int feature_layer) {
  if (!ctx || !specs || n_layers <= 0 || in_h <= 0 || in_w <= 0 || in_c <= 0) return NNAL_ERR_INVALID;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  free_layers(ctx);
  ctx->weights_version++;
  ctx->in_h = in_h; ctx->in_w = in_w; ctx->in_c = in_c;
  int H = in_h, W = in_w, C = in_c;
  int flat = 0;            // >0 once flattened: current vector length
  ctx->fc_first = -1;
  for (int i = 0; i < n_layers; ++i) {
    Layer L;
    L.type = specs[i].type;
    if (L.type == NNAL_LAYER_CONV) {
      if (flat) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "conv layer after an fc layer");
      if (specs[i].kh <= 0 || specs[i].kw <= 0 || !(specs[i].kh & 1) || !(specs[i].kw & 1) || specs[i].out <= 0)
        NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "conv kernels must be odd-sized (SAME, stride 1)");
      L.kh = specs[i].kh; L.kw = specs[i].kw;
      L.in_h = H; L.in_w = W; L.in_c = C;
      L.out_h = H; L.out_w = W; L.out_c = specs[i].out;
      L.relu = 1;
      C = L.out_c;
    } else if (L.type == NNAL_LAYER_POOL) {
      if (flat) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "pool layer after an fc layer");
      if (specs[i].kh <= 0 || specs[i].kh != specs[i].kw) NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "pool window must be square");
      L.kh = L.kw = specs[i].kh;
      L.in_h = H; L.in_w = W; L.in_c = C;
      L.out_h = (H + L.kh - 1) / L.kh; L.out_w = (W + L.kw - 1) / L.kw; L.out_c = C;
      // tf.nn.max_pool SAME: the pad_total = out*s - in missing cells are split, the smaller half BEFORE the first
      // row / column (nonzero only when s >= 3 leaves two or more cells over)
      L.pad_t = (L.out_h * L.kh - H) / 2; L.pad_l = (L.out_w * L.kw - W) / 2;
      H = L.out_h; W = L.out_w;
    } else if (L.type == NNAL_LAYER_FC) {
      if (specs[i].out <= 0) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "fc layer needs out > 0");
      if (!flat) { flat = H * W * C; ctx->fc_first = i; L.in_h = H; L.in_w = W; L.in_c = C; }
      L.in_dim = flat;
      L.out_dim = specs[i].out;
      L.relu = (i != n_layers - 1);
      flat = L.out_dim;
    } else {
      NNAL_FAIL(ctx, NNAL_ERR_INVALID, "Layer's type should be either 'fc', 'conv' or 'pool'.");
    }
    ctx->layers.push_back(L);
  }
  if (ctx->layers.back().type != NNAL_LAYER_FC) NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "last layer must be fc");
  ctx->n_class = ctx->layers.back().out_dim;
  if (feature_layer < 0) feature_layer = n_layers - 2;
  ctx->feature_layer = feature_layer;
  ctx->feat_dim = 0; ctx->prev_dim = 0;
  if (feature_layer >= 0 && feature_layer < n_layers - 1 && ctx->layers[feature_layer].type == NNAL_LAYER_FC) {
    ctx->feat_dim = ctx->layers[feature_layer].out_dim;
    ctx->prev_dim = ctx->layers[feature_layer].in_dim;
  }
  return NNAL_OK;
}

extern "C" int nnal_model_info(nnal_ctx* ctx, int* n_class, int* feat_dim, int* prev_dim) {
  if (!ctx || ctx->layers.empty()) return NNAL_ERR_STATE;
  if (n_class) *n_class = ctx->n_class;
  if (feat_dim) *feat_dim = ctx->feat_dim;
  if (prev_dim) *prev_dim = ctx->prev_dim;
  return NNAL_OK;
}

// power-of-two scale that lifts max|W| to [2^13, 2^14): fp16 hi terms stay far from overflow and the
// lo terms (2^-11 of hi) stay out of the subnormal range for all but negligible weights
void nnal_set_weight_scale(Layer& L, const float* W, size_t n) {
  float mx = 0.f;
  for (size_t i = 0; i < n; ++i) { float a = fabsf(W[i]); if (a > mx && a < 3.0e38f) mx = a; }
  int e = 0;
  if (mx > 0.f) { int ex; frexpf(mx, &ex); e = 14 - ex; }       // mx = f * 2^ex, f in [0.5,1)
  if (e > 24) e = 24;
  if (e < -24) e = -24;
  L.w_scale = ldexpf(1.f, e);
  L.w_scale_inv = ldexpf(1.f, -e);
}

extern "C" int nnal_model_set_weights(nnal_ctx* ctx, int layer, const float* W, const float* b) {
  if (!ctx || !W || !b) return NNAL_ERR_INVALID;
  if (layer < 0 || layer >= (int)ctx->layers.size()) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "layer index out of range");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  Layer& L = ctx->layers[layer];
  size_t wn, bn;
  if (L.type == NNAL_LAYER_CONV) { wn = (size_t)L.kh * L.kw * L.in_c * L.out_c; bn = L.out_c; }
  else if (L.type == NNAL_LAYER_FC) { wn = (size_t)L.in_dim * L.out_dim; bn = L.out_dim; }
  else NNAL_FAIL(ctx, NNAL_ERR_INVALID, "pool layers have no weights");
  if (!L.W) CUDA_TRY(ctx, cudaMalloc(&L.W, wn * sizeof(float)));
  if (!L.b) CUDA_TRY(ctx, cudaMalloc(&L.b, bn * sizeof(float)));
  CUDA_TRY(ctx, cudaMemcpyAsync(L.b, b, bn * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  if (L.type == NNAL_LAYER_FC && layer == ctx->fc_first && L.in_h * L.in_w > 1) {
    NNAL_TRY(devbuf_reserve(ctx, ctx->stage, wn * sizeof(float)));
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->stage.p, W, wn * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    NNAL_TRY(nnal_k_permute_fc_weight(ctx, (const float*)ctx->stage.p, L.W, L.out_dim, L.in_c, L.in_h, L.in_w));
  } else {
    CUDA_TRY(ctx, cudaMemcpyAsync(L.W, W, wn * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  }
  L.has_weights = true;
  ctx->weights_version++;
  nnal_set_weight_scale(L, W, wn);
  NNAL_TRY(nnal_tc_prepare_layer(ctx, L));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return NNAL_OK;
}

// ---------------------------------------------------------------------------------------------
// host -> device copies of large PAGEABLE arrays (what np.pad hands the reference's callers): the driver's own staging
// moves them at ~9 GB/s on this box (one thread), a pinned source at 51 GB/s.  Here T host threads copy 4 MB pieces into
// their own pinned double buffers and issue the DMA of each piece on their own stream, so the link, not one core's memcpy,
// is the bound.  Pinned (or registered) sources take the plain cudaMemcpyAsync path.
// ---------------------------------------------------------------------------------------------
struct UploadStage {
  static constexpr int T = 8, SLOTS = 2;
  static constexpr size_t PIECE = (size_t)4 << 20;
  unsigned char* pinned = nullptr;             // [T][SLOTS][PIECE]
  cudaStream_t streams[T] = {};
  cudaEvent_t ev[T][SLOTS] = {};
};
struct H2DSeg { void* dst; const void* src; size_t bytes; };

static void upload_stage_release(nnal_ctx* ctx) {
  UploadStage* u = (UploadStage*)ctx->upload_state;
  if (!u) return;
  for (int t = 0; t < UploadStage::T; ++t) {
    if (u->streams[t]) cudaStreamDestroy(u->streams[t]);
    for (int s = 0; s < UploadStage::SLOTS; ++s) if (u->ev[t][s]) cudaEventDestroy(u->ev[t][s]);
  }
  if (u->pinned) cudaFreeHost(u->pinned);
  delete u;
  ctx->upload_state = nullptr;
}

static bool host_ptr_is_pageable(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return true; }
  return a.type == cudaMemoryTypeUnregistered;
}

// copies every segment into device memory; returns with all copies COMPLETE or enqueued on ctx->stream
static int h2d_segments(nnal_ctx* ctx, const std::vector<H2DSeg>& segs) {
  size_t total = 0;
  bool pageable = false;
  for (const H2DSeg& s : segs) { total += s.bytes; pageable = pageable || host_ptr_is_pageable(s.src); }
  unsigned hw = std::thread::hardware_concurrency();
  const int nt = (int)std::max(1u, std::min(hw ? hw : 1u, (unsigned)UploadStage::T));
  if (!pageable || total < 4 * UploadStage::PIECE || nt < 2 || ctx->dbg.plain_upload) {
    for (const H2DSeg& s : segs) CUDA_TRY(ctx, cudaMemcpyAsync(s.dst, s.src, s.bytes, cudaMemcpyHostToDevice, ctx->stream));
    return NNAL_OK;
  }
  UploadStage* u = (UploadStage*)ctx->upload_state;
  if (!u) {
    u = new UploadStage();
    ctx->upload_state = u;
    CUDA_TRY(ctx, cudaHostAlloc((void**)&u->pinned, (size_t)UploadStage::T * UploadStage::SLOTS * UploadStage::PIECE, cudaHostAllocDefault));
    for (int t = 0; t < UploadStage::T; ++t) {
      CUDA_TRY(ctx, cudaStreamCreateWithFlags(&u->streams[t], cudaStreamNonBlocking));
      for (int s = 0; s < UploadStage::SLOTS; ++s) CUDA_TRY(ctx, cudaEventCreateWithFlags(&u->ev[t][s], cudaEventDisableTiming));
    }
  }
  // the destination may still be read by work queued on the library's stream (the previous subject's re-layout)
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  std::vector<H2DSeg> pieces;
  for (const H2DSeg& s : segs)
    for (size_t o = 0; o < s.bytes; o += UploadStage::PIECE)
      pieces.push_back({(char*)s.dst + o, (const char*)s.src + o, std::min(UploadStage::PIECE, s.bytes - o)});
  std::vector<cudaError_t> errs(nt, cudaSuccess);
  auto work = [&](int t) {
    cudaError_t e = cudaSetDevice(ctx->device);
    int used = 0;
    for (size_t c = t; c < pieces.size() && e == cudaSuccess; c += nt, ++used) {
      const int s = used % UploadStage::SLOTS;
      unsigned char* slot = u->pinned + ((size_t)t * UploadStage::SLOTS + s) * UploadStage::PIECE;
      if (used >= UploadStage::SLOTS) e = cudaEventSynchronize(u->ev[t][s]);       // the slot's previous DMA has drained
      if (e != cudaSuccess) break;
      memcpy(slot, pieces[c].src, pieces[c].bytes);
      e = cudaMemcpyAsync(pieces[c].dst, slot, pieces[c].bytes, cudaMemcpyHostToDevice, u->streams[t]);
      if (e == cudaSuccess) e = cudaEventRecord(u->ev[t][s], u->streams[t]);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(u->streams[t]);
    errs[t] = e;
  };
  std::vector<std::thread> th;
  for (int t = 1; t < nt; ++t) th.emplace_back(work, t);
  work(0);
  for (auto& t : th) t.join();
  for (int t = 0; t < nt; ++t)
    if (errs[t] != cudaSuccess) { ctx->err = std::string("staged host->device copy: ") + cudaGetErrorString(errs[t]); return NNAL_ERR_CUDA; }
  return NNAL_OK;
}

// ---------------------------------------------------------------------------------------------
// volumes
// ---------------------------------------------------------------------------------------------
static int volume_finish(nnal_ctx* ctx, Volume& v, const void* d_stage, int m, int dtype, int64_t X, int64_t Y, int64_t Z,
                         int64_t px, int64_t py, int64_t pz, size_t out_bytes) {
  if (v.bytes < out_bytes) {
    if (v.data) { CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream)); CUDA_TRY(ctx, cudaFree(v.data)); v.data = nullptr; }
    CUDA_TRY(ctx, cudaMalloc(&v.data, out_bytes));
    v.bytes = out_bytes;
  }
  v.m = m; v.X = X + 2 * px; v.Y = Y + 2 * py; v.Z = Z + 2 * pz; v.dtype = dtype;
  NNAL_TRY(nnal_k_relayout(ctx, d_stage, dtype, m, X, Y, Z, px, py, pz, v.data));
  return NNAL_OK;
}

extern "C" int nnal_volume_set(nnal_ctx* ctx, int subject, int m, const void* const* mods, int dtype, int64_t X, int64_t Y,
                               int64_t Z, int64_t px, int64_t py, int64_t pz) {
  if (!ctx || !mods || m <= 0 || subject < 0 || X <= 0 || Y <= 0 || Z <= 0 || px < 0 || py < 0 || pz < 0) return NNAL_ERR_INVALID;
  if (dtype != NNAL_F32 && dtype != NNAL_F64) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "volume dtype must be NNAL_F32 or NNAL_F64");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if ((int)ctx->vols.size() <= subject) ctx->vols.resize(subject + 1);
  Volume& v = ctx->vols[subject];
  size_t esz = dtype == NNAL_F64 ? 8 : 4;
  size_t in_elems = (size_t)X * Y * Z;
  size_t out_bytes = (size_t)(X + 2 * px) * (Y + 2 * py) * (Z + 2 * pz) * m * esz;
  NNAL_TRY(devbuf_reserve(ctx, ctx->stage, in_elems * m * esz));
  std::vector<H2DSeg> segs;
  for (int j = 0; j < m; ++j) {
    if (!mods[j]) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "null modality pointer");
    segs.push_back({(char*)ctx->stage.p + (size_t)j * in_elems * esz, mods[j], in_elems * esz});
  }
  NNAL_TRY(h2d_segments(ctx, segs));
  return volume_finish(ctx, v, ctx->stage.p, m, dtype, X, Y, Z, px, py, pz, out_bytes);
}

// Same, with the m modality arrays already in DEVICE memory (d_stage: m consecutive C-contiguous (X,Y,Z) arrays).  Used
// by the multi-GPU host layer: every rank copies 1/world of each volume over PCIe and the parts are all-gathered over
// NVLink (NCCL, on nnal_stream()) instead of every rank pulling the same volume through its own PCIe link.
extern "C" int nnal_volume_set_device(nnal_ctx* ctx, int subject, int m, const void* d_stage, int dtype, int64_t X, int64_t Y,
                                      int64_t Z, int64_t px, int64_t py, int64_t pz) {
  if (!ctx || !d_stage || m <= 0 || subject < 0 || X <= 0 || Y <= 0 || Z <= 0 || px < 0 || py < 0 || pz < 0) return NNAL_ERR_INVALID;
  if (dtype != NNAL_F32 && dtype != NNAL_F64) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "volume dtype must be NNAL_F32 or NNAL_F64");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if ((int)ctx->vols.size() <= subject) ctx->vols.resize(subject + 1);
  Volume& v = ctx->vols[subject];
  const size_t esz = dtype == NNAL_F64 ? 8 : 4;
  const size_t out_bytes = (size_t)(X + 2 * px) * (Y + 2 * py) * (Z + 2 * pz) * m * esz;
  return volume_finish(ctx, v, d_stage, m, dtype, X, Y, Z, px, py, pz, out_bytes);
}

static int check_gather_args(nnal_ctx* ctx, int subject, int64_t n, int d1, int d2, int d3, const Volume** vout) {
  if (subject < 0 || subject >= (int)ctx->vols.size() || !ctx->vols[subject].data)
    NNAL_FAIL(ctx, NNAL_ERR_STATE, "subject volume not set");
  const Volume& v = ctx->vols[subject];
  if (n < 0 || d1 <= 0 || d2 <= 0 || d3 <= 0 || !(d1 & 1) || !(d2 & 1) || !(d3 & 1))
    NNAL_FAIL(ctx, NNAL_ERR_INVALID, "patch shape must be odd and positive");
  if (v.X - (d1 - 1) <= 0 || v.Y - (d2 - 1) <= 0 || v.Z - (d3 - 1) <= 0)
    NNAL_FAIL(ctx, NNAL_ERR_INVALID, "patch larger than padded volume");
  *vout = &v;
  return NNAL_OK;
}

// Uploads the per-modality normalisation table [m][3] = (mu, sigma, y): y = RN(1/sigma) drives the
// correctly-rounded Markstein division of the gather kernels; y = NaN makes them fall back to a true division
// (sigma zero / non-finite, or a significand of all ones, where the Markstein sequence is not proven).
static int upload_stats(nnal_ctx* ctx, const double* stats, int m, int norm_mode, double** d_stats) {
  *d_stats = nullptr;
  if (norm_mode == NNAL_NORM_NONE) return NNAL_OK;
  if (!stats) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "normalisation requested without stats");
  if ((size_t)m * 3 * sizeof(double) > 4096) NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "too many modalities");
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));       // earlier async copies from stats_host must be done before it is rewritten
  ctx->stats_host.resize((size_t)m * 3);
  for (int j = 0; j < m; ++j) {
    const double mu = stats[2 * j], sg = stats[2 * j + 1];
    uint64_t bits;
    memcpy(&bits, &sg, 8);
    const bool ok = std::isfinite(sg) && sg != 0.0 && (bits & 0xfffffffffffffull) != 0xfffffffffffffull;
    ctx->stats_host[3 * j] = mu;
    ctx->stats_host[3 * j + 1] = sg;
    ctx->stats_host[3 * j + 2] = ok ? 1.0 / sg : std::nan("");
  }
  NNAL_TRY(devbuf_reserve(ctx, ctx->logits, 4096));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->logits.p, ctx->stats_host.data(), (size_t)m * 3 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  *d_stats = (double*)ctx->logits.p;
  return NNAL_OK;
}

int nnal_upload_stats(nnal_ctx* ctx, const double* stats, int m, int norm_mode, double** d_stats) {
  return upload_stats(ctx, stats, m, norm_mode, d_stats);
}
int nnal_check_gather_args(nnal_ctx* ctx, int subject, int64_t n, int d1, int d2, int d3, const Volume** vout) {
  return check_gather_args(ctx, subject, n, d1, d2, d3, vout);
}

extern "C" int nnal_gather(nnal_ctx* ctx, int subject, const int64_t* inds, int64_t n, int d1, int d2, int d3,
                           const double* stats, int norm_mode, double* out) {
  if (!ctx) return NNAL_ERR_INVALID;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const Volume* v;
  NNAL_TRY(check_gather_args(ctx, subject, n, d1, d2, d3, &v));
  if (n == 0) return NNAL_OK;
  if (!inds || !out) return NNAL_ERR_INVALID;
  double* d_stats;
  NNAL_TRY(upload_stats(ctx, stats, v->m, norm_mode, &d_stats));
  const int64_t per = (int64_t)d1 * d2 * d3 * v->m;
  const int64_t chunk = std::max<int64_t>(1, std::min<int64_t>(n, (int64_t)(1ll << 28) / (per * 8)));   // <= 256 MiB staging
  NNAL_TRY(devbuf_reserve(ctx, ctx->inds, (size_t)chunk * 8));
  NNAL_TRY(devbuf_reserve(ctx, ctx->act[0], (size_t)chunk * per * 8));
  for (int64_t o = 0; o < n; o += chunk) {
    int64_t nb = std::min(chunk, n - o);
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->inds.p, inds + o, (size_t)nb * 8, cudaMemcpyHostToDevice, ctx->stream));
    NNAL_TRY(nnal_k_gather_f64(ctx, *v, (const int64_t*)ctx->inds.p, nb, d1, d2, d3, d_stats, norm_mode, (double*)ctx->act[0].p));
    CUDA_TRY(ctx, cudaMemcpyAsync(out + o * per, ctx->act[0].p, (size_t)nb * per * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  }
  return NNAL_OK;
}

// device-resident variants (memory-bound path of config 4: full-volume patch gather, pixel-wise entropy map)
extern "C" int nnal_gather_device_f32(nnal_ctx* ctx, int subject, const int64_t* d_inds, int64_t n, int d1, int d2, int d3,
                                      const double* stats, int norm_mode, float* d_out) {
  if (!ctx) return NNAL_ERR_INVALID;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const Volume* v;
  NNAL_TRY(check_gather_args(ctx, subject, n, d1, d2, d3, &v));
  if (n == 0) return NNAL_OK;
  if (!d_inds || !d_out) return NNAL_ERR_INVALID;
  double* d_stats;
  NNAL_TRY(upload_stats(ctx, stats, v->m, norm_mode, &d_stats));
  prof_begin(ctx, NNAL_PROF_GATHER);
  int rc = nnal_k_gather_norm_f32(ctx, *v, d_inds, n, d1, d2, d3, d_stats, norm_mode, d_out);
  prof_end(ctx);
  return rc;
}

extern "C" int nnal_entropy_device_f32(nnal_ctx* ctx, const float* d_post, int c, int64_t n, double eps, float* d_out) {
  if (!ctx || c <= 0 || n < 0) return NNAL_ERR_INVALID;
  if (n == 0) return NNAL_OK;
  if (!d_post || !d_out) return NNAL_ERR_INVALID;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  prof_begin(ctx, NNAL_PROF_SCORE);
  int rc = nnal_k_entropy_f32(ctx, d_post, c, n, (float)eps, d_out);
  prof_end(ctx);
  return rc;
}

// ---------------------------------------------------------------------------------------------
// pool pass
// ---------------------------------------------------------------------------------------------
// MC-dropout and committee statistics: c = 2 keeps the binary running means (P(class 1), PW_NNAL.py:80); 3 <= c <= 32
// and c >= 64 keep the running mean of every class.  33 <= c <= 63 has no head (nnal_k_head).
static int check_mc_classes(nnal_ctx* ctx) {
  const int c = ctx->n_class;
  if (c < 2 || (c > 32 && c < NNAL_WIDE_HEAD_MIN))
    NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "MC-dropout and committee scores need 2 to 32 or at least 64 classes");
  return NNAL_OK;
}
// Running-mean storage for n pool samples; free_pool resets the capacity when the class count changes.
static int reserve_mc(nnal_ctx* ctx, int64_t n) {
  if ((size_t)n <= ctx->pool_cap_mc) return NNAL_OK;
  const size_t rows = ctx->n_class == 2 ? 1 : (size_t)ctx->n_class;
  if (ctx->pool_mc_post) { CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream)); cudaFree(ctx->pool_mc_post); cudaFree(ctx->pool_mc_ent); }
  ctx->pool_mc_post = ctx->pool_mc_ent = nullptr;
  ctx->pool_cap_mc = 0;
  CUDA_TRY(ctx, cudaMalloc(&ctx->pool_mc_post, (size_t)n * rows * sizeof(double)));
  CUDA_TRY(ctx, cudaMalloc(&ctx->pool_mc_ent, (size_t)n * sizeof(double)));
  ctx->pool_cap_mc = (size_t)n;
  return NNAL_OK;
}

extern "C" int nnal_pool_begin(nnal_ctx* ctx, int64_t n_total, int keep) {
  if (!ctx || n_total < 0 || keep < 0 || keep > 2) return NNAL_ERR_INVALID;
  if (ctx->layers.empty()) NNAL_FAIL(ctx, NNAL_ERR_STATE, "model not set");
  for (auto& L : ctx->layers)
    if (L.type != NNAL_LAYER_POOL && !L.has_weights) NNAL_FAIL(ctx, NNAL_ERR_STATE, "weights not set for every layer");
  if (keep > 0 && ctx->feat_dim == 0) NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "feature layer must be an fc layer before the last");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  // Every pool array has its own grow-only capacity, so alternating rounds of different shape (a large
  // posterior-only pass, then a small candidate pass that keeps the FC factors) never re-allocate.
  const size_t n = (size_t)std::max<int64_t>(n_total, 1);
  if (ctx->pool_cap_class != ctx->n_class || ctx->pool_cap_feat != ctx->feat_dim || ctx->pool_cap_prev != ctx->prev_dim) {
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    free_pool(ctx);
    ctx->pool_cap_class = ctx->n_class; ctx->pool_cap_feat = ctx->feat_dim; ctx->pool_cap_prev = ctx->prev_dim;
  }
  auto grow = [&](void** p, size_t& cap, size_t elem_bytes) -> int {
    if (*p && cap >= n) return NNAL_OK;
    if (*p) { CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream)); CUDA_TRY(ctx, cudaFree(*p)); *p = nullptr; cap = 0; }
    CUDA_TRY(ctx, cudaMalloc(p, n * elem_bytes));
    cap = n;
    return NNAL_OK;
  };
  NNAL_TRY(grow((void**)&ctx->pool_post, ctx->pool_cap_n, (size_t)ctx->n_class * sizeof(float)));
  NNAL_TRY(grow((void**)&ctx->pool_score, ctx->pool_cap_score, sizeof(double)));
  if (keep >= 1) NNAL_TRY(grow((void**)&ctx->pool_feat, ctx->pool_cap_nfeat, (size_t)ctx->feat_dim * sizeof(float)));
  if (keep >= 2) NNAL_TRY(grow((void**)&ctx->pool_prev, ctx->pool_cap_nprev, (size_t)ctx->prev_dim * sizeof(float)));
  if (ctx->mc_T > 0) {
    if (keep != 0) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "MC-dropout passes do not keep features");
    NNAL_TRY(check_mc_classes(ctx));
    NNAL_TRY(reserve_mc(ctx, n_total));
  }
  if (!ctx->ens_open) ctx->mc_have = ctx->mc_T > 0;
  ctx->pool_n = n_total;
  ctx->keep = keep;
  return NNAL_OK;
}

// MC-dropout configuration for the following nnal_pool_begin / nnal_pool_eval* calls (T = 0 switches it off).
// layers: indices of the layers whose output is dropped out (model.dropout_layers); they must be FC layers.
extern "C" int nnal_pool_mc_config(nnal_ctx* ctx, int T, double keep_prob, unsigned long long seed, unsigned int first_pass,
                                   long long pos0, const int* layers, int n_layers) {
  if (!ctx || T < 0) return NNAL_ERR_INVALID;
  ctx->mc_T = 0;
  if (T == 0) return NNAL_OK;
  if (!(keep_prob > 0.0 && keep_prob <= 1.0) || n_layers < 0 || (n_layers > 0 && !layers)) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "keep_prob must be in (0, 1]");
  if (ctx->fc_first < 0) NNAL_FAIL(ctx, NNAL_ERR_STATE, "model not set");
  NNAL_TRY(check_mc_classes(ctx));
  for (int j = ctx->fc_first; j < (int)ctx->layers.size() - 1; ++j)
    if (!nnal_layer_on_tc(ctx, j))
      NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "MC-dropout: the hidden FC layers must run on the tensor-core path");
  ctx->mc_sites.clear();
  for (int i = 0; i < n_layers; ++i) {
    if (layers[i] < ctx->fc_first || layers[i] >= (int)ctx->layers.size())
      NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "dropout sites must be FC layers (the conv trunk is evaluated once)");
    ctx->mc_sites.push_back(layers[i]);
    // a wide head drops out its logits in the tensor-core GEMM's epilogue
    if (layers[i] == (int)ctx->layers.size() - 1 && ctx->n_class >= NNAL_WIDE_HEAD_MIN && !nnal_layer_on_tc(ctx, layers[i]))
      NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "MC-dropout on the logits of a head with 64 or more classes needs the tensor-core path");
  }
  DropSpec d;
  d.keep = (float)keep_prob;
  // keep_prob == 1: tf.nn.dropout is the identity; thresh 0 = off
  d.thresh = keep_prob >= 1.0 ? 0u : (uint32_t)(keep_prob * 4294967296.0);
  d.k0 = (uint32_t)(seed & 0xffffffffull);
  d.k1 = (uint32_t)(seed >> 32);
  d.pass = first_pass;
  d.row0 = pos0;
  ctx->mc_drop = d;
  ctx->mc_T = T;
  return NNAL_OK;
}

// Committee scorers ('ensemble', 'QBC-JS'; PW_NNAL.py:453-545): member t's DETERMINISTIC pool pass (current posteriors)
// is folded into the same float64 running means the MC-dropout passes use:  av = (x + t * av) / (t + 1).
// t = 0 opens the accumulation, nnal_pool_ensemble_end closes it; every member must score the same pool.
extern "C" int nnal_pool_ensemble_accumulate(nnal_ctx* ctx, int t) {
  if (!ctx || t < 0) return NNAL_ERR_INVALID;
  if (!ctx->pool_post || ctx->pool_n <= 0) NNAL_FAIL(ctx, NNAL_ERR_STATE, "no pool pass");
  NNAL_TRY(check_mc_classes(ctx));
  if (t > 0 && !ctx->ens_open) NNAL_FAIL(ctx, NNAL_ERR_STATE, "committee accumulation starts with member 0");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if ((size_t)ctx->pool_n > ctx->pool_cap_mc) {
    if (t > 0) NNAL_FAIL(ctx, NNAL_ERR_STATE, "committee members must score the same pool");
    NNAL_TRY(reserve_mc(ctx, ctx->pool_n));
  }
  prof_begin(ctx, NNAL_PROF_MC_ACCUM);
  NNAL_TRY(nnal_k_mc_accumulate(ctx, ctx->pool_post, ctx->n_class, ctx->pool_n, 0, ctx->pool_n, t, ctx->pool_mc_post,
                                ctx->pool_mc_ent));
  prof_end(ctx);
  ctx->ens_open = 1;
  ctx->mc_have = 1;
  return NNAL_OK;
}
extern "C" int nnal_pool_ensemble_end(nnal_ctx* ctx) {
  if (!ctx) return NNAL_ERR_INVALID;
  ctx->ens_open = 0;
  return NNAL_OK;
}

extern "C" int nnal_pool_mc_read(nnal_ctx* ctx, double* av_post, double* av_ent) {
  if (!ctx) return NNAL_ERR_INVALID;
  if (!ctx->pool_mc_post || !ctx->mc_have) NNAL_FAIL(ctx, NNAL_ERR_STATE, "no MC-dropout pass has run");
  if (ctx->n_class != 2) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "binary running means need a 2-class model (nnal_pool_mc_read_classes)");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (av_post) CUDA_TRY(ctx, cudaMemcpyAsync(av_post, ctx->pool_mc_post, (size_t)ctx->pool_n * 8, cudaMemcpyDeviceToHost, ctx->stream));
  if (av_ent) CUDA_TRY(ctx, cudaMemcpyAsync(av_ent, ctx->pool_mc_ent, (size_t)ctx->pool_n * 8, cudaMemcpyDeviceToHost, ctx->stream));
  NNAL_SYNC_CHECKED(ctx);
  return NNAL_OK;
}

extern "C" int nnal_pool_mc_read_classes(nnal_ctx* ctx, double* av_post, double* av_ent) {
  if (!ctx) return NNAL_ERR_INVALID;
  if (!ctx->pool_mc_post || !ctx->mc_have) NNAL_FAIL(ctx, NNAL_ERR_STATE, "no MC-dropout pass has run");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  const size_t n = (size_t)ctx->pool_n;
  const bool binary = ctx->n_class == 2;
  // c = 2 keeps P(class 1) only: it goes to row 1, and row 0 is 1 - row 1 as the binary scores take it
  if (av_post) CUDA_TRY(ctx, cudaMemcpyAsync(binary ? av_post + n : av_post, ctx->pool_mc_post, (binary ? n : n * ctx->n_class) * 8,
                                             cudaMemcpyDeviceToHost, ctx->stream));
  if (av_ent) CUDA_TRY(ctx, cudaMemcpyAsync(av_ent, ctx->pool_mc_ent, n * 8, cudaMemcpyDeviceToHost, ctx->stream));
  NNAL_SYNC_CHECKED(ctx);
  if (av_post && binary)
    for (size_t i = 0; i < n; ++i) av_post[i] = 1.0 - av_post[n + i];
  return NNAL_OK;
}

static int reserve_forward(nnal_ctx* ctx, int64_t nb) {
  size_t mx = (size_t)ctx->in_h * ctx->in_w * std::max(16, (ctx->in_c + 7) / 8 * 8);   // padded / x-im2col'd input planes
  for (auto& L : ctx->layers) {
    size_t o = L.type == NNAL_LAYER_FC ? (size_t)L.out_dim : (size_t)L.out_h * L.out_w * L.out_c;
    mx = std::max(mx, o);
  }
  NNAL_TRY(devbuf_reserve(ctx, ctx->act[0], (size_t)nb * mx * sizeof(float)));
  NNAL_TRY(devbuf_reserve(ctx, ctx->act[1], (size_t)nb * mx * sizeof(float)));
  // input staging: fp32 NHWC, or (fused gather) fp16 hi/lo planes padded to 8 channels
  NNAL_TRY(devbuf_reserve(ctx, ctx->xin, (size_t)nb * ctx->in_h * ctx->in_w * std::max<size_t>((size_t)ctx->in_c * sizeof(float), 64)));
  return NNAL_OK;
}

static int pool_eval_impl(nnal_ctx* ctx, int subject, const int64_t* inds, bool inds_on_device, int64_t n, int64_t offset,
                          int d1, int d2, int d3, const double* stats, int norm_mode) {
  if (!ctx) return NNAL_ERR_INVALID;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (!ctx->pool_post) NNAL_FAIL(ctx, NNAL_ERR_STATE, "nnal_pool_begin not called");
  const Volume* v;
  NNAL_TRY(check_gather_args(ctx, subject, n, d1, d2, d3, &v));
  if (offset < 0 || offset + n > ctx->pool_n) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "pool range out of bounds");
  if (d1 != ctx->in_h || d2 != ctx->in_w || d3 * v->m != ctx->in_c)
    NNAL_FAIL(ctx, NNAL_ERR_INVALID, "patch shape does not match the model input");
  if (n == 0) return NNAL_OK;
  if (!inds) return NNAL_ERR_INVALID;
  double* d_stats;
  NNAL_TRY(upload_stats(ctx, stats, v->m, norm_mode, &d_stats));
  const int64_t chunk = std::min(chunk_size(ctx), n);
  NNAL_TRY(reserve_forward(ctx, chunk));
  // gather straight into the first conv's tensor-core input planes when it takes them
  const bool fused_ok = !ctx->dbg.no_fused_gather;
  // conv1 gathers its own input when it can (PW1's first layer on a 3-modality float32 volume): no gather kernel at all
  const bool fusedc1 = fused_ok && !ctx->dbg.no_fused_conv1 && nnal_layer_on_tc(ctx, 0) &&
                       nnal_tc_conv1_fused_supported(ctx, ctx->layers[0], *v, d1, d2, d3);
  const bool fused16 = fused_ok && !fusedc1 && nnal_first_layer_wants_x16(ctx) && nnal_k_gather_x16_supported(*v, d1, d2, d3);
  const bool fused = fused_ok && !fusedc1 && !fused16 && nnal_first_layer_wants_split8(ctx) && nnal_k_gather_split_supported(*v, d3);
  const int64_t* d_inds = inds;
  if (!inds_on_device) {
    NNAL_TRY(devbuf_reserve(ctx, ctx->inds, (size_t)n * 8));
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->inds.p, inds, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
    d_inds = (const int64_t*)ctx->inds.p;
  }
  for (int64_t o = 0; o < n; o += chunk) {
    int64_t nb = std::min(chunk, n - o);
    if (fusedc1) {
      ctx->fg.vol = v; ctx->fg.d_inds = d_inds + o; ctx->fg.h_stats = stats; ctx->fg.norm_mode = norm_mode;
      ctx->fg.d1 = d1; ctx->fg.d2 = d2; ctx->fg.d3 = d3;
      NNAL_TRY(nnal_forward_chunk(ctx, nb, offset + o, 3));
      continue;
    }
    prof_begin(ctx, NNAL_PROF_GATHER);
    if (fused16) {
      nnal_h* hi = (nnal_h*)ctx->xin.p;
      NNAL_TRY(nnal_k_gather_x16(ctx, *v, d_inds + o, nb, d1, d2, d3, stats, norm_mode, hi, hi + (size_t)nb * d1 * d2 * 16));
    } else if (fused) {
      nnal_h* hi = (nnal_h*)ctx->xin.p;
      NNAL_TRY(nnal_k_gather_split(ctx, *v, d_inds + o, nb, d1, d2, d3, stats, norm_mode, hi, hi + (size_t)nb * d1 * d2 * 8));
    } else {
      NNAL_TRY(nnal_k_gather_norm_f32(ctx, *v, d_inds + o, nb, d1, d2, d3, d_stats, norm_mode, (float*)ctx->xin.p));
    }
    prof_end(ctx);
    NNAL_TRY(nnal_forward_chunk(ctx, nb, offset + o, fused16 ? 2 : fused ? 1 : 0));
  }
  return NNAL_OK;
}

extern "C" int nnal_pool_eval(nnal_ctx* ctx, int subject, const int64_t* inds, int64_t n, int64_t offset, int d1, int d2,
                              int d3, const double* stats, int norm_mode) {
  return pool_eval_impl(ctx, subject, inds, false, n, offset, d1, d2, d3, stats, norm_mode);
}
extern "C" int nnal_pool_eval_device_inds(nnal_ctx* ctx, int subject, const int64_t* d_inds, int64_t n, int64_t offset,
                                          int d1, int d2, int d3, const double* stats, int norm_mode) {
  return pool_eval_impl(ctx, subject, d_inds, true, n, offset, d1, d2, d3, stats, norm_mode);
}

extern "C" int nnal_pool_eval_images(nnal_ctx* ctx, const float* x, int64_t n, int64_t offset) {
  if (!ctx) return NNAL_ERR_INVALID;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (!ctx->pool_post) NNAL_FAIL(ctx, NNAL_ERR_STATE, "nnal_pool_begin not called");
  if (n < 0 || offset < 0 || offset + n > ctx->pool_n) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "pool range out of bounds");
  if (n == 0) return NNAL_OK;
  if (!x) return NNAL_ERR_INVALID;
  const int64_t chunk = std::min(chunk_size(ctx), n);
  NNAL_TRY(reserve_forward(ctx, chunk));
  const size_t per = (size_t)ctx->in_h * ctx->in_w * ctx->in_c;
  for (int64_t o = 0; o < n; o += chunk) {
    int64_t nb = std::min(chunk, n - o);
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->xin.p, x + o * per, (size_t)nb * per * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    NNAL_TRY(nnal_forward_chunk(ctx, nb, offset + o));
  }
  return NNAL_OK;
}

extern "C" int nnal_pool_posteriors(nnal_ctx* ctx, float* out) {
  if (!ctx || !out) return NNAL_ERR_INVALID;
  if (!ctx->pool_post) NNAL_FAIL(ctx, NNAL_ERR_STATE, "no pool pass");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  CUDA_TRY(ctx, cudaMemcpyAsync(out, ctx->pool_post, (size_t)ctx->pool_n * ctx->n_class * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  NNAL_SYNC_CHECKED(ctx);
  return NNAL_OK;
}

__global__ void transpose_feat_kernel(const float* __restrict__ in, float* __restrict__ out, int64_t n, int d) {
  __shared__ float t[32][33];
  int64_t s0 = (int64_t)blockIdx.x * 32;
  int f0 = blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += 8) {
    int64_t s = s0 + r; int f = f0 + threadIdx.x;
    t[r][threadIdx.x] = (s < n && f < d) ? in[s * d + f] : 0.f;
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += 8) {
    int f = f0 + r; int64_t s = s0 + threadIdx.x;
    if (s < n && f < d) out[(int64_t)f * n + s] = t[threadIdx.x][r];
  }
}

extern "C" int nnal_pool_features(nnal_ctx* ctx, int64_t start, int64_t n, float* out) {
  if (!ctx || !out) return NNAL_ERR_INVALID;
  if (!ctx->pool_feat || ctx->keep < 1) NNAL_FAIL(ctx, NNAL_ERR_STATE, "pool pass did not keep features");
  if (start < 0 || n < 0 || start + n > ctx->pool_n) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "feature range out of bounds");
  if (n == 0) return NNAL_OK;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  int d = ctx->feat_dim;
  NNAL_TRY(devbuf_reserve(ctx, ctx->act[0], (size_t)n * d * sizeof(float)));
  dim3 grid(cdiv(n, 32), cdiv(d, 32)), block(32, 8);
  transpose_feat_kernel<<<grid, block, 0, ctx->stream>>>(ctx->pool_feat + start * d, (float*)ctx->act[0].p, n, d);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  CUDA_TRY(ctx, cudaMemcpyAsync(out, ctx->act[0].p, (size_t)n * d * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  NNAL_SYNC_CHECKED(ctx);
  return NNAL_OK;
}

__global__ void gather_rows_f32_kernel(const float* __restrict__ src, const int64_t* __restrict__ pos, int64_t n, int d,
                                       float* __restrict__ out) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n * d; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = e / d;
    out[e] = src[pos[r] * d + (e - r * d)];
  }
}

// rows `pos` of a kept pool matrix src [pool_n][d] -> out [n][d] (host)
static int gather_pool_rows(nnal_ctx* ctx, const float* src, int d, const int64_t* pos, int64_t n, float* out) {
  if (n == 0) return NNAL_OK;
  if (!pos || !out) return NNAL_ERR_INVALID;
  for (int64_t i = 0; i < n; ++i)
    if (pos[i] < 0 || pos[i] >= ctx->pool_n) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "feature row position outside the pool");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  NNAL_TRY(devbuf_reserve(ctx, ctx->act[0], (size_t)n * d * sizeof(float)));
  NNAL_TRY(devbuf_reserve(ctx, ctx->inds, (size_t)n * 8));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->inds.p, pos, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
  gather_rows_f32_kernel<<<std::min(cdiv(n * d, 256), ctx->sm_count * 16), 256, 0, ctx->stream>>>(src, (const int64_t*)ctx->inds.p, n, d,
                                                                                                 (float*)ctx->act[0].p);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  CUDA_TRY(ctx, cudaMemcpyAsync(out, ctx->act[0].p, (size_t)n * d * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  NNAL_SYNC_CHECKED(ctx);
  return NNAL_OK;
}

extern "C" int nnal_pool_feature_rows(nnal_ctx* ctx, const int64_t* pos, int64_t n, float* out) {
  if (!ctx || n < 0) return NNAL_ERR_INVALID;
  if (!ctx->pool_feat || ctx->keep < 1) NNAL_FAIL(ctx, NNAL_ERR_STATE, "pool pass did not keep features");
  return gather_pool_rows(ctx, ctx->pool_feat, ctx->feat_dim, pos, n, out);
}

extern "C" int nnal_pool_prev_rows(nnal_ctx* ctx, const int64_t* pos, int64_t n, float* out) {
  if (!ctx || n < 0) return NNAL_ERR_INVALID;
  if (!ctx->pool_prev || ctx->keep < 2) NNAL_FAIL(ctx, NNAL_ERR_STATE, "pool pass did not keep the previous FC output");
  if (ctx->feature_layer < 1 || ctx->layers[ctx->feature_layer - 1].type != NNAL_LAYER_FC)
    NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "the layer before the feature layer is not an FC layer");     // pool_prev is not written
  return gather_pool_rows(ctx, ctx->pool_prev, ctx->prev_dim, pos, n, out);
}

extern "C" int nnal_pool_score(nnal_ctx* ctx, int kind, double eps) {
  if (!ctx) return NNAL_ERR_INVALID;
  if (!ctx->pool_post) NNAL_FAIL(ctx, NNAL_ERR_STATE, "no pool pass");
  if (kind == NNAL_SCORE_MC_BINARY || kind == NNAL_SCORE_NEG_BALD || kind == NNAL_SCORE_MC_NEG_ENTROPY ||
      kind == NNAL_SCORE_MC_NEG_BALD) {
    if (kind < NNAL_SCORE_MC_NEG_ENTROPY && ctx->n_class != 2)
      NNAL_FAIL(ctx, NNAL_ERR_INVALID, "binary MC scores need a 2-class model (NNAL_SCORE_MC_NEG_ENTROPY / _MC_NEG_BALD)");
    if (!ctx->pool_mc_post || !ctx->mc_have) NNAL_FAIL(ctx, NNAL_ERR_STATE, "MC scores need an MC-dropout pool pass");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    prof_begin(ctx, NNAL_PROF_SCORE);
    int rc = nnal_k_scores_mc(ctx, ctx->pool_mc_post, ctx->pool_mc_ent, ctx->n_class, ctx->pool_n, kind, ctx->pool_score);
    prof_end(ctx);
    return rc;
  }
  if (kind < 0 || kind > 3) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "unknown score kind");
  if (kind == NNAL_SCORE_BINARY && ctx->n_class != 2) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "binary uncertainty needs a 2-class model");
  if (kind == NNAL_SCORE_NEG_FI_TRACE && (!ctx->pool_feat || ctx->keep < 1))
    NNAL_FAIL(ctx, NNAL_ERR_STATE, "the FI trace score needs a pool pass that kept the feature layer");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  prof_begin(ctx, NNAL_PROF_SCORE);
  int rc = kind == NNAL_SCORE_NEG_FI_TRACE
               ? nnal_k_fi_trace_scores(ctx, ctx->pool_post, ctx->n_class, ctx->pool_n, ctx->pool_feat, ctx->feat_dim, ctx->pool_score)
               : nnal_k_scores_f32(ctx, ctx->pool_post, ctx->n_class, ctx->pool_n, kind, eps, ctx->pool_score);
  prof_end(ctx);
  return rc;
}

extern "C" int nnal_pool_scores_read(nnal_ctx* ctx, double* out) {
  if (!ctx || !out) return NNAL_ERR_INVALID;
  if (!ctx->pool_score) NNAL_FAIL(ctx, NNAL_ERR_STATE, "no pool pass");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  CUDA_TRY(ctx, cudaMemcpyAsync(out, ctx->pool_score, (size_t)ctx->pool_n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  NNAL_SYNC_CHECKED(ctx);
  return NNAL_OK;
}

static int topk_to_host(nnal_ctx* ctx, const double* d_score, int64_t n, int64_t k, int64_t* idx_out, double* score_out) {
  if (k > n) k = n;
  if (k <= 0) return NNAL_OK;
  NNAL_TRY(devbuf_reserve(ctx, ctx->inds, (size_t)k * 16));
  int64_t* d_idx = (int64_t*)ctx->inds.p;
  double* d_sc = (double*)((char*)ctx->inds.p + (size_t)k * 8);
  prof_begin(ctx, NNAL_PROF_TOPK);
  NNAL_TRY(nnal_k_topk(ctx, d_score, n, k, d_idx, d_sc));
  prof_end(ctx);
  CUDA_TRY(ctx, cudaMemcpyAsync(idx_out, d_idx, (size_t)k * 8, cudaMemcpyDeviceToHost, ctx->stream));
  if (score_out) CUDA_TRY(ctx, cudaMemcpyAsync(score_out, d_sc, (size_t)k * 8, cudaMemcpyDeviceToHost, ctx->stream));
  NNAL_SYNC_CHECKED(ctx);
  return NNAL_OK;
}

extern "C" int nnal_pool_topk(nnal_ctx* ctx, int64_t k, int64_t* idx_out, double* score_out) {
  if (!ctx || !idx_out || k < 0) return NNAL_ERR_INVALID;
  if (!ctx->pool_score) NNAL_FAIL(ctx, NNAL_ERR_STATE, "no pool pass");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  return topk_to_host(ctx, ctx->pool_score, ctx->pool_n, k, idx_out, score_out);
}

// Device-resident top-k for the multi-GPU merge (SURVEY.md 8e, collective 1): the k best (score, global position)
// pairs of this rank stay in DEVICE memory, the host layer all-gathers the pair buffers with NCCL on nnal_stream() and
// nnal_topk_merge_pairs picks the global top-k -- one small device-to-host copy per query instead of a host-staged
// exchange.  Pair = {float64 score, int64 position}; unused slots are {+inf, INT64_MAX}.
struct TopkPair { double score; long long pos; };

__global__ void topk_pack_pairs_kernel(const int64_t* __restrict__ idx, const double* __restrict__ sc, int64_t k, int64_t k_pad,
                                       long long pos_offset, TopkPair* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < k_pad; i += (int64_t)gridDim.x * blockDim.x) {
    TopkPair p;
    if (i < k) { p.score = sc[i]; p.pos = (long long)idx[i] + pos_offset; }
    else { p.score = INFINITY; p.pos = 0x7fffffffffffffffll; }
    out[i] = p;
  }
}
__global__ void topk_pair_scores_kernel(const TopkPair* __restrict__ in, int64_t n, double* __restrict__ sc) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) sc[i] = in[i].score;
}
__global__ void topk_pair_pos_kernel(const TopkPair* __restrict__ in, const int64_t* __restrict__ idx, int64_t k,
                                     int64_t* __restrict__ pos) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < k; i += (int64_t)gridDim.x * blockDim.x) pos[i] = in[idx[i]].pos;
}

extern "C" int nnal_pool_topk_device(nnal_ctx* ctx, int64_t k, int64_t k_pad, int64_t pos_offset, void* d_pairs) {
  if (!ctx || !d_pairs || k < 0 || k_pad < k) return NNAL_ERR_INVALID;
  if (!ctx->pool_score) NNAL_FAIL(ctx, NNAL_ERR_STATE, "no pool pass");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (k > ctx->pool_n) k = ctx->pool_n;
  if (k_pad == 0) return NNAL_OK;
  NNAL_TRY(devbuf_reserve(ctx, ctx->inds, (size_t)std::max<int64_t>(k, 1) * 16));
  int64_t* d_idx = (int64_t*)ctx->inds.p;
  double* d_sc = (double*)((char*)ctx->inds.p + (size_t)std::max<int64_t>(k, 1) * 8);
  prof_begin(ctx, NNAL_PROF_TOPK);
  if (k > 0) NNAL_TRY(nnal_k_topk(ctx, ctx->pool_score, ctx->pool_n, k, d_idx, d_sc));
  topk_pack_pairs_kernel<<<std::min(cdiv(k_pad, 256), 1024), 256, 0, ctx->stream>>>(d_idx, d_sc, k, k_pad, (long long)pos_offset,
                                                                                  (TopkPair*)d_pairs);
  ctx->launches++;
  prof_end(ctx);
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}

// Global top-k of n_pairs gathered pairs [world][k_pad] (rank-major; every rank's list ascending by (score, position)
// and the ranks owning ascending position blocks, so that array order breaks score ties by position, as
// np.argsort(kind='stable') does on the concatenated pool).  pos_out / score_out: HOST arrays [k].
extern "C" int nnal_topk_merge_pairs(nnal_ctx* ctx, const void* d_pairs, int64_t n_pairs, int64_t k, int64_t* pos_out,
                                     double* score_out) {
  if (!ctx || !d_pairs || n_pairs < 0 || k < 0 || k > n_pairs) return NNAL_ERR_INVALID;
  if (k == 0) return NNAL_OK;
  if (!pos_out) return NNAL_ERR_INVALID;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  NNAL_TRY(devbuf_reserve(ctx, ctx->inds, (size_t)n_pairs * 8 + (size_t)k * 24));
  double* d_all = (double*)ctx->inds.p;
  int64_t* d_idx = (int64_t*)(d_all + n_pairs);
  double* d_sc = (double*)(d_idx + k);
  int64_t* d_pos = (int64_t*)(d_sc + k);
  prof_begin(ctx, NNAL_PROF_TOPK);
  topk_pair_scores_kernel<<<std::min(cdiv(n_pairs, 256), 1024), 256, 0, ctx->stream>>>((const TopkPair*)d_pairs, n_pairs, d_all);
  NNAL_TRY(nnal_k_topk(ctx, d_all, n_pairs, k, d_idx, d_sc));
  topk_pair_pos_kernel<<<std::min(cdiv(k, 256), 1024), 256, 0, ctx->stream>>>((const TopkPair*)d_pairs, d_idx, k, d_pos);
  ctx->launches += 2;
  prof_end(ctx);
  CUDA_TRY(ctx, cudaGetLastError());
  CUDA_TRY(ctx, cudaMemcpyAsync(pos_out, d_pos, (size_t)k * 8, cudaMemcpyDeviceToHost, ctx->stream));
  if (score_out) CUDA_TRY(ctx, cudaMemcpyAsync(score_out, d_sc, (size_t)k * 8, cudaMemcpyDeviceToHost, ctx->stream));
  NNAL_SYNC_CHECKED(ctx);
  return NNAL_OK;
}

// ---------------------------------------------------------------------------------------------
// stand-alone helpers
// ---------------------------------------------------------------------------------------------
extern "C" int nnal_entropy(nnal_ctx* ctx, const double* P, int c, int64_t n, int kind, double eps, double* out) {
  if (!ctx || c <= 0 || n < 0) return NNAL_ERR_INVALID;
  if (n == 0) return NNAL_OK;
  if (!P || !out) return NNAL_ERR_INVALID;
  if (kind == NNAL_SCORE_BINARY && c != 2) NNAL_FAIL(ctx, NNAL_ERR_INVALID, "binary uncertainty needs c == 2");
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  NNAL_TRY(devbuf_reserve(ctx, ctx->act[0], (size_t)n * c * 8));
  NNAL_TRY(devbuf_reserve(ctx, ctx->act[1], (size_t)n * 8));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->act[0].p, P, (size_t)n * c * 8, cudaMemcpyHostToDevice, ctx->stream));
  NNAL_TRY(nnal_k_scores_f64(ctx, (const double*)ctx->act[0].p, c, n, kind, eps, (double*)ctx->act[1].p));
  CUDA_TRY(ctx, cudaMemcpyAsync(out, ctx->act[1].p, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return NNAL_OK;
}

extern "C" int nnal_topk(nnal_ctx* ctx, const double* scores, int64_t n, int64_t k, int64_t* idx_out) {
  if (!ctx || n < 0 || k < 0) return NNAL_ERR_INVALID;
  if (n == 0 || k == 0) return NNAL_OK;
  if (!scores || !idx_out) return NNAL_ERR_INVALID;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  NNAL_TRY(devbuf_reserve(ctx, ctx->act[1], (size_t)n * 8));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->act[1].p, scores, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
  return topk_to_host(ctx, (const double*)ctx->act[1].p, n, k, idx_out, nullptr);
}

// test hook: declare a pool of n samples whose SCORES are given (no model, no pool pass) -- lets tests drive the top-k /
// merge kernels with arbitrary scores (exact ties, ragged ranks)
extern "C" int nnal_debug_set_pool_scores(nnal_ctx* ctx, const double* scores, int64_t n) {
  if (!ctx || n < 0 || (n > 0 && !scores)) return NNAL_ERR_INVALID;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (ctx->pool_cap_score < (size_t)std::max<int64_t>(n, 1)) {
    if (ctx->pool_score) { CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream)); CUDA_TRY(ctx, cudaFree(ctx->pool_score)); ctx->pool_score = nullptr; }
    CUDA_TRY(ctx, cudaMalloc(&ctx->pool_score, (size_t)std::max<int64_t>(n, 1) * sizeof(double)));
    ctx->pool_cap_score = (size_t)std::max<int64_t>(n, 1);
  }
  if (n) CUDA_TRY(ctx, cudaMemcpyAsync(ctx->pool_score, scores, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->pool_n = n;
  return NNAL_OK;
}

// ---------------------------------------------------------------------------------------------
// test hook: one FC layer out = act(A W^T + b) on host buffers (used by tests to compare the
// tcgen05 GEMM with the FP32 CUDA-core GEMM and the oracle in isolation)
// ---------------------------------------------------------------------------------------------
extern "C" int nnal_debug_fc(nnal_ctx* ctx, const float* A, const float* W, const float* b, int64_t M, int N, int K,
                             int relu, int use_tc, float* out) {
  if (!ctx || !A || !W || !b || !out || M <= 0 || N <= 0 || K <= 0) return NNAL_ERR_INVALID;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  Layer L;
  L.type = NNAL_LAYER_FC; L.in_dim = K; L.out_dim = N; L.relu = relu;
  float *dA = nullptr, *dO = nullptr;
  int rc = NNAL_OK;
  auto cleanup = [&]() {
    cudaStreamSynchronize(ctx->stream);
    if (dA) cudaFree(dA); if (dO) cudaFree(dO);
    if (L.W) cudaFree(L.W); if (L.b) cudaFree(L.b); if (L.Wh) cudaFree(L.Wh); if (L.Wl) cudaFree(L.Wl); if (L.Wt) cudaFree(L.Wt); if (L.Wx) cudaFree(L.Wx);
  };
  if (cudaMalloc(&dA, (size_t)M * K * 4) != cudaSuccess || cudaMalloc(&dO, (size_t)M * N * 4) != cudaSuccess ||
      cudaMalloc(&L.W, (size_t)N * K * 4) != cudaSuccess || cudaMalloc(&L.b, (size_t)N * 4) != cudaSuccess) {
    cleanup(); NNAL_FAIL(ctx, NNAL_ERR_CUDA, "debug_fc allocation failed");
  }
  cudaMemcpyAsync(dA, A, (size_t)M * K * 4, cudaMemcpyHostToDevice, ctx->stream);
  cudaMemcpyAsync(L.W, W, (size_t)N * K * 4, cudaMemcpyHostToDevice, ctx->stream);
  cudaMemcpyAsync(L.b, b, (size_t)N * 4, cudaMemcpyHostToDevice, ctx->stream);
  L.has_weights = true;
  nnal_set_weight_scale(L, W, (size_t)N * K);
  if (use_tc) {
    rc = nnal_tc_prepare_layer(ctx, L);
    if (rc == NNAL_OK && !nnal_tc_fc_supported(ctx, L)) { ctx->err = "shape not supported by the tensor-core FC"; rc = NNAL_ERR_UNSUPPORTED; }
    if (rc == NNAL_OK) rc = nnal_tc_fc(ctx, L, dA, dO, M);
  } else {
    rc = nnal_k_fc_simt(ctx, L, dA, dO, M);
  }
  if (rc == NNAL_OK) {
    if (cudaMemcpyAsync(out, dO, (size_t)M * N * 4, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess ||
        cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
      ctx->err = std::string("debug_fc: ") + cudaGetErrorString(cudaGetLastError()); rc = NNAL_ERR_CUDA;
    }
  }
  if (rc == NNAL_OK && nnal_ovf_enqueue(ctx) == NNAL_OK && cudaStreamSynchronize(ctx->stream) == cudaSuccess) rc = nnal_ovf_test(ctx);
  cleanup();
  return rc;
}

// test hook: one conv layer (SAME, stride 1, bias, ReLU) on host NHWC buffers
extern "C" int nnal_debug_conv(nnal_ctx* ctx, const float* x, const float* W, const float* b, int64_t n, int H, int Wd,
                               int Cin, int Cout, int ks, int use_tc, float* out) {
  if (!ctx || !x || !W || !b || !out || n <= 0) return NNAL_ERR_INVALID;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  Layer L;
  L.type = NNAL_LAYER_CONV; L.kh = L.kw = ks; L.in_h = L.out_h = H; L.in_w = L.out_w = Wd; L.in_c = Cin; L.out_c = Cout; L.relu = 1;
  const size_t ie = (size_t)n * H * Wd * Cin, oe = (size_t)n * H * Wd * Cout;
  size_t oe_out = oe;
  float *dX = nullptr, *dO = nullptr;
  nnal_h *ih = nullptr, *oh = nullptr;
  int rc = NNAL_OK;
  auto cleanup = [&]() {
    cudaStreamSynchronize(ctx->stream);
    if (dX) cudaFree(dX); if (dO) cudaFree(dO); if (ih) cudaFree(ih); if (oh) cudaFree(oh);
    if (L.W) cudaFree(L.W); if (L.b) cudaFree(L.b); if (L.Wh) cudaFree(L.Wh); if (L.Wl) cudaFree(L.Wl); if (L.Wt) cudaFree(L.Wt); if (L.Wx) cudaFree(L.Wx);
  };
  if (cudaMalloc(&dX, ie * 4) != cudaSuccess || cudaMalloc(&dO, oe * 4) != cudaSuccess || cudaMalloc(&ih, ie * 4) != cudaSuccess ||
      cudaMalloc(&oh, oe * 4) != cudaSuccess || cudaMalloc(&L.W, (size_t)ks * ks * Cin * Cout * 4) != cudaSuccess ||
      cudaMalloc(&L.b, (size_t)Cout * 4) != cudaSuccess) {
    cleanup(); NNAL_FAIL(ctx, NNAL_ERR_CUDA, "debug_conv allocation failed");
  }
  cudaMemcpyAsync(dX, x, ie * 4, cudaMemcpyHostToDevice, ctx->stream);
  cudaMemcpyAsync(L.W, W, (size_t)ks * ks * Cin * Cout * 4, cudaMemcpyHostToDevice, ctx->stream);
  cudaMemcpyAsync(L.b, b, (size_t)Cout * 4, cudaMemcpyHostToDevice, ctx->stream);
  L.has_weights = true;
  nnal_set_weight_scale(L, W, (size_t)ks * ks * Cin * Cout);
  if (use_tc) {
    rc = nnal_tc_prepare_layer(ctx, L);
    if (rc == NNAL_OK && !nnal_tc_conv_supported(ctx, L)) { ctx->err = "shape not supported by the tensor-core conv"; rc = NNAL_ERR_UNSUPPORTED; }
    bool x16done = false;
    if (rc == NNAL_OK && use_tc == 5) {
      // conv1 on the x-im2col'd input: fp32 -> [n][H][W][16] hi/lo planes -> CfgConv1X
      if (!nnal_tc_conv_x16_supported(ctx, L)) { ctx->err = "shape not supported by the x-im2col'd conv"; rc = NNAL_ERR_UNSUPPORTED; }
      const size_t iex = (size_t)n * H * Wd * 16;
      nnal_h* ix = nullptr;
      if (rc == NNAL_OK && cudaMalloc(&ix, iex * 4) != cudaSuccess) { cleanup(); NNAL_FAIL(ctx, NNAL_ERR_CUDA, "debug_conv allocation failed"); }
      if (rc == NNAL_OK) rc = nnal_k_split_x16(ctx, dX, ix, ix + iex, (int64_t)n * H * Wd, Wd, Cin, ks);
      if (rc == NNAL_OK) rc = nnal_tc_conv_x16(ctx, L, ix, ix + iex, oh, oh + oe, n);
      if (rc == NNAL_OK) rc = nnal_k_merge_flat(ctx, oh, oh + oe, dO, (int64_t)oe);
      cudaStreamSynchronize(ctx->stream);
      if (ix) cudaFree(ix);
      x16done = true;
    }
    const int cp = (Cin + 7) / 8 * 8;
    const size_t iep = (size_t)n * H * Wd * cp;
    if (cp != Cin) { cudaFree(ih); ih = nullptr; if (cudaMalloc(&ih, iep * 4) != cudaSuccess) { cleanup(); NNAL_FAIL(ctx, NNAL_ERR_CUDA, "debug_conv allocation failed"); } }
    if (rc == NNAL_OK && !x16done) rc = nnal_k_split_pad(ctx, dX, ih, ih + iep, (int64_t)n * H * Wd, Cin, cp);
    if (rc == NNAL_OK && (use_tc == 2 || use_tc == 3) &&
        !(use_tc == 3 ? nnal_wt_conv_pool_supported(ctx, L) : nnal_wt_conv_supported(ctx, L))) {
      ctx->err = "shape not supported by the weight-stationary conv"; rc = NNAL_ERR_UNSUPPORTED;
    }
    if (rc == NNAL_OK && use_tc == 4 && !nnal_tc_conv_pool_supported(ctx, L)) {
      ctx->err = "conv+pool shape not supported by the tensor-core conv"; rc = NNAL_ERR_UNSUPPORTED;
    }
    if (use_tc == 3 || use_tc == 4) oe_out = (size_t)n * ((H + 1) / 2) * ((Wd + 1) / 2) * Cout;      // fused 2x2/s2 SAME max-pool
    if (rc == NNAL_OK && !x16done)
      rc = use_tc == 4 ? nnal_tc_conv_pool(ctx, L, ih, ih + iep, oh, oh + oe_out, n)
         : use_tc >= 2 ? nnal_wt_conv(ctx, L, ih, ih + iep, oh, oh + oe_out, n, use_tc == 3)
                       : nnal_tc_conv(ctx, L, ih, ih + iep, oh, oh + oe, n);
    if (rc == NNAL_OK && !x16done) rc = nnal_k_merge_flat(ctx, oh, oh + oe_out, dO, (int64_t)oe_out);
  } else {
    rc = nnal_k_conv_simt(ctx, L, dX, dO, n);
  }
  if (rc == NNAL_OK) {
    if (cudaMemcpyAsync(out, dO, oe_out * 4, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess ||
        cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
      ctx->err = std::string("debug_conv: ") + cudaGetErrorString(cudaGetLastError()); rc = NNAL_ERR_CUDA;
    }
  }
  if (rc == NNAL_OK && nnal_ovf_enqueue(ctx) == NNAL_OK && cudaStreamSynchronize(ctx->stream) == cudaSuccess) rc = nnal_ovf_test(ctx);
  cleanup();
  return rc;
}

// test hook: conv1 of the model with the patch gather fused in (conv_tc.cu CfgConv1XG) over `n` voxels of an uploaded volume:
// conv1's float32 output [n][25][25][24] (merged fp16 hi/lo planes) on the host
extern "C" int nnal_debug_conv1_gather(nnal_ctx* ctx, int subject, const int64_t* inds, int64_t n, const double* stats,
                                       int norm_mode, float* out) {
  if (!ctx || !inds || !out || n <= 0) return NNAL_ERR_INVALID;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (ctx->layers.empty() || !ctx->layers[0].has_weights) NNAL_FAIL(ctx, NNAL_ERR_STATE, "model weights not set");
  const Volume* v;
  NNAL_TRY(check_gather_args(ctx, subject, n, 25, 25, 1, &v));
  const Layer& L = ctx->layers[0];
  if (!nnal_tc_conv1_fused_supported(ctx, L, *v, 25, 25, 1))
    NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "first layer / volume not covered by the conv1 that gathers its own input");
  double* d_stats;
  NNAL_TRY(upload_stats(ctx, stats, v->m, norm_mode, &d_stats));
  const size_t oe = (size_t)n * 25 * 25 * L.out_c;
  int64_t* dI = nullptr;
  nnal_h* oh = nullptr;
  float* dO = nullptr;
  auto cleanup = [&]() {
    cudaStreamSynchronize(ctx->stream);
    if (dI) cudaFree(dI); if (oh) cudaFree(oh); if (dO) cudaFree(dO);
  };
  if (cudaMalloc(&dI, (size_t)n * 8) != cudaSuccess || cudaMalloc(&oh, oe * 4) != cudaSuccess || cudaMalloc(&dO, oe * 4) != cudaSuccess) {
    cleanup(); NNAL_FAIL(ctx, NNAL_ERR_CUDA, "debug_conv1_gather allocation failed");
  }
  int rc = NNAL_OK;
  if (cudaMemcpyAsync(dI, inds, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess) {
    ctx->err = std::string("debug_conv1_gather: ") + cudaGetErrorString(cudaGetLastError()); rc = NNAL_ERR_CUDA;
  }
  FusedGather fg;
  fg.vol = v; fg.d_inds = dI; fg.h_stats = stats; fg.norm_mode = norm_mode; fg.d1 = 25; fg.d2 = 25; fg.d3 = 1;
  if (rc == NNAL_OK) rc = nnal_tc_conv1_fused(ctx, L, fg, oh, oh + oe, n);
  if (rc == NNAL_OK) rc = nnal_k_merge_flat(ctx, oh, oh + oe, dO, (int64_t)oe);
  if (rc == NNAL_OK) {
    if (cudaMemcpyAsync(out, dO, oe * 4, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess ||
        cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
      ctx->err = std::string("debug_conv1_gather: ") + cudaGetErrorString(cudaGetLastError()); rc = NNAL_ERR_CUDA;
    }
  }
  if (rc == NNAL_OK && nnal_ovf_enqueue(ctx) == NNAL_OK && cudaStreamSynchronize(ctx->stream) == cudaSuccess) rc = nnal_ovf_test(ctx);
  cleanup();
  return rc;
}
