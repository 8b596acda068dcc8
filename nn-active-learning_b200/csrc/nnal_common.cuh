// Shared declarations of libnnal_b200 (sm_100a only).  See include/nnal_b200.h for the C ABI.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cstdint>
#include <cstdio>
#include "philox.cuh"
#include <cstring>
#include <string>
#include <vector>

#define NNAL_OK 0
#define NNAL_ERR_INVALID 1
#define NNAL_ERR_CUDA 2
#define NNAL_ERR_STATE 3
#define NNAL_ERR_UNSUPPORTED 4
#define NNAL_ERR_NO_DEVICE 5
#define NNAL_ERR_OVERFLOW 6

enum { NNAL_LAYER_CONV = 0, NNAL_LAYER_POOL = 1, NNAL_LAYER_FC = 2 };
enum { NNAL_F32 = 0, NNAL_F64 = 1 };

// Operand element type of the tensor-core path.  Every fp32 value x is carried as two fp16 terms
// x ~= hi + lo (hi = fp16(x), lo = fp16(x - hi)): 22 significant bits, products hi.hi + hi.lo + lo.hi.
// (bf16 terms were measured first: 2^-18 relative operand error, too coarse for the 1e-4 posterior
// tolerance at 1e5-sample pools; fp16 terms have the same MMA rate.)  Weights are pre-scaled by a
// power of two so that their lo terms stay in fp16's normal range; epilogues undo the scale.
typedef __half nnal_h;
// fp16 range guard.  Operands are clamped to +-65504 before the hi/lo split; a value that hits the clamp (or is not
// finite) sets a device flag, and every entry point that hands results to the caller returns NNAL_ERR_OVERFLOW when the
// flag is up -- a model or input outside fp16's range fails loudly instead of returning saturated posteriors.  The flag
// word is one per device (capi.cu); every translation unit holds a pointer to it in a static __device__ variable that is
// bound when a context is created (nnal_ovf_register collects the per-unit binders at load time).
void nnal_ovf_register(int (*bind)(unsigned int*));
#ifdef __CUDACC__
static __device__ unsigned int* nnal_ovf_ptr;
__device__ __forceinline__ void nnal_ovf_note(float x) {
  if (!(fabsf(x) <= 65504.f)) {
    unsigned int* p = nnal_ovf_ptr;
    if (p) atomicOr(p, 1u);
  }
}
static int nnal_ovf_bind_tu(unsigned int* word) {
  return cudaMemcpyToSymbol(nnal_ovf_ptr, &word, sizeof(word)) == cudaSuccess ? 0 : 1;
}
namespace {
struct NnalOvfRegistrar { NnalOvfRegistrar() { nnal_ovf_register(&nnal_ovf_bind_tu); } };
static NnalOvfRegistrar nnal_ovf_registrar_instance;
}
// hot epilogues: track the largest |x| bit pattern of a thread's tile (NaN / Inf patterns sort above every finite value:
// two integer ops per element, no branch) and test it once per tile
__device__ __forceinline__ void nnal_ovf_track(uint32_t& m, float x) { m = max(m, __float_as_uint(x) & 0x7fffffffu); }
__device__ __forceinline__ void nnal_ovf_commit(uint32_t m) {
  if (m > 0x477fe000u) {                      // bits of 65504.f
    unsigned int* p = nnal_ovf_ptr;
    if (p) atomicOr(p, 1u);
  }
}
// epilogues that round post-ReLU values (>= 0) to fp16 pairs: the largest hi-term bit pattern per 16-bit lane (one SIMD
// max per pair), tested once per tile -- an Inf (the rounding of anything >= 65520) or NaN pattern raises the flag
__device__ __forceinline__ void nnal_ovf_track_h2(uint32_t& m, uint32_t h2bits) { m = __vmaxu2(m, h2bits); }
__device__ __forceinline__ void nnal_ovf_commit_h2(uint32_t m) {
  if ((m & 0xffffu) >= 0x7c00u || (m >> 16) >= 0x7c00u) {
    unsigned int* p = nnal_ovf_ptr;
    if (p) atomicOr(p, 1u);
  }
}
__device__ __forceinline__ void nnal_split_unchecked(float x, nnal_h& h, nnal_h& l) {
  x = fminf(fmaxf(x, -65504.f), 65504.f);
  h = __float2half_rn(x);
  l = __float2half_rn(x - __half2float(h));
}
__device__ __forceinline__ void nnal_split(float x, nnal_h& h, nnal_h& l) {
  nnal_ovf_note(x);
  x = fminf(fmaxf(x, -65504.f), 65504.f);
  h = __float2half_rn(x);
  l = __float2half_rn(x - __half2float(h));
}
__device__ __forceinline__ float nnal_merge(nnal_h h, nnal_h l) { return __half2float(h) + __half2float(l); }
__device__ __forceinline__ uint32_t nnal_pack2(nnal_h a, nnal_h b) {
  return (uint32_t)__half_as_ushort(a) | ((uint32_t)__half_as_ushort(b) << 16);
}
#endif

struct LayerSpec { int type, out, kh, kw; };

struct Layer {
  int type = 0;
  int kh = 0, kw = 0;
  int in_h = 0, in_w = 0, in_c = 0;      // conv/pool input geometry (NHWC)
  int out_h = 0, out_w = 0, out_c = 0;   // conv/pool output geometry
  int pad_t = 0, pad_l = 0;              // pool: TF SAME padding before the first row / column (0 for 2x2)
  int in_dim = 0, out_dim = 0;           // fc
  int relu = 0;
  bool has_weights = false;
  float* W = nullptr;                    // conv: [kh][kw][cin][cout]; fc: [out][in_native]
  float* b = nullptr;
  // fp16 split planes for the tensor-core path (hi = fp16(x), lo = fp16(x - hi))
  nnal_h* Wh = nullptr;
  nnal_h* Wl = nullptr;
  void* Wt = nullptr;                    // conv: weight blocks of the weight-stationary kernel (conv_wt.cu)
  void* Wx = nullptr;                    // conv1: packed weights of the x-im2col'd form (conv_tc.cu, CfgConv1X)
  int k_pad = 0;                         // padded K of the split planes
  int n_pad = 0;                         // padded N (rows) of the split planes
  float w_scale = 1.f, w_scale_inv = 1.f; // power-of-two scale applied to the fp16 weight planes
};

struct Volume {
  int m = 0;                             // modalities
  int64_t X = 0, Y = 0, Z = 0;           // padded extents (as the reference passes them)
  int dtype = NNAL_F32;                  // device storage type
  void* data = nullptr;                  // [Z][X][Y][m]
  size_t bytes = 0;
};

// per OUTPUT channel (C <= 8) normalisation table of the fused gathers: (x - mu) / sigma in float64 (volume.cu)
struct NormTab { double mu[8], sg[8], rs[8]; int on[8]; };
#ifdef __CUDACC__
__device__ __forceinline__ double norm_apply(double v, double mu, double sg, double rs) {
  const double a = v - mu;
  if (rs != rs) return a / sg;               // no usable reciprocal: true division
  const double q0 = a * rs;
  const double r = fma(-q0, sg, a);
  return fma(r, rs, q0);
}
#endif
// what the first conv layer needs to gather its own input (conv_tc.cu, gather fused into conv1): set by the pool pass
struct FusedGather {
  const Volume* vol = nullptr;
  const int64_t* d_inds = nullptr;       // raveled voxel ids of the chunk (device)
  const double* h_stats = nullptr;       // [m][2] (host)
  int norm_mode = 0, d1 = 0, d2 = 0, d3 = 0;
};

struct ProfRec { int cls; cudaEvent_t a, b; };

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
};

// Test-only switches (nnal_debug_option): they select FALLBACK kernels or chunk sizes so that tests can hold every code path
// to the same parity bar.  The product never sets them; there are no environment variables.
struct DebugOpts {
  long chunk = 0;              // samples per forward chunk (0: default)
  long bw_chunk = 0;           // samples per chunk of the shrunk-gradient pass (0: default)
  int no_fused_gather = 0;     // fp32 gather + separate split pass instead of the gather that writes conv1's planes
  int no_fused_conv1 = 0;      // stand-alone gather kernel + conv1 instead of the conv1 that gathers its own input
  int wt_flags = 0;            // conv_wt.cu timing experiments: 1 skip the epilogue stores, 2 skip the lo plane
  int sdp_no_coop = 0;         // one launch per SDP iteration instead of the cooperative loop
  int bw_no_ws = 0, bw_no_tc8 = 0, bw_no_tc = 0, bw_simt_fwd = 0;   // shrunk.cu fallbacks
  int plain_upload = 0;        // volumes: one cudaMemcpyAsync per modality even from pageable memory (instead of the threaded pinned staging)
  int fi_flags = 0;            // fi.cu: 1 skip the column pass, 2 skip the evaluation, 4 skip stand-alone inversions (timing experiments, results are garbage);
                               // 8 one-pivot-at-a-time inverse inside the column kernel instead of the pipelined step, 16 no speculative columns (tests)
};

struct nnal_ctx {
  DebugOpts dbg;
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  std::string err;
  // model
  std::vector<Layer> layers;
  int in_h = 0, in_w = 0, in_c = 0, n_class = 0, feature_layer = -1, feat_dim = 0;
  int fc_first = -1;                     // index of first fc layer
  int use_tc = 1;                        // tensor-core (tcgen05) path for conv/fc where supported
  FusedGather fg;                        // valid during nnal_forward_chunk(.., input_format 3)
  int use_x16 = 0;                       // conv1 on x-im2col'd input (3 channels x 5 filter columns folded into 16 channels); NNAL_CONV_X16=1
  int use_wt = 2;                        // conv_wt.cu: 0 never, 1 where it is the faster kernel, 2 (default) + fused max-pool, 3 wherever it covers the layer
  // volumes
  std::vector<Volume> vols;
  DevBuf stage;                          // upload staging
  std::vector<double> stats_host;        // normalisation table being uploaded (mu, sigma, 1/sigma per modality)
  // workspaces
  DevBuf inds, act[2], xin, featbuf, prevbuf, logits;
  DevBuf splitA[2];                      // fp16 hi/lo activation planes
  // pool state
  int64_t pool_n = 0;
  int keep = 0;                          // 0: posteriors only, 1: + features (fc_{L-1} out), 2: + previous fc out
  float* pool_post = nullptr;            // [c][pool_n]
  double* pool_score = nullptr;           // [pool_n] float64 like the reference's ranking
  float* pool_feat = nullptr;            // [pool_n][feat_dim]
  float* pool_prev = nullptr;            // [pool_n][prev_dim]
  int prev_dim = 0;
  DevBuf topk_ws;
  // FI state
  DevBuf fi_ws;
  // counters / per-kernel-class device timing (bench.py roofline leg)
  long long launches = 0;
  int profile = 0;
  std::vector<ProfRec> prof;
  size_t pool_cap_n = 0, pool_cap_score = 0, pool_cap_nfeat = 0, pool_cap_nprev = 0;   // per-array capacities (samples)
  int pool_cap_class = 0, pool_cap_feat = 0, pool_cap_prev = 0;                        // widths they were sized for
  void* tc_state = nullptr;              // tensor-map cache etc. (gemm_tc.cu)
  void* sims_state = nullptr;            // representativeness queries (sims.cu)
  void* fi_state = nullptr;              // Fisher-information candidate set / greedy state (fi.cu)
  void* fi_block_state = nullptr;        // multi-class block-form FI candidates / greedy state (fi_block.cu)
  unsigned long long weights_version = 0; // bumped by nnal_model_set / nnal_model_set_weights: derived weight copies (shrunk.cu) are rebuilt
  void* bw_state = nullptr;              // shrunk class-score gradients: kept activations and gradient buffers (shrunk.cu)
  void* sdp_state = nullptr;             // query-distribution solver workspaces (sdp.cu)
  // MC-dropout (MC-entropy / BALD): T stochastic passes of the FC tail per chunk, running means per pool sample
  int mc_T = 0;                          // 0: deterministic forward
  int mc_have = 0;                       // the current pool pass ran in MC mode: running means are valid
  int ens_open = 0;                      // committee accumulation in progress: pool passes of the members keep the running means
  DropSpec mc_drop;                      // keep, threshold, seed, first pass id, global position of pool offset 0
  std::vector<int> mc_sites;             // layer indices whose OUTPUT is dropped out (NN.py:167-171)
  double* pool_mc_post = nullptr;        // [pool_n] running mean of P(class 1) over the passes (float64, PW_NNAL.py:80)
  double* pool_mc_ent = nullptr;         // [pool_n] running mean of the per-pass binary entropies (PW_NNAL.py:262-268)
  size_t pool_cap_mc = 0;
  DevBuf act_mc;                         // third activation buffer: the conv trunk's output must survive the T tail passes
  unsigned int* ovf_word = nullptr;      // device flag set by nnal_ovf_note (shared by the contexts of one device)
  unsigned int* ovf_host = nullptr;      // pinned host copy read by nnal_ovf_test
  void* upload_state = nullptr;          // pinned staging ring + copy streams for pageable volumes (capi.cu)
  void* p2p_state = nullptr;             // peer-memory exchange buffers of the multi-GPU greedy step (p2p.cu)
};

#define CUDA_TRY(ctx, expr)                                                            \
  do {                                                                                 \
    cudaError_t _e = (expr);                                                           \
    if (_e != cudaSuccess) {                                                           \
      (ctx)->err = std::string(#expr) + ": " + cudaGetErrorString(_e);                 \
      return NNAL_ERR_CUDA;                                                            \
    }                                                                                  \
  } while (0)

#define NNAL_FAIL(ctx, code, msg)                                                      \
  do { (ctx)->err = (msg); return (code); } while (0)

#define NNAL_TRY(expr)                                                                 \
  do { int _r = (expr); if (_r != NNAL_OK) return _r; } while (0)

static inline int devbuf_reserve(nnal_ctx* ctx, DevBuf& b, size_t bytes) {
  if (b.cap >= bytes) return NNAL_OK;
  if (b.p) { CUDA_TRY(ctx, cudaFree(b.p)); b.p = nullptr; b.cap = 0; }
  size_t want = bytes + (bytes >> 3) + 256;
  CUDA_TRY(ctx, cudaMalloc(&b.p, want));
  b.cap = want;
  return NNAL_OK;
}

static inline void prof_begin(nnal_ctx* ctx, int cls) {
  if (!ctx->profile) return;
  ProfRec r; r.cls = cls;
  cudaEventCreate(&r.a); cudaEventCreate(&r.b);
  cudaEventRecord(r.a, ctx->stream);
  ctx->prof.push_back(r);
}
static inline void prof_end(nnal_ctx* ctx) {
  if (!ctx->profile || ctx->prof.empty()) return;
  cudaEventRecord(ctx->prof.back().b, ctx->stream);
}
#define NNAL_PROF_GATHER 100
#define NNAL_PROF_SCORE 101
#define NNAL_PROF_TOPK 102
#define NNAL_PROF_FI_SETUP 110
#define NNAL_PROF_FI_GRAM 111
#define NNAL_PROF_FI_GREEDY 112
#define NNAL_PROF_FI_SOLVE 113
#define NNAL_PROF_FIB_SYSTEM 114         // fi_block.cu: K_SS row, alpha I + K_SS, inversion, Z, tr C
#define NNAL_PROF_FIB_EVAL 115           // fi_block.cu: per-candidate losses + arg-min
#define NNAL_PROF_FIB_COLUMN 116         // fi_block.cu: the winner's column s_{., w}
#define NNAL_PROF_BW_FORWARD 120
#define NNAL_PROF_BW_BACKWARD 121

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

// fp16 range guard: enqueue the flag read on the stream (before a synchronisation the caller does anyway), then test it
int nnal_ovf_enqueue(nnal_ctx* ctx);
int nnal_ovf_test(nnal_ctx* ctx);
#define NNAL_SYNC_CHECKED(ctx)                                                         \
  do {                                                                                 \
    NNAL_TRY(nnal_ovf_enqueue(ctx));                                                   \
    CUDA_TRY(ctx, cudaStreamSynchronize((ctx)->stream));                               \
    NNAL_TRY(nnal_ovf_test(ctx));                                                      \
  } while (0)

// ---- kernels launchers (defined in the individual .cu files) -------------------------
// volume.cu
int nnal_k_relayout(nnal_ctx*, const void* stage, int dtype, int m, int64_t X, int64_t Y, int64_t Z,
                    int64_t px, int64_t py, int64_t pz, void* out);
int nnal_k_gather_f64(nnal_ctx*, const Volume&, const int64_t* d_inds, int64_t n, int d1, int d2, int d3,
                      const double* d_stats, int norm_mode, double* d_out);
int nnal_k_gather_norm_f32(nnal_ctx*, const Volume&, const int64_t* d_inds, int64_t n, int d1, int d2, int d3,
                           const double* d_stats, int norm_mode, float* d_out);
bool nnal_k_gather_split_supported(const Volume&, int d3);
int nnal_k_gather_split(nnal_ctx*, const Volume&, const int64_t* d_inds, int64_t n, int d1, int d2, int d3,
                        const double* h_stats, int norm_mode, nnal_h* out_hi, nnal_h* out_lo);
// forward_simt.cu
int nnal_k_conv_simt(nnal_ctx*, const Layer&, const float* in, float* out, int64_t n);
int nnal_k_pool(nnal_ctx*, const Layer&, const float* in, float* out, int64_t n);
int nnal_k_fc_simt(nnal_ctx*, const Layer&, const float* in, float* out, int64_t n);
int nnal_k_permute_fc_weight(nnal_ctx*, const float* Wtf, float* Wnative, int out, int C, int H, int W);
// score.cu
int nnal_k_head(nnal_ctx*, const Layer& fc_last, const float* feat, int64_t n, int64_t pool_n, int64_t offset,
                float* post /*[c][pool_n]*/, float* logits_out /*[n][c] or null*/, const DropSpec* drop = nullptr);
int nnal_k_mc_accumulate(nnal_ctx*, const float* post, int64_t pool_n, int64_t offset, int64_t n, int t,
                         double* av_post, double* av_ent);
int nnal_k_scores_mc(nnal_ctx*, const double* av_post, const double* av_ent, int64_t n, int kind, double* score);
int nnal_k_scores_f32(nnal_ctx*, const float* post, int c, int64_t n, int kind, double eps, double* score);
int nnal_k_scores_f64(nnal_ctx*, const double* post, int c, int64_t n, int kind, double eps, double* score);
int nnal_k_entropy_f32(nnal_ctx*, const float* post, int c, int64_t n, float eps, float* H);
int nnal_k_topk(nnal_ctx*, const double* score, int64_t n, int64_t k, int64_t* d_idx_out, double* d_score_out);
// gemm_tc.cu / conv_tc.cu (tcgen05 path)
int nnal_tc_prepare_layer(nnal_ctx*, Layer&);
bool nnal_tc_fc_supported(const nnal_ctx*, const Layer&);
int nnal_tc_release(nnal_ctx*);
int nnal_tc_fc(nnal_ctx*, const Layer&, const float* in, float* out, int64_t n);
int nnal_tc_fc_planes(nnal_ctx*, const Layer&, const nnal_h* Ah, const nnal_h* Al, int lda, float* out,
                      nnal_h* out_hi, nnal_h* out_lo, int64_t n, const DropSpec* drop = nullptr);
int nnal_tc_gemm_planes(nnal_ctx*, const nnal_h* Ah, const nnal_h* Al, int64_t lda, int64_t M, const nnal_h* Bh,
                        const nnal_h* Bl, int64_t ldb, int N, int64_t K, const float* bias, float scale, int relu,
                        int accum, float* out, int ldo, nnal_h* out_hi, nnal_h* out_lo, int ld_split,
                        const DropSpec* drop = nullptr);
int nnal_k_split_flat(nnal_ctx*, const float* in, nnal_h* hi, nnal_h* lo, int64_t count);
int nnal_k_split_pad(nnal_ctx*, const float* in, nnal_h* hi, nnal_h* lo, int64_t rows, int C, int Cp);
int nnal_k_merge_flat(nnal_ctx*, const nnal_h* hi, const nnal_h* lo, float* out, int64_t count);
bool nnal_tc_conv_supported(const nnal_ctx*, const Layer&);
bool nnal_tc_conv_x16_supported(const nnal_ctx*, const Layer&);
// conv1 that gathers, normalises and x-im2col's its own input from the volume (no gather kernel, no input planes in HBM)
bool nnal_tc_conv1_fused_supported(const nnal_ctx*, const Layer&, const Volume&, int d1, int d2, int d3);
int nnal_tc_conv1_fused(nnal_ctx*, const Layer&, const FusedGather&, nnal_h* out_hi, nnal_h* out_lo, int64_t n);
NormTab nnal_make_norm_tab(const Volume& v, int d3, const double* h_stats, int norm_mode);
int nnal_tc_prepare_conv_x16(nnal_ctx*, Layer&);
int nnal_tc_conv_x16(nnal_ctx*, const Layer&, const nnal_h* in_hi, const nnal_h* in_lo, nnal_h* out_hi, nnal_h* out_lo, int64_t n);
int nnal_k_split_x16(nnal_ctx*, const float* in, nnal_h* hi, nnal_h* lo, int64_t rows, int W, int C, int KW);
bool nnal_k_gather_x16_supported(const Volume&, int d1, int d2, int d3);
int nnal_k_gather_x16(nnal_ctx*, const Volume&, const int64_t* d_inds, int64_t n, int d1, int d2, int d3,
                      const double* h_stats, int norm_mode, nnal_h* out_hi, nnal_h* out_lo);
// data-gradient convolutions on the tensor cores (conv_tc.cu; used by shrunk.cu)
bool nnal_tc_conv_bwd_supported(const nnal_ctx*, const Layer&);
int nnal_tc_conv_bwd_prepare(nnal_ctx*, const Layer&, void** packed);
int nnal_tc_conv_bwd(nnal_ctx*, const Layer&, const void* packed, const nnal_h* dz_hi, const nnal_h* dz_lo, float* d_in, int64_t n,
                     float scale_inv);
bool nnal_tc_conv_pool_supported(const nnal_ctx*, const Layer&);
int nnal_tc_conv_pool(nnal_ctx*, const Layer&, const nnal_h* in_hi, const nnal_h* in_lo, nnal_h* out_hi, nnal_h* out_lo,
                      int64_t n);
int nnal_tc_conv(nnal_ctx*, const Layer&, const nnal_h* in_hi, const nnal_h* in_lo, nnal_h* out_hi,
                 nnal_h* out_lo, int64_t n);
// conv_wt.cu (weight-stationary tcgen05 conv, optional fused 2x2 max-pool)
bool nnal_wt_conv_supported(const nnal_ctx*, const Layer&);
bool nnal_wt_conv_preferred(const nnal_ctx*, const Layer&);
bool nnal_wt_conv_pool_supported(const nnal_ctx*, const Layer&);
int nnal_wt_prepare_conv(nnal_ctx*, Layer&);
int nnal_wt_conv(nnal_ctx*, const Layer&, const nnal_h* in_hi, const nnal_h* in_lo, nnal_h* out_hi, nnal_h* out_lo,
                 int64_t n, int fuse_pool);
int nnal_k_conv_simt_split(nnal_ctx*, const Layer&, const float* in, nnal_h* out_hi, nnal_h* out_lo, int64_t n);
int nnal_k_pool_split(nnal_ctx*, const Layer&, const nnal_h* in_hi, const nnal_h* in_lo, nnal_h* out_hi,
                      nnal_h* out_lo, int64_t n);
// input_format: 0 fp32 NHWC in xin, 1 fp16 hi/lo planes padded to 8 channels, 2 x-im2col'd fp16 hi/lo planes (16 per position),
// 3 none: the first conv gathers its input from the volume (ctx->fg)
int nnal_forward_chunk(nnal_ctx*, int64_t nb, int64_t offset, int input_format = 0);
bool nnal_first_layer_wants_split8(const nnal_ctx*);
bool nnal_first_layer_wants_x16(const nnal_ctx*);
// shrunk.cu / sdp.cu
int nnal_bw_release(nnal_ctx*);
int nnal_sdp_release(nnal_ctx*);
int nnal_upload_stats(nnal_ctx*, const double* stats, int m, int norm_mode, double** d_stats);
int nnal_check_gather_args(nnal_ctx*, int subject, int64_t n, int d1, int d2, int d3, const Volume** vout);
// fi.cu
int nnal_gj64_invert(nnal_ctx*, double* M, int np);      // in-place inverse of an SPD float64 matrix, np % 64 == 0
int nnal_k_fi_trace_scores(nnal_ctx*, const float* post, int c, int64_t n, const float* feat, int d, double* score);
