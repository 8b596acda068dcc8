/* libnnal_b200 -- C ABI of the B200-native query-scoring path of nn-active-learning.
 *
 * This is the drop-in boundary (SURVEY.md §8b): plain pointers and sizes, int status codes,
 * caller-owned HOST buffers unless a parameter is named d_* (device pointer).  One context per
 * process and GPU; calls on one context are serialised by the caller.  No exceptions cross the
 * boundary; nnal_last_error() returns the message of the last failing call.
 *
 * The reference is pure Python (TensorFlow 1.x + NumPy); each entry point cites the reference
 * function (file:line in jsourati/nn-active-learning) whose work it replaces.  The Python package
 * nn-active-learning_b200 (import name nnal_b200) binds these with ctypes and re-exposes them under
 * the reference's own module/function names; INTEGRATION.md shows the binding.
 */
#ifndef NNAL_B200_H
#define NNAL_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct nnal_ctx nnal_ctx;

/* status codes */
#define NNAL_OK 0
#define NNAL_ERR_INVALID 1      /* bad argument (the reference would raise ValueError/IndexError) */
#define NNAL_ERR_CUDA 2         /* CUDA runtime error; context is unusable afterwards */
#define NNAL_ERR_STATE 3        /* call order violated (e.g. scoring before a pool pass) */
#define NNAL_ERR_UNSUPPORTED 4  /* shape outside what the kernels cover */
#define NNAL_ERR_NO_DEVICE 5    /* no CUDA device / not an sm_100 part: there is NO CPU fallback */
#define NNAL_ERR_OVERFLOW 6     /* an input, weight or activation left the fp16 operand range of the tensor-core path
                                   (|x| > 65504 or not finite): results of the pass are invalid.  Returned by the calls that
                                   hand pool results to the caller; the reference's fp32 TF path has no such limit --
                                   rescale the input or switch to the FP32 kernels with nnal_set_tensor_cores(ctx, 0). */

/* layer kinds of NN.CNN's layer_dict (NN.py:98-108): [out,'conv',[kh,kw]] / [[p,p],'pool'] / [out,'fc'] */
#define NNAL_LAYER_CONV 0
#define NNAL_LAYER_POOL 1
#define NNAL_LAYER_FC 2
typedef struct { int32_t type, out, kh, kw; } nnal_layer_spec;

/* element types of volumes handed to nnal_volume_set */
#define NNAL_F32 0
#define NNAL_F64 1

/* normalisation applied by the gather */
#define NNAL_NORM_NONE 0
#define NNAL_NORM_BATCH_EVAL 1  /* PW_NN.py:503-506: channel ch<m uses stats[ch] */
#define NNAL_NORM_MULTIMG 2     /* patch_utils.py:1203-1207: block ch/d3 uses stats[ch/d3] */

/* score kinds */
#define NNAL_SCORE_BINARY 0     /* |P(class1) - 0.5|          (PW_NNAL.py:64,109-110,724-730) */
#define NNAL_SCORE_NEG_ENTROPY 1 /* sum_c p log p = -H        (NNAL.py:309-310, NNAL_tools.py:32-34) */
#define NNAL_SCORE_ENTROPY 2    /* H                          (NNAL_tools.py:71-85) */
#define NNAL_SCORE_NEG_FI_TRACE 3 /* -(1-|pi|^2)(|u|^2+1): minus the trace of the last-layer FI (NNAL.py:121-139);
                                     needs a pool pass that kept the feature layer */

#define NNAL_SCORE_MC_BINARY 10 /* |mean_t P_t(class1) - 0.5| over the MC-dropout passes (PW_NNAL.py:67-87, 232-244) */
#define NNAL_SCORE_NEG_BALD 11  /* -(H(mean_t P_t) - mean_t H(P_t)), zeros bumped by 1e-6 (PW_NNAL.py:247-282): ascending
                                   top-k of it = np.argsort(-scores)[:k] */

/* ---- context ------------------------------------------------------------------------------- */
int nnal_version(void);
/* Creates a context on CUDA device `device`.  Fails with NNAL_ERR_NO_DEVICE when there is no
 * usable sm_100 GPU: the product path has no CPU fallback. */
int nnal_ctx_create(int device, nnal_ctx** out);
int nnal_ctx_destroy(nnal_ctx* ctx);
const char* nnal_last_error(nnal_ctx* ctx);
/* kernels launched by this context so far (bench.py's gpu_launches) */
long long nnal_launch_count(nnal_ctx* ctx);
/* 0: every conv/fc layer on the FP32 CUDA-core kernels (no fp16 operand range limit); 1 (default): tcgen05 tensor-core
 * kernels (fp16 hi/lo split operands, 3 MMAs per product, FP32 accumulate) for the shapes they cover. */
int nnal_set_tensor_cores(nnal_ctx* ctx, int enable);
int nnal_synchronize(nnal_ctx* ctx);
/* the context's CUDA stream (cudaStream_t) so host code can record CUDA events on it */
void* nnal_stream(nnal_ctx* ctx);

/* free / total bytes of the context's device (cudaMemGetInfo): the host layer sizes what it keeps resident with it */
int nnal_device_memory(nnal_ctx* ctx, uint64_t* free_bytes, uint64_t* total_bytes);
/* 64-bit content hash of a caller-owned HOST array (multi-threaded, ~50 GB/s): the host layer re-uploads a volume or a
 * weight set exactly when its full content changed since the last query (the reference passes the same padded volumes
 * every AL iteration, PW_AL.py:848-853, and fine-tunes the weights in between). */
int nnal_host_hash(const void* data, uint64_t bytes, uint64_t* out);

/* Per-kernel-class device timing (CUDA events on the context stream) for bench.py's roofline leg.
 * cls: layer index (0..n_layers-1), 100 gather, 101 scores, 102 top-k, 110-113 FI setup / Gram / greedy / Gram solve,
 * 120 / 121 forward / backward of the shrunk-gradient pass. */
int nnal_profile(nnal_ctx* ctx, int enable);
int nnal_profile_read(nnal_ctx* ctx, int cls, double* total_ms, long long* count);

/* ---- model: replaces the TF graph built by NN.CNN / NN.create_PW1 (NN.py:56-345, 1319-1359) --- */
/* Input is NHWC [*, in_h, in_w, in_c]; conv = SAME/stride 1 + bias + ReLU (NN.py:285-290); pool =
 * max, SAME, window=stride (NN.py:1473-1477); fc = W x + b with ReLU except on the last layer
 * (NN.py:213-241, 322-327).  feature_layer is the index into `specs` whose output is
 * model.feature_layer (NN.py:173-176); -1 = second to last. */
int nnal_model_set(nnal_ctx* ctx, const nnal_layer_spec* specs, int n_layers, int in_h, int in_w, int in_c,
                   int feature_layer);
/* Weights in the reference's TF variable layouts (NN.py:270-283, 311-320; the HDF5 layout of
 * NN.save_weights NN.py:379-396): conv W[kh][kw][cin][cout], b[cout]; fc W[out][in] with the
 * reference's flatten order in = c*(W*H)+w*H+h (NN.py:296-301), b[out]. */
int nnal_model_set_weights(nnal_ctx* ctx, int layer, const float* W, const float* b);
int nnal_model_info(nnal_ctx* ctx, int* n_class, int* feat_dim, int* prev_dim);
/* multiply-accumulates per sample of layer `layer` and the kernel family it runs on: 0 FP32 CUDA cores, 1 tcgen05
 * (conv_tc_kernel / fc_tc_kernel), 2 tcgen05 weight-stationary conv (conv_wt_kernel) */
int nnal_model_layer_info(nnal_ctx* ctx, int layer, int* type, long long* macs_per_sample, int* uses_tc);

/* ---- volumes: the padded multi-modality images the query functions receive ----------------- */
/* Uploads subject `subject` (m modality arrays, each C-contiguous (X,Y,Z), z fastest, as
 * PW_AL.py:737-761 builds them) and re-lays it out as [Z][X][Y][m] in HBM.  pad_* > 0 adds zero
 * padding on the device (get_patches(..., padded=False), patch_utils.py:1118-1132). */
int nnal_volume_set(nnal_ctx* ctx, int subject, int m, const void* const* mods, int dtype, int64_t X, int64_t Y,
                    int64_t Z, int64_t pad_x, int64_t pad_y, int64_t pad_z);
/* Same, from DEVICE memory: d_stage = the m modality arrays back to back, each C-contiguous (X,Y,Z).  Multi-GPU host
 * layer: every rank copies 1/world of each volume host->device and the parts are all-gathered over NVLink (NCCL on
 * nnal_stream()), so a volume crosses PCIe once per box instead of once per GPU. */
int nnal_volume_set_device(nnal_ctx* ctx, int subject, int m, const void* d_stage, int dtype, int64_t X, int64_t Y,
                           int64_t Z, int64_t pad_x, int64_t pad_y, int64_t pad_z);
int nnal_volume_clear(nnal_ctx* ctx);

/* ---- patch gather: replaces patch_utils.get_patches (patch_utils.py:1087-1173) --------------- */
/* inds: raveled C-order voxel ids of the UNPADDED volume (:1144).  out: float64
 * [n][d1][d2][m*d3], channel j*d3+dz (:1156-1165); bit-exact.  stats: [m][2] (mu,sigma) or NULL. */
int nnal_gather(nnal_ctx* ctx, int subject, const int64_t* inds, int64_t n, int d1, int d2, int d3,
                const double* stats, int norm_mode, double* out);

/* Device-resident variants for the memory-bound full-volume path (PW_analyze_results.full_slice_eval
 * PW_analyze_results.py:689-715 gathers every voxel of a slice; eval_utils.py:153-175 holds posteriors as
 * [c,h,w,z]): d_inds / d_out / d_post are DEVICE pointers, float32 patches [n][d1][d2][m*d3] resp. a float32
 * entropy map [n] from float32 posteriors [c][n] (zeros -> eps as compute_entropy). */
int nnal_gather_device_f32(nnal_ctx* ctx, int subject, const int64_t* d_inds, int64_t n, int d1, int d2, int d3,
                           const double* stats, int norm_mode, float* d_out);
int nnal_entropy_device_f32(nnal_ctx* ctx, const float* d_post, int c, int64_t n, double eps, float* d_out);

/* ---- pool pass: replaces PW_NN.batch_eval (PW_NN.py:357-539) + the TF forward --------------- */
/* Declares a pool of n_total samples scored in this query round.  keep = 0: posteriors only; 1: also
 * model.feature_layer; 2: also the input of the feature layer's FC (needed for two-layer FI). */
int nnal_pool_begin(nnal_ctx* ctx, int64_t n_total, int keep);
/* Gathers + normalises (float64 arithmetic, cast to float32 like the TF feed) + runs the forward
 * pass for n voxels of `subject`, writing pool positions [offset, offset+n). */
int nnal_pool_eval(nnal_ctx* ctx, int subject, const int64_t* inds, int64_t n, int64_t offset, int d1, int d2,
                   int d3, const double* stats, int norm_mode);
/* Same, for samples already in host memory as float32 NHWC [n][in_h][in_w][in_c] (whole-image
 * pools of NNAL.CNN_query, NNAL.py:298-306). */
int nnal_pool_eval_images(nnal_ctx* ctx, const float* x, int64_t n, int64_t offset);
/* Same, for samples resident in device memory (d_inds int64 device pointer) */
int nnal_pool_eval_device_inds(nnal_ctx* ctx, int subject, const int64_t* d_inds, int64_t n, int64_t offset, int d1,
                               int d2, int d3, const double* stats, int norm_mode);
/* MC-dropout (replaces feeding x_feed_dict = {model.keep_prob: model.dropout_rate} to PW_NN.batch_eval T times,
 * PW_NNAL.py:67-87, 232-282).  Configure BEFORE nnal_pool_begin; the following nnal_pool_eval* calls evaluate the conv
 * trunk once per chunk and the FC tail T times with tf.nn.dropout semantics (x / keep_prob where kept, NN.py:167-171)
 * on the outputs of `layers` (model.dropout_layers: FC layers only), keeping float64 running means of P(class 1) and of
 * the per-pass binary entropies for every pool sample.  Masks are Philox4x32-10 words keyed by `seed`, counter
 * {unit/4, pos0 + pool position, first_pass + t, layer}: independent of chunking and of how the pool is sharded.
 * T = 0 switches MC mode off.  Binary models only. */
int nnal_pool_mc_config(nnal_ctx* ctx, int T, double keep_prob, unsigned long long seed, unsigned int first_pass,
                        long long pos0, const int* layers, int n_layers);
/* Committee scorers 'ensemble' / 'QBC-JS' (PW_NNAL.py:453-545): fold member t's deterministic pool pass (the current
 * posteriors) into the same running means, av = (x + t av) / (t + 1).  t = 0 opens the accumulation,
 * nnal_pool_ensemble_end closes it; every member scores the same pool.  Scores: NNAL_SCORE_MC_BINARY / _NEG_BALD. */
int nnal_pool_ensemble_accumulate(nnal_ctx* ctx, int t);
int nnal_pool_ensemble_end(nnal_ctx* ctx);
/* running means after the pool pass: av_post [n_total], av_ent [n_total] (either may be NULL) */
int nnal_pool_mc_read(nnal_ctx* ctx, double* av_post, double* av_ent);
/* posteriors [c][n_total] float32 (layout of model.posteriors, NN.py:184-188) */
int nnal_pool_posteriors(nnal_ctx* ctx, float* out);
/* model.feature_layer as [feat_dim][n] columns start..start+n (PW_NN.py:530-531 layout) */
int nnal_pool_features(nnal_ctx* ctx, int64_t start, int64_t n, float* out);
/* score every pool sample (float64 like the reference) and keep the scores on the device */
int nnal_pool_score(nnal_ctx* ctx, int kind, double eps);
int nnal_pool_scores_read(nnal_ctx* ctx, double* out);
/* k smallest scores, ascending, ties -> lowest pool position: np.argsort(score)[:k] */
int nnal_pool_topk(nnal_ctx* ctx, int64_t k, int64_t* idx_out, double* score_out);

/* Device-resident form for the multi-GPU merge (SURVEY.md 8e collective 1; the reference ranks one concatenated
 * pool, PW_NNAL.py:724-730): writes k_pad pairs {float64 score, int64 pos_offset + pool position} of the k best
 * samples into DEVICE memory (slots k..k_pad-1 = {+inf, INT64_MAX}); the host layer all-gathers the pair buffers of
 * all ranks with NCCL on nnal_stream(); nnal_topk_merge_pairs then returns the global k smallest by (score,
 * position) to HOST arrays.  d_pairs of the merge is [world][k_pad], ranks owning ascending position blocks. */
int nnal_pool_topk_device(nnal_ctx* ctx, int64_t k, int64_t k_pad, int64_t pos_offset, void* d_pairs);
int nnal_topk_merge_pairs(nnal_ctx* ctx, const void* d_pairs, int64_t n_pairs, int64_t k, int64_t* pos_out,
                          double* score_out);

/* ---- stand-alone scoring helpers (host float64 in/out like the NumPy originals) -------------- */
/* NNAL_tools.compute_entropy (NNAL_tools.py:71-85): P [c][n]; zeros are treated as eps (the
 * in-place bump of the caller's array is done by the Python shim). kind as NNAL_SCORE_*. */
int nnal_entropy(nnal_ctx* ctx, const double* P, int c, int64_t n, int kind, double eps, double* out);
/* np.argsort(scores)[:k] */
int nnal_topk(nnal_ctx* ctx, const double* scores, int64_t n, int64_t k, int64_t* idx_out);

/* ---- Fisher-information scoring (PW_NNAL.py:89-163, 547-627, 738-816; NN.py:874-955) ---------- */
/* The conditional FI of a sample over the parameters of the last 1 or 2 FC layers is kept in FACTORED
 * form (NN.LLFC_grads NN.py:905-955, NNAL_tools.FC_gradnorms_batch NNAL_tools.py:725-775): for the
 * binary model Abar_i = w_i gbar_i gbar_i^T, w_i = p_i(1-p_i), <gbar_i,gbar_j> = 2(u_i.u_j+1) +
 * (delta2_i.delta2_j)(a_i.a_j+1).  Selection is the deterministic greedy restatement of the reference's
 * SDP objective tr((sum_i q_i A_i)^-1) (NNAL_tools.py:576-659) at q = uniform(S); see DESIGN.md.
 *
 * Candidate set from the current pool pass (nnal_pool_begin keep >= n_layers): cand = n_cand pool
 * positions, or NULL for every pool sample.  Candidate indices used below are positions in this list. */
int nnal_fi_set_candidates(nnal_ctx* ctx, const int64_t* cand, int64_t n_cand, int n_layers /*1 or 2*/);
/* Candidate set from host factors: p1[n] = P(class 1), U[n][d] = feature-layer activations (input of the
 * last FC), A_prev[n][d_prev] = input of the feature layer's FC and w_last[2][d] = last FC weights (both
 * NULL for last-layer-only FI). */
int nnal_fi_set_factors(nnal_ctx* ctx, int64_t n, int d, int d_prev, const double* p1, const float* U,
                        const float* A_prev, const float* w_last);
/* n candidates, layers covered, widths and the parameter count D = 2(d+1) [+ d(d_prev+1)] */
int nnal_fi_info(nnal_ctx* ctx, int64_t* n_cand, int* n_layers, int* d, int* d_prev, double* param_dim);
/* Weighted penultimate-feature Gram  H = sum_i wq_i [u_i;1][u_i;1]^T over the candidates ((d+1)x(d+1)
 * float32, row-major) on tensor cores -- the last-layer FI of NN.LLFC_hess (NN.py:891-901) is
 * (v v^T) (x) H, never formed.  wq_i = q_i p_i(1-p_i), q from the host (n_cand) or uniform 1/n_cand if
 * NULL.  The result stays on the device (nnal_fi_gram_ptr: base pointer, rows = d+1, row stride ld, for
 * the NCCL all-reduce of per-GPU partials by the host layer) and is copied to H_out if non-NULL. */
int nnal_fi_gram(nnal_ctx* ctx, const double* q, float* H_out);
/* Same Gram over a SUBSET of the candidates -- the support of a query distribution such as the greedy selection:
 * cand[n_sub] = candidate indices, q_sub[n_sub] their weights (n_sub = 0: H = 0, a rank that owns no selected sample). */
int nnal_fi_gram_subset(nnal_ctx* ctx, const int64_t* cand, int64_t n_sub, const double* q_sub, float* H_out);
void* nnal_fi_gram_ptr(nnal_ctx* ctx, int64_t* rows, int64_t* ld);
int nnal_fi_gram_read(nnal_ctx* ctx, float* H_out);
/* Primal FI objective through the Gram currently on the device (i.e. after the host layer's NCCL all-reduce):
 * *tr_out = tr((delta I + scale H)^-1) by a blocked float64 Gauss-Jordan inversion on the device.  With scale = 2,
 * tr_out + (d+1)/delta = tr((sum_i q_i F_i + delta I)^-1) for the last-layer FI F_i = (v v^T) (x) w_i [u_i;1][u_i;1]^T of
 * NN.LLFC_hess (NN.py:891-901), the objective of NNAL_tools.py:589-602.  d_G2: optional DEVICE pointer to a second Gram
 * of the same layout (e.g. a copy of the pool-wide one): *ratio_out = tr((delta I + scale H)^-1 (delta I + scale G2)). */
int nnal_fi_gram_solve(nnal_ctx* ctx, double delta, double scale, const float* d_G2, double* tr_out, double* ratio_out);
/* Greedy FI selection: k candidates minimising f(S) = tr(((1/|S|) sum_{i in S} Abar_i + delta I)^-1) step
 * by step (ties: lowest candidate index).  sel_out[k]: candidate indices in selection order; obj_out[k]:
 * f(S_t) after each step; red_out[k]: its kernel-dependent part tr((delta I + K_SS/s)^-1).  Any of
 * obj_out / red_out may be NULL.  Fewer than k candidates: only n_cand entries are written. */
int nnal_fi_greedy(nnal_ctx* ctx, int64_t k, double delta, int64_t* sel_out, double* obj_out, double* red_out);
/* Multi-GPU greedy, one step split so that the host layer can combine ranks (NCCL): nnal_fi_begin once;
 * per step (1) local best candidate: loss, local candidate index (-1 if none) and tr C of the shared
 * winners' system (objective after the step = (D-s)/delta + s (trC + global loss), s = step+1);
 * (2) the owner exports its winner's message [u (d) | a (d_prev) | sqrt(w) as one double | row `step` of the
 * winners' kernel K_SS as step+1 doubles]; (3) every rank applies the global winner. */
int nnal_fi_begin(nnal_ctx* ctx, int64_t k, double delta);
int nnal_fi_step_local_best(nnal_ctx* ctx, int64_t step, double* loss_out, int64_t* cand_out, double* trC_out);
int nnal_fi_winner_factors(nnal_ctx* ctx, int64_t step, int64_t cand, float* factors_out /*NULL: size query*/,
                           int64_t* n_floats);
int nnal_fi_step_apply(nnal_ctx* ctx, int64_t step, const float* winner_factors, int64_t n_floats, int owner_is_local,
                       int64_t cand_local);

/* Device-resident form of the same step (no host round trip inside the loop): every rank packs its local best
 * into a fixed-size message in DEVICE memory (nnal_fi_msg_bytes), the host layer all-gathers the messages with
 * NCCL on nnal_stream(), and every rank applies the global winner (min loss, ties -> lowest global id) from the
 * gathered buffer [world][msg_bytes].  nnal_fi_set_gids gives the global ids of the local candidates (NULL:
 * local index); nnal_fi_result reads the selected global ids and the reduced objective per step. */
int nnal_fi_set_gids(nnal_ctx* ctx, const int64_t* gids, int64_t n);
int nnal_fi_msg_bytes(nnal_ctx* ctx, int64_t* bytes);
int nnal_fi_step_pack(nnal_ctx* ctx, int64_t step, void* d_msg);
int nnal_fi_step_apply_gathered(nnal_ctx* ctx, int64_t step, const void* d_msgs, int world, int rank);
int nnal_fi_result(nnal_ctx* ctx, int64_t k, int64_t* gids_out, double* red_out);

/* Greedy FI selection for multi-class models (2 <= c <= 32), last FC layer only, in block form (csrc/fi_block.cu):
 * F_i = A(pi_i) (x) [u_i;1][u_i;1]^T with A(pi) = diag pi - pi pi^T = L_i L_i^T (closed-form c x (c-1) factor of the
 * float64-renormalised posteriors), block kernel K_ij = (L_i^T L_j)(u_i.u_j + 1), D = c(d+1), r = c-1.  Same objective
 * f(S) = tr((sum_{i in S} F_i/|S| + delta I)^-1) = (D - |S| r)/delta + red(S), red(S) = tr((delta I + K_SS/|S|)^-1), and
 * the same conventions as nnal_fi_set_candidates / nnal_fi_set_factors / nnal_fi_greedy (ties: lowest candidate index;
 * fewer than k candidates: only n_cand entries written).  k (c-1) <= 4096.
 * Candidates from the current pool pass (keep >= 1; NULL = every pool sample), or from host factors:
 * post[c][n] posteriors, U[n][d] feature-layer activations (input of the last FC). */
int nnal_fi_block_set_candidates(nnal_ctx* ctx, const int64_t* cand, int64_t n_cand);
int nnal_fi_block_set_factors(nnal_ctx* ctx, int64_t n, int c, int d, const float* post, const float* U);
int nnal_fi_block_greedy(nnal_ctx* ctx, int64_t k, double delta, int64_t* sel_out, double* obj_out, double* red_out);

/* All-gather of the per-step messages over NVLink peer memory instead of NCCL (csrc/p2p.cu): 100 dependent steps of one small
 * message each are latency bound, and one kernel that stores into the peers' buffers and spins on their flags costs a third of
 * an NCCL call.  The reference has no distributed code; the contract is SURVEY.md 8e, collective 3.
 * nnal_p2p_alloc: (collective) allocate this rank's receive buffer for `world` slots of `slot_bytes` (multiple of 16) and return
 * its 64-byte CUDA IPC handle; nnal_p2p_open: open the peers' handles (`handles` = world x 64 bytes in rank order, own entry
 * ignored); nnal_p2p_allgather: enqueue exchange number `seq` (the same, increasing by one per call, on every rank) of the
 * `nbytes` at `d_send` on nnal_stream(); *d_recv = device address of the gathered [world][slot_bytes] buffer, valid for the
 * kernels enqueued after it until exchange seq + 2. */
int nnal_p2p_alloc(nnal_ctx* ctx, int world, int rank, int64_t slot_bytes, unsigned char* handle_out);
int nnal_p2p_open(nnal_ctx* ctx, const unsigned char* handles);
int nnal_p2p_allgather(nnal_ctx* ctx, const void* d_send, int64_t nbytes, uint64_t seq, void** d_recv);
/* same-process variant of nnal_p2p_open (several contexts in one process): nnal_p2p_base returns this context's buffer,
 * nnal_p2p_open_local takes the `world` buffers in rank order */
int nnal_p2p_base(nnal_ctx* ctx, void** own_base);
int nnal_p2p_open_local(nnal_ctx* ctx, void* const* bases);

/* ---- the reference's own FI coordinates: shrunk class-score gradients + SDP query distribution ------------------ */
/* Replaces the 2B single-sample sess.run(model.grad_posts[y]) calls of PW_NNAL.gen_A_matrices (PW_NNAL.py:773-807;
 * graph built by NN.get_gradients NN.py:621-645, all trainable layers) followed by NNAL_tools.shrink_gradient(grad,'sum')
 * (NNAL_tools.py:784-796): g_out[y][i][t] = (sum dlog p_y(x_i)/dW_t + sum dlog p_y(x_i)/db_t) / (size W_t + size b_t) for
 * every class y, sample i and parameterised layer t (creation order; tau of them), float64 [c][n][tau]; post_out (may be
 * NULL) = posteriors [c][n] float32.  One batched data-gradient backward pass, no parameter gradient is formed.
 * _images: samples as float32 NHWC [n][in_h][in_w][in_c] on the host (the normalised sel_patches of PW_NNAL.py:121-131);
 * _voxels: gathered and normalised on the device like nnal_pool_eval. */
int nnal_fi_shrunk_tau(nnal_ctx* ctx, int* tau);
int nnal_fi_shrunk_images(nnal_ctx* ctx, const float* x, int64_t n, float* post_out, double* g_out);
int nnal_fi_shrunk_voxels(nnal_ctx* ctx, int subject, const int64_t* inds, int64_t n, int d1, int d2, int d3,
                          const double* stats, int norm_mode, float* post_out, double* g_out);
/* Replaces NNAL_tools.SDP_query_distribution with lambda_ = 0 (NNAL_tools.py:612-659; solve_FIAL_SDP :576-610):
 * minimise sum_j t_j s.t. [[sum_i q_i A_i, e_j],[e_j^T, t_j]] >= 0, q >= 0, sum q = 1, i.e. tr((sum_i q_i A_i)^-1) over the
 * simplex.  A: n symmetric positive-definite tau x tau matrices (float64 [n][tau][tau], tau <= 16).  First-order
 * multiplicative algorithm on the device, q_i <- q_i (d_i/phi)^gamma (gamma in (0,1]; 0.5 is monotone, a larger value is
 * used until the objective increases once and 0.5 from then on), stopped at the
 * duality certificate max_i tr(M^-1 A_i M^-1) / tr(M^-1) - 1 <= tol or after max_iter iterations.  q_out [n];
 * t_out [tau] = diag((sum q_i A_i)^-1) (the SDP's t); *obj_out = sum_j t_j; *gap_out = the certificate of the returned q
 * (objective within gap, relative, of the optimum); any of t_out/obj_out/gap_out/iters_out may be NULL. */
int nnal_sdp_query_distribution(nnal_ctx* ctx, const double* A, int64_t n, int tau, double tol, int64_t max_iter,
                                double gamma, double* q_out, double* t_out, double* obj_out, double* gap_out,
                                int64_t* iters_out);
/* NNAL_tools.SDP_query_distribution with lambda_ > 0 (NNAL_tools.py:625-644): objective sum_j t_j - lambda_ sum_i q_i |x_i|^2
 * and the extra equalities X q = 0, X [d][n] (float64, row-major) = the zero-mean refined feature matrix ref_F of
 * PW_NNAL.py:146-151 / NNAL.py:417-447 (d < n, d <= 4096).  Feasible multiplicative natural-gradient method on the device
 * (every iterate satisfies q >= 0, sum q = 1, X q = 0 to rounding), stopped at the convexity certificate
 * (max_i g_i - nu) / max(|objective|, tr M^-1) <= tol.  *obj_out = tr((sum q_i A_i)^-1) - lambda_ sum_i q_i |x_i|^2. */
int nnal_sdp_query_distribution_reg(nnal_ctx* ctx, const double* A, int64_t n, int tau, double lambda_, const double* X, int d,
                                    double tol, int64_t max_iter, double* q_out, double* t_out, double* obj_out, double* gap_out,
                                    int64_t* iters_out);
/* Same solver, with the binary A-matrices of PW_NNAL.gen_A_matrices (PW_NNAL.py:766-814) assembled on the device from
 * the shrunk gradients g [2][n][tau] and p1 [n] = P(class 1): p < 1e-6 -> only g0, p > 1-1e-6 -> only g1,
 * A_i = (1-p) g0 g0^T + p g1 g1^T + diag_load I (bit-identical to the host assembly); saves the n tau^2 upload. */
int nnal_sdp_from_shrunk(nnal_ctx* ctx, const double* g, const double* p1, int64_t n, int tau, double diag_load, double tol,
                         int64_t max_iter, double gamma, double* q_out, double* t_out, double* obj_out, double* gap_out,
                         int64_t* iters_out);

/* ---- last-layer influence recursion (SURVEY.md 8f rank 4) ---------------------------------------------------------- */
/* Replaces PW_NNAL.stoch_approx_IF (PW_NNAL.py:851-881) with NN.LLFC_grads / NN.LLFC_hess (NN.py:874-955): V_0 = G,
 * V_{t+1} = (G + V_t) - H_t V_t / scale for t < T, where column i of G is the last-layer log-loss gradient of pool sample i
 * at label labels[i], [(e_y - pi) (x) u ; (e_y - pi)], and H_t = -LLFC_hess of training sample t = (diag pi - pi pi^T) (x)
 * [u;1][u;1]^T (the iteration's random draw: the caller passes the factors in iteration order).  Factored on the device:
 * the ((d+1)c)^2 Hessian is never formed.  pool_post [c][n], pool_U [n][d], tr_post [T][c], tr_U [T][d] float32 (what
 * model.posteriors / model.feature_layer return); V_out [(d+1)c][n] float64, rows = W (class-major, a*d+k) then biases. */
int nnal_if_lissa(nnal_ctx* ctx, int64_t n, int c, int d, const float* pool_post, const float* pool_U, const int64_t* labels,
                  int64_t T, const float* tr_post, const float* tr_U, double scale, double* V_out);

/* ---- representativeness queries over the feature layer (SURVEY.md 8f rank 1) ------------------------------- */
/* Rows = the samples of the current pool pass (nnal_pool_begin keep >= 1; feature width multiple of 8).
 * 'rep-entropy' (NNAL.py:466-523, PW_NNAL.py:284-351): cols [B][d] = feature rows of the B most uncertain samples
 * (every rank passes the same array), excl_pos = pool positions of this rank that belong to them (they are not
 * rows).  nnal_rep_set builds the cosine similarities [rows][B] on tensor cores; each greedy step is
 * nnal_rep_step_scores (local partial sums sum_rows max(cur_row, sims[row][j]) into a DEVICE float64 [B] array
 * that the host layer all-reduces) + nnal_rep_step_pick (arg-max, ties -> lowest column, update).
 * nnal_rep_greedy runs k steps in one process.  nnal_sel_result reads the selected columns / global ids. */
int nnal_rep_set(nnal_ctx* ctx, const float* cols, int64_t B, const int64_t* excl_pos, int64_t n_excl, int64_t k);
int nnal_rep_step_scores(nnal_ctx* ctx, double* d_scores);
int nnal_rep_step_pick(nnal_ctx* ctx, int64_t step, const double* d_scores);
int nnal_rep_greedy(nnal_ctx* ctx, int64_t k, int64_t* sel_out, double* val_out);
int nnal_sel_result(nnal_ctx* ctx, int64_t k, int64_t* sel_out, double* val_out);
/* PW_NNAL.get_cross_sims (PW_NNAL.py:1093-1136): out[i] = max_j cos(pool row i, F2[j]) (float64 [n] on the host);
 * the result also stays on the device as the starting point of a core-set selection (init = 2 below). */
int nnal_cross_sims(nnal_ctx* ctx, const float* F2, int64_t n2, double* out);
/* 'core-set' (PW_NNAL.py:353-451): k-center over the pool rows: q = argmin(sims) (ties -> lowest id),
 * sims = max(sims, cos(f_q, F_u)), sims[q] = inf.  init 0: sims = -inf; 1: host array sims0[n]; 2: device result
 * of the last nnal_cross_sims.  Multi-rank: per step nnal_cs_step_pack writes this rank's best (similarity, global
 * id, feature row) into a DEVICE message, the messages are all-gathered, nnal_cs_step_apply_gathered applies the
 * global winner.  nnal_cs_greedy runs k steps in one process. */
int nnal_cs_begin(nnal_ctx* ctx, int init, const double* sims0, const int64_t* gids, int64_t k);
int nnal_cs_msg_bytes(nnal_ctx* ctx, int64_t* bytes);
int nnal_cs_step_pack(nnal_ctx* ctx, int64_t step, void* d_msg);
int nnal_cs_step_apply_gathered(nnal_ctx* ctx, int64_t step, const void* d_msgs, int world, int rank);
int nnal_cs_greedy(nnal_ctx* ctx, int64_t k, int64_t* sel_out, double* val_out);
/* feature rows of the given pool positions as [n][d] float32 on the host (row-major) */
int nnal_pool_feature_rows(nnal_ctx* ctx, const int64_t* pos, int64_t n, float* out);

/* ---- test hooks --------------------------------------------------------------------------- */
/* Kernel-selection switches for TESTS (there are no environment variables): "chunk" / "bw_chunk" (samples per chunk of the
 * forward / shrunk-gradient pass), "no_fused_gather", "conv_wt" (0..3), "conv_x16" (set before the weights are uploaded),
 * "wt_flags", "sdp_no_coop", "bw_no_ws", "bw_no_tc8", "bw_no_tc", "bw_simt_fwd" select fallback kernels so that every code
 * path can be held to the same parity bar.  The product path never calls this. */
int nnal_debug_option(nnal_ctx* ctx, const char* name, long value);
/* Declares a pool of n samples with the given float64 scores (no model, no pool pass): drives nnal_pool_topk /
 * nnal_pool_topk_device with arbitrary scores in tests. */
int nnal_debug_set_pool_scores(nnal_ctx* ctx, const double* scores, int64_t n);

/* One FC layer out[M][N] = act(A[M][K] W[N][K]^T + b) on host buffers, on the tcgen05 GEMM
 * (use_tc=1) or the FP32 CUDA-core GEMM (use_tc=0); lets tests check the kernels in isolation. */
int nnal_debug_fc(nnal_ctx* ctx, const float* A, const float* W, const float* b, int64_t M, int N, int K, int relu,
                  int use_tc, float* out);

/* One conv layer (SAME, stride 1, bias, ReLU; NN.py:285-290) on host NHWC buffers.  use_tc: 0 CUDA-core kernel,
 * 1 tcgen05 kernel with positions on M (conv_tc.cu), 2 weight-stationary tcgen05 kernel (conv_wt.cu), 3 = 2 and 4 = 1 with
 * the following 2x2/s2 SAME max-pool (NN.py:1473-1477) fused: out is then [n][ceil(H/2)][ceil(Wd/2)][Cout];
 * 5 = PW1 conv1 with the 5 filter columns folded into the channel axis (x-im2col'd input, conv_tc.cu CfgConv1X). */
int nnal_debug_conv(nnal_ctx* ctx, const float* x, const float* W, const float* b, int64_t n, int H, int Wd, int Cin,
                    int Cout, int ks, int use_tc, float* out);

#ifdef __cplusplus
}
#endif
#endif /* NNAL_B200_H */
