// Forward driver: walks the layer list for one chunk of samples and picks, per layer, the tensor-core
// kernel (fp16 hi/lo operand planes) or the FP32 CUDA-core kernel, converting the activation format
// only where two neighbouring layers disagree.  Replaces one sess.run(model.posteriors / feature_layer)
// of PW_NN.batch_eval (PW_NN.py:522-524).
#include "nnal_common.cuh"
#include <algorithm>

namespace {

struct Act {
  float* f32 = nullptr;
  nnal_h* hi = nullptr;
  nnal_h* lo = nullptr;
  bool split = false;
  int64_t elems = 0;        // per sample
};

bool layer_on_tc(const nnal_ctx* ctx, int i) {
  if (!ctx->use_tc) return false;
  const int nl = (int)ctx->layers.size();
  if (i < 0 || i >= nl) return false;
  const Layer& L = ctx->layers[i];
  // the last FC: c <= 32 runs in the fused head kernel, c >= 64 as the wide head's logits GEMM where it is supported
  if (i == nl - 1) return L.out_dim >= NNAL_WIDE_HEAD_MIN && nnal_tc_head_supported(ctx, L);
  if (L.type == NNAL_LAYER_CONV) return nnal_tc_conv_supported(ctx, L);
  if (L.type == NNAL_LAYER_FC) return nnal_tc_fc_supported(ctx, L);
  return false;
}

// does the consumer of layer i's output (skipping pools) want fp16 hi/lo planes?
bool consumer_wants_split(const nnal_ctx* ctx, int i) {
  const int nl = (int)ctx->layers.size();
  int j = i + 1;
  while (j < nl && ctx->layers[j].type == NNAL_LAYER_POOL) ++j;
  return layer_on_tc(ctx, j);
}

// wide head on the tensor cores from split features [nb][elems]: logits GEMM into the head's scratch, then the softmax
// into the pool posteriors at `offset`
int wide_head_planes(nnal_ctx* ctx, const Layer& L, const Act& a, int64_t nb, int64_t offset, const DropSpec* drop) {
  const int ldz = nnal_head_ldz(L.out_dim);
  NNAL_TRY(devbuf_reserve(ctx, ctx->head_logits, (size_t)nb * ldz * sizeof(float)));
  float* z = (float*)ctx->head_logits.p;
  NNAL_TRY(nnal_tc_head_planes(ctx, L, a.hi, a.lo, (int)a.elems, z, nb, drop));
  return nnal_k_softmax_wide(ctx, z, ldz, nb, L.out_dim, ctx->pool_n, offset, ctx->pool_post);
}

}  // namespace

bool nnal_layer_on_tc(const nnal_ctx* ctx, int i) { return layer_on_tc(ctx, i); }

bool nnal_first_layer_wants_split8(const nnal_ctx* ctx) {
  if (ctx->layers.empty()) return false;
  const Layer& L = ctx->layers[0];
  return L.type == NNAL_LAYER_CONV && L.in_c % 8 != 0 && L.in_c <= 8 && layer_on_tc(ctx, 0);
}

// conv1 on the x-im2col'd input (conv_tc.cu CfgConv1X): 3x fewer MMAs (conv1 4.2 -> 3.2 ms per 100k patches), but the
// gather then writes 40 KB instead of 20 KB per patch (0.84 -> 1.6 ms) and conv1 becomes bound by its 16-byte-row TMA
// loads and its epilogue: a net 0.3 ms.  Kept behind NNAL_CONV_X16=1 (tests cover it), off by default.
bool nnal_first_layer_wants_x16(const nnal_ctx* ctx) {
  if (ctx->layers.empty() || !ctx->use_x16) return false;
  return layer_on_tc(ctx, 0) && nnal_tc_conv_x16_supported(ctx, ctx->layers[0]);
}

int nnal_forward_chunk(nnal_ctx* ctx, int64_t nb, int64_t offset, int input_format) {
  const bool input_is_split8 = input_format == 1;
  bool input_is_x16 = input_format == 2;
  const bool fused_conv1 = input_format == 3;           // the first conv gathers its own input (ctx->fg)
  const int nl = (int)ctx->layers.size();
  Act cur;
  cur.f32 = (float*)ctx->xin.p;
  cur.elems = (int64_t)ctx->in_h * ctx->in_w * ctx->in_c;
  if (input_is_split8) {                  // the fused gather already wrote the first conv's 8-channel hi/lo planes
    cur.elems = (int64_t)ctx->in_h * ctx->in_w * 8;
    cur.hi = (nnal_h*)ctx->xin.p;
    cur.lo = cur.hi + nb * cur.elems;
    cur.split = true;
  }
  if (input_is_x16) {                     // the fused gather wrote conv1's x-im2col'd hi/lo planes
    cur.elems = (int64_t)ctx->in_h * ctx->in_w * 16;
    cur.hi = (nnal_h*)ctx->xin.p;
    cur.lo = cur.hi + nb * cur.elems;
    cur.split = true;
  }
  int pp = 0;
  auto next_buf = [&](int64_t elems, Act& o) {
    // both formats occupy 4 bytes per element: fp32, or an fp16 hi plane followed by an fp16 lo plane
    o.f32 = (float*)ctx->act[pp].p;
    o.hi = (nnal_h*)ctx->act[pp].p;
    o.lo = o.hi + nb * elems;
    o.elems = elems;
    pp ^= 1;
  };
  auto to_split = [&](Act& a) -> int {
    if (a.split) return NNAL_OK;
    Act o; next_buf(a.elems, o);
    NNAL_TRY(nnal_k_split_flat(ctx, a.f32, o.hi, o.lo, nb * a.elems));
    o.split = true; a = o;
    return NNAL_OK;
  };
  auto to_f32 = [&](Act& a) -> int {
    if (!a.split) return NNAL_OK;
    Act o; next_buf(a.elems, o);
    NNAL_TRY(nnal_k_merge_flat(ctx, a.hi, a.lo, o.f32, nb * a.elems));
    o.split = false; a = o;
    return NNAL_OK;
  };

  for (int i = 0; i < nl; ++i) {
    const Layer& L = ctx->layers[i];
    if (ctx->mc_T > 0 && i == ctx->fc_first) {
      // MC-dropout: the conv trunk is deterministic (PW1 drops out the FC outputs only, NN.py:1338) and was computed
      // once; the FC tail runs T times with fresh masks.  The tail ping-pongs between the activation buffer that does
      // not hold the trunk output and a third buffer.  The trunk's last layer writes the split planes the tail's first
      // FC layer takes, on either path; an FC-only net's fp32 input is split once here, not once per pass.
      if (layer_on_tc(ctx, i)) NNAL_TRY(to_split(cur));
      else NNAL_TRY(to_f32(cur));
      size_t maxfc = 0;
      for (int j = i; j < nl; ++j) maxfc = std::max(maxfc, (size_t)ctx->layers[j].out_dim);
      NNAL_TRY(devbuf_reserve(ctx, ctx->act_mc, (size_t)nb * maxfc * sizeof(float)));
      void* bufs[2] = {ctx->act[pp].p, ctx->act_mc.p};
      for (int t = 0; t < ctx->mc_T; ++t) {
        Act h = cur;
        int q = 0;
        for (int j = i; j < nl; ++j) {
          const Layer& F = ctx->layers[j];
          DropSpec d = ctx->mc_drop;
          d.pass += (uint32_t)t;
          d.site = (uint32_t)j;
          bool site = false;
          for (int sj : ctx->mc_sites) site |= (sj == j);
          prof_begin(ctx, j);
          if (j == nl - 1 && layer_on_tc(ctx, j)) {
            // wide head on the tensor cores: the logits' dropout runs in the GEMM epilogue (rows are chunk-relative)
            if (!h.split) NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "MC-dropout: the wide head expects split features");
            d.row0 += offset;
            NNAL_TRY(wide_head_planes(ctx, F, h, nb, offset, site ? &d : nullptr));
          } else if (j == nl - 1) {
            if (h.split) NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "MC-dropout: the head expects fp32 features");
            NNAL_TRY(nnal_k_head(ctx, F, h.f32, nb, ctx->pool_n, offset, ctx->pool_post, nullptr, site ? &d : nullptr));
          } else {
            if (F.type != NNAL_LAYER_FC || !layer_on_tc(ctx, j) || !h.split)
              NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "MC-dropout: FC tail must run on the tensor-core path");
            Act o;
            o.f32 = (float*)bufs[q]; o.hi = (nnal_h*)bufs[q]; o.lo = o.hi + nb * F.out_dim; o.elems = F.out_dim;
            q ^= 1;
            const bool ws = consumer_wants_split(ctx, j);
            d.row0 += offset;                    // FC rows are chunk-relative; the head adds the offset itself
            NNAL_TRY(nnal_tc_fc_planes(ctx, F, h.hi, h.lo, F.in_dim, ws ? nullptr : o.f32, ws ? o.hi : nullptr,
                                       ws ? o.lo : nullptr, nb, site ? &d : nullptr));
            o.split = ws;
            h = o;
          }
          prof_end(ctx);
        }
        prof_begin(ctx, NNAL_PROF_MC_ACCUM);
        NNAL_TRY(nnal_k_mc_accumulate(ctx, ctx->pool_post, ctx->n_class, ctx->pool_n, offset, nb, t, ctx->pool_mc_post,
                                      ctx->pool_mc_ent));
        prof_end(ctx);
      }
      return NNAL_OK;
    }
    prof_begin(ctx, i);
    if (i == nl - 1) {
      if (layer_on_tc(ctx, i)) {
        NNAL_TRY(to_split(cur));
        NNAL_TRY(wide_head_planes(ctx, L, cur, nb, offset, nullptr));
      } else {
        NNAL_TRY(to_f32(cur));
        NNAL_TRY(nnal_k_head(ctx, L, cur.f32, nb, ctx->pool_n, offset, ctx->pool_post, nullptr));
      }
      prof_end(ctx);
      break;
    }
    const bool want_split = consumer_wants_split(ctx, i);
    if (L.type == NNAL_LAYER_CONV) {
      const int64_t oe = (int64_t)L.out_h * L.out_w * L.out_c;
      if (layer_on_tc(ctx, i)) {
        if (i == 0 && !input_is_split8 && !input_is_x16 && nnal_first_layer_wants_x16(ctx)) {
          // fp32 input (images, unfused gather): x-im2col + split in one pass
          NNAL_TRY(to_f32(cur));
          Act o2; next_buf((int64_t)L.in_h * L.in_w * 16, o2);
          NNAL_TRY(nnal_k_split_x16(ctx, cur.f32, o2.hi, o2.lo, nb * L.in_h * L.in_w, L.in_w, L.in_c, L.kw));
          o2.split = true; cur = o2;
          input_is_x16 = true;
        }
        if (i == 0 && fused_conv1) {
          Act o; next_buf(oe, o);
          NNAL_TRY(nnal_tc_conv1_fused(ctx, L, ctx->fg, o.hi, o.lo, nb));
          o.split = true; cur = o;
          prof_end(ctx);
          continue;
        }
        if (i == 0 && input_is_x16) {
          Act o; next_buf(oe, o);
          NNAL_TRY(nnal_tc_conv_x16(ctx, L, cur.hi, cur.lo, o.hi, o.lo, nb));
          o.split = true; cur = o;
          prof_end(ctx);
          continue;
        }
        if (i == 0 && input_is_split8) {
          // nothing to do: planes come from the gather
        } else if (L.in_c % 8 != 0) {
          // the tensor-core conv consumes whole 8-channel chunks: zero-pad the channels while splitting
          NNAL_TRY(to_f32(cur));
          const int cp = (L.in_c + 7) / 8 * 8;
          Act o2; next_buf((int64_t)L.in_h * L.in_w * cp, o2);
          NNAL_TRY(nnal_k_split_pad(ctx, cur.f32, o2.hi, o2.lo, nb * L.in_h * L.in_w, L.in_c, cp));
          o2.split = true; cur = o2;
        } else {
          NNAL_TRY(to_split(cur));
        }
        // narrow layers: weight-stationary kernel; when a 2x2 max-pool follows it is fused into the epilogue
        const bool wt = ctx->use_wt >= 3 ? nnal_wt_conv_supported(ctx, L) : ctx->use_wt >= 1 && nnal_wt_conv_preferred(ctx, L);
        const bool fuse = wt && ctx->use_wt >= 2 && i + 1 < nl - 1 && ctx->layers[i + 1].type == NNAL_LAYER_POOL &&
                          ctx->layers[i + 1].kh == 2 && ctx->layers[i + 1].kw == 2 && nnal_wt_conv_pool_supported(ctx, L);
        const bool fuse_tc = !wt && ctx->use_wt >= 2 && i + 1 < nl - 1 && ctx->layers[i + 1].type == NNAL_LAYER_POOL &&
                             ctx->layers[i + 1].kh == 2 && ctx->layers[i + 1].kw == 2 && nnal_tc_conv_pool_supported(ctx, L);
        if (fuse || fuse_tc) {
          const Layer& P = ctx->layers[i + 1];
          Act o; next_buf((int64_t)P.out_h * P.out_w * P.out_c, o);
          if (fuse) NNAL_TRY(nnal_wt_conv(ctx, L, cur.hi, cur.lo, o.hi, o.lo, nb, 1));
          else NNAL_TRY(nnal_tc_conv_pool(ctx, L, cur.hi, cur.lo, o.hi, o.lo, nb));
          o.split = true; cur = o;
          prof_end(ctx);
          ++i;                                  // the pool layer is done
          continue;
        }
        Act o; next_buf(oe, o);
        if (wt) NNAL_TRY(nnal_wt_conv(ctx, L, cur.hi, cur.lo, o.hi, o.lo, nb, 0));
        else NNAL_TRY(nnal_tc_conv(ctx, L, cur.hi, cur.lo, o.hi, o.lo, nb));
        o.split = true; cur = o;
      } else {
        NNAL_TRY(to_f32(cur));
        Act o; next_buf(oe, o);
        if (want_split) { NNAL_TRY(nnal_k_conv_simt_split(ctx, L, cur.f32, o.hi, o.lo, nb)); o.split = true; }
        else { NNAL_TRY(nnal_k_conv_simt(ctx, L, cur.f32, o.f32, nb)); o.split = false; }
        cur = o;
      }
    } else if (L.type == NNAL_LAYER_POOL) {
      const int64_t oe = (int64_t)L.out_h * L.out_w * L.out_c;
      Act o; next_buf(oe, o);
      if (cur.split) { NNAL_TRY(nnal_k_pool_split(ctx, L, cur.hi, cur.lo, o.hi, o.lo, nb)); o.split = true; }
      else { NNAL_TRY(nnal_k_pool(ctx, L, cur.f32, o.f32, nb)); o.split = false; }
      cur = o;
    } else {
      // FC (not the last).  fp32 copies wanted by the pool state go straight to their final place.
      float* keep_dst = nullptr;
      if (ctx->keep >= 1 && i == ctx->feature_layer) keep_dst = ctx->pool_feat + offset * (int64_t)ctx->feat_dim;
      else if (ctx->keep >= 2 && i == ctx->feature_layer - 1 && L.out_dim == ctx->prev_dim)
        keep_dst = ctx->pool_prev + offset * (int64_t)ctx->prev_dim;
      if (layer_on_tc(ctx, i)) {
        NNAL_TRY(to_split(cur));
        Act o; next_buf(L.out_dim, o);
        float* f32_dst = keep_dst ? keep_dst : (want_split ? nullptr : o.f32);
        NNAL_TRY(nnal_tc_fc_planes(ctx, L, cur.hi, cur.lo, L.in_dim, f32_dst, want_split ? o.hi : nullptr,
                                   want_split ? o.lo : nullptr, nb));
        if (want_split) { o.split = true; }
        else { o.split = false; if (keep_dst) o.f32 = keep_dst; }
        cur = o;
      } else {
        NNAL_TRY(to_f32(cur));
        Act o; next_buf(L.out_dim, o);
        float* dst = keep_dst ? keep_dst : o.f32;
        NNAL_TRY(nnal_k_fc_simt(ctx, L, cur.f32, dst, nb));
        o.f32 = dst; o.split = false;
        cur = o;
      }
    }
    prof_end(ctx);
  }
  return NNAL_OK;
}
