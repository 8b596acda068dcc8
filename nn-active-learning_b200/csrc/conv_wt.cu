// Weight-stationary ("transposed") tcgen05 implicit-GEMM convolution (SAME, stride 1, bias, ReLU, optional fused
// 2x2/s2 SAME max-pool) for the narrow conv layers of the patch CNN (sm_100a).
//
// Replaces tf.nn.conv2d + bias + relu (+ tf.nn.max_pool) of NN.CNN.add_conv / add_pool (NN.py:258-301, 329-340,
// 1473-1477) for layers with few output channels (PW1 conv1: 24, conv2: 32, conv3: 48).
//
// Why a second conv kernel.  conv_tc.cu puts raster positions on the MMA's M axis and output channels on N.  With
// N = Cout = 24..48 every 128x16 A tile (4 KB of shared memory) feeds only 16-32 tensor-core cycles, so the layer is
// bound by the tensor core's shared-memory operand fetch (128 B/clk), not by math: profiles/r1_forward_full.md
// reads 41 % tensor-pipe active for conv2.  Here the roles are swapped:
//
//     D[row, p] = sum_k  Wstack[row, k] * X[p + shift(k), k]          M = 128 stacked weight rows,  N = 256 positions
//
//   * B operand = 256 consecutive positions of the zero-padded raster (the same no-swizzle K-major layout and the
//     same "shift = descriptor start address" trick as conv_tc.cu: no im2col), so one MMA runs 128 tensor-core
//     cycles against 96 cycles of operand fetch (4 KB of weights + 8 KB of positions): math bound.
//   * A operand = weights.  Cout is far below 128, so the 128 rows stack what would otherwise be separate MMAs:
//     TAPS = 2:  rows = [W_hi(tap a) | W_lo(tap a) | W_hi(tap b) | W_lo(tap b)],  b = a + (0,2)   (conv1, conv2)
//     TAPS = 1:  rows = [W_hi(tap a) | W_lo(tap a)]                                             (conv3)
//     One MMA with B = X_hi therefore yields hi.hi and hi.lo of two taps at once; a second MMA with the SAME A
//     block and B = X_lo adds lo.hi (and the harmless 2^-22 lo.lo).  The partial sums of tap b belong to the
//     output two positions to the left: out[p] = D_a[p] + D_b[p + 2].  A shift along N is a TMEM *column* offset,
//     i.e. free for tcgen05.ld; tiles advance by 248 positions so that the shifted columns always exist.
//     (scripts/microbench/mma_rate.cu: an M = 128, K = 16 MMA costs max(N/2, (4 KB + 32 N) / 128 B/clk) cycles, so below
//     N = 128 the 4 KB A read dominates and the tensor core idles: N = 32 runs at 40 % of the math rate at best.)
//   * All weight blocks of the layer (conv2: 23 x 4 KB) stay resident in shared memory for the life of the CTA:
//     no weight streaming at all.  That leaves room for only ONE input raster (conv2: 81 KB), which is loaded in
//     two row bands with separate full/empty barriers: the lower band of the next sample arrives while the last
//     tile of the current sample is still being multiplied.
//   * Epilogue (NEW warpgroups on alternate 32-column sub-blocks, each warp on its own TMEM lane quadrant): the
//     partial sums of a channel (hi/lo weight rows, two tap groups) are stacked 8 rows apart, and
//     tcgen05.ld.16x256b delivers rows r and r + 8 to the SAME thread, so they add up in registers -- no shuffles,
//     no shared-memory staging, no barriers between epilogue warps.  Then bias, ReLU, and either fp16 hi/lo planes
//     in global memory or (POOL) an atomicMax into a pooled raster in shared memory that is written out once per
//     sample: the separate max-pool pass and the full-size activation round trip through HBM disappear.
//     (History, profiles/r1_conv_wt.md: a shared-memory staged epilogue cost 30 % of the MMA rate through the
//     bandwidth it took from the operand fetch; a shuffle transpose-reduce was instruction bound.)
// Precision: fp16 hi/lo split operands, FP32 accumulation in TMEM, as conv_tc.cu / gemm_tc.cu (DESIGN.md §4).
// Warp roles: warp 0 input TMA, warp 1 MMA issuer, warp 2 TMEM allocator + one-off weight load, warps 4.. epilogue
// (the next sub-block's tcgen05.ld is in flight while the current one is stored).
#include "nnal_common.cuh"
#include "tc_ptx.cuh"

namespace cwt {
using namespace tcx;

template <int H_, int W_, int CIN_REAL_, int COUT_REAL_, int KS_, int TAPS_, int G_, int RL_, bool POOL_, int NEW_ = 2>
struct Cfg {
  static constexpr int NEW = NEW_;                        // epilogue warpgroups
  static constexpr int THREADS = 128 + 128 * NEW_;
  static constexpr int H = H_, W = W_, KS = KS_, TAPS = TAPS_, G = G_, RL = RL_;
  static constexpr bool POOL = POOL_, SPLIT = RL_ > 0;
  static constexpr int CIN_REAL = CIN_REAL_, COUT_REAL = COUT_REAL_;
  static constexpr int CIN = (CIN_REAL + 7) / 8 * 8, Q = CIN / 8;
  static constexpr int CBT = 4 / TAPS;                    // 16-channel blocks (one epilogue warp each) per tap group
  static constexpr int COUT_MAX = 16 * CBT;
  static constexpr int PH = KS / 2, HP = H + KS - 1, WP = W + KS - 1;
  static constexpr int RASTER1 = HP * WP, RASTER = G * RASTER1;
  // B shifts per filter row.  TAPS == 2 pairs the taps (dx, dx + 2): dx_a = 0, 1, 4, 5, 8, ... (the TMEM column offset
  // of tcgen05.ld.16x256b must be even, so the pair distance is 2, not 1)
  static constexpr int NSLOT_ROW = TAPS == 1 ? KS : (KS / 4) * 2 + (KS % 4 < 2 ? KS % 4 : 2);
  __host__ __device__ static constexpr int dx_a(int pr) { return TAPS == 1 ? pr : 4 * (pr / 2) + pr % 2; }
  static constexpr int NSLOT = KS * NSLOT_ROW;
  static constexpr int NCS = NSLOT * Q;                   // (slot, 8-channel chunk) pairs = K / 8
  static constexpr int NBLK = (NCS + 1) / 2;              // K = 16 weight blocks (4 KB each)
  static constexpr int TILE_N = 256, TILE_OUT = TAPS == 2 ? TILE_N - 8 : TILE_N;   // TAPS == 2: tap group b is read 2 columns further; its last 8-column block is not
  static constexpr int LAST_VALID = (G - 1) * RASTER1 + (H - 1) * WP + (W - 1);
  static constexpr int T = LAST_VALID / TILE_OUT + 1;     // position tiles per sample group
  static constexpr int MAX_OFF = (KS - 1) * WP + (KS - 1);
  static constexpr int PLANE = (RASTER * 16 + 127) / 128 * 128;
  static constexpr int READ_END = (T - 1) * TILE_OUT + TILE_N + MAX_OFF + 1;   // positions a plane is read up to
  static constexpr int OVERRUN = READ_END * 16 > PLANE ? READ_END * 16 - PLANE : 0;
  static constexpr int IN_BYTES = (2 * Q * PLANE + OVERRUN + 1023) / 1024 * 1024;   // hi planes then lo planes
  static constexpr int NBUF = SPLIT ? 1 : 2;
  static constexpr int W_BYTES = NBLK * 4096;
  static constexpr int PHO = (H + 1) / 2, PWO = (W + 1) / 2;
  static constexpr int PSTRIDE = COUT_MAX + 8;             // pooled-cell stride (words), = 8 mod 32: the 4 cells a warp touches per atomic land in different banks
  static constexpr int POOL_BYTES = POOL ? (PHO * PWO * PSTRIDE * 4 + 15) / 16 * 16 : 0;
  static constexpr int SMEM = NBUF * IN_BYTES + W_BYTES + POOL_BYTES + 1024 + 256;
  static constexpr int BYTES_L = 2 * Q * (SPLIT ? RL : HP) * WP * 16 * G;        // TMA bytes of the first band / whole raster
  static constexpr int BYTES_U = SPLIT ? 2 * Q * (HP - RL) * WP * 16 * G : 0;
  static_assert(TAPS == 1 || TAPS == 2, "tap stacking");
  static_assert(COUT_REAL <= COUT_MAX && COUT_REAL % 8 == 0, "output channels");
  static_assert(SMEM <= 232448, "shared memory budget");
  static_assert(T >= 1, "tiles");
  // band protocol: band L (raster rows < RL) must hold everything tile 0 reads and nothing tile T-1 reads
  static_assert(!SPLIT || (G == 1 && T >= 2), "row bands need a single-sample raster with at least two tiles");
  static_assert(!SPLIT || (TILE_N + MAX_OFF + 1 <= RL * WP), "tile 0 must read only band L");
  static_assert(!SPLIT || ((T - 1) * TILE_OUT >= RL * WP), "the last tile must read only band U");
  static_assert((RL * WP * 16) % 128 == 0, "TMA shared-memory destinations are 128-byte aligned");
  static_assert(!POOL || G == 1, "fused pooling works on single-sample groups");
};

struct Params {
  const uint8_t* wpack;     // [NBLK][2 K-halves][128 rows][8] fp16
  const float* bias;
  nnal_h* out_hi;           // [n][H][W][COUT_REAL]  or (POOL) [n][PHO][PWO][COUT_REAL]
  nnal_h* out_lo;
  int n;
  float w_scale_inv;
  int flags;                // diagnostics (NNAL_WT_FLAGS): 1 = skip the output stores / pool atomics (timing experiments only)
};

template <class C>
__global__ void __launch_bounds__(C::THREADS, 1)
conv_wt_kernel(const __grid_constant__ CUtensorMap tmHiL, const __grid_constant__ CUtensorMap tmLoL,
               const __grid_constant__ CUtensorMap tmHiU, const __grid_constant__ CUtensorMap tmLoU, Params p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* base_ptr = smem_raw + (base - raw);
  const uint32_t in_base = base;
  const uint32_t w_base = in_base + C::NBUF * C::IN_BYTES;
  constexpr int POOL_OFF = C::NBUF * C::IN_BYTES + C::W_BYTES;
  constexpr int BAR_OFF = POOL_OFF + C::POOL_BYTES;
  uint32_t* pooled = reinterpret_cast<uint32_t*>(base_ptr + POOL_OFF);
  const uint32_t bar0 = base + BAR_OFF;
  // barrier map: in_full[buf][band], in_empty[buf][band], w_full, acc_full[2], acc_empty[2]
  auto in_full = [&](int b, int h) { return bar0 + 8u * (b * 2 + h); };
  auto in_empty = [&](int b, int h) { return bar0 + 8u * (4 + b * 2 + h); };
  const uint32_t w_full = bar0 + 8u * 8;
  auto acc_full = [&](int a) { return bar0 + 8u * (9 + a); };
  auto acc_empty = [&](int a) { return bar0 + 8u * (11 + a); };
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(base_ptr + BAR_OFF + 8 * 13);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ngroups = (p.n + C::G - 1) / C::G;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmHiL));
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmLoL));
    if (C::SPLIT) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(&tmHiU));
      asm volatile("prefetch.tensormap [%0];" ::"l"(&tmLoU));
    }
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < 8; ++i) mbar_init(bar0 + 8u * i, 1);
    mbar_init(w_full, 1);
    for (int a = 0; a < 2; ++a) { mbar_init(acc_full(a), 1); mbar_init(acc_empty(a), 4 * C::NEW); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  // Zero the raster buffers (slack after each plane is read, never written by TMA) and the pooled raster.
  {
    uint4* z = reinterpret_cast<uint4*>(base_ptr);
    for (int i = threadIdx.x; i < C::NBUF * C::IN_BYTES / 16; i += blockDim.x) z[i] = make_uint4(0, 0, 0, 0);
    for (int i = threadIdx.x; i < C::POOL_BYTES / 4; i += blockDim.x) pooled[i] = 0u;
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  // Weight-block table: block -> B descriptor words of its two (slot, chunk) K halves.  Chunk-major order
  // (cs = q * NSLOT + slot, slots sorted by shift) keeps every leading-byte offset positive.
  __shared__ uint2 ktab[C::NBLK];
  for (int blk = threadIdx.x; blk < C::NBLK; blk += blockDim.x) {
    auto off_of = [](int cs) {
      const int q = cs / C::NSLOT, s = cs % C::NSLOT;
      const int dy = s / C::NSLOT_ROW, dx = C::dx_a(s % C::NSLOT_ROW);
      return (uint32_t)(q * C::PLANE + (dy * C::WP + dx) * 16);
    };
    const uint32_t off0 = off_of(2 * blk);
    uint32_t lbo = 16;                      // dummy second half of an odd K tail (zero weights): stay in-plane
    if (2 * blk + 1 < C::NCS) lbo = off_of(2 * blk + 1) - off0;
    ktab[blk] = make_uint2(off0 >> 4, ((lbo >> 4) & 0x3fffu) << 16);
  }
  // Output-offset table: (tile, column) -> element offset of that raster position inside the sample group's output
  // (POOL: word offset of its pooled cell), -1 for padding columns / rows and for the overlap column of a tile.
  __shared__ __align__(16) int otab[C::T * C::TILE_N];
  for (int i = threadIdx.x; i < C::T * C::TILE_N; i += blockDim.x) {
    const int t = i / C::TILE_N, col = i % C::TILE_N;
    const int pp = t * C::TILE_OUT + col;
    const int gs = pp / C::RASTER1, rem = pp % C::RASTER1;
    const int y = rem / C::WP, x = rem % C::WP;
    int o = -1;
    if (col < C::TILE_OUT && gs < C::G && y < C::H && x < C::W)
      o = C::POOL ? ((y >> 1) * C::PWO + (x >> 1)) * C::PSTRIDE : ((gs * C::H + y) * C::W + x) * C::COUT_REAL;
    otab[i] = o;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== input producer: per 8-channel plane one 4-D box {8ch, WP, rows, G} for hi and lo; OOB zero fill = SAME padding =====
    if (lane == 0) {
      uint32_t it = 0;
      for (int g = blockIdx.x; g < ngroups; g += gridDim.x, ++it) {
        const int b = it % C::NBUF;
        const uint32_t ph = (it / C::NBUF) & 1;
        const uint32_t dst = in_base + b * C::IN_BYTES;
        mbar_wait(in_empty(b, 0), ph ^ 1);
        mbar_arrive_expect_tx(in_full(b, 0), C::BYTES_L);
#pragma unroll 1
        for (int q = 0; q < C::Q; ++q) {
          tma_load_4d(dst + q * C::PLANE, &tmHiL, in_full(b, 0), q * 8, -C::PH, -C::PH, g * C::G);
          tma_load_4d(dst + (C::Q + q) * C::PLANE, &tmLoL, in_full(b, 0), q * 8, -C::PH, -C::PH, g * C::G);
        }
        if (C::SPLIT) {
          mbar_wait(in_empty(b, 1), ph ^ 1);
          mbar_arrive_expect_tx(in_full(b, 1), C::BYTES_U);
#pragma unroll 1
          for (int q = 0; q < C::Q; ++q) {
            tma_load_4d(dst + q * C::PLANE + C::RL * C::WP * 16, &tmHiU, in_full(b, 1), q * 8, -C::PH, -C::PH + C::RL, g * C::G);
            tma_load_4d(dst + (C::Q + q) * C::PLANE + C::RL * C::WP * 16, &tmLoU, in_full(b, 1), q * 8, -C::PH, -C::PH + C::RL, g * C::G);
          }
        }
      }
    }
  } else if (warp == 2) {
    // ===== one-off weight load: the whole layer stays in shared memory =====
    if (lane == 0) {
      mbar_arrive_expect_tx(w_full, C::W_BYTES);
      for (int o = 0; o < C::W_BYTES; o += 16384) {
        const int nbytes = C::W_BYTES - o < 16384 ? C::W_BYTES - o : 16384;
        bulk_load(w_base + o, p.wpack + o, nbytes, w_full);
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    const uint32_t idesc = make_idesc_bf16(128, C::TILE_N);
    constexpr uint32_t DESC_HI = 8u /*SBO 128 B*/ | (1u << 14) /*version*/;
    constexpr uint32_t A_LBO = (2048u >> 4) << 16;              // K-half stride of a weight block
    const uint32_t wb16 = w_base >> 4;
    mbar_wait(w_full, 0);
    uint32_t it_in = 0, it_acc = 0;
    for (int g = blockIdx.x; g < ngroups; g += gridDim.x, ++it_in) {
      const int b = it_in % C::NBUF;
      const uint32_t ph_in = (it_in / C::NBUF) & 1;
      const uint32_t r16 = (in_base + b * C::IN_BYTES) >> 4;
#pragma unroll 1
      for (int t = 0; t < C::T; ++t, ++it_acc) {
        if (t == 0) mbar_wait(in_full(b, 0), ph_in);
        if (C::SPLIT && t == 1) mbar_wait(in_full(b, 1), ph_in);
        const int a = it_acc & 1;
        const uint32_t ph_acc = (it_acc >> 1) & 1;
        mbar_wait(acc_empty(a), ph_acc ^ 1);
        tc_fence_after();
        if (elect_one_sync()) {
          const uint32_t d = tmem_base + a * C::TILE_N;
          const uint32_t tile16 = (uint32_t)(t * C::TILE_OUT);   // 16-byte units == positions
#pragma unroll 1
          for (int blk = 0; blk < C::NBLK; ++blk) {
            const uint2 e = ktab[blk];
            const uint32_t bh = (r16 + e.x + tile16) | e.y;
            const uint32_t bl = bh + ((C::Q * C::PLANE) >> 4);
            const uint64_t dA = ((uint64_t)DESC_HI << 32) | ((wb16 + blk * 256u) | A_LBO);
            umma_bf16(d, dA, ((uint64_t)DESC_HI << 32) | bh, idesc, blk != 0);    // [W_hi|W_lo] x X_hi
            umma_bf16(d, dA, ((uint64_t)DESC_HI << 32) | bl, idesc, 1);           // [W_hi|W_lo] x X_lo
          }
          umma_commit(acc_full(a));
          if (C::SPLIT) {
            if (t == C::T - 2) umma_commit(in_empty(b, 0));
            if (t == C::T - 1) umma_commit(in_empty(b, 1));
          } else {
            if (t == C::T - 1) umma_commit(in_empty(b, 0));
          }
        }
        __syncwarp();
      }
    }
  } else if (warp >= 4) {
    // ===== epilogue: NEW warpgroups, each takes every NEW-th 32-column sub-block of every tile; warps never meet =====
    // A warp owns one TMEM lane quadrant = 32 stacked weight rows, read as two 16-lane halves with tcgen05.ld.16x256b,
    // which hands rows r and r + 8 of a half to the SAME thread (thread T: rows T/4, T/4 + 8; columns 2 (T%4) + {0,1} of
    // every 8-column block).  The weight rows are ordered so that everything a thread receives belongs together:
    //   TAPS == 2: half = tap group, rows 0-7 W_hi / rows 8-15 W_lo of channels 8 w + 0..7; tap group b is read two
    //              columns further (out[p] = D_a[p] + D_b[p + 2]): 4 partial sums, 3 adds, no shuffles, no selects
    //   TAPS == 1: half = channel block, rows 0-7 W_hi / rows 8-15 W_lo of channels 16 w + 8 half + 0..7
    // so a thread ends up with 8 output positions of one channel (two channels for TAPS == 1).
    const int wgi = (warp - 4) >> 2;
    const int w = warp & 3;
    constexpr int NSB = C::TILE_N / 32;
    constexpr int NCH = C::TAPS == 2 ? 1 : 2;               // channels per thread
    const int cq = lane >> 2, m = lane & 3;
    int co[NCH];
    float bias[NCH];
    uint32_t chlim[NCH];
#pragma unroll
    for (int h = 0; h < NCH; ++h) {
      co[h] = C::TAPS == 2 ? 8 * w + cq : 16 * w + 8 * h + cq;
      bias[h] = co[h] < C::COUT_REAL ? __ldg(p.bias + co[h]) : 0.f;
    }
    uint32_t it = 0;
    for (int g = blockIdx.x; g < ngroups; g += gridDim.x) {
      // outputs of this sample group: table offsets are relative to its first sample; a partly filled last group
      // (or a channel beyond COUT_REAL) is cut off by the limit
      constexpr int SAMPLE_ELEMS = C::H * C::W * C::COUT_REAL;
      nnal_h* ghi = p.out_hi + (size_t)g * C::G * SAMPLE_ELEMS;
      nnal_h* glo = p.out_lo + (size_t)g * C::G * SAMPLE_ELEMS;
      const int left = p.n - g * C::G;
      const uint32_t glim = (uint32_t)((left < C::G ? left : C::G) * SAMPLE_ELEMS);   // a partly filled last group ends here
#pragma unroll
      for (int h = 0; h < NCH; ++h) chlim[h] = co[h] >= C::COUT_REAL ? 0u : C::POOL ? 0x7fffffffu : glim;
#pragma unroll 1
      for (int t = 0; t < C::T; ++t, ++it) {
        const int a = it & 1;
        const uint32_t ph_acc = (it >> 1) & 1;
        mbar_wait(acc_full(a), ph_acc);
        tc_fence_after();
        const uint32_t trowA = tmem_base + ((uint32_t)(w * 32) << 16) + (uint32_t)(a * C::TILE_N);
        const uint32_t trowB = trowA + (16u << 16) + (C::TAPS == 2 ? 2u : 0u);
        uint32_t ra[16], rb[16];
        auto issue = [&](int sb) {
          tmem_ld16x256_x4_issue(trowA + sb * 32, ra);
          if (C::TAPS == 2 && sb == NSB - 1) {
            // columns TILE_N, TILE_N + 1 do not exist: the last 8-column block of tap group b (outputs >= TILE_OUT) is skipped
            tmem_ld16x256_x2_issue(trowB + sb * 32, rb);
            tmem_ld16x256_x1_issue(trowB + sb * 32 + 16, rb + 8);
            rb[12] = rb[13] = rb[14] = rb[15] = 0u;
          } else {
            tmem_ld16x256_x4_issue(trowB + sb * 32, rb);
          }
        };
        issue(wgi);
#pragma unroll 1
        for (int sb = wgi; sb < NSB; sb += C::NEW) {
          tmem_ld_wait_2x16(ra, rb);
          float z[NCH][8];                         // [channel][block i, column k]: position 8 i + 2 m + k of the sub-block
#pragma unroll
          for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int k = 0; k < 2; ++k) {
              const float sa = __uint_as_float(ra[4 * i + k]) + __uint_as_float(ra[4 * i + 2 + k]);
              const float sb_ = __uint_as_float(rb[4 * i + k]) + __uint_as_float(rb[4 * i + 2 + k]);
              if (C::TAPS == 2) z[0][2 * i + k] = sa + sb_;
              else { z[0][2 * i + k] = sa; z[NCH - 1][2 * i + k] = sb_; }
            }
          if (sb + C::NEW < NSB) issue(sb + C::NEW);                      // next sub-block in flight during the stores
          uint32_t amax = 0u;                                             // fp16 range guard: largest |value| of the sub-block
          if (C::POOL) {
            // output offsets (or -1) of this thread's positions from the table; one shared-memory atomicMax per output
            const int* ot = otab + t * C::TILE_N + sb * 32 + 2 * m;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int2 o2 = *reinterpret_cast<const int2*>(ot + 8 * i);
#pragma unroll
              for (int k = 0; k < 2; ++k) {
                const uint32_t off = (uint32_t)(k ? o2.y : o2.x);
#pragma unroll
                for (int h = 0; h < NCH; ++h) {
                  if (off < chlim[h] && !(p.flags & 1)) {                 // -1 (padding / garbage column) fails too
                    const float rr = z[h][2 * i + k] * p.w_scale_inv + bias[h];
                    nnal_ovf_track(amax, rr);
                    const float o = rr > 0.f ? fminf(rr, 65504.f) : 0.f;
                    atomicMax(pooled + off + co[h], __float_as_uint(o));  // o >= +0: uint order == float order
                  }
                }
              }
            }
          } else {
            // fp16 hi/lo planes in global memory.  A thread holds 8 positions of ONE channel (2-byte scattered stores:
            // measured store bound); an 8x8 register transpose among the 8 lanes that share m (lane ^ 4, ^ 8, ^ 16)
            // turns that into ONE position with 8 consecutive channels: a 16-byte store per plane.
#pragma unroll
            for (int h = 0; h < NCH; ++h) {
              uint32_t P[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const float rr = z[h][j] * p.w_scale_inv + bias[h];
                nnal_ovf_track(amax, rr);
                const float o = rr > 0.f ? fminf(rr, 65504.f) : 0.f;
                const nnal_h hh = __float2half_rn(o);
                P[j] = nnal_pack2(hh, __float2half_rn(o - __half2float(hh)));
              }
#pragma unroll
              for (int sft = 1; sft < 8; sft <<= 1) {
                const bool up = (cq & sft) != 0;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  if (j & sft) continue;
                  const uint32_t recv = __shfl_xor_sync(0xffffffffu, up ? P[j] : P[j ^ sft], 4 * sft);
                  if (up) P[j] = recv; else P[j ^ sft] = recv;
                }
              }
              // now P[c'] = channel (base + c') of position index cq of this m group
              const int col = sb * 32 + 8 * (cq >> 1) + 2 * m + (cq & 1);
              const uint32_t off = (uint32_t)otab[t * C::TILE_N + col];
              const int chbase = C::TAPS == 2 ? 8 * w : 16 * w + 8 * h;
              if (off < glim && chbase < C::COUT_REAL && !(p.flags & 1)) {
                uint4 vh, vl;
                vh.x = __byte_perm(P[0], P[1], 0x5410); vl.x = __byte_perm(P[0], P[1], 0x7632);
                vh.y = __byte_perm(P[2], P[3], 0x5410); vl.y = __byte_perm(P[2], P[3], 0x7632);
                vh.z = __byte_perm(P[4], P[5], 0x5410); vl.z = __byte_perm(P[4], P[5], 0x7632);
                vh.w = __byte_perm(P[6], P[7], 0x5410); vl.w = __byte_perm(P[6], P[7], 0x7632);
                *reinterpret_cast<uint4*>(ghi + off + chbase) = vh;
                if (!(p.flags & 2)) *reinterpret_cast<uint4*>(glo + off + chbase) = vl;
              }
            }
          }
          nnal_ovf_commit(amax);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(acc_empty(a));
        if (C::POOL && t == C::T - 1) {
          // the sample's pooled raster is complete: write it out (hi/lo planes) and clear it for the next sample
          named_bar_sync(1, 128 * C::NEW);
          constexpr int OCT_REAL = C::COUT_REAL / 8;
          for (int item = threadIdx.x - 128; item < C::PHO * C::PWO * OCT_REAL; item += 128 * C::NEW) {
            const int cell = item / OCT_REAL, oct = item % OCT_REAL;
            uint32_t* pc = pooled + cell * C::PSTRIDE + 8 * oct;
            uint32_t hi[4], lo[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float o0 = __uint_as_float(pc[2 * j]), o1 = __uint_as_float(pc[2 * j + 1]);
              pc[2 * j] = 0u; pc[2 * j + 1] = 0u;
              const nnal_h h0_ = __float2half_rn(o0), h1_ = __float2half_rn(o1);
              hi[j] = nnal_pack2(h0_, h1_);
              lo[j] = nnal_pack2(__float2half_rn(o0 - __half2float(h0_)), __float2half_rn(o1 - __half2float(h1_)));
            }
            const size_t ob = ((size_t)g * C::PHO * C::PWO + cell) * C::COUT_REAL + 8 * oct;
            *reinterpret_cast<uint4*>(p.out_hi + ob) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            *reinterpret_cast<uint4*>(p.out_lo + ob) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
          }
          named_bar_sync(1, 128 * C::NEW);
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
  }
}

// W fp32 [kh][kw][cin][cout] -> fp16 weight blocks [NBLK][2 K-halves][128 rows][8].
template <class C>
__global__ void pack_weights_kernel(const float* __restrict__ W, nnal_h* __restrict__ out, float scale) {
  const int total = C::NBLK * 2 * 128 * 8;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    const int k8 = e % 8;
    const int row = (e / 8) % 128;
    const int h = (e / (8 * 128)) % 2;
    const int blk = e / (8 * 128 * 2);
    const int cs = 2 * blk + h;
    float w = 0.f;
    // row = 32 w + lane;  TAPS == 2: lane = 16 * tg + 8 * term + c, channel 8 w + c
    //                     TAPS == 1: lane = 16 * half + 8 * term + c, channel 16 w + 8 * half + c
    const int wq = row / 32, ln = row % 32;
    const int tg = C::TAPS == 2 ? ln / 16 : 0;
    const int term = (ln / 8) % 2;
    const int co = C::TAPS == 2 ? 8 * wq + ln % 8 : 16 * wq + 8 * (ln / 16) + ln % 8;
    if (cs < C::NCS) {
      const int q = cs / C::NSLOT, s = cs % C::NSLOT;
      const int dy = s / C::NSLOT_ROW, dx = C::dx_a(s % C::NSLOT_ROW) + 2 * tg;
      const int ci = q * 8 + k8;
      if (dx < C::KS && ci < C::CIN_REAL && co < C::COUT_REAL)
        w = W[(((size_t)dy * C::KS + dx) * C::CIN_REAL + ci) * C::COUT_REAL + co] * scale;
    }
    nnal_h hh, ll;
    w = fminf(fmaxf(w, -65504.f), 65504.f);
    hh = __float2half_rn(w);
    ll = __float2half_rn(w - __half2float(hh));
    out[e] = term ? ll : hh;
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess) fn = (EncodeTiledFn)f;
  }
  return fn;
}

// activation tensor [n][H][W][C] fp16 viewed as 4-D (c, x, y, sample) with box {8, WP, rows, G}
static int make_act_tmap(nnal_ctx* ctx, CUtensorMap* tm, const void* ptr, int n, int H, int W, int C, int WP, int rows, int G) {
  EncodeTiledFn enc = get_encode();
  if (!enc) NNAL_FAIL(ctx, NNAL_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)n};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t box[4] = {8, (cuuint32_t)WP, (cuuint32_t)rows, (cuuint32_t)G};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) NNAL_FAIL(ctx, NNAL_ERR_CUDA, "cuTensorMapEncodeTiled (conv_wt activations) failed");
  return NNAL_OK;
}

//            H   W  CIN COUT KS TAPS G  RL  POOL
typedef Cfg<25, 25, 24, 32, 5, 2, 1, 16, false, 4> CfgConv2;     // PW1 conv2: 23 resident weight blocks, single raster in two bands
typedef Cfg<25, 25, 24, 32, 5, 2, 1, 16, true, 4> CfgConv2Pool;  // ... with the following 2x2 max-pool fused
typedef Cfg<25, 25, 3, 24, 5, 2, 1, 0, false, 4> CfgConv1;       // PW1 conv1: 3 input channels zero-padded to one chunk
typedef Cfg<13, 13, 32, 48, 3, 1, 2, 0, false, 4> CfgConv3;      // PW1 conv3: 2 samples per group

template <class C>
static bool matches(const Layer& L) {
  return L.in_h == C::H && L.in_w == C::W && L.in_c == C::CIN_REAL && L.out_c == C::COUT_REAL && L.kh == C::KS && L.kw == C::KS;
}

template <class C>
static int pack(nnal_ctx* ctx, Layer& L) {
  if (!L.Wt) CUDA_TRY(ctx, cudaMalloc(&L.Wt, (size_t)C::W_BYTES));
  const int total = C::NBLK * 2 * 128 * 8;
  pack_weights_kernel<C><<<(total + 255) / 256, 256, 0, ctx->stream>>>(L.W, (nnal_h*)L.Wt, L.w_scale);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}

template <class C>
static int launch(nnal_ctx* ctx, const Layer& L, const nnal_h* in_hi, const nnal_h* in_lo, nnal_h* out_hi,
                  nnal_h* out_lo, int64_t n) {
  CUtensorMap tmHiL, tmLoL, tmHiU, tmLoU;
  const int rowsL = C::SPLIT ? C::RL : C::HP;
  NNAL_TRY(make_act_tmap(ctx, &tmHiL, in_hi, (int)n, C::H, C::W, C::CIN, C::WP, rowsL, C::G));
  NNAL_TRY(make_act_tmap(ctx, &tmLoL, in_lo, (int)n, C::H, C::W, C::CIN, C::WP, rowsL, C::G));
  if (C::SPLIT) {
    NNAL_TRY(make_act_tmap(ctx, &tmHiU, in_hi, (int)n, C::H, C::W, C::CIN, C::WP, C::HP - C::RL, C::G));
    NNAL_TRY(make_act_tmap(ctx, &tmLoU, in_lo, (int)n, C::H, C::W, C::CIN, C::WP, C::HP - C::RL, C::G));
  } else {
    tmHiU = tmHiL; tmLoU = tmLoL;
  }
  static bool attr = false;
  if (!attr) {
    CUDA_TRY(ctx, cudaFuncSetAttribute(conv_wt_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM));
    attr = true;
  }
  Params p;
  p.wpack = (const uint8_t*)L.Wt; p.bias = L.b; p.out_hi = out_hi; p.out_lo = out_lo; p.n = (int)n; p.w_scale_inv = L.w_scale_inv;
  p.flags = ctx->dbg.wt_flags;
  const int grid = nnal_conv_grid(ctx, (n + C::G - 1) / C::G);
  conv_wt_kernel<C><<<grid, C::THREADS, C::SMEM, ctx->stream>>>(tmHiL, tmLoL, tmHiU, tmLoU, p);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}

}  // namespace cwt

// which layers the weight-stationary kernel covers (bias must hold a multiple of 8 floats: COUT_REAL % 8 == 0)
bool nnal_wt_conv_supported(const nnal_ctx*, const Layer& L) {
  if (L.type != NNAL_LAYER_CONV || !L.Wt) return false;
  return cwt::matches<cwt::CfgConv1>(L) || cwt::matches<cwt::CfgConv2>(L) || cwt::matches<cwt::CfgConv3>(L);
}
// ... and where it is the faster kernel (measured, profiles/r1_conv_wt.md): conv2 only.  conv1 (K = 25 taps x 8 channels)
// and conv3 have so little MMA work per tile that the 4x larger accumulator read-out makes them epilogue bound.
bool nnal_wt_conv_preferred(const nnal_ctx* ctx, const Layer& L) {
  return nnal_wt_conv_supported(ctx, L) && cwt::matches<cwt::CfgConv2>(L);
}
bool nnal_wt_conv_pool_supported(const nnal_ctx*, const Layer& L) {
  return L.type == NNAL_LAYER_CONV && L.Wt && cwt::matches<cwt::CfgConv2Pool>(L);
}

int nnal_wt_prepare_conv(nnal_ctx* ctx, Layer& L) {
  if (L.type != NNAL_LAYER_CONV) return NNAL_OK;
  if (cwt::matches<cwt::CfgConv1>(L)) return cwt::pack<cwt::CfgConv1>(ctx, L);
  if (cwt::matches<cwt::CfgConv2>(L)) return cwt::pack<cwt::CfgConv2>(ctx, L);
  if (cwt::matches<cwt::CfgConv3>(L)) return cwt::pack<cwt::CfgConv3>(ctx, L);
  return NNAL_OK;
}

// fuse_pool: the layer's output goes through the following 2x2/s2 SAME max-pool before it is written
// ([n][ceil(H/2)][ceil(W/2)][Cout] planes)
int nnal_wt_conv(nnal_ctx* ctx, const Layer& L, const nnal_h* in_hi, const nnal_h* in_lo, nnal_h* out_hi,
                 nnal_h* out_lo, int64_t n, int fuse_pool) {
  if (n == 0) return NNAL_OK;
  if (fuse_pool) {
    if (cwt::matches<cwt::CfgConv2Pool>(L)) return cwt::launch<cwt::CfgConv2Pool>(ctx, L, in_hi, in_lo, out_hi, out_lo, n);
    NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "conv+pool shape not covered by the weight-stationary kernel");
  }
  if (cwt::matches<cwt::CfgConv1>(L)) return cwt::launch<cwt::CfgConv1>(ctx, L, in_hi, in_lo, out_hi, out_lo, n);
  if (cwt::matches<cwt::CfgConv2>(L)) return cwt::launch<cwt::CfgConv2>(ctx, L, in_hi, in_lo, out_hi, out_lo, n);
  if (cwt::matches<cwt::CfgConv3>(L)) return cwt::launch<cwt::CfgConv3>(ctx, L, in_hi, in_lo, out_hi, out_lo, n);
  NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "conv shape not covered by the weight-stationary kernel");
}
