// tcgen05 implicit-GEMM convolution (SAME, stride 1, bias, ReLU) for the patch CNN (sm_100a).
//
// Replaces tf.nn.conv2d + bias + relu of NN.CNN.add_conv (NN.py:258-301) -- conv1 (with the patch gather of
// patch_utils.get_patches / PW_NN.batch_eval fused in), conv3, conv4 (+ max2) of PW1, the same layer dict on 28 x 28 x 1 images
// (BASELINE config 1), and the conv DATA gradients of the shrunk-gradient pass (tf.gradients, NN.py:621-645) as forward
// convolutions with the flipped, transposed filter (raw float32 epilogue).  conv2 of PW1 runs on conv_wt.cu.
// Precision: fp16 hi/lo split operands, three products per term, FP32 accumulation in TMEM, as gemm_tc.cu (DESIGN.md 4).
//
// "Shift" implicit GEMM -- no im2col is ever materialised:
//   * A group of G samples is TMA-loaded ONCE into shared memory as zero-padded rasters (TMA
//     out-of-bounds zero fill reproduces SAME padding), in the no-swizzle K-major UMMA layout built
//     from 16-byte "chunks": plane q holds channels 8q..8q+7 of every padded position,
//     addr = q*PLANE + pos*16.  Eight consecutive positions form one 128-byte UMMA core matrix.
//   * The GEMM rows are padded-raster positions (M tile = 128 consecutive positions); for filter tap
//     (dy,dx) the A operand is the SAME buffer shifted by (dy*Wp+dx) positions, i.e. only the
//     descriptor start address changes.  Columns x >= W / rows y >= H of the raster produce garbage
//     that the epilogue discards.
//   * One K=16 MMA consumes two chunks (tap,q) whose addresses may be unrelated: the descriptor's
//     leading-byte-offset is set per instruction, so K = (#taps * Cin/8) chunks is only padded to an
//     even count (75 -> 76 for conv2), not per tap.
//   * Weights are pre-arranged per K-step as [2 chunks][2*Cout][8] fp16 -- rows 0..Cout-1 the hi terms, rows
//     Cout..2Cout-1 the lo terms -- and streamed through a 3-stage ring with cp.async.bulk.  The three
//     products hi.hi + hi.lo + lo.hi take TWO MMAs per K-step: A_hi x [W_hi;W_lo] (N = 2 Cout: hi.hi lands in
//     accumulator columns 0..Cout-1, hi.lo in Cout..2Cout-1) and A_lo x W_hi (N = Cout, first Cout rows of the
//     same block, accumulated into columns 0..Cout-1); the epilogue adds the two column halves.  With N as
//     small as 32 the MMA is bound by SHARED-MEMORY operand reads (4 KB of A per 16-cycle MMA at 128 B/clk),
//     so reading A_hi once instead of twice is worth 27 % (profiles/).
//   * The T M-tiles of a sample group are processed in NG groups of TG tiles (the weight ring is streamed
//     once per tile group): 2 x TG x 2Cout accumulator columns fit TMEM, so the epilogue of one tile group
//     overlaps the MMAs of the next.
// Warp roles: warp 0 input TMA, warp 3 weight producer, warps 1 and 12 MMA issuers, warp 2 TMEM allocator,
// warps 4-11 epilogue (TMEM -> +bias, ReLU -> fp16 hi/lo NHWC in global memory, the fused max-pool raster, or raw float32):
// two warpgroups, each draining one (NACC = 2) or two (NACC = 4) accumulators in rotation; GATHER: warps 13-20 are the
// input producers instead of the TMA (volume -> normalise -> split -> x-im2col'd operand planes in shared memory).
// What bounds these kernels is the SM's shared-memory data path -- the tensor core's operand fetch of narrow-N MMAs plus
// everything the LSU moves -- not tensor math (profiles/r2_conv1_fused.md).
#include "nnal_common.cuh"
#include <cuda.h>

namespace ctc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// try_wait with a suspend-time hint: the thread is parked by the hardware until the phase completes (or the hint, 10 ms,
// runs out) -- it takes no issue slots from the warps that share its scheduler and wakes up at once.  (Round 2 had
// __nanosleep(200) between polls for the warps "off the critical path": with two input buffers and two to four accumulators
// every hand-off IS on the critical path, and the sleeps made the empty synchronisation skeleton of the fused conv1 cost
// 1800 cycles per sample -- flags 55 experiment in profiles/r2_conv1_fused.md.)  `backoff_ns` > 0 selects the old polling.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, unsigned backoff_ns = 0) {
  uint32_t ok = 0;
  long long t0 = 0;
  for (uint32_t spin = 0;; ++spin) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity), "r"(0x989680u)
        : "memory");
    if (ok) return;
    if (backoff_ns) __nanosleep(backoff_ns);
    if ((spin & 0xfff) == 0xfff) {
      long long now = clock64();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 4000000000ll) __trap();     // protocol bug -> CUDA error, never a hung GPU
    }
  }
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* tmap, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(tmap), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
// no-swizzle K-major descriptor: start>>4 | LBO>>4 at [16,30) | SBO>>4 at [32,46) | version 1 | layout 0
__device__ __forceinline__ uint64_t make_desc_none(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3ffff) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3fff) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3fff) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N) {       // A/B format 0 = F16
  return (1u << 4) | (0u << 7) | (0u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// one elected lane of a converged warp (lets ptxas issue tcgen05/TMA ops without per-thread retry loops)
__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld8_issue(uint32_t taddr, uint32_t* r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld8_wait(uint32_t* a, uint32_t* b) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7]), "+r"(b[0]),
                 "+r"(b[1]), "+r"(b[2]), "+r"(b[3]), "+r"(b[4]), "+r"(b[5]), "+r"(b[6]), "+r"(b[7])
               :
               : "memory");
}
// waits for every outstanding tcgen05.ld of the thread; both register sets are in/out operands so that their uses stay below
__device__ __forceinline__ void tmem_ld16_wait(uint32_t* a, uint32_t* b) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7]), "+r"(a[8]),
                 "+r"(a[9]), "+r"(a[10]), "+r"(a[11]), "+r"(a[12]), "+r"(a[13]), "+r"(a[14]), "+r"(a[15]), "+r"(b[0]),
                 "+r"(b[1]), "+r"(b[2]), "+r"(b[3]), "+r"(b[4]), "+r"(b[5]), "+r"(b[6]), "+r"(b[7]), "+r"(b[8]),
                 "+r"(b[9]), "+r"(b[10]), "+r"(b[11]), "+r"(b[12]), "+r"(b[13]), "+r"(b[14]), "+r"(b[15])
               :
               : "memory");
}

// Compile-time geometry of one conv layer
template <int H_, int W_, int CIN_REAL_, int COUT_REAL_, int KS_, int G_, int KPS_, int NBUF_, int TG_, bool CAT_, bool POOL_ = false, bool DUAL_ = false, int KW_ = 0, int NWG_ = 2, bool GATHER_ = false, int NACC_ = 2, bool RAW_ = false>
struct Cfg {
  static constexpr bool RAW = RAW_;                       // epilogue writes acc * scale as float32, no bias, no ReLU (data-gradient convolutions)
  static constexpr bool GATHER = GATHER_;                 // the input is gathered from the volume by producer warps (x-im2col'd conv1)
  static constexpr int NGW = GATHER_ ? 8 : 0;             // ... this many of them
  static constexpr int GW0 = 4 + 4 * NWG_ + 1;            // first gather warp
  static constexpr int NWG = 2;                           // epilogue warpgroups, one per accumulator: warpgroup wg drains every other tile group
  static_assert(NWG_ == 2, "tile-level splits over more warpgroups were measured slower: extra warps on the issuing warp's scheduler delay the MMAs");
  static constexpr int THREADS = 32 * (4 + 4 * NWG_ + 1 + NGW); // 4 service warps, 4 * NWG epilogue warps, the second MMA issuer, gather warps
  static constexpr int NISSUE = DUAL_ ? 2 : 1;            // MMA-issuing threads that share a tile group (its tiles alternate between them)
  static constexpr bool POOL = POOL_;                     // fuse the following 2x2/s2 SAME max-pool into the epilogue
  // CIN / COUT are the padded operand extents (multiples of 8 / 16); the *_REAL values are the layer's
  static constexpr int CIN_REAL = CIN_REAL_, COUT_REAL = COUT_REAL_;
  static constexpr int CIN = (CIN_REAL + 7) / 8 * 8, COUT = (COUT_REAL + 15) / 16 * 16;
  static constexpr int H = H_, W = W_, KS = KS_, G = G_;
  static constexpr int KPS = KPS_;                       // K-steps per weight stage
  // NACC accumulators in rotation, tile group it -> accumulator it % NACC -> epilogue warpgroup it % 2.  With NACC = 2 a
  // warpgroup owns ONE accumulator: it idles while the tensor core refills it (conv1: the epilogue warps waited 50 % of the
  // time, profiles/r2_conv1_fused.md); with NACC = 4 it alternates between two and the MMAs run a tile group ahead.
  static constexpr int NBUF = NBUF_, NACC = NACC_, TG = TG_;  // TG: M tiles per accumulator (tile group)
  static_assert(NACC_ == 2 || NACC_ == 4, "accumulators in rotation");
  static constexpr bool CAT = CAT_;                      // A_hi x [W_hi;W_lo] in one MMA (2 MMAs per K-step) or three separate MMAs
  static constexpr int KH = KS_, KW = KW_ > 0 ? KW_ : KS_;   // KW_ = 1: filter columns folded into the channels by an x-im2col'd input
  static constexpr int PH = KH / 2, PW = KW / 2;
  static constexpr int HP = H + KH - 1, WP = W + KW - 1;
  static constexpr int Q = CIN / 8;
  static constexpr int NTAPS = KH * KW;
  static constexpr int NCH = NTAPS * Q;                  // 16-byte chunks along K
  static constexpr int NK = (NCH + 1) / 2;               // K=16 MMA steps
  static constexpr int NSTAGE_W = (NK + KPS - 1) / KPS;  // weight stages per group
  static constexpr int RASTER = G * HP * WP;
  static constexpr int LAST_VALID = (G - 1) * HP * WP + (H - 1) * WP + (W - 1);
  static constexpr int T = LAST_VALID / 128 + 1;         // M tiles per sample group
  static constexpr int NG = (T + TG - 1) / TG;           // tile groups per sample group
  static constexpr int TILE_COLS = CAT ? 2 * COUT : COUT; // TMEM columns of one M tile (CAT: hi.hi+lo.hi | hi.lo halves)
  static constexpr int ACC_COLS = TG * TILE_COLS;        // TMEM columns of one accumulator
  static constexpr int MAX_OFF = (KH - 1) * WP + (KW - 1);
  static constexpr int PLANE = ((RASTER * 16 + 127) / 128) * 128;                 // bytes
  static constexpr int OVERRUN = (T * 128 + MAX_OFF + 8 - RASTER) > 0 ? (T * 128 + MAX_OFF + 8 - RASTER) : 0;
  static constexpr int IN_BYTES = ((2 * Q * PLANE + OVERRUN * 16 + 1023) / 1024) * 1024;   // hi planes then lo planes
  static constexpr int W_KSTEP_BYTES = 2 * (2 * COUT) * 16;   // one K-step: [2 chunks][hi rows | lo rows][8] fp16
  static constexpr int W_STAGE_BYTES = KPS * W_KSTEP_BYTES;
  static constexpr int WSTAGES = 3;
  static constexpr bool WRES = NSTAGE_W <= WSTAGES;       // the whole weight set fits the ring: load it once, keep it resident
  static constexpr int PHO = (H + 1) / 2, PWO = (W + 1) / 2;
  static constexpr int PSTRIDE = COUT_REAL | 1;           // pooled-cell stride in words: odd, so neighbouring cells hit different banks
  static constexpr int POOL_WORDS = (PHO * PWO * PSTRIDE + 3) / 4 * 4;    // one pooled raster per epilogue warpgroup
  static constexpr int POOL_BYTES = POOL ? 2 * POOL_WORDS * 4 : 0;
  static constexpr int SMEM = NBUF * IN_BYTES + WSTAGES * W_STAGE_BYTES + 1024 + 256 + POOL_BYTES;
  static constexpr int TMEM_COLS_USED = NACC * ACC_COLS;
  static_assert(CIN % 8 == 0, "input channels must be a multiple of 8");
  static_assert(COUT % 16 == 0 && 2 * COUT <= 256, "UMMA N");
  static_assert(TMEM_COLS_USED <= 512, "TMEM budget");
  static_assert(SMEM <= 232448, "shared memory budget");
  static_assert(!(POOL && RAW_), "raw float32 output: unpooled");
  static_assert(!POOL || (G == 1 && NG == 1 && NACC == 2), "fused pooling: one sample = one tile group = one epilogue warpgroup");
  static_assert(!GATHER || (G == 1 && KW == 1 && CIN == 16 && KH == 5 && H == 25 && W == 25), "fused gather: conv1 of PW1 in the x-im2col'd form");
};

// fused gather (Cfg::GATHER): the [Z][X][Y][m] float32 volume, the raveled voxel ids of the samples, normalisation table
struct GatherArgs {
  const float* vol;
  int64_t Xp, Yp, Zp;
  const int64_t* inds;
  NormTab tab;
  int flags;                 // debug option wt_flags -- timing experiments: 1 no normalise/split, 2 no operand assembly, 4 no fetch; tests: 8 float64 normalisation
};

struct ConvParams {
  const uint8_t* wpack;      // [NSTAGE_W][KPS][2 chunks][hi COUT | lo COUT][8] fp16
  const float* bias;
  nnal_h* out_hi;     // [n][H][W][COUT]
  nnal_h* out_lo;
  float* out_f32;     // RAW: [n][H][W][COUT_REAL] float32
  int n;
  float w_scale_inv;
};

template <class C>
__global__ void __launch_bounds__(C::THREADS, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmHi, const __grid_constant__ CUtensorMap tmLo, ConvParams p, GatherArgs ga) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* base_ptr = smem_raw + (base - raw);
  const uint32_t in_base = base;
  const uint32_t w_base = base + C::NBUF * C::IN_BYTES;
  const uint32_t bar0 = w_base + C::WSTAGES * C::W_STAGE_BYTES;
  // barrier map
  auto in_full = [&](int b) { return bar0 + 8u * b; };
  auto in_empty = [&](int b) { return bar0 + 8u * (2 + b); };
  auto w_full = [&](int s) { return bar0 + 8u * (4 + s); };
  auto w_empty = [&](int s) { return bar0 + 8u * (7 + s); };
  auto acc_full = [&](int a) { return bar0 + 8u * (10 + a); };
  auto acc_empty = [&](int a) { return bar0 + 8u * (14 + a); };
  volatile uint32_t* tmem_slot =
      reinterpret_cast<volatile uint32_t*>(base_ptr + C::NBUF * C::IN_BYTES + C::WSTAGES * C::W_STAGE_BYTES + 8 * 18);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ngroups = (p.n + C::G - 1) / C::G;
  uint32_t* pooled = reinterpret_cast<uint32_t*>(base_ptr + C::NBUF * C::IN_BYTES + C::WSTAGES * C::W_STAGE_BYTES + 256);
  for (int i = threadIdx.x; i < C::POOL_BYTES / 4; i += blockDim.x) pooled[i] = 0u;
  __shared__ __align__(16) float sbias[(C::COUT + 15) / 16 * 16];
  for (int i = threadIdx.x; i < (C::COUT + 15) / 16 * 16; i += blockDim.x) sbias[i] = (!C::RAW && i < C::COUT_REAL) ? p.bias[i] : 0.f;

  if (warp == 0 && lane == 0 && !C::GATHER) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmHi));
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmLo));
  }
  if (warp == 1 && lane == 0) {
    // two MMA-issuing threads (see below): every "MMAs retired" barrier collects one commit from each
    for (int b = 0; b < 2; ++b) { mbar_init(in_full(b), C::GATHER ? C::NGW : 1); mbar_init(in_empty(b), C::NISSUE); }
    for (int s = 0; s < 3; ++s) { mbar_init(w_full(s), 1); mbar_init(w_empty(s), C::NISSUE); }
    for (int a = 0; a < C::NACC; ++a) { mbar_init(acc_full(a), C::NISSUE); mbar_init(acc_empty(a), 4); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  // Zero the input buffers once: the slack after each plane and after the last plane is never written
  // by TMA but IS read (second chunk of an odd K tail, overrun rows of the last tile).  Those reads
  // only ever meet zero weights or discarded rows, but NaN bit patterns in stale shared memory would
  // still poison valid rows (NaN x 0 = NaN).
  {
    uint4* z = reinterpret_cast<uint4*>(base_ptr);
    for (int i = threadIdx.x; i < C::NBUF * C::IN_BYTES / 16; i += blockDim.x) z[i] = make_uint4(0, 0, 0, 0);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  // K-step table: chunk c -> (q = c / NTAPS, tap = c % NTAPS); q-major order keeps every LBO positive
  __shared__ uint2 ktab[C::NK];
  for (int ks = threadIdx.x; ks < C::NK; ks += blockDim.x) {
    const int c0 = 2 * ks, c1 = 2 * ks + 1;
    const int q0 = c0 / C::NTAPS, t0 = c0 % C::NTAPS;
    const uint32_t off0 = q0 * C::PLANE + ((t0 / C::KW) * C::WP + (t0 % C::KW)) * 16;
    uint32_t lbo = 16;                    // dummy second chunk of an odd K tail (zero weights) stays in-plane
    if (c1 < C::NCH) {
      const int q1 = c1 / C::NTAPS, t1 = c1 % C::NTAPS;
      lbo = q1 * C::PLANE + ((t1 / C::KW) * C::WP + (t1 % C::KW)) * 16 - off0;
    }
    ktab[ks] = make_uint2(off0 >> 4, ((lbo >> 4) & 0x3fffu) << 16);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (C::GATHER && warp >= C::GW0) {
    // ===== input producers (fused gather): the patch is read from the volume, normalised (float64, as batch_eval) and split
    // ONCE into a packed staging array, then every thread assembles the x-im2col'd rows of its positions -- element
    // dx * 3 + ch of position (i, k) = value (i, k + dx - 2, ch), zero outside the patch, element 15 = 0 -- straight into the
    // UMMA operand planes (plane q = elements 8q..8q+7, 16 bytes per raster position; rows -2, -1, 25, 26 of the raster stay
    // zero from the initial clear).  What the stand-alone gather wrote to HBM (and conv1 read back through 16-byte TMA rows)
    // never leaves the SM.
    constexpr int NPOS = C::H * C::W, CH = 3, ROW = C::W * CH, NT = C::GATHER ? 32 * C::NGW : 32;
    constexpr int NE = NPOS * CH, PER = (NE + NT - 1) / NT, NPP = (NPOS + NT - 1) / NT;
    // staging: fp16 hi and lo terms of the patch, row-major [25][RS] with 6 zero halves before and after the 75 values of a
    // row, so that the 15 values a position needs -- (k - 2 .. k + 2) x 3 channels -- are 15 CONSECUTIVE halves starting at
    // half 3 k: eight 32-bit words per plane, shifted by one half when k is odd (funnel shift), no bounds tests.  Two copies:
    // sample s is staged while the stragglers still assemble sample s - 1 (one named barrier per sample).
    constexpr int RS = 88, RSW = RS / 2;
    __shared__ __align__(16) uint16_t svh[2][C::H * RS], svl[2][C::H * RS];
    const int pt = threadIdx.x - 32 * C::GW0;
    const int64_t Y0 = ga.Yp - (C::W - 1), Z0 = ga.Zp;
    const bool small = Y0 < (1ll << 31) && Z0 < (1ll << 31);
    // this thread's elements of a patch: e = pt + u NT -> (row i, offset r in the row, channel); the same for every sample
    int eoff[PER];
    short srow[PER];                                     // index of the element in the staging rows
    for (int e = pt; e < 2 * C::H * RS; e += NT) { (&svh[0][0])[e] = 0; (&svl[0][0])[e] = 0; }   // (pads stay zero; the values are rewritten per patch)
    asm volatile("bar.sync 3, %0;" ::"n"(NT) : "memory");
    static_assert(!C::GATHER || (NT % 3 != 0 && ROW % 3 == 0), "channel pattern of the per-thread elements");
#pragma unroll
    for (int u = 0; u < PER; ++u) {
      const int e = pt + u * NT;
      const int i = e / ROW, r = e - i * ROW;
      eoff[u] = e < NE ? (int)(i * ga.Yp * CH + r) : -1;
      srow[u] = (short)(i * RS + 6 + r);
    }
    // this thread's raster positions pos = pt + j NT: first staging word, odd-column flag, byte offset in an operand plane
    short aw0[NPP], aodd[NPP];
    int aoff[NPP];
#pragma unroll
    for (int j = 0; j < NPP; ++j) {
      const int pos = pt + j * NT;
      const int i = pos / C::W, k = pos - i * C::W;
      aw0[j] = pos < NPOS ? (short)(i * RSW + ((3 * k) >> 1)) : (short)0;
      aodd[j] = (short)(k & 1);
      aoff[j] = pos < NPOS ? ((i + C::PH) * C::WP + k) * 16 : -1;
    }
    // normalisation (x - mu) / sigma of channel q = u % 3 (element u has channel (pt + (NT % 3) u) % 3, ROW = 0 mod 3).
    // Default: float32 two-term arithmetic, ((x - mu_hi) - mu_lo) * (r_hi + r_lo) with r = 1 / sigma: within 2^-22 of the
    // float64 quotient, i.e. below what the fp16 hi/lo split keeps anyway -- the float64 pipe is 30x slower than the float32
    // one on this chip and its eight divisions per thread took 44 % of the producers' time (profiles/r2_conv1_fused.md).
    // exact (debug option wt_flags & 8, or a sigma without a usable reciprocal): the float64 sequence of batch_eval.
    double mu[3], sg[3], rs[3];
    float mh[3], ml[3], rh[3], rl[3];
    bool exact = (ga.flags & 8) != 0;
#pragma unroll
    for (int q = 0; q < 3; ++q) {
      const int ch = (pt + (NT % 3) * q) % 3;
      const bool on = ga.tab.on[ch];
      mu[q] = on ? ga.tab.mu[ch] : 0.0;
      sg[q] = on ? ga.tab.sg[ch] : 1.0;
      rs[q] = on ? ga.tab.rs[ch] : 1.0;                  // (x - 0) / 1 = x, exactly
      mh[q] = (float)mu[q]; ml[q] = (float)(mu[q] - (double)mh[q]);
      rh[q] = (float)rs[q]; rl[q] = (float)(rs[q] - (double)rh[q]);
    }
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) exact = exact || (ga.tab.on[ch] && !(ga.tab.rs[ch] == ga.tab.rs[ch]));
    // voxel id -> address of the patch corner (32-bit divisions whenever the id fits)
    auto corner = [&](int64_t ind) -> const float* {
      int64_t x, y, z;
      if (small && (uint64_t)ind <= 0xffffffffull) {
        const uint32_t i32 = (uint32_t)ind, z0 = (uint32_t)Z0, y0 = (uint32_t)Y0;
        const uint32_t t = i32 / z0, xx = t / y0;
        z = i32 - t * z0; y = t - xx * y0; x = xx;
      } else {
        z = ind % Z0;
        const int64_t t = ind / Z0;
        y = t % Y0;
        x = t / Y0;
      }
      return ga.vol + ((z * ga.Xp + x) * ga.Yp + y) * CH;
    };
    // all loads of a patch are issued before the first is used, the NEXT patch is fetched while this one is assembled, and
    // the voxel id of the patch after that is already on its way (its latency was 10 % of the producers' time)
    float raw[PER];
    auto fetch = [&](int64_t ind) {
      const float* pbase = corner(ind);
#pragma unroll
      for (int u = 0; u < PER; ++u) raw[u] = eoff[u] >= 0 ? pbase[eoff[u]] : 0.f;
    };
    const int stride = (int)gridDim.x;
    int64_t ind_next = 0;
    if ((int)blockIdx.x < ngroups) fetch(ga.inds[blockIdx.x]);
    if ((int)blockIdx.x + stride < ngroups) ind_next = ga.inds[blockIdx.x + stride];
    uint32_t it = 0;
    for (int g = blockIdx.x; g < ngroups; g += stride, ++it) {
      const int b = it % C::NBUF, sb = it & 1;
      const uint32_t ph = (it / C::NBUF) & 1;
      uint16_t* sh_ = svh[sb];
      uint16_t* sl_ = svl[sb];
      if (!(ga.flags & 1)) {
        // branch-free per element (the fp16 range check is one test per thread and patch): independent chains
        uint32_t amax = 0u;
#pragma unroll
        for (int u = 0; u < PER; ++u) {
          const int e = pt + u * NT;
          float v;
          if (exact) v = (float)norm_apply((double)raw[u], mu[u % 3], sg[u % 3], rs[u % 3]);
          else {
            const float d = (raw[u] - mh[u % 3]) - ml[u % 3];
            v = fmaf(d, rl[u % 3], d * rh[u % 3]);
          }
          nnal_ovf_track(amax, v);
          nnal_h h, l;
          nnal_split_unchecked(v, h, l);
          if (e < NE) { sh_[srow[u]] = __half_as_ushort(h); sl_[srow[u]] = __half_as_ushort(l); }
        }
        nnal_ovf_commit(amax);
      }
      asm volatile("bar.sync 3, %0;" ::"n"(NT) : "memory");
      if (g + stride < ngroups && !(ga.flags & 4)) {
        // (the id is warp-uniform and ptxas would move it to a uniform register -- i.e. wait for the load -- right where it
        // was issued, a whole sample earlier; the empty asm hides that it is the load's result until here)
        asm volatile("" : "+l"(ind_next));
        fetch(ind_next);
        if (g + 2 * stride < ngroups) ind_next = ga.inds[g + 2 * stride];
      }
      mbar_wait(in_empty(b), ph ^ 1, 0);
      uint8_t* dst = base_ptr + (size_t)b * C::IN_BYTES;
      const uint32_t* wh = reinterpret_cast<const uint32_t*>(sh_);
      const uint32_t* wl = reinterpret_cast<const uint32_t*>(sl_);
      // (the loads of position j + 1 are issued before the stores of position j: the compiler cannot move shared-memory
      // loads above shared-memory stores by itself, and their latency was a third of the assembly time)
      uint32_t a[9], c[9];
      a[8] = 0u; c[8] = 0u;
#pragma unroll
      for (int t = 0; t < 8; ++t) { a[t] = wh[aw0[0] + t]; c[t] = wl[aw0[0] + t]; }
#pragma unroll
      for (int j = 0; j < NPP; ++j) {
        const uint32_t sh = (uint32_t)aodd[j] * 16u, top = aodd[j] ? 0xffffffffu : 0x0000ffffu;     // element 15 of a position is zero
        uint32_t hw[8], lw[8];
#pragma unroll
        for (int t = 0; t < 8; ++t) { hw[t] = __funnelshift_r(a[t], a[t + 1], sh); lw[t] = __funnelshift_r(c[t], c[t + 1], sh); }
        hw[7] &= top; lw[7] &= top;
        if (j + 1 < NPP) {
#pragma unroll
          for (int t = 0; t < 8; ++t) { a[t] = wh[aw0[j + 1] + t]; c[t] = wl[aw0[j + 1] + t]; }
        }
        if (aoff[j] < 0 || (ga.flags & 2)) continue;
        uint8_t* o = dst + aoff[j];
        *reinterpret_cast<uint4*>(o) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
        *reinterpret_cast<uint4*>(o + C::PLANE) = make_uint4(hw[4], hw[5], hw[6], hw[7]);
        *reinterpret_cast<uint4*>(o + 2 * C::PLANE) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
        *reinterpret_cast<uint4*>(o + 3 * C::PLANE) = make_uint4(lw[4], lw[5], lw[6], lw[7]);
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic-proxy stores -> visible to the tensor core's reads
      __syncwarp();
      if (lane == 0) mbar_arrive(in_full(b));
    }
  } else if (warp == 0) {
    // ===== input producer: Q 4-D TMA boxes {8ch, WP, HP, G} per (hi|lo), zero-filled borders =====
    if (lane == 0 && !C::GATHER) {
      uint32_t it = 0;
      for (int g = blockIdx.x; g < ngroups; g += gridDim.x, ++it) {
        const int b = it % C::NBUF;
        const uint32_t ph = (it / C::NBUF) & 1;
        mbar_wait(in_empty(b), ph ^ 1);
        const uint32_t dst = in_base + b * C::IN_BYTES;
        mbar_arrive_expect_tx(in_full(b), 2 * C::Q * C::RASTER * 16);
#pragma unroll 1
        for (int q = 0; q < C::Q; ++q) {
          tma_load_4d(dst + q * C::PLANE, &tmHi, in_full(b), q * 8, -C::PW, -C::PH, g * C::G);
          tma_load_4d(dst + (C::Q + q) * C::PLANE, &tmLo, in_full(b), q * 8, -C::PW, -C::PH, g * C::G);
        }
      }
    }
  } else if (warp == 3) {
    // ===== weight producer: one contiguous bulk copy per stage =====
    if (lane == 0 && C::WRES) {
      for (int ws = 0; ws < C::NSTAGE_W; ++ws) {
        mbar_arrive_expect_tx(w_full(ws), C::W_STAGE_BYTES);
        bulk_load(w_base + ws * C::W_STAGE_BYTES, p.wpack + (size_t)ws * C::W_STAGE_BYTES, C::W_STAGE_BYTES, w_full(ws));
      }
    } else if (lane == 0) {
      uint32_t it = 0;
      for (int g = blockIdx.x; g < ngroups; g += gridDim.x) {
        for (int ws = 0; ws < C::NG * C::NSTAGE_W; ++ws, ++it) {
          const int s = it % C::WSTAGES;
          const uint32_t ph = (it / C::WSTAGES) & 1;
          mbar_wait(w_empty(s), ph ^ 1);
          mbar_arrive_expect_tx(w_full(s), C::W_STAGE_BYTES);
          bulk_load(w_base + s * C::W_STAGE_BYTES, p.wpack + (size_t)(ws % C::NSTAGE_W) * C::W_STAGE_BYTES, C::W_STAGE_BYTES, w_full(s));
        }
      }
    }
  } else if (warp == 1 || (warp == 4 + 4 * C::NWG && C::NISSUE == 2)) {
    // ===== MMA issuers =====
    // tcgen05.mma does not run ahead of the tensor pipe: the issuing thread is held until the instruction is accepted,
    // and every cycle it spends on anything else (descriptor arithmetic, barrier waits, commits) is a cycle the pipe
    // idles (scripts/microbench/mma_rate.cu: a gap of g cycles between bursts costs g cycles; clock64 probes put
    // these gaps at 20-30 % of conv1/conv3/conv4).  With NISSUE == 2 two threads issue concurrently, each for every
    // other tile of the tile group (independent accumulator columns, same operands): one thread's gaps are filled by
    // the other's MMAs -- conv4 5.3 -> 4.6 ms per 100k patches.  The concatenated configurations keep one issuer:
    // halving the tiles per thread halves the distance between two MMAs on the same accumulator, and that costs more
    // than the filled gaps gain (conv1 4.4 -> 6.3 ms).  Per-K-step descriptor words come from the table built above,
    // per-tile descriptors differ by a compile-time constant.
    const int mi = warp == 1 ? 0 : 1;
    {
      const uint32_t idesc_cat = make_idesc_bf16(128, 2 * C::COUT);   // A_hi x [W_hi;W_lo]
      const uint32_t idesc_hi = make_idesc_bf16(128, C::COUT);        // A_lo x W_hi
      constexpr uint32_t DESC_HI = 8u /*SBO 128 B*/ | (1u << 14) /*version*/;
      constexpr uint32_t B_LBO = (uint32_t)(2 * C::COUT) << 16;      // chunk stride (2*COUT*16 B) >> 4 in the LBO field
      uint32_t it_in = 0, it_w = 0, it_acc = 0;
      for (int g = blockIdx.x; g < ngroups; g += gridDim.x, ++it_in) {
        const int b = it_in % C::NBUF;
        const uint32_t ph_in = (it_in / C::NBUF) & 1;
        mbar_wait(in_full(b), ph_in);
        tc_fence_after();
        const uint32_t a_hi16 = (in_base + b * C::IN_BYTES) >> 4;
#pragma unroll 1
        for (int tgi = 0; tgi < C::NG; ++tgi, ++it_acc) {
          // two tile groups of unequal size (conv1: 3 + 2 tiles): every other sample takes them in reverse order, so that
          // the two epilogue warpgroups (one per accumulator) drain 5 tiles each per two samples instead of 6 and 4
          const int tg = (C::NG == 2 && (it_in & 1)) ? C::NG - 1 - tgi : tgi;
          const int a = it_acc % C::NACC;
          const uint32_t ph_acc = (it_acc / C::NACC) & 1;
          mbar_wait(acc_empty(a), ph_acc ^ 1);
          tc_fence_after();
          const uint32_t d_base = tmem_base + a * C::ACC_COLS;
          const uint32_t tile0 = (uint32_t)(tg * C::TG) * 128u;       // first raster position of the tile group (>>4 units: x128 = 16 B x 128 / 16)
          for (int ws = 0; ws < C::NSTAGE_W; ++ws, ++it_w) {
            const int s = C::WRES ? ws : it_w % C::WSTAGES;
            const uint32_t ph = C::WRES ? 0u : (it_w / C::WSTAGES) & 1;      // resident: phase 0 completes once and stays complete
            mbar_wait(w_full(s), ph);
            tc_fence_after();
            const uint32_t wb16 = (w_base + s * C::W_STAGE_BYTES) >> 4;
            if (elect_one_sync()) {
#pragma unroll
              for (int j = 0; j < C::KPS; ++j) {
                const int ks = ws * C::KPS + j;
                if (ks < C::NK) {
                  const uint2 e = ktab[ks];                           // {start offset >> 4, LBO field}
                  const uint32_t ah = (a_hi16 + e.x + tile0) | e.y;
                  const uint32_t al = ah + ((C::Q * C::PLANE) >> 4);
                  const uint64_t dB = ((uint64_t)DESC_HI << 32) | ((wb16 + j * (C::W_KSTEP_BYTES >> 4)) | B_LBO);
                  const uint32_t acc0 = ks != 0;
                  if (C::CAT) {
                    // the two MMAs of a tile accumulate into the same columns: issue them TG MMAs apart
#pragma unroll
                    for (int t = 0; t < C::TG; ++t) {
                      if ((t % C::NISSUE) == mi && tg * C::TG + t < C::T) {
                        const uint64_t dAh = ((uint64_t)DESC_HI << 32) | (ah + t * 128);
                        umma_bf16(d_base + t * C::TILE_COLS, dAh, dB, idesc_cat, acc0);   // cols [0,COUT): hi.hi  [COUT,2COUT): hi.lo
                      }
                    }
#pragma unroll
                    for (int t = 0; t < C::TG; ++t) {
                      if ((t % C::NISSUE) == mi && tg * C::TG + t < C::T) {
                        const uint64_t dAl = ((uint64_t)DESC_HI << 32) | (al + t * 128);
                        umma_bf16(d_base + t * C::TILE_COLS, dAl, dB, idesc_hi, 1);       // cols [0,COUT) += lo.hi
                      }
                    }
                  } else {
                    const uint64_t dBl = dB + (uint64_t)C::COUT;                          // lo rows start COUT*16 B further
#pragma unroll
                    for (int t = 0; t < C::TG; ++t) {
                      if ((t % C::NISSUE) == mi && tg * C::TG + t < C::T) {
                        const uint64_t dAh = ((uint64_t)DESC_HI << 32) | (ah + t * 128);
                        const uint64_t dAl = ((uint64_t)DESC_HI << 32) | (al + t * 128);
                        const uint32_t d = d_base + t * C::TILE_COLS;
                        umma_bf16(d, dAl, dB, idesc_hi, acc0);
                        umma_bf16(d, dAh, dBl, idesc_hi, 1);
                        umma_bf16(d, dAh, dB, idesc_hi, 1);
                      }
                    }
                  }
                }
              }
              if (!C::WRES) umma_commit(w_empty(s));
            }
            __syncwarp();
          }
          if (elect_one_sync()) {
            if (tgi == C::NG - 1) umma_commit(in_empty(b));
            umma_commit(acc_full(a));
          }
          __syncwarp();
        }
      }
    }
  } else if (warp >= 4 && warp < 4 + 4 * C::NWG) {
    // ===== epilogue: two warpgroups, warpgroup wg drains accumulator wg (every other tile group) =====
    const int qd = warp & 3;
    const int wg = (warp - 4) >> 2;
    uint32_t it = 0, it_s = 0;
    for (int g = blockIdx.x; g < ngroups; g += gridDim.x, ++it_s) {
#pragma unroll 1
      for (int tgi = 0; tgi < C::NG; ++tgi, ++it) {
        if ((int)(it & 1) != wg) continue;
        const int tg = (C::NG == 2 && (it_s & 1)) ? C::NG - 1 - tgi : tgi;       // (same order as the MMA issuer)
        const int a = it % C::NACC;
        uint32_t* my_pooled = pooled + a * C::POOL_WORDS;           // one pooled raster per accumulator (= per sample in flight)
        const uint32_t ph_acc = (it / C::NACC) & 1;
        mbar_wait(acc_full(a), ph_acc, 0);
        tc_fence_after();
        // The epilogue warps are latency bound (one or two warps per scheduler, every TMEM load ~100 and every bias load ~30
        // cycles away): the accumulator loads run ONE 16-channel piece ahead of the arithmetic -- the load of the next piece
        // (or of the next tile's first piece) is issued before the current one is converted and stored -- and the bias is
        // fetched before the wait.  Pieces: NC16 of 16 channels + one of 8 when COUT_REAL = 8 mod 16 (conv1: 24 = 16 + 8).
        constexpr int NC16 = C::COUT_REAL / 16, TAIL8 = (C::COUT_REAL % 16 == 8) ? 1 : 0, NPC = NC16 + TAIL8;
        static_assert(C::COUT_REAL % 8 == 0 && (!C::POOL || TAIL8 == 0), "output channels: multiples of 8 (16 with the fused pool)");
        const int ntl = (C::T - tg * C::TG) < C::TG ? (C::T - tg * C::TG) : C::TG;
        const uint32_t tcol0 = tmem_base + ((uint32_t)(qd * 32) << 16) + (uint32_t)(a * C::ACC_COLS);
        uint32_t rv[16], rw[16];
        tmem_ld16_issue(tcol0, rv);                              // hi.hi + lo.hi (CAT) or the full sum
        if (C::CAT) tmem_ld16_issue(tcol0 + C::COUT, rw);        // hi.lo
#pragma unroll 1
        for (int tl = 0; tl < ntl; ++tl) {
          const int t = tg * C::TG + tl;
          const int pos = t * 128 + qd * 32 + lane;              // padded-raster position of this thread's row
          const int gs = pos / (C::HP * C::WP);
          const int rem = pos - gs * (C::HP * C::WP);
          const int y = rem / C::WP, x = rem - y * C::WP;
          const int sample = g * C::G + gs;
          const bool valid = gs < C::G && y < C::H && x < C::W && sample < p.n;
          const size_t obase = (((size_t)sample * C::H + y) * C::W + x) * C::COUT_REAL;
          const uint32_t tcol = tcol0 + (uint32_t)(tl * C::TILE_COLS);
#pragma unroll
          for (int ci = 0; ci < NPC; ++ci) {
            const int c0 = ci * 16;
            const bool is8 = TAIL8 && ci == NC16;                // (compile-time after unrolling)
            float bb[16];
#pragma unroll
            for (int j = 0; j < (is8 ? 2 : 4); ++j) {
              const float4 b4 = *reinterpret_cast<const float4*>(sbias + c0 + 4 * j);
              bb[4 * j] = b4.x; bb[4 * j + 1] = b4.y; bb[4 * j + 2] = b4.z; bb[4 * j + 3] = b4.w;
            }
            tmem_ld16_wait(rv, rw);
            float v[16];
#pragma unroll
            for (int j = 0; j < (is8 ? 8 : 16); ++j) v[j] = C::CAT ? __uint_as_float(rv[j]) + __uint_as_float(rw[j]) : __uint_as_float(rv[j]);
            // next piece: the following one of this tile, or the first of the next tile
            if (ci + 1 < NPC) {
              if (TAIL8 && ci + 1 == NC16) {
                tmem_ld8_issue(tcol + c0 + 16, rv);
                if (C::CAT) tmem_ld8_issue(tcol + C::COUT + c0 + 16, rw);
              } else {
                tmem_ld16_issue(tcol + c0 + 16, rv);
                if (C::CAT) tmem_ld16_issue(tcol + C::COUT + c0 + 16, rw);
              }
            } else if (tl + 1 < ntl) {
              tmem_ld16_issue(tcol + C::TILE_COLS, rv);
              if (C::CAT) tmem_ld16_issue(tcol + C::TILE_COLS + C::COUT, rw);
            }
            if (valid && C::POOL) {
              // post-ReLU values are >= +0, so their bit patterns order like unsigned integers
              uint32_t* pc = my_pooled + ((y >> 1) * C::PWO + (x >> 1)) * C::PSTRIDE + c0;
              uint32_t amax = 0u;
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                const float r = v[j] * p.w_scale_inv + bb[j];
                nnal_ovf_track(amax, r);
                atomicMax(pc + j, __float_as_uint(r > 0.f ? fminf(r, 65504.f) : 0.f));
              }
              nnal_ovf_commit(amax);
            } else if (valid && C::RAW) {
              float4* d4 = reinterpret_cast<float4*>(p.out_f32 + obase + c0);
#pragma unroll
              for (int j = 0; j < (is8 ? 2 : 4); ++j)
                d4[j] = make_float4(v[4 * j] * p.w_scale_inv, v[4 * j + 1] * p.w_scale_inv, v[4 * j + 2] * p.w_scale_inv,
                                    v[4 * j + 3] * p.w_scale_inv);
            } else if (valid) {
              // post-ReLU values are >= 0: no clamp; a value beyond fp16 rounds to Inf, which the SIMD max below catches (the
              // lo term is garbage then, and the call fails with NNAL_ERR_OVERFLOW) -- 7 instead of 10 instructions per output
              uint32_t hi[8], lo[8], hmax = 0u;
#pragma unroll
              for (int j = 0; j < (is8 ? 4 : 8); ++j) {
                const float x0 = fmaxf(fmaf(v[2 * j], p.w_scale_inv, bb[2 * j]), 0.f);
                const float x1 = fmaxf(fmaf(v[2 * j + 1], p.w_scale_inv, bb[2 * j + 1]), 0.f);
                const __half2 h = __floats2half2_rn(x0, x1);              // .x (low half) = x0
                const float2 hf = __half22float2(h);
                const __half2 l = __floats2half2_rn(x0 - hf.x, x1 - hf.y);
                hi[j] = *reinterpret_cast<const uint32_t*>(&h);
                lo[j] = *reinterpret_cast<const uint32_t*>(&l);
                nnal_ovf_track_h2(hmax, hi[j]);
              }
              nnal_ovf_commit_h2(hmax);
              uint4* dh = reinterpret_cast<uint4*>(p.out_hi + obase + c0);
              uint4* dl = reinterpret_cast<uint4*>(p.out_lo + obase + c0);
              dh[0] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
              dl[0] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
              if (!is8) {
                dh[1] = make_uint4(hi[4], hi[5], hi[6], hi[7]);
                dl[1] = make_uint4(lo[4], lo[5], lo[6], lo[7]);
              }
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(acc_empty(a));
        if (C::POOL && tg == C::NG - 1) {
          // the sample's pooled raster is complete: write it out as fp16 hi/lo planes [n][PHO][PWO][COUT] and clear it
          asm volatile("bar.sync %0, 128;" ::"r"(1 + wg) : "memory");
          constexpr int OCT = C::COUT_REAL / 8;
          for (int item = (threadIdx.x - 128) & 127; item < C::PHO * C::PWO * OCT; item += 128) {
            const int cell = item / OCT, oct = item % OCT;
            uint32_t* pc = my_pooled + cell * C::PSTRIDE + 8 * oct;
            uint32_t hi[4], lo[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float o0 = __uint_as_float(pc[2 * j]), o1 = __uint_as_float(pc[2 * j + 1]);
              pc[2 * j] = 0u; pc[2 * j + 1] = 0u;
              nnal_h h0, h1, l0, l1;
              nnal_split_unchecked(o0, h0, l0);                    // clamped (and flagged) when they entered the raster
              nnal_split_unchecked(o1, h1, l1);
              hi[j] = nnal_pack2(h0, h1);
              lo[j] = nnal_pack2(l0, l1);
            }
            const size_t ob = ((size_t)g * C::PHO * C::PWO + cell) * C::COUT_REAL + 8 * oct;
            *reinterpret_cast<uint4*>(p.out_hi + ob) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            *reinterpret_cast<uint4*>(p.out_lo + ob) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
          }
          asm volatile("bar.sync %0, 128;" ::"r"(1 + wg) : "memory");
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

// W fp32 [kh][kw][cin][cout] -> packed fp16 [NSTAGE_W][KPS][2 chunks][hi COUT rows | lo COUT rows][8]
__global__ void pack_conv_weights_kernel(const float* __restrict__ W, uint8_t* __restrict__ out, int NTAPS, int CIN, int COUT,
                                         int CIN_REAL, int COUT_REAL, int KPS, int NK, int NSTAGE, float scale) {
  const int Q = CIN / 8, NCH = NTAPS * Q;
  const int64_t total = (int64_t)NSTAGE * KPS * 2 * COUT * 8;
  nnal_h* o = reinterpret_cast<nnal_h*>(out);
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    int k8 = e % 8;
    int64_t t = e / 8;
    int co = t % COUT; t /= COUT;
    int half = t % 2; t /= 2;
    int ks = (int)t;                         // global K-step index (ws * KPS + j)
    int c = 2 * ks + half;
    float w = 0.f;
    if (ks < NK && c < NCH) {
      int q = c / NTAPS, tap = c % NTAPS;
      int ci = q * 8 + k8;
      if (ci < CIN_REAL && co < COUT_REAL) w = W[((int64_t)tap * CIN_REAL + ci) * COUT_REAL + co] * scale;
    }
    nnal_h h, l;
    nnal_split(w, h, l);
    const int64_t kstep_elems = (int64_t)2 * (2 * COUT) * 8;
    const int64_t base = ks * kstep_elems + (int64_t)half * (2 * COUT) * 8;
    o[base + (int64_t)co * 8 + k8] = h;
    o[base + (int64_t)(COUT + co) * 8 + k8] = l;
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

// activation tensor [n][H][W][C] fp16 viewed as 4-D (c, x, y, sample) with box {8, WP, HP, G}
static int make_act_tmap(nnal_ctx* ctx, CUtensorMap* tm, const void* ptr, int n, int H, int W, int C, int WP, int HP, int G) {
  EncodeTiledFn enc = get_encode();
  if (!enc) NNAL_FAIL(ctx, NNAL_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)n};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t box[4] = {8, (cuuint32_t)WP, (cuuint32_t)HP, (cuuint32_t)G};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) NNAL_FAIL(ctx, NNAL_ERR_CUDA, "cuTensorMapEncodeTiled (conv activations) failed");
  return NNAL_OK;
}

//                 H   W  CIN COUT KS G KPS NBUF TG CAT
typedef Cfg<25, 25, 3, 24, 5, 1, 7, 2, 3, true> CfgConv1;     // PW1 conv1: 3 input channels zero-padded to one 8-channel chunk
// conv1 with the filter COLUMNS folded into the channel axis: the input is x-im2col'd to 16 "channels"
// (element dx * 3 + ch of position (y, x) = in[y][x + dx - 2][ch], zero outside the patch, element 15 = 0), the filter
// becomes 5 x 1 over 16 channels: K = 5 taps x 16 = 80 instead of 25 taps x 8 (3 real) = 200, no x padding (5 M tiles
// instead of 6): 50 MMAs per sample instead of 156
typedef Cfg<25, 25, 16, 24, 5, 1, 5, 2, 3, true, false, false, 1> CfgConv1X;
// ... and with the gather fused in (the kernel reads the volume itself)
typedef Cfg<25, 25, 16, 24, 5, 1, 5, 2, 2, true, false, false, 1, 2, true, 4> CfgConv1XG;   // 5 M tiles in groups of 2 + 2 + 1, four accumulators of 2 x 64 columns
typedef Cfg<25, 25, 24, 32, 5, 1, 8, 2, 3, true> CfgConv2;    // PW1 conv2: 6 M tiles in 2 groups of 3
// conv3/conv4: the concatenated form was measured for conv3 (TG = 2, N = 96 + 48): 2.63 ms vs 2.61 ms per 100k samples
// -- with only two accumulators in rotation the MMAs wait on each other (scripts/microbench/mma_rate.cu: 129 cycles
// per K-step and tile at TG = 2 against 100 at TG = 4), and four tiles of 96 columns do not fit TMEM twice.  conv4
// would need 2 x 192 columns per tile and its 166 KB weight set streamed once per tile (L2-bound).
typedef Cfg<13, 13, 32, 48, 3, 2, 6, 2, 4, false> CfgConv3;   // PW1 conv3: 2 samples, 4 M tiles
typedef Cfg<13, 13, 48, 96, 3, 1, 3, 2, 2, false, false, true> CfgConv4;   // PW1 conv4: 2 M tiles, one per issuing thread
typedef Cfg<13, 13, 48, 96, 3, 1, 3, 2, 2, false, true, true> CfgConv4Pool;   // ... with the following 2x2 max-pool fused (shared-memory atomicMax raster)
// The same layer dict on a 28 x 28 x 1 input (BASELINE config 1, the reference's small CNN on MNIST-sized images): 28 x 28 and
// 14 x 14 rasters.  Round 2 ran these on the FP32 CUDA-core kernels; the kernel template is shape-generic, a shape only needs
// its tile plan.  conv2's 96 KB raster leaves room for one input buffer.
typedef Cfg<28, 28, 1, 24, 5, 1, 7, 2, 3, true> CfgS1Conv1;    // 7 M tiles in groups of 3 + 3 + 1, weights resident
typedef Cfg<28, 28, 24, 32, 5, 1, 8, 1, 3, true> CfgS1Conv2;
typedef Cfg<14, 14, 32, 48, 3, 2, 6, 2, 4, false> CfgS1Conv3;  // 2 samples, 4 M tiles
typedef Cfg<14, 14, 48, 96, 3, 1, 3, 2, 2, false, false, true> CfgS1Conv4;
typedef Cfg<14, 14, 48, 96, 3, 1, 3, 2, 2, false, true, true> CfgS1Conv4Pool;
// every forward configuration / every configuration with the fused pool
#define NNAL_CTC_FWD(X) X(CfgConv1) X(CfgConv2) X(CfgConv3) X(CfgConv4) X(CfgS1Conv1) X(CfgS1Conv2) X(CfgS1Conv3) X(CfgS1Conv4)
#define NNAL_CTC_POOL(X) X(CfgConv4Pool) X(CfgS1Conv4Pool)

template <class C>
static bool matches(const Layer& L) {
  return L.in_h == C::H && L.in_w == C::W && L.in_c == C::CIN_REAL && L.out_c == C::COUT_REAL && L.kh == C::KS && L.kw == C::KS;
}

template <class C>
static int pack_from(nnal_ctx* ctx, const float* W, void** dst, float w_scale) {
  size_t bytes = (size_t)C::NSTAGE_W * C::W_STAGE_BYTES;
  if (!*dst) CUDA_TRY(ctx, cudaMalloc(dst, bytes));
  int64_t total = (int64_t)C::NSTAGE_W * C::KPS * 2 * C::COUT * 8;
  int grid = (int)((total + 255) / 256);
  pack_conv_weights_kernel<<<grid, 256, 0, ctx->stream>>>(W, (uint8_t*)*dst, C::NTAPS, C::CIN, C::COUT, C::CIN_REAL, C::COUT_REAL, C::KPS, C::NK,
                                                          C::NSTAGE_W, w_scale);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}
template <class C>
static int pack(nnal_ctx* ctx, Layer& L) { return pack_from<C>(ctx, L.W, (void**)&L.Wh, L.w_scale); }

template <class C>
static int launch(nnal_ctx* ctx, const Layer& L, const nnal_h* in_hi, const nnal_h* in_lo, nnal_h* out_hi,
                  nnal_h* out_lo, int64_t n, const void* wpack = nullptr, const GatherArgs* gather = nullptr, float* out_f32 = nullptr,
                  float scale_inv = 0.f) {
  CUtensorMap tmHi, tmLo;
  GatherArgs ga;
  memset(&ga, 0, sizeof(ga));
  if (C::GATHER) {
    memset(&tmHi, 0, sizeof(tmHi));
    memset(&tmLo, 0, sizeof(tmLo));
    ga = *gather;
  } else {
    NNAL_TRY(make_act_tmap(ctx, &tmHi, in_hi, (int)n, C::H, C::W, C::CIN, C::WP, C::HP, C::G));
    NNAL_TRY(make_act_tmap(ctx, &tmLo, in_lo, (int)n, C::H, C::W, C::CIN, C::WP, C::HP, C::G));
  }
  static bool attr = false;
  if (!attr) {
    CUDA_TRY(ctx, cudaFuncSetAttribute(conv_tc_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM));
    attr = true;
  }
  ConvParams p;
  p.wpack = (const uint8_t*)(wpack ? wpack : L.Wh); p.bias = L.b; p.out_hi = out_hi; p.out_lo = out_lo; p.out_f32 = out_f32; p.n = (int)n; p.w_scale_inv = C::RAW ? scale_inv : L.w_scale_inv;
  const int grid = nnal_conv_grid(ctx, (n + C::G - 1) / C::G);
  conv_tc_kernel<C><<<grid, C::THREADS, C::SMEM, ctx->stream>>>(tmHi, tmLo, p, ga);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}

}  // namespace ctc

bool nnal_tc_conv_supported(const nnal_ctx*, const Layer& L) {
  if (L.type != NNAL_LAYER_CONV || !L.Wh) return false;
#define X(C) if (ctc::matches<ctc::C>(L)) return true;
  NNAL_CTC_FWD(X)
#undef X
  return false;
}

int nnal_tc_prepare_conv(nnal_ctx* ctx, Layer& L) {
  if (L.type != NNAL_LAYER_CONV) return NNAL_OK;
#define X(C) if (ctc::matches<ctc::C>(L)) return ctc::pack<ctc::C>(ctx, L);
  NNAL_CTC_FWD(X)
#undef X
  return NNAL_OK;
}

// ---- conv1 on x-im2col'd input ("x16") -------------------------------------------------------------------------
namespace ctc {
// W fp32 [5][5][C][cout] -> W' fp32 [5][1][16][cout]:  W'[dy][0][dx * C + ch][co] = W[dy][dx][ch][co], rest 0
__global__ void rearrange_x16_kernel(const float* __restrict__ W, float* __restrict__ Wx, int KH, int KW, int C, int COUT) {
  const int total = KH * 16 * COUT;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    const int co = e % COUT, j = (e / COUT) % 16, dy = e / (COUT * 16);
    const int dx = j / C, ch = j % C;
    Wx[e] = (dx < KW) ? W[(((size_t)dy * KW + dx) * C + ch) * COUT + co] : 0.f;
  }
}
// fp32 NHWC [n][H][W][C] -> x-im2col'd fp16 hi/lo planes [n][H][W][16] (inputs that do not come from the fused gather)
__global__ void __launch_bounds__(256) split_x16_kernel(const float* __restrict__ in, nnal_h* __restrict__ hi,
                                                         nnal_h* __restrict__ lo, int64_t rows, int W, int C, int KW) {
  const int64_t total = rows * 16;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = e / 16;
    const int j = (int)(e - r * 16);
    const int dx = j / C, ch = j % C;
    const int x = (int)(r % W) + dx - KW / 2;
    const float v = (dx < KW && x >= 0 && x < W) ? in[(r + dx - KW / 2) * C + ch] : 0.f;
    nnal_h h, l;
    nnal_split(v, h, l);
    hi[e] = h;
    lo[e] = l;
  }
}
}  // namespace ctc

bool nnal_tc_conv_x16_supported(const nnal_ctx*, const Layer& L) {
  return L.type == NNAL_LAYER_CONV && L.Wx && L.in_h == 25 && L.in_w == 25 && L.in_c == 3 && L.out_c == 24 && L.kh == 5 && L.kw == 5;
}
int nnal_tc_prepare_conv_x16(nnal_ctx* ctx, Layer& L) {
  if (!(L.type == NNAL_LAYER_CONV && L.in_h == 25 && L.in_w == 25 && L.in_c == 3 && L.out_c == 24 && L.kh == 5 && L.kw == 5)) return NNAL_OK;
  float* Wx = nullptr;
  const int total = 5 * 16 * 24;
  CUDA_TRY(ctx, cudaMalloc(&Wx, total * sizeof(float)));
  ctc::rearrange_x16_kernel<<<(total + 255) / 256, 256, 0, ctx->stream>>>(L.W, Wx, 5, 5, 3, 24);
  ctx->launches++;
  int rc = ctc::pack_from<ctc::CfgConv1X>(ctx, Wx, &L.Wx, L.w_scale);
  cudaStreamSynchronize(ctx->stream);
  cudaFree(Wx);
  return rc;
}
int nnal_k_split_x16(nnal_ctx* ctx, const float* in, nnal_h* hi, nnal_h* lo, int64_t rows, int W, int C, int KW) {
  const int64_t total = rows * 16;
  if (total == 0) return NNAL_OK;
  int grid = (int)((total + 255) / 256 < (int64_t)ctx->sm_count * 16 ? (total + 255) / 256 : (int64_t)ctx->sm_count * 16);
  ctc::split_x16_kernel<<<grid, 256, 0, ctx->stream>>>(in, hi, lo, rows, W, C, KW);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}
// in_hi / in_lo: x-im2col'd planes [n][25][25][16]
int nnal_tc_conv_x16(nnal_ctx* ctx, const Layer& L, const nnal_h* in_hi, const nnal_h* in_lo, nnal_h* out_hi, nnal_h* out_lo,
                     int64_t n) {
  if (n == 0) return NNAL_OK;
  return ctc::launch<ctc::CfgConv1X>(ctx, L, in_hi, in_lo, out_hi, out_lo, n, L.Wx);
}
bool nnal_tc_conv1_fused_supported(const nnal_ctx* ctx, const Layer& L, const Volume& v, int d1, int d2, int d3) {
  return nnal_tc_conv_x16_supported(ctx, L) && v.dtype == NNAL_F32 && v.m == 3 && d1 == 25 && d2 == 25 && d3 == 1;
}
int nnal_tc_conv1_fused(nnal_ctx* ctx, const Layer& L, const FusedGather& fg, nnal_h* out_hi, nnal_h* out_lo, int64_t n) {
  if (n == 0) return NNAL_OK;
  ctc::GatherArgs ga;
  ga.vol = (const float*)fg.vol->data; ga.Xp = fg.vol->X; ga.Yp = fg.vol->Y; ga.Zp = fg.vol->Z; ga.inds = fg.d_inds;
  ga.tab = nnal_make_norm_tab(*fg.vol, fg.d3, fg.h_stats, fg.norm_mode);
  ga.flags = ctx->dbg.wt_flags;
  return ctc::launch<ctc::CfgConv1XG>(ctx, L, nullptr, nullptr, out_hi, out_lo, n, L.Wx, &ga);
}
// conv + the following 2x2/s2 SAME max-pool in one kernel: output planes are [n][ceil(H/2)][ceil(W/2)][Cout]
bool nnal_tc_conv_pool_supported(const nnal_ctx*, const Layer& L) {
  if (L.type != NNAL_LAYER_CONV || !L.Wh) return false;
#define X(C) if (ctc::matches<ctc::C>(L)) return true;
  NNAL_CTC_POOL(X)
#undef X
  return false;
}
int nnal_tc_conv_pool(nnal_ctx* ctx, const Layer& L, const nnal_h* in_hi, const nnal_h* in_lo, nnal_h* out_hi,
                      nnal_h* out_lo, int64_t n) {
  if (n == 0) return NNAL_OK;
#define X(C) if (ctc::matches<ctc::C>(L)) return ctc::launch<ctc::C>(ctx, L, in_hi, in_lo, out_hi, out_lo, n);
  NNAL_CTC_POOL(X)
#undef X
  NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "conv+pool shape not covered by the tensor-core kernel");
}

int nnal_tc_conv(nnal_ctx* ctx, const Layer& L, const nnal_h* in_hi, const nnal_h* in_lo, nnal_h* out_hi,
                 nnal_h* out_lo, int64_t n) {
  if (n == 0) return NNAL_OK;
#define X(C) if (ctc::matches<ctc::C>(L)) return ctc::launch<ctc::C>(ctx, L, in_hi, in_lo, out_hi, out_lo, n);
  NNAL_CTC_FWD(X)
#undef X
  NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "conv shape not covered by the tensor-core kernel");
}

// ---- data-gradient convolutions (shrunk.cu): d_in = correlation of dz with the flipped, transposed filter ------------------
// d_in[y][x][ci] = sum_{dy,dx,co} dz[y - dy + ph][x - dx + pw][co] W[dy][dx][ci][co] is the SAME-padded forward convolution of dz
// (Cout channels) with W'[dy'][dx'][co][ci] = W[kh-1-dy'][kw-1-dx'][ci][co]: the same shift-GEMM kernel with the roles of the
// channel counts swapped, a raw float32 epilogue (no bias, no ReLU) and dz as power-of-two scaled fp16 hi/lo planes.
namespace ctc {
//                 H   W  CIN COUT KS G KPS NBUF TG CAT  POOL   DUAL  KW NWG GATHER NACC RAW
typedef Cfg<25, 25, 32, 24, 5, 1, 5, 1, 3, true, false, false, 0, 2, false, 2, true> CfgBwd2;   // PW1 conv2: one 108 KB input raster (no room for two)
typedef Cfg<13, 13, 48, 32, 3, 1, 9, 2, 2, true, false, false, 0, 2, false, 2, true> CfgBwd3;   // PW1 conv3 (weights resident)
typedef Cfg<13, 13, 96, 48, 3, 1, 3, 2, 2, true, false, false, 0, 2, false, 2, true> CfgBwd4;   // PW1 conv4
// ... and of the same layer dict on a 28 x 28 x 1 input (config 1)
typedef Cfg<28, 28, 32, 24, 5, 1, 5, 1, 3, true, false, false, 0, 2, false, 2, true> CfgS1Bwd2;
typedef Cfg<14, 14, 48, 32, 3, 1, 9, 2, 2, true, false, false, 0, 2, false, 2, true> CfgS1Bwd3;
typedef Cfg<14, 14, 96, 48, 3, 1, 3, 2, 2, true, false, false, 0, 2, false, 2, true> CfgS1Bwd4;
#define NNAL_CTC_BWD(X) X(CfgBwd2) X(CfgBwd3) X(CfgBwd4) X(CfgS1Bwd2) X(CfgS1Bwd3) X(CfgS1Bwd4)

template <class C>
static bool matches_bwd(const Layer& L) {
  return L.type == NNAL_LAYER_CONV && L.in_h == C::H && L.in_w == C::W && L.out_c == C::CIN_REAL && L.in_c == C::COUT_REAL &&
         L.kh == C::KS && L.kw == C::KS;
}
// W fp32 [kh][kw][cin][cout] -> W' fp32 [kh][kw][cout][cin], taps reversed
__global__ void flip_transpose_kernel(const float* __restrict__ W, float* __restrict__ Wf, int KH, int KW, int CIN, int COUT) {
  const int total = KH * KW * CIN * COUT;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    const int ci = e % CIN, co = (e / CIN) % COUT, tap = e / (CIN * COUT);
    const int dy = tap / KW, dx = tap % KW;
    Wf[e] = W[((size_t)((KH - 1 - dy) * KW + (KW - 1 - dx)) * CIN + ci) * COUT + co];
  }
}
template <class C>
static int prepare_bwd(nnal_ctx* ctx, const Layer& L, void** packed) {
  float* Wf = nullptr;
  const int total = L.kh * L.kw * L.in_c * L.out_c;
  CUDA_TRY(ctx, cudaMalloc(&Wf, (size_t)total * sizeof(float)));
  flip_transpose_kernel<<<(total + 255) / 256, 256, 0, ctx->stream>>>(L.W, Wf, L.kh, L.kw, L.in_c, L.out_c);
  ctx->launches++;
  int rc = pack_from<C>(ctx, Wf, packed, L.w_scale);
  cudaStreamSynchronize(ctx->stream);
  cudaFree(Wf);
  return rc;
}
}  // namespace ctc

bool nnal_tc_conv_bwd_supported(const nnal_ctx*, const Layer& L) {
  if (!L.has_weights) return false;
#define X(C) if (ctc::matches_bwd<ctc::C>(L)) return true;
  NNAL_CTC_BWD(X)
#undef X
  return false;
}
// *packed: device buffer with the flipped, transposed filter in the kernel's operand layout (allocated here when null)
int nnal_tc_conv_bwd_prepare(nnal_ctx* ctx, const Layer& L, void** packed) {
#define X(C) if (ctc::matches_bwd<ctc::C>(L)) return ctc::prepare_bwd<ctc::C>(ctx, L, packed);
  NNAL_CTC_BWD(X)
#undef X
  NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "conv gradient shape not covered by the tensor-core kernel");
}
// dz_hi / dz_lo: planes [n][H][W][Cout] of dz * 2^e; d_in [n][H][W][Cin] float32 = acc * scale_inv (scale_inv = 2^-e / w_scale)
int nnal_tc_conv_bwd(nnal_ctx* ctx, const Layer& L, const void* packed, const nnal_h* dz_hi, const nnal_h* dz_lo, float* d_in,
                     int64_t n, float scale_inv) {
  if (n == 0) return NNAL_OK;
#define X(C) if (ctc::matches_bwd<ctc::C>(L)) return ctc::launch<ctc::C>(ctx, L, dz_hi, dz_lo, nullptr, nullptr, n, packed, nullptr, d_in, scale_inv);
  NNAL_CTC_BWD(X)
#undef X
  NNAL_FAIL(ctx, NNAL_ERR_UNSUPPORTED, "conv gradient shape not covered by the tensor-core kernel");
}
