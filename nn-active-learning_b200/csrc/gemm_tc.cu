// tcgen05 / TMEM / TMA GEMM for the fully-connected layers (sm_100a).
//
//   out[M][N] = act( A[M][K] . W[N][K]^T + b )          (sample-major restatement of W@x+b, NN.py:322-327)
//
// Precision: the north-star tolerance (posteriors within 1e-4 absolute of the float64 oracle) rules out
// single-pass bf16 / fp16 / tf32 operands (measured: 2e-3 / 1.2e-4 / 1.1e-4 max posterior error on PW1,
// DESIGN.md 4).  Operands are therefore split into two fp16 terms x = hi + lo
// (hi = fp16(x), lo = fp16(x - hi); weights scaled by a power of two so that the lo terms stay normal) and each K-step issues
// three kind::f16 MMAs
//   hi.hi + hi.lo + lo.hi      (lo.lo ~ 2^-22 relative is dropped)
// into FP32 TMEM accumulators (chunks of 8 k-blocks, summed with round-to-nearest in registers: the tensor core accumulates
// with round-toward-zero): 1.1e-5 ... 2.3e-5 max posterior error measured on PW1.
//
// Structure: persistent CTA pairs (clusters of 2, one pair per two SMs), 384 threads per CTA.  A pair computes a
// 256 (M) x 256 (N) tile with the 2-SM MMA: each CTA holds its own 128 rows of A and half (128) of the 256 W rows, so a
// CTA reads 64 KB per 64-wide k-block for the MMA work that needed 96 KB with one CTA per 128x256 tile.
//   warp 0    : TMA producer (both CTAs) -- cp.async.bulk.tensor 2-D tiles (SWIZZLE_128B) of A_hi, A_lo, W_hi, W_lo; the
//               loads of both CTAs complete on the leader CTA's full barrier
//   warp 1    : MMA issuer (leader CTA only) -- one elected lane issues tcgen05.mma.cta_group::2.kind::f16, M=256 N=256 K=16;
//               tcgen05.commit ... multicast frees the stage in both CTAs and signals both accumulator-full barriers
//   warp 2    : TMEM allocator (cta_group::2, 512 columns per CTA = two 128x256 FP32 accumulators)
//   warps 4-11: epilogue (both CTAs, own 128 rows) -- tcgen05.ld -> FP32 register sums -> +bias, ReLU -> global (fp32 / fp16
//               hi,lo); the 16 epilogue warps of the pair release an accumulator on the leader's empty barrier
// smem ring per CTA: 3 stages x (2 x 16 KB A + 2 x 16 KB W) = 192 KB, mbarrier full/empty pairs.
//
// Chunked accumulation.  The tensor core adds into its FP32 accumulator with round-toward-zero
// (measured on B200: signed bias -1.1e-5 of the output rms at K=4704, shrinking linearly with the
// number of accumulations -- profiles/r1_precision.md).  The K loop is therefore cut into chunks of
// CHUNK_KB k-blocks; each chunk accumulates from zero into one of the two TMEM buffers while the
// epilogue warps drain the other one and add it to per-thread FP32 sums with round-to-nearest.
#include "nnal_common.cuh"
#include <cuda.h>

namespace tc {

constexpr int BM = 128, BN = 256, BK = 64, STAGES = 3;  // BM: rows per CTA; a pair tile is 2 BM x BN
constexpr int PAIR_M = 2 * BM;
constexpr int A_BYTES = BM * BK * 2;                  // 16 KB
constexpr int B_BYTES = (BN / 2) * BK * 2;            // 16 KB: this CTA's half of the W rows
constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;   // 64 KB per CTA; the leader's full barrier expects both CTAs' bytes
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
constexpr int NUM_THREADS = 384;
constexpr int CHUNK_KB = 8;                           // k-blocks (of 64) accumulated inside the tensor core

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// Bounded wait: a protocol bug must surface as a CUDA error (trap), never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok = 0;
  long long t0 = 0;
  for (uint32_t spin = 0;; ++spin) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    if (ok) return;
    if ((spin & 0xfff) == 0xfff) {
      long long now = clock64();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 4000000000ll) __trap();     // ~2 s
    }
  }
}

// Arrive on the barrier at the same offset in CTA `rank` of the cluster (the pair's leader for the accumulator-empty barrier).
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar, uint32_t rank) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t}"
      ::"r"(bar), "r"(rank)
      : "memory");
}
__device__ __forceinline__ uint32_t map_to_rank(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// 2-SM form: lands in this CTA's shared memory and completes on `bar`, which may be the peer (leader) CTA's barrier
// (a shared::cluster address from map_to_rank).
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tmap, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(tmap), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
// start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) | version=1 [46,48) | base_offset [49,52) | layout [61,64)
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3ffff) >> 4);
  d |= (uint64_t)1 << 16;                  // LBO (ignored for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;        // SBO: 8 rows x 128 B
  d |= (uint64_t)1 << 46;                  // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                  // SWIZZLE_128B
  return d;
}

// kind::f16 instruction descriptor: D=F32, A=B=BF16, both K-major, N>>3 at [17,23), M>>4 at [24,29)
// (A/B format field 0 = F16; 1 would be BF16)
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N) {
  return (1u << 4) | (0u << 7) | (0u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives on the barrier at this offset in both CTAs of the pair once the leader's issued MMAs retire
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"((uint16_t)0x3) : "memory");
}
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

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

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

struct FcParams {
  const float* bias;
  float* out;
  nnal_h* out_hi;     // optional: fp16 split planes of the activated output (next layer's A operand)
  nnal_h* out_lo;
  int ld_split;              // row stride (elements) of the split planes
  int M, N, num_kb, relu, ldo;
  float w_scale_inv;
  int accum;                 // out += result (Gram partial sums over sample chunks)
  DropSpec drop;             // tf.nn.dropout on the activated output (thresh == 0: off)
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
fc_tc_pair_kernel(const __grid_constant__ CUtensorMap tmAh, const __grid_constant__ CUtensorMap tmAl,
                  const __grid_constant__ CUtensorMap tmBh, const __grid_constant__ CUtensorMap tmBl, FcParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;            // SWIZZLE_128B tiles need 1024-B alignment
  uint8_t* base_ptr = smem_raw + (base - raw);
  // Both CTAs of a pair use the same offsets: the leader's MMA descriptors and commits address the peer's stages and barriers
  // at the offsets of its own.
  const uint32_t bar0 = base + STAGES * STAGE_BYTES;
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (STAGES + s); };
  auto tfull_bar = [&](int a) { return bar0 + 8u * (2 * STAGES + a); };
  auto tempty_bar = [&](int a) { return bar0 + 8u * (2 * STAGES + 2 + a); };
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(base_ptr + STAGES * STAGE_BYTES + 8 * (2 * STAGES + 4));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();                 // 0: leader (issues the MMAs), 1: peer
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const int mblocks = (p.M + PAIR_M - 1) / PAIR_M, nblocks = (p.N + BN - 1) / BN;
  const int ntiles = mblocks * nblocks;
  // Tile order (in pair tiles): N is cut into bands of NBAND column blocks and a band is finished (all row blocks) before the next
  // starts.  With the plain row-major order the tiles in flight touch EVERY column block: fc1's weight planes (77 MB) went through
  // the L2 once per wave and were re-read from HBM 14 times per launch (1.42 GB read against 0.39 GB algorithmic,
  // profiles/r2_traffic.json); with bands, fc1 reads 1.22 GB and fc2 0.99 GB (was 1.22) and both run 2-3 % faster.  (The band's
  // planes still do not survive from one wave to the next -- L2 evict_last / evict_first hints on the TMA loads changed nothing
  // for fc1 and cost fc2 20 % more reads.)
  constexpr int NBAND = 8;
  auto tile_blocks = [&](int t, int& m_blk, int& n_blk) {
    const int full = mblocks * NBAND;
    int b = t / full;
    const int nbands = (nblocks + NBAND - 1) / NBAND;
    if (b > nbands - 1) b = nbands - 1;
    const int r = t - b * full;
    const int wb = nblocks - b * NBAND < NBAND ? nblocks - b * NBAND : NBAND;
    m_blk = r / wb;
    n_blk = b * NBAND + r % wb;
  };

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmAh));
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmAl));
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmBh));
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmBl));
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    // accumulator-empty: released by the 8 epilogue warps of each CTA (only the leader's barrier is used)
    for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 16); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
  }
  // the peer's TMA and epilogue signal the leader's barriers: both CTAs' barriers must be initialised first
  tc_fence_before();
  cluster_sync();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer (both CTAs): own 128 rows of A, own 128 of the tile's 256 W rows =====
    if (lane == 0) {
      uint32_t it = 0;
      const int a_row = (int)rank * BM, b_row = (int)rank * (BN / 2);
      for (int t = pair; t < ntiles; t += npairs) {
        int n_blk, m_blk;
        tile_blocks(t, m_blk, n_blk);
        for (int kb = 0; kb < p.num_kb; ++kb, ++it) {
          const int s = it % STAGES;
          const uint32_t ph = (it / STAGES) & 1;
          mbar_wait(empty_bar(s), ph ^ 1);
          const uint32_t sa = base + s * STAGE_BYTES;
          const uint32_t fb = map_to_rank(full_bar(s), 0);
          if (rank == 0) mbar_arrive_expect_tx(full_bar(s), 2 * STAGE_BYTES);
          tma_load_2d(sa, &tmAh, fb, kb * BK, m_blk * PAIR_M + a_row);
          tma_load_2d(sa + A_BYTES, &tmAl, fb, kb * BK, m_blk * PAIR_M + a_row);
          tma_load_2d(sa + 2 * A_BYTES, &tmBh, fb, kb * BK, n_blk * BN + b_row);
          tma_load_2d(sa + 2 * A_BYTES + B_BYTES, &tmBl, fb, kb * BK, n_blk * BN + b_row);
        }
      }
    }
  } else if (warp == 1 && rank == 0) {
    // ===== MMA issuer (leader): warp-uniform control flow, one elected lane issues =====
    const uint32_t idesc = make_idesc_bf16(PAIR_M, BN);
    uint32_t it = 0, cc = 0;                                     // smem-stage counter, accumulation-chunk counter
    for (int t = pair; t < ntiles; t += npairs) {
      for (int kb0 = 0; kb0 < p.num_kb; kb0 += CHUNK_KB, ++cc) {
        const int acc = cc & 1;
        const uint32_t acc_ph = (cc >> 1) & 1;
        mbar_wait(tempty_bar(acc), acc_ph ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        const int kb1 = kb0 + CHUNK_KB < p.num_kb ? kb0 + CHUNK_KB : p.num_kb;
        for (int kb = kb0; kb < kb1; ++kb, ++it) {
          const int s = it % STAGES;
          const uint32_t ph = (it / STAGES) & 1;
          mbar_wait(full_bar(s), ph);
          tc_fence_after();
          if (elect_one_sync()) {
            const uint32_t sa = base + s * STAGE_BYTES;
            const uint64_t dAh = make_desc_sw128(sa), dAl = make_desc_sw128(sa + A_BYTES);
            const uint64_t dBh = make_desc_sw128(sa + 2 * A_BYTES), dBl = make_desc_sw128(sa + 2 * A_BYTES + B_BYTES);
#pragma unroll
            for (int k = 0; k < BK / 16; ++k) {
              const uint64_t adv = (uint64_t)(k * 2);            // +32 B per K=16 step (start address >> 4)
              umma_bf16(d_tmem, dAl + adv, dBh + adv, idesc, ((kb - kb0) | k) != 0);
              umma_bf16(d_tmem, dAh + adv, dBl + adv, idesc, 1);
              umma_bf16(d_tmem, dAh + adv, dBh + adv, idesc, 1);
            }
            umma_commit_pair(empty_bar(s));                      // frees the smem stage of both CTAs when the MMAs retire
            if (kb == kb1 - 1) umma_commit_pair(tfull_bar(acc)); // chunk complete -> both epilogues
          }
          __syncwarp();
        }
      }
    }
  } else if (warp >= 4) {
    // ===== epilogue: drain each chunk from TMEM into FP32 register sums (round-to-nearest adds) =====
    const int q = warp & 3;                                      // TMEM lane quarter owned by this warp
    const int half = (warp - 4) >> 2;                            // which 128 of the 256 accumulator columns
    uint32_t cc = 0;
    for (int t = pair; t < ntiles; t += npairs) {
      int n_blk, m_blk;
      tile_blocks(t, m_blk, n_blk);
      float sum[128];
#pragma unroll
      for (int j = 0; j < 128; ++j) sum[j] = 0.f;
      for (int kb0 = 0; kb0 < p.num_kb; kb0 += CHUNK_KB, ++cc) {
        const int acc = cc & 1;
        const uint32_t acc_ph = (cc >> 1) & 1;
        mbar_wait(tfull_bar(acc), acc_ph);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BN + half * 128);
#pragma unroll
        for (int c = 0; c < 128; c += 16) {
          float v[16];
          tmem_ld16(taddr + c, v);
#pragma unroll
          for (int j = 0; j < 16; ++j) sum[c + j] += v[j];
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(tempty_bar(acc), 0);
      }
      const int row = m_blk * PAIR_M + (int)rank * BM + q * 32 + lane;
      if (row < p.M) {
#pragma unroll
        for (int c = 0; c < 128; c += 16) {
          const int col0 = n_blk * BN + half * 128 + c;
          if (col0 >= p.N) continue;
          float v[16];
          if (col0 + 16 <= p.N) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              float x = sum[c + j] * p.w_scale_inv + (p.bias ? __ldg(p.bias + col0 + j) : 0.f);
              v[j] = p.relu ? fmaxf(x, 0.f) : x;
            }
            if (p.drop.thresh) {                                   // NN.py:169-171: dropout on the layer's output
              const uint32_t pos = (uint32_t)(p.drop.row0 + row);
#pragma unroll
              for (int jb = 0; jb < 4; ++jb) {
                uint32_t r4[4];
                philox4x32_10((uint32_t)(col0 + 4 * jb) >> 2, pos, p.drop.pass, p.drop.site, p.drop.k0, p.drop.k1, r4);
#pragma unroll
                for (int k = 0; k < 4; ++k) v[4 * jb + k] = r4[k] < p.drop.thresh ? v[4 * jb + k] / p.drop.keep : 0.f;
              }
            }
            if (p.out) {
              float4* dst = reinterpret_cast<float4*>(p.out + (size_t)row * p.ldo + col0);
              if (p.accum) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                  const float4 o = dst[j];
                  v[4 * j] += o.x; v[4 * j + 1] += o.y; v[4 * j + 2] += o.z; v[4 * j + 3] += o.w;
                }
              }
#pragma unroll
              for (int j = 0; j < 4; ++j) dst[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            }
            if (p.out_hi) {
              uint32_t hi[8], lo[8], amax = 0u;
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                nnal_h h0, h1, l0, l1;
                nnal_ovf_track(amax, v[2 * j]);
                nnal_ovf_track(amax, v[2 * j + 1]);
                nnal_split_unchecked(v[2 * j], h0, l0);
                nnal_split_unchecked(v[2 * j + 1], h1, l1);
                hi[j] = nnal_pack2(h0, h1);
                lo[j] = nnal_pack2(l0, l1);
              }
              nnal_ovf_commit(amax);
              uint4* dh = reinterpret_cast<uint4*>(p.out_hi + (size_t)row * p.ld_split + col0);
              uint4* dl = reinterpret_cast<uint4*>(p.out_lo + (size_t)row * p.ld_split + col0);
              dh[0] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
              dh[1] = make_uint4(hi[4], hi[5], hi[6], hi[7]);
              dl[0] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
              dl[1] = make_uint4(lo[4], lo[5], lo[6], lo[7]);
            }
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              if (col0 + j < p.N) {
                float x = sum[c + j] * p.w_scale_inv + (p.bias ? __ldg(p.bias + col0 + j) : 0.f);
                x = p.relu ? fmaxf(x, 0.f) : x;
                if (p.drop.thresh) {
                  uint32_t r4[4];
                  philox4x32_10((uint32_t)(col0 + j) >> 2, (uint32_t)(p.drop.row0 + row), p.drop.pass, p.drop.site, p.drop.k0,
                                p.drop.k1, r4);
                  x = r4[(col0 + j) & 3] < p.drop.thresh ? x / p.drop.keep : 0.f;
                }
                if (p.out && p.accum) x += p.out[(size_t)row * p.ldo + col0 + j];
                if (p.out) p.out[(size_t)row * p.ldo + col0 + j] = x;
                if (p.out_hi) {
                  nnal_h h, l;
                  nnal_split(x, h, l);
                  p.out_hi[(size_t)row * p.ld_split + col0 + j] = h;
                  p.out_lo[(size_t)row * p.ld_split + col0 + j] = l;
                }
              }
            }
          }
        }
      }
    }
  }

  // Neither CTA leaves while the other may still signal its barriers or (leader MMAs) use its shared and tensor memory.
  __syncwarp();
  tc_fence_before();
  cluster_sync();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
  }
}

// fp32 [M][K] -> fp16 hi/lo planes [M][Kp] (zero padded columns)
__global__ void __launch_bounds__(256) split_kernel(const float* __restrict__ in, nnal_h* __restrict__ hi,
                                                     nnal_h* __restrict__ lo, int64_t M, int K, int Kp, float scale) {
  const int64_t total = M * (int64_t)(Kp / 2);
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    int64_t r = e / (Kp / 2);
    int c = (int)(e - r * (Kp / 2)) * 2;
    float x0 = c < K ? in[r * K + c] * scale : 0.f;
    float x1 = c + 1 < K ? in[r * K + c + 1] * scale : 0.f;
    nnal_h h0, h1, l0, l1;
    nnal_split(x0, h0, l0);
    nnal_split(x1, h1, l1);
    *reinterpret_cast<uint32_t*>(hi + r * Kp + c) = nnal_pack2(h0, h1);
    *reinterpret_cast<uint32_t*>(lo + r * Kp + c) = nnal_pack2(l0, l1);
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct TcState {
  EncodeTiledFn encode = nullptr;
  int max_pairs = 0;         // co-resident CTA pairs of fc_tc_pair_kernel (0: not queried yet)
};

static int get_state(nnal_ctx* ctx, TcState** out) {
  if (!ctx->tc_state) {
    TcState* st = new TcState();
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || !fn) { delete st; NNAL_FAIL(ctx, NNAL_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available"); }
    st->encode = (EncodeTiledFn)fn;
    ctx->tc_state = st;
  }
  *out = (TcState*)ctx->tc_state;
  return NNAL_OK;
}

// 2-D fp16 tensor [rows][ld] (ld elements per row, `cols` valid) with a {64, box_rows} SWIZZLE_128B box
static int make_tmap(nnal_ctx* ctx, TcState* st, CUtensorMap* tm, const void* ptr, uint64_t cols, uint64_t rows, uint64_t ld,
                     uint32_t box_rows) {
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)BK, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = st->encode(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) NNAL_FAIL(ctx, NNAL_ERR_CUDA, "cuTensorMapEncodeTiled failed");
  return NNAL_OK;
}

}  // namespace tc

static inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

bool nnal_tc_fc_supported(const nnal_ctx*, const Layer& L) {
  return L.type == NNAL_LAYER_FC && L.Wh != nullptr && L.out_dim >= 64 && L.in_dim >= 64 && (L.out_dim % 8) == 0 &&
         (L.in_dim % 8) == 0;
}

// Builds the fp16 hi/lo planes of an FC weight (called from nnal_model_set_weights).
int nnal_tc_prepare_conv(nnal_ctx* ctx, Layer& L);
int nnal_tc_prepare_layer(nnal_ctx* ctx, Layer& L) {
  if (L.type == NNAL_LAYER_CONV) {
    NNAL_TRY(nnal_tc_prepare_conv(ctx, L));
    NNAL_TRY(nnal_tc_prepare_conv_x16(ctx, L));
    return nnal_wt_prepare_conv(ctx, L);
  }
  if (L.type != NNAL_LAYER_FC || L.out_dim < 64 || L.in_dim < 64) return NNAL_OK;
  const int Kp = round_up(L.in_dim, tc::BK);
  if (!L.Wh) {
    CUDA_TRY(ctx, cudaMalloc(&L.Wh, (size_t)L.out_dim * Kp * 2));
    CUDA_TRY(ctx, cudaMalloc(&L.Wl, (size_t)L.out_dim * Kp * 2));
  }
  L.k_pad = Kp;
  L.n_pad = L.out_dim;
  int64_t total = (int64_t)L.out_dim * (Kp / 2);
  int grid = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
  tc::split_kernel<<<grid, 256, 0, ctx->stream>>>(L.W, L.Wh, L.Wl, L.out_dim, L.in_dim, Kp, L.w_scale);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}

// Generic split-plane GEMM  out[M][N] (+)= scale * A[M][K] . B[N][K]^T (+ bias, ReLU): both operands are
// fp16 hi/lo planes, K-major, row strides lda/ldb elements (multiples of 8); the K tail of the last
// 64-wide block and rows beyond M/N are zero-filled by TMA.
int nnal_tc_gemm_planes(nnal_ctx* ctx, const nnal_h* Ah, const nnal_h* Al, int64_t lda, int64_t M, const nnal_h* Bh,
                        const nnal_h* Bl, int64_t ldb, int N, int64_t K, const float* bias, float scale, int relu,
                        int accum, float* out, int ldo, nnal_h* out_hi, nnal_h* out_lo, int ld_split,
                        const DropSpec* drop) {
  if (M == 0 || N == 0) return NNAL_OK;
  tc::TcState* st;
  NNAL_TRY(tc::get_state(ctx, &st));
  CUtensorMap tmAh, tmAl, tmBh, tmBl;
  NNAL_TRY(tc::make_tmap(ctx, st, &tmAh, Ah, (uint64_t)K, (uint64_t)M, (uint64_t)lda, tc::BM));
  NNAL_TRY(tc::make_tmap(ctx, st, &tmAl, Al, (uint64_t)K, (uint64_t)M, (uint64_t)lda, tc::BM));
  NNAL_TRY(tc::make_tmap(ctx, st, &tmBh, Bh, (uint64_t)K, (uint64_t)N, (uint64_t)ldb, tc::BN / 2));
  NNAL_TRY(tc::make_tmap(ctx, st, &tmBl, Bl, (uint64_t)K, (uint64_t)N, (uint64_t)ldb, tc::BN / 2));
  if (!st->max_pairs) {
    CUDA_TRY(ctx, cudaFuncSetAttribute(tc::fc_tc_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SMEM_BYTES));
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = 2; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
    cfg.gridDim = dim3(2 * ctx->sm_count);
    cfg.blockDim = dim3(tc::NUM_THREADS);
    cfg.dynamicSmemBytes = tc::SMEM_BYTES;
    cfg.stream = ctx->stream;
    cfg.attrs = &attr;
    cfg.numAttrs = 1;
    int n = 0;
    CUDA_TRY(ctx, cudaOccupancyMaxActiveClusters(&n, (void*)tc::fc_tc_pair_kernel, &cfg));
    if (n < 1) NNAL_FAIL(ctx, NNAL_ERR_CUDA, "fc_tc_pair_kernel: no CTA pair fits on the device");
    st->max_pairs = n;
  }
  tc::FcParams p;
  p.bias = bias; p.out = out; p.out_hi = out_hi; p.out_lo = out_lo; p.ld_split = ld_split;
  p.M = (int)M; p.N = N; p.num_kb = (int)((K + tc::BK - 1) / tc::BK); p.relu = relu; p.ldo = ldo; p.w_scale_inv = scale;
  p.accum = accum;
  p.drop = drop ? *drop : DropSpec();
  const int ntiles = cdiv(M, tc::PAIR_M) * cdiv(N, tc::BN);
  const int pairs = ntiles < st->max_pairs ? ntiles : st->max_pairs;
  tc::fc_tc_pair_kernel<<<2 * pairs, tc::NUM_THREADS, tc::SMEM_BYTES, ctx->stream>>>(tmAh, tmAl, tmBh, tmBl, p);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}

// A operand given as fp16 hi/lo planes [n][lda] (lda >= K, K % 8 == 0; the K tail of the last 64-wide
// block is zero-filled by TMA).  Outputs: fp32 [n][N] (out, may be null) and/or fp16 hi/lo planes
// [n][N] of the activated result (the next tensor-core layer's A operand).
int nnal_tc_fc_planes(nnal_ctx* ctx, const Layer& L, const nnal_h* Ah, const nnal_h* Al, int lda, float* out,
                      nnal_h* out_hi, nnal_h* out_lo, int64_t n, const DropSpec* drop) {
  return nnal_tc_gemm_planes(ctx, Ah, Al, lda, n, L.Wh, L.Wl, L.k_pad, L.out_dim, L.in_dim, L.b, L.w_scale_inv, L.relu, 0,
                             out, L.out_dim, out_hi, out_lo, L.out_dim, drop);
}

// Wide classifier head (c >= 64 classes): the logits GEMM.  Its own predicate, so the hidden layers keep theirs: the class
// count need not be a multiple of 8 (W's planes have c rows; TMA zero-fills the last 256-row block), the input width must
// be (16-byte rows of the A planes).  The planes are built by nnal_tc_prepare_layer for every FC with in, out >= 64.
bool nnal_tc_head_supported(const nnal_ctx*, const Layer& L) {
  return L.type == NNAL_LAYER_FC && L.Wh != nullptr && L.out_dim >= NNAL_WIDE_HEAD_MIN && L.in_dim >= 64 && (L.in_dim % 8) == 0;
}

// logits [n][ldz] = A . W^T + b, ldz = nnal_head_ldz(c): the epilogue's full 16-column groups store float4 at row * ldz + col0,
// so the row stride must keep 16-byte alignment for any c; columns >= c are not written.  No ReLU; `drop` (MC-dropout on
// the logits) uses the epilogue's tf.nn.dropout with drop->row0 the global position of chunk row 0.
int nnal_tc_head_planes(nnal_ctx* ctx, const Layer& L, const nnal_h* Ah, const nnal_h* Al, int lda, float* logits, int64_t n,
                        const DropSpec* drop) {
  return nnal_tc_gemm_planes(ctx, Ah, Al, lda, n, L.Wh, L.Wl, L.k_pad, L.out_dim, L.in_dim, L.b, L.w_scale_inv, 0, 0, logits,
                             nnal_head_ldz(L.out_dim), nullptr, nullptr, 0, drop);
}

// fp32 A operand [n][K] -> hi/lo planes [n][Kp] in ctx->splitA
static int split_operand(nnal_ctx* ctx, const Layer& L, const float* in, int64_t n, nnal_h** Ah, nnal_h** Al) {
  const int K = L.in_dim, Kp = L.k_pad;
  const size_t plane = (size_t)n * Kp * 2;
  NNAL_TRY(devbuf_reserve(ctx, ctx->splitA[0], plane));
  NNAL_TRY(devbuf_reserve(ctx, ctx->splitA[1], plane));
  *Ah = (nnal_h*)ctx->splitA[0].p;
  *Al = (nnal_h*)ctx->splitA[1].p;
  int64_t total = n * (int64_t)(Kp / 2);
  int grid = (int)((total + 255) / 256 < (int64_t)ctx->sm_count * 16 ? (total + 255) / 256 : (int64_t)ctx->sm_count * 16);
  tc::split_kernel<<<grid, 256, 0, ctx->stream>>>(in, *Ah, *Al, n, K, Kp, 1.f);
  ctx->launches++;
  return NNAL_OK;
}

// fp32 A operand [n][K]: split into planes first (used by the isolated test hook and mixed pipelines)
int nnal_tc_fc(nnal_ctx* ctx, const Layer& L, const float* in, float* out, int64_t n) {
  if (n == 0) return NNAL_OK;
  nnal_h *Ah, *Al;
  NNAL_TRY(split_operand(ctx, L, in, n, &Ah, &Al));
  return nnal_tc_fc_planes(ctx, L, Ah, Al, L.k_pad, out, nullptr, nullptr, n);
}

// the wide head's logits from fp32 features (shrunk-gradient forward, fp32 activations)
int nnal_tc_head(nnal_ctx* ctx, const Layer& L, const float* in, float* logits, int64_t n, const DropSpec* drop) {
  if (n == 0) return NNAL_OK;
  nnal_h *Ah, *Al;
  NNAL_TRY(split_operand(ctx, L, in, n, &Ah, &Al));
  return nnal_tc_head_planes(ctx, L, Ah, Al, L.k_pad, logits, n, drop);
}

// flat fp32 <-> fp16 hi/lo conversions (format changes between CUDA-core and tensor-core layers)
__global__ void __launch_bounds__(256) split_flat_kernel(const float* __restrict__ in, nnal_h* __restrict__ hi,
                                                          nnal_h* __restrict__ lo, int64_t count) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < count; e += (int64_t)gridDim.x * blockDim.x) {
    nnal_h h, l;
    nnal_split(in[e], h, l);
    hi[e] = h;
    lo[e] = l;
  }
}
__global__ void __launch_bounds__(256) merge_flat_kernel(const nnal_h* __restrict__ hi, const nnal_h* __restrict__ lo,
                                                          float* __restrict__ out, int64_t count) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < count; e += (int64_t)gridDim.x * blockDim.x)
    out[e] = nnal_merge(hi[e], lo[e]);
}
// fp32 [rows][C] -> fp16 hi/lo [rows][Cp] with zero-padded channels (conv1: 3 -> 8, one UMMA chunk per pixel)
__global__ void __launch_bounds__(256) split_pad_kernel(const float* __restrict__ in, nnal_h* __restrict__ hi,
                                                         nnal_h* __restrict__ lo, int64_t rows, int C, int Cp) {
  const int64_t total = rows * Cp;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = e / Cp;
    const int c = (int)(e - r * Cp);
    const float x = c < C ? in[r * C + c] : 0.f;
    nnal_h h, l;
    nnal_split(x, h, l);
    hi[e] = h;
    lo[e] = l;
  }
}
int nnal_k_split_pad(nnal_ctx* ctx, const float* in, nnal_h* hi, nnal_h* lo, int64_t rows, int C, int Cp) {
  const int64_t total = rows * Cp;
  if (total == 0) return NNAL_OK;
  int grid = (int)((total + 255) / 256 < (int64_t)ctx->sm_count * 16 ? (total + 255) / 256 : (int64_t)ctx->sm_count * 16);
  split_pad_kernel<<<grid, 256, 0, ctx->stream>>>(in, hi, lo, rows, C, Cp);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}

int nnal_k_split_flat(nnal_ctx* ctx, const float* in, nnal_h* hi, nnal_h* lo, int64_t count) {
  if (count == 0) return NNAL_OK;
  int grid = (int)((count + 255) / 256 < (int64_t)ctx->sm_count * 16 ? (count + 255) / 256 : (int64_t)ctx->sm_count * 16);
  split_flat_kernel<<<grid, 256, 0, ctx->stream>>>(in, hi, lo, count);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}
int nnal_k_merge_flat(nnal_ctx* ctx, const nnal_h* hi, const nnal_h* lo, float* out, int64_t count) {
  if (count == 0) return NNAL_OK;
  int grid = (int)((count + 255) / 256 < (int64_t)ctx->sm_count * 16 ? (count + 255) / 256 : (int64_t)ctx->sm_count * 16);
  merge_flat_kernel<<<grid, 256, 0, ctx->stream>>>(hi, lo, out, count);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return NNAL_OK;
}

int nnal_tc_release(nnal_ctx* ctx) {
  if (ctx->tc_state) { delete (tc::TcState*)ctx->tc_state; ctx->tc_state = nullptr; }
  return NNAL_OK;
}
