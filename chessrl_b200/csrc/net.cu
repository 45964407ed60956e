// net.cu -- forward pass of the policy/value ResNet (model.ChessModel, model.py:31-63, 111-122) for sm_100a.
//
// The 21 3x3 convolutions (1 stem + 10 residual blocks x 2) are >99.9% of the FLOPs (1.548 GFLOP/position) and run as
// ONE persistent kernel per evaluation batch, k_trunk4: implicit GEMMs on the 5th-generation tensor cores
// (tcgen05.mma.cta_group::2 across a CTA pair, fp32 accumulators in tensor memory), activations kept in an L2-resident
// scratch between layers, the three 1x1 head convolutions fused into the last layer's epilogue.  Then the policy head's
// Dense 128->1968 runs as a tcgen05 GEMM through k_conv_v2 (taps = 1), and k_softmax_value finishes the softmax and the
// value head (Dense 64->256->1 tanh).  k_conv_v2 with taps = 9 is one convolution layer on its own (crl_debug_conv).
#include "engine.cuh"

#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_fp8.h>
#include <math.h>
#include <type_traits>
#include <string.h>

namespace crl {

// ======================================================================================================
// PTX wrappers
// ======================================================================================================
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// bounded spin: a protocol bug traps (reported as a CUDA error) instead of hanging the GPU
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0;
  const uint32_t addr = smem_u32(bar);
#pragma unroll 1
  for (uint32_t spin = 0; spin < (1u << 26); ++spin) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
    if (done) return;
  }
  __trap();
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)map) : "memory");
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, 128-byte-swizzled shared-memory operand descriptor (cute::UMMA::SmemDescriptor bit layout):
// [0,14) start>>4 | [16,30) LBO>>4 (unused here) | [32,46) SBO>>4 = 8 rows * 128 B | [46,48) version=1 |
// [61,64) layout = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_kmajor_sw128_desc(uint32_t smem_addr) {
  return (uint64_t)((smem_addr >> 4) & 0x3FFF) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}

static constexpr int CONV_THREADS = 256;
static constexpr int TILE_N = 256;                       // all filters
static constexpr int BLOCK_K = 64;                       // one 128-byte swizzle atom of bf16

// ======================================================================================================
// k_conv_v2: CTA-pair (cta_group::2) implicit-GEMM kernel.  Two CTAs of a cluster share one 256-row tile: each loads
// its own 128 rows of A and HALF of the weight tile (128 of the 256 filters), so a stage is 32 KB and the ring has
// 6 stages.  The leader CTA issues tcgen05.mma.cta_group::2 (M=256 across the pair, N=256, K=16); tcgen05.commit
// multicasts stage-release and accumulator-ready to both CTAs; both CTAs run their own epilogue out of their own
// tensor memory.  With taps = 9 it is one 3x3 convolution layer (A: one TMA box per tap and 64-channel slice, the
// im2col tile with 'same' padding from the TMA unit's zero fill); with taps = 1 a plain GEMM (A through a 2-D map),
// the policy head's dense layer.  Its epilogue can also fuse the three 1x1 head convolutions (+BN+ReLU, head_w).
// ======================================================================================================
static constexpr int V2_STAGES = 6;
static constexpr int V2_A_BYTES = 128 * BLOCK_K * 2;      // 16 KB: this CTA's 128 rows
static constexpr int V2_B_BYTES = 128 * BLOCK_K * 2;      // 16 KB: this CTA's half of the 256 filters
static constexpr int V2_STAGE_BYTES = V2_A_BYTES + V2_B_BYTES;
static constexpr int V2_SMEM_BYTES = 1024 + V2_STAGES * V2_STAGE_BYTES + 2 * TILE_N * 4 + 3 * 256 * 4 + 64 + 512;
static constexpr uint32_t V2_IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((TILE_N >> 3) << 17) | ((256u >> 4) << 24);
static constexpr uint32_t PEER_MASK = 0xFEFFFFFFu;        // clears the CTA-rank bit of a shared::cluster address

struct ConvParams2 {
  const int* n_units_dev;       // boards (conv) or rows (gemm) on the device, or null
  int n_units_host;
  int rows_per_unit;            // 64 for convolutions (squares per board), 1 for the dense GEMM
  int taps;                     // 9 or 1
  int k_chunks;                 // K per tap / 64
  int n_tiles;                  // output tiles of 256 columns
  const float* scale;           // [n_tiles*256]
  const float* shift;           // [n_tiles*256]
  const __nv_bfloat16* residual;
  __nv_bfloat16* out;           // bf16 [rows][256] (may be null when only the fused heads are wanted)
  float* out_f32;               // gemm mode: fp32 [rows][out_ld]
  int out_ld;
  int relu;
  // fused heads (last convolution only)
  const float* head_w;          // [3][256]  policy ch0, policy ch1, value ch (1x1 conv kernels)
  const float* head_s;          // [6]       folded scale x3, shift x3
  __nv_bfloat16* pf_out;        // [boards][128] policy features, Keras flatten order (h*8+w)*2+c
  float* vf_out;                // [boards][64]
};

__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// arrive on the barrier at the same offset in CTA `cta` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t cta) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}"
      ::"r"(smem_u32(bar)), "r"(cta)
      : "memory");
}
// TMA loads of a CTA pair: the bytes are accounted on the LEADER's barrier
__device__ __forceinline__ void tma2_load_4d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1,
                                             int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"((uint64_t)map), "r"(smem_u32(bar) & PEER_MASK), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma2_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"((uint64_t)map), "r"(smem_u32(bar) & PEER_MASK), "r"(c0), "r"(c1)
      : "memory");
}
// the same loads with an L2 eviction-priority hint (createpolicy encodings, as CUTLASS's TMA::CacheHintSm90)
static constexpr uint64_t L2_EVICT_NORMAL = 0x1000000000000000ull;
static constexpr uint64_t L2_EVICT_FIRST = 0x12F0000000000000ull;
static constexpr uint64_t L2_EVICT_LAST = 0x14F0000000000000ull;
__device__ __forceinline__ void tma2_load_4d_hint(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1,
                                                  int c2, int c3, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint "
      "[%0], [%1, {%3, %4, %5, %6}], [%2], %7;"
      ::"r"(smem_u32(smem_dst)), "l"((uint64_t)map), "r"(smem_u32(bar) & PEER_MASK), "r"(c0), "r"(c1), "r"(c2), "r"(c3),
        "l"(policy)
      : "memory");
}
__device__ __forceinline__ void tma2_load_2d_hint(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1,
                                                  uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint "
      "[%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_u32(smem_dst)), "l"((uint64_t)map), "r"(smem_u32(bar) & PEER_MASK), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void umma2_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// e4m3 x e4m3 -> fp32, K = 32 per instruction (the same 32 bytes of a swizzle row as a bf16 K = 16 step)
__device__ __forceinline__ void umma2_fp8(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// instruction descriptor: fp32 accumulate, A = B = E4M3 (format 0), both K-major, N = 256, M = 256 (CTA pair)
static constexpr uint32_t V2_IDESC_FP8 = (1u << 4) | ((TILE_N >> 3) << 17) | ((256u >> 4) << 24);
// arrive (once the issued MMAs retire) on the barrier at this offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma2_commit_both(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(smem_u32(bar)), "h"((uint16_t)3)
      : "memory");
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(CONV_THREADS, 1)
k_conv_v2(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_w, ConvParams2 p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + V2_STAGES * V2_A_BYTES;
  float* s_scale = (float*)(smem + V2_STAGES * V2_STAGE_BYTES);
  float* s_shift = s_scale + TILE_N;
  float* s_hw = s_shift + TILE_N;               // [3][256]
  float* s_hs = s_hw + 3 * 256;                 // [8]
  uint64_t* bars = (uint64_t*)(s_hs + 16);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + V2_STAGES;
  uint64_t* tmem_full = bars + 2 * V2_STAGES;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_slot = (uint32_t*)(tmem_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  int n_units = p.n_units_host;
  if (p.n_units_dev) n_units = min(n_units, *p.n_units_dev);
  const long long total_rows = (long long)n_units * p.rows_per_unit;
  const int m_tiles = (int)((total_rows + 255) >> 8);
  const int n_work = m_tiles * p.n_tiles;
  const int n_kblocks = p.taps * p.k_chunks;
  const bool fused_heads = p.head_w != nullptr;

  if (threadIdx.x == 0) {
    prefetch_tmap(&map_a);
    prefetch_tmap(&map_w);
  }
  if (threadIdx.x == 32) {
    for (int i = 0; i < V2_STAGES; ++i) {
      mbar_init(&full_bar[i], 2);        // leader's arrive.expect_tx + the peer's remote arrive
      mbar_init(&empty_bar[i], 1);       // one multicast commit
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], 256);    // 128 epilogue threads of each CTA arrive on the leader's barrier
    }
    fence_barrier_init();
  }
  cluster_sync_all();
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  if (fused_heads) {
    for (int i = threadIdx.x; i < 3 * 256; i += CONV_THREADS) s_hw[i] = p.head_w[i];
    if (threadIdx.x < 6) s_hs[threadIdx.x] = p.head_s[threadIdx.x];
  }
  tcgen05_fence_before();
  cluster_sync_all();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (threadIdx.x == 0) {
    // ================= TMA producer (one per CTA) =================
    int stage = 0;
    uint32_t phase = 0;
    for (int w = pair; w < n_work; w += n_pairs) {
      const int mt = w / p.n_tiles, nt = w - mt * p.n_tiles;
      for (int kb = 0; kb < n_kblocks; ++kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * V2_STAGE_BYTES);
        if (p.taps == 9) {
          const int tap = kb / p.k_chunks, kc = kb - tap * p.k_chunks;
          tma2_load_4d(smem_a + stage * V2_A_BYTES, &map_a, &full_bar[stage], kc * BLOCK_K, tap % 3 - 1, tap / 3 - 1,
                       mt * 4 + (int)rank * 2);
        } else {
          tma2_load_2d(smem_a + stage * V2_A_BYTES, &map_a, &full_bar[stage], kb * BLOCK_K, mt * 256 + (int)rank * 128);
        }
        tma2_load_2d(smem_b + stage * V2_B_BYTES, &map_w, &full_bar[stage], kb * BLOCK_K, nt * TILE_N + (int)rank * 128);
        if (rank != 0) mbar_arrive_remote(&full_bar[stage], 0);
        if (++stage == V2_STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (threadIdx.x == 32 && rank == 0) {
    // ================= MMA issuer (leader CTA only) =================
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int w = pair; w < n_work; w += n_pairs, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
      tcgen05_fence_after();
      const uint32_t tmem_d = tmem_base + acc * TILE_N;
      for (int kb = 0; kb < n_kblocks; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tcgen05_fence_after();
        const uint64_t da = make_kmajor_sw128_desc(smem_u32(smem_a + stage * V2_A_BYTES));
        const uint64_t db = make_kmajor_sw128_desc(smem_u32(smem_b + stage * V2_B_BYTES));
#pragma unroll
        for (int k = 0; k < BLOCK_K / 16; ++k) umma2_bf16(tmem_d, da + 2 * k, db + 2 * k, V2_IDESC, (kb | k) != 0);
        umma2_commit_both(&empty_bar[stage]);
        if (kb == n_kblocks - 1) umma2_commit_both(&tmem_full[acc]);
        if (++stage == V2_STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
    // the peer's epilogue threads arrive on OUR tmem_empty barriers: drain them before this CTA may exit
    for (int a = 0; a < 2; ++a) {
      const int used = (it + 1 - a) >> 1;           // accumulator a served iterations a, a+2, ...
      if (used > 0) mbar_wait(&tmem_empty[a], (uint32_t)((used - 1) & 1));
    }
  } else if (warp >= 4) {
    // ================= epilogue (both CTAs, own tensor memory) =================
    const int q = warp & 3;
    const int row_in_cta = q * 32 + lane;
    int it = 0;
    for (int w = pair; w < n_work; w += n_pairs, ++it) {
      const int mt = w / p.n_tiles, nt = w - mt * p.n_tiles;
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      // the first tile of this CTA needs this layer's per-column constants; they are per n-tile
      if (it == 0 || p.n_tiles > 1) {
        // all 128 epilogue threads cooperate; named barrier 1 keeps the other warps out of it
        asm volatile("bar.sync 1, 128;" ::: "memory");
        for (int i = threadIdx.x - 128; i < TILE_N; i += 128) {
          s_scale[i] = p.scale[nt * TILE_N + i];
          s_shift[i] = p.shift[nt * TILE_N + i];
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");
      }
      mbar_wait(&tmem_full[acc], acc_phase);
      tcgen05_fence_after();
      const long long grow = (long long)mt * 256 + rank * 128 + row_in_cta;
      const bool valid = grow < total_rows;
      __nv_bfloat16* orow = p.out ? p.out + grow * TILE_N : nullptr;
      float* frow = p.out_f32 ? p.out_f32 + grow * p.out_ld + nt * TILE_N : nullptr;
      const __nv_bfloat16* rrow = p.residual ? p.residual + grow * TILE_N : nullptr;
      float h0 = 0.f, h1 = 0.f, h2 = 0.f;
#pragma unroll 1
      for (int c0 = 0; c0 < TILE_N; c0 += 32) {
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + acc * TILE_N + c0, v);
        tmem_ld_wait();
        if (!valid) continue;
        uint4 res[4];
        if (rrow) {
#pragma unroll
          for (int j = 0; j < 4; ++j) res[j] = *reinterpret_cast<const uint4*>(rrow + c0 + 8 * j);
        }
        float a[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) a[j] = __uint_as_float(v[j]) * s_scale[c0 + j] + s_shift[c0 + j];
        if (rrow) {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint32_t* rj = reinterpret_cast<const uint32_t*>(&res[j]);
#pragma unroll
            for (int h = 0; h < 4; ++h) {
              a[8 * j + 2 * h] += __uint_as_float(rj[h] << 16);
              a[8 * j + 2 * h + 1] += __uint_as_float(rj[h] & 0xFFFF0000u);
            }
          }
        }
        if (p.relu) {
#pragma unroll
          for (int j = 0; j < 32; ++j) a[j] = fmaxf(a[j], 0.f);
        }
        if (fused_heads) {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            // the heads see the bf16-rounded trunk output, like every other consumer of an activation
            const float x = __bfloat162float(__float2bfloat16_rn(a[j]));
            h0 = fmaf(x, s_hw[c0 + j], h0);
            h1 = fmaf(x, s_hw[256 + c0 + j], h1);
            h2 = fmaf(x, s_hw[512 + c0 + j], h2);
          }
        }
        if (orow) {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            uint32_t pk[4];
#pragma unroll
            for (int h = 0; h < 4; ++h) {
              __nv_bfloat162 b2 = __floats2bfloat162_rn(a[8 * j + 2 * h], a[8 * j + 2 * h + 1]);
              pk[h] = *reinterpret_cast<uint32_t*>(&b2);
            }
            *reinterpret_cast<uint4*>(orow + c0 + 8 * j) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
          }
        }
        if (frow) {
#pragma unroll
          for (int j = 0; j < 8; ++j)
            *reinterpret_cast<float4*>(frow + c0 + 4 * j) = make_float4(a[4 * j], a[4 * j + 1], a[4 * j + 2], a[4 * j + 3]);
        }
      }
      tcgen05_fence_before();
      mbar_arrive_remote(&tmem_empty[acc], 0);
      if (fused_heads && valid) {
        // row = board*64 + square: policy features in Keras flatten order (h*8+w)*2+c, value features [square]
        const float f0 = fmaxf(h0 * s_hs[0] + s_hs[3], 0.f), f1 = fmaxf(h1 * s_hs[1] + s_hs[4], 0.f);
        __nv_bfloat162 b2 = __floats2bfloat162_rn(f0, f1);
        reinterpret_cast<__nv_bfloat162*>(p.pf_out)[grow] = b2;
        p.vf_out[grow] = fmaxf(h2 * s_hs[2] + s_hs[5], 0.f);
      }
    }
  }

  tcgen05_fence_before();
  cluster_sync_all();
  if (warp == 2) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

struct LayerDesc {
  int map_in;            // index into the tensor-map table: 0 planes, 1 act4[0], 2 act4[1]
  int map_w;             // 3 + layer
  int k_chunks;
  int relu;
  int fuse_heads;
  int write_out;
  const float* scale;
  const float* shift;
  const __nv_bfloat16* residual;
  __nv_bfloat16* out;
};
// the fp8 tower's layer table (k_trunk4<..., FP8 = true>): activations are e4m3 codes x a power-of-two scale per layer.
// scale[n] already holds weight scale x input scale x folded BatchNorm scale; the residual is the block input, stored
// with its own layer's scale s_res; the output is stored as e4m3(a * inv_out) and means code x s_out.
struct LayerDesc8 {
  int map_in;
  int map_w;
  int k_chunks;          // Cin / 128
  int relu;
  int fuse_heads;
  int write_out;
  const float* scale;
  const float* shift;
  const uint8_t* residual;
  uint8_t* out;
  float s_res;
  float s_out;
  float inv_out;
};
struct TrunkParams {
  const int* n_dev;
  int n_host;
  int n_layers;
  const float* head_w;
  const float* head_s;
  __nv_bfloat16* pf_out;
  float* vf_out;
  __nv_bfloat16* dbg_out;   // test tap (crl_debug_tower): layer dbg_layer's output [boards][64][256], else null
  int dbg_layer;
  // L2 eviction priorities of the tower's TMA loads: the planes are read once (evict first), the weights are re-read
  // by every CTA pair for every group (evict last), the activation scratch keeps the default.  Kernel parameters
  // rather than compile-time constants: as immediates they compile to 8 more instructions per instantiation.
  uint64_t hint_planes, hint_weights;
};

// ======================================================================================================
// k_trunk4: the whole residual tower in ONE persistent kernel.
// A 3x3 'same' convolution of a board only reads that board, so a CTA pair can carry its boards through all 21
// layers without any grid-wide synchronisation.  Each pair works on a GROUP of two 256-row tiles (2 x 4 boards),
// tile X bound to tensor-memory accumulator X, and walks  for layer: for tile in (A, B): k-blocks .  While the
// tensor cores run tile B of layer L, the epilogue warps drain tile A of layer L and publish its activations, so
// the producer can prefetch tile A of layer L+1 as ring slots free up: no kernel boundaries, no pipeline ramp,
// no tail wave between layers, and activations never leave L2.
//   extra barrier: act_ready[X] (128 local epilogue arrivals) = "tile X's output of the previous layer is in global
//   memory"; the epilogue makes its generic-proxy stores visible to the TMA (async proxy) with
//   __threadfence + fence.proxy.async before arriving.
//
// The im2col operand is REUSED across the nine filter taps: the TMA unit loads, once per 64-channel slice, the
// zero-padded IMAGE of the CTA's two boards
//     rows [y = -1..8][board 0..1][x = -1..8] x 64 channels  (200 rows of 128 bytes, 128-byte swizzle)
// through a tensor map whose dimensions are ordered (C, W, B, H), so that out-of-board rows / columns are zero-filled
// by the TMA unit.  The A operand of tap (dy, dx) is then the SAME image addressed through a shifted shared-memory
// descriptor: start row (1+dy)*20 + (1+dx), 8-row groups 1,280 bytes apart (one image row of ten pixels), group
// g = 2*y + board.  Rows of a tile are therefore ordered (y, board, x) instead of (board, y, x); the epilogue
// un-permutes when it computes its global row.  Per (tile, layer) a CTA reads 4 x 25.6 KB of activations where one
// box per (tap, slice) would read 36 x 16 KB; the weight stream (36 x 16 KB) has its own, deeper ring.
//
// Activation scratch is indexed by CTA-PAIR SLOT, not by board: a pair carries its group of 8 boards through all 21
// layers before it takes the next group, so the two ping-pong buffers only need 8 boards per pair
// (74 pairs x 8 boards x 32 KB x 2 = 39 MB).  That footprint stays resident in the 126 MB L2 and every line is
// overwritten by the next layer before it is evicted, so the activations stop being written back to HBM
// (board-indexed buffers: 2 x 134 MB per 4,096-position batch, 4.85 x the algorithmic DRAM traffic).
// ======================================================================================================
static constexpr int T4_NA = 3;                           // padded-image slots
static constexpr int T4_NB = 7;                           // weight stages
static constexpr int T4_IMG_ROWS = 200;                   // 10 x 2 x 10
static constexpr int T4_IMG_BYTES = T4_IMG_ROWS * 128;    // 25,600
static constexpr int T4_A_SLOT = 26 * 1024;               // slot pitch (1,024-byte aligned)
static constexpr int T4_B_BYTES = 128 * BLOCK_K * 2;      // 16 KB: this CTA's half of the 256 filters
static constexpr int T4_SMEM_BYTES = 1024 + T4_NA * T4_A_SLOT + T4_NB * T4_B_BYTES + 2 * TILE_N * 4 + 3 * 256 * 4 + 64 + 512;

// K-major SWIZZLE_128B descriptor with an explicit stride between 8-row groups
__device__ __forceinline__ uint64_t make_kmajor_sw128_desc_sbo(uint32_t smem_addr, uint32_t sbo_bytes) {
  return (uint64_t)((smem_addr >> 4) & 0x3FFF) | ((uint64_t)(sbo_bytes >> 4) << 32) | (1ull << 46) | (2ull << 61);
}

// FP8 (a separate instantiation): the same pipeline on e4m3 operands.  A 128-byte swizzle row then holds
// 128 channels, so a slice is 128 channels and the boxes keep their byte sizes; each MMA is kind::f8f6f4 with K = 32.
// The epilogue applies the per-layer scales of LayerDesc8 and stores e4m3 codes; the last convolution (fused heads only)
// rounds to bf16 exactly as the bf16 tower does.
template <bool SINGLE, bool FP8>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(CONV_THREADS, 1)
k_trunk4(const __grid_constant__ CUtensorMap map_planes, const CUtensorMap* __restrict__ maps,
         const typename std::conditional<FP8, LayerDesc8, LayerDesc>::type* __restrict__ layers, TrunkParams p) {
  using LD = typename std::conditional<FP8, LayerDesc8, LayerDesc>::type;
  using ActT = typename std::conditional<FP8, uint8_t, __nv_bfloat16>::type;
  constexpr int KSLICE = FP8 ? 128 : BLOCK_K;         // channels per 128-byte swizzle row
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + T4_NA * T4_A_SLOT;
  float* s_scale = (float*)(smem_b + T4_NB * T4_B_BYTES);
  float* s_shift = s_scale + TILE_N;
  float* s_hw = s_shift + TILE_N;
  float* s_hs = s_hw + 3 * 256;
  uint64_t* bars = (uint64_t*)(s_hs + 16);
  uint64_t* a_full = bars;
  uint64_t* a_empty = a_full + T4_NA;
  uint64_t* b_full = a_empty + T4_NA;
  uint64_t* b_empty = b_full + T4_NB;
  uint64_t* tmem_full = b_empty + T4_NB;
  uint64_t* tmem_empty = tmem_full + 2;
  uint64_t* act_ready = tmem_empty + 2;
  uint32_t* tmem_slot = (uint32_t*)(act_ready + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  int n_boards = p.n_host;
  if (p.n_dev) n_boards = min(n_boards, *p.n_dev);
  const int n_tiles = (n_boards + 3) >> 2;          // 256-row tiles (4 boards)
  // SINGLE (a separate instantiation, chosen by the host when the batch bound gives every tile a CTA pair of its own:
  // <= 4 boards per pair -- one game, small lane counts): ONE tile per group.  A second tile would only be padding, and a
  // pair working through two tiles takes twice as long as two pairs with one each.  (The epilogue then has no other tile's
  // MMAs to hide behind; the weight stages of the next layer still stream in meanwhile.)  Same arithmetic per tile, same
  // results.  The two-tile instantiation is untouched (a run-time switch measured 0.5 % slower at 4,096 positions).
  constexpr bool single = SINGLE;
  constexpr int XN = SINGLE ? 1 : 2;
  const int n_groups = single ? n_tiles : (n_tiles + 1) >> 1;
  const int NL = p.n_layers;

  if (threadIdx.x == 0) prefetch_tmap(&map_planes);
  if (threadIdx.x == 32) {
    for (int i = 0; i < T4_NA; ++i) {
      mbar_init(&a_full[i], 2);
      mbar_init(&a_empty[i], 1);
    }
    for (int i = 0; i < T4_NB; ++i) {
      mbar_init(&b_full[i], 2);
      mbar_init(&b_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], 256);
      mbar_init(&act_ready[i], 128);
    }
    fence_barrier_init();
  }
  cluster_sync_all();
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  for (int i = threadIdx.x; i < 3 * 256; i += CONV_THREADS) s_hw[i] = p.head_w[i];
  if (threadIdx.x < 6) s_hs[threadIdx.x] = p.head_s[threadIdx.x];
  tcgen05_fence_before();
  cluster_sync_all();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (threadIdx.x == 0) {
    // ================= TMA producer =================
    int as = 0, bs = 0;
    uint32_t aphase = 0, bphase = 0;
    int uses = 0;
    for (int grp = pair; grp < n_groups; grp += n_pairs) {
      for (int L = 0; L < NL; ++L, ++uses) {
        const LD ld = layers[L];
        const CUtensorMap* map_a = ld.map_in == 0 ? &map_planes : maps + ld.map_in;
        const CUtensorMap* map_w = maps + ld.map_w;
        for (int X = 0; X < XN; ++X) {
          const int tile = single ? grp : 2 * grp + X;
          if (L > 0) mbar_wait(&act_ready[X], (uint32_t)((uses - 1) & 1));
          for (int kc = 0; kc < ld.k_chunks; ++kc) {
            mbar_wait(&a_empty[as], aphase ^ 1);
            if (rank == 0) mbar_arrive_expect_tx(&a_full[as], 2 * T4_IMG_BYTES);
            // coordinates (channel, x, board, y): the box {64, 10, 2, 10} starts one pixel outside the board.
            // The planes are indexed by board, the activation scratch by this pair's slot.
            const int b0 = (ld.map_in == 0 ? tile * 4 : pair * 8 + X * 4) + (int)rank * 2;
            tma2_load_4d_hint(smem_a + as * T4_A_SLOT, map_a, &a_full[as], kc * KSLICE, -1, b0, -1,
                              ld.map_in == 0 ? p.hint_planes : L2_EVICT_NORMAL);
            if (rank != 0) mbar_arrive_remote(&a_full[as], 0);
            if (++as == T4_NA) {
              as = 0;
              aphase ^= 1;
            }
            for (int tap = 0; tap < 9; ++tap) {
              mbar_wait(&b_empty[bs], bphase ^ 1);
              if (rank == 0) mbar_arrive_expect_tx(&b_full[bs], 2 * T4_B_BYTES);
              tma2_load_2d_hint(smem_b + bs * T4_B_BYTES, map_w, &b_full[bs], (tap * ld.k_chunks + kc) * KSLICE,
                                (int)rank * 128, p.hint_weights);
              if (rank != 0) mbar_arrive_remote(&b_full[bs], 0);
              if (++bs == T4_NB) {
                bs = 0;
                bphase ^= 1;
              }
            }
          }
        }
      }
    }
  } else if (threadIdx.x == 32 && rank == 0) {
    // ================= MMA issuer (leader CTA) =================
    int as = 0, bs = 0;
    uint32_t aphase = 0, bphase = 0;
    int uses = 0;
    for (int grp = pair; grp < n_groups; grp += n_pairs) {
      for (int L = 0; L < NL; ++L, ++uses) {
        const int k_chunks = layers[L].k_chunks;
        for (int X = 0; X < XN; ++X) {
          mbar_wait(&tmem_empty[X], (uint32_t)((uses & 1) ^ 1));
          tcgen05_fence_after();
          const uint32_t tmem_d = tmem_base + X * TILE_N;
          for (int kc = 0; kc < k_chunks; ++kc) {
            mbar_wait(&a_full[as], aphase);
            const uint32_t img = smem_u32(smem_a + as * T4_A_SLOT);
            for (int tap = 0; tap < 9; ++tap) {
              mbar_wait(&b_full[bs], bphase);
              tcgen05_fence_after();
              const int dy = tap / 3, dx = tap - 3 * dy;                 // already offset by +1
              const uint64_t da = make_kmajor_sw128_desc_sbo(img + (uint32_t)(dy * 20 + dx) * 128u, 1280u);
              const uint64_t db = make_kmajor_sw128_desc(smem_u32(smem_b + bs * T4_B_BYTES));
              if constexpr (FP8) {
#pragma unroll
                for (int k = 0; k < 4; ++k) umma2_fp8(tmem_d, da + 2 * k, db + 2 * k, V2_IDESC_FP8, (kc | tap | k) != 0);
              } else {
#pragma unroll
                for (int k = 0; k < BLOCK_K / 16; ++k) umma2_bf16(tmem_d, da + 2 * k, db + 2 * k, V2_IDESC, (kc | tap | k) != 0);
              }
              umma2_commit_both(&b_empty[bs]);
              if (++bs == T4_NB) {
                bs = 0;
                bphase ^= 1;
              }
            }
            umma2_commit_both(&a_empty[as]);
            if (kc == k_chunks - 1) umma2_commit_both(&tmem_full[X]);
            if (++as == T4_NA) {
              as = 0;
              aphase ^= 1;
            }
          }
        }
      }
    }
    if (uses > 0) {
      mbar_wait(&tmem_empty[0], (uint32_t)((uses - 1) & 1));
      if (!single) mbar_wait(&tmem_empty[1], (uint32_t)((uses - 1) & 1));
    }
  } else if (warp >= 4) {
    // ================= epilogue (both CTAs) =================
    const int q = warp & 3;
    const int m = q * 32 + lane;                       // accumulator row = (y, board, x): g = m / 8 = 2*y + board
    const int eb = (m >> 3) & 1, ey = m >> 4, ex = m & 7;
    int uses = 0;
    for (int grp = pair; grp < n_groups; grp += n_pairs) {
      for (int L = 0; L < NL; ++L, ++uses) {
        const LD ld = layers[L];
        asm volatile("bar.sync 1, 128;" ::: "memory");
        for (int i = threadIdx.x - 128; i < TILE_N; i += 128) {
          s_scale[i] = ld.scale[i];
          s_shift[i] = ld.shift[i];
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");
        for (int X = 0; X < XN; ++X) {
          const int tile = single ? grp : 2 * grp + X;
          mbar_wait(&tmem_full[X], (uint32_t)(uses & 1));
          tcgen05_fence_after();
          const int board = tile * 4 + (int)rank * 2 + eb;
          const long long grow = (long long)board * 64 + ey * 8 + ex;                    // row by board (heads, tap)
          const long long srow = (long long)(pair * 8 + X * 4 + (int)rank * 2 + eb) * 64 + ey * 8 + ex;   // row by slot
          const bool valid = board < n_boards;
          ActT* orow = ld.write_out ? ld.out + srow * TILE_N : nullptr;
          const ActT* rrow = ld.residual ? ld.residual + srow * TILE_N : nullptr;
          __nv_bfloat16* drow = (p.dbg_out && L == p.dbg_layer) ? p.dbg_out + grow * TILE_N : nullptr;
          float h0 = 0.f, h1 = 0.f, h2 = 0.f;
          if constexpr (FP8) {
#pragma unroll 1
            for (int c0 = 0; c0 < TILE_N; c0 += 32) {
              uint32_t v[32];
              tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + X * TILE_N + c0, v);
              tmem_ld_wait();
              if (!valid) continue;
              uint4 res[2];
              if (rrow) {
                res[0] = *reinterpret_cast<const uint4*>(rrow + c0);
                res[1] = *reinterpret_cast<const uint4*>(rrow + c0 + 16);
              }
              float a[32];
#pragma unroll
              for (int j = 0; j < 32; ++j) a[j] = __uint_as_float(v[j]) * s_scale[c0 + j] + s_shift[c0 + j];
              if (rrow) {
                const __nv_fp8x2_storage_t* r2 = reinterpret_cast<const __nv_fp8x2_storage_t*>(res);
#pragma unroll
                for (int h = 0; h < 16; ++h) {
                  const float2 f = __half22float2(__half2(__nv_cvt_fp8x2_to_halfraw2(r2[h], __NV_E4M3)));
                  a[2 * h] += f.x * ld.s_res;
                  a[2 * h + 1] += f.y * ld.s_res;
                }
              }
              if (ld.relu) {
#pragma unroll
                for (int j = 0; j < 32; ++j) a[j] = fmaxf(a[j], 0.f);
              }
              if (ld.fuse_heads) {
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                  const float x = __bfloat162float(__float2bfloat16_rn(a[j]));
                  h0 = fmaf(x, s_hw[c0 + j], h0);
                  h1 = fmaf(x, s_hw[256 + c0 + j], h1);
                  h2 = fmaf(x, s_hw[512 + c0 + j], h2);
                }
                if (drow) {
#pragma unroll
                  for (int j = 0; j < 16; ++j)
                    reinterpret_cast<__nv_bfloat162*>(drow + c0)[j] = __floats2bfloat162_rn(a[2 * j], a[2 * j + 1]);
                }
              } else if (orow || drow) {
                alignas(16) __nv_fp8x2_storage_t pk[16];   // read back as two uint4
#pragma unroll
                for (int h = 0; h < 16; ++h)
                  pk[h] = __nv_cvt_float2_to_fp8x2(make_float2(a[2 * h] * ld.inv_out, a[2 * h + 1] * ld.inv_out),
                                                   __NV_SATFINITE, __NV_E4M3);
                if (orow) {
                  const uint4* src = reinterpret_cast<const uint4*>(pk);
                  *reinterpret_cast<uint4*>(orow + c0) = src[0];
                  *reinterpret_cast<uint4*>(orow + c0 + 16) = src[1];
                }
                if (drow) {   // the stored value code x s_out is exact in bf16
#pragma unroll
                  for (int h = 0; h < 16; ++h) {
                    const float2 f = __half22float2(__half2(__nv_cvt_fp8x2_to_halfraw2(pk[h], __NV_E4M3)));
                    reinterpret_cast<__nv_bfloat162*>(drow + c0)[h] = __floats2bfloat162_rn(f.x * ld.s_out, f.y * ld.s_out);
                  }
                }
              }
            }
          } else {
#pragma unroll 1
          for (int c0 = 0; c0 < TILE_N; c0 += 32) {
            uint32_t v[32];
            tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + X * TILE_N + c0, v);
            tmem_ld_wait();
            if (!valid) continue;
            uint4 res[4];
            if (rrow) {
#pragma unroll
              for (int j = 0; j < 4; ++j) res[j] = *reinterpret_cast<const uint4*>(rrow + c0 + 8 * j);
            }
            float a[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) a[j] = __uint_as_float(v[j]) * s_scale[c0 + j] + s_shift[c0 + j];
            if (rrow) {
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const uint32_t* rj = reinterpret_cast<const uint32_t*>(&res[j]);
#pragma unroll
                for (int h = 0; h < 4; ++h) {
                  a[8 * j + 2 * h] += __uint_as_float(rj[h] << 16);
                  a[8 * j + 2 * h + 1] += __uint_as_float(rj[h] & 0xFFFF0000u);
                }
              }
            }
            if (ld.relu) {
#pragma unroll
              for (int j = 0; j < 32; ++j) a[j] = fmaxf(a[j], 0.f);
            }
            if (ld.fuse_heads) {
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                const float x = __bfloat162float(__float2bfloat16_rn(a[j]));
                h0 = fmaf(x, s_hw[c0 + j], h0);
                h1 = fmaf(x, s_hw[256 + c0 + j], h1);
                h2 = fmaf(x, s_hw[512 + c0 + j], h2);
              }
            }
            if (orow || drow) {
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                uint32_t pk[4];
#pragma unroll
                for (int h = 0; h < 4; ++h) {
                  __nv_bfloat162 b2 = __floats2bfloat162_rn(a[8 * j + 2 * h], a[8 * j + 2 * h + 1]);
                  pk[h] = *reinterpret_cast<uint32_t*>(&b2);
                }
                if (orow) *reinterpret_cast<uint4*>(orow + c0 + 8 * j) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                if (drow) *reinterpret_cast<uint4*>(drow + c0 + 8 * j) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
              }
            }
          }
          }
          tcgen05_fence_before();
          mbar_arrive_remote(&tmem_empty[X], 0);
          if (ld.fuse_heads && valid) {
            const float f0 = fmaxf(h0 * s_hs[0] + s_hs[3], 0.f), f1 = fmaxf(h1 * s_hs[1] + s_hs[4], 0.f);
            reinterpret_cast<__nv_bfloat162*>(p.pf_out)[grow] = __floats2bfloat162_rn(f0, f1);
            p.vf_out[grow] = fmaxf(h2 * s_hs[2] + s_hs[5], 0.f);
          }
          __threadfence();
          asm volatile("fence.proxy.async.global;" ::: "memory");
          mbar_arrive(&act_ready[X]);
        }
      }
    }
  }

  tcgen05_fence_before();
  cluster_sync_all();
  if (warp == 2) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// softmax over the policy logits + the value head's two dense layers; 8 positions per block, one warp each
struct TailParams {
  const int* n_rows_dev;
  int n_rows_host;
  const float* logits;   // [rows][ld]
  int ld;
  const float* vf;       // [rows][64]
  const float* wv1;      // [64][256]
  const float* bv1;      // [256]
  const float* wv2;      // [256]
  const float* bv2;      // [1]
  float* policy;         // [rows][1968]
  float* value;          // [rows]
  float* stats;          // null, or [rows][2]: write (max logit, 1 / sum exp) INSTEAD of the probability row
};
__global__ void __launch_bounds__(256) k_softmax_value(TailParams p) {
  __shared__ float s_vf[8][64];
  __shared__ float s_hid[8][256];
  int n_rows = p.n_rows_host;
  if (p.n_rows_dev) n_rows = min(n_rows, *p.n_rows_dev);
  const int pos0 = blockIdx.x * 8;
  if (pos0 >= n_rows) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < 8 * 64; i += 256) {
    const int q = i >> 6;
    s_vf[q][i & 63] = (pos0 + q < n_rows) ? p.vf[(long long)(pos0 + q) * 64 + (i & 63)] : 0.f;
  }
  __syncthreads();
  {
    const int j = threadIdx.x;
    float acc[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) acc[q] = 0.f;
    for (int i = 0; i < 64; ++i) {
      const float w = p.wv1[i * 256 + j];
#pragma unroll
      for (int q = 0; q < 8; ++q) acc[q] = fmaf(s_vf[q][i], w, acc[q]);
    }
    const float b = p.bv1[j];
#pragma unroll
    for (int q = 0; q < 8; ++q) s_hid[q][j] = fmaxf(acc[q] + b, 0.f);
  }
  __syncthreads();
  const int pos = pos0 + warp;
  if (pos >= n_rows) return;
  const float* lg = p.logits + (long long)pos * p.ld;
  float x[62];
  float m = -INFINITY;
#pragma unroll
  for (int k = 0; k < 62; ++k) {
    const int j = lane + 32 * k;
    x[k] = j < CRL_N_LABELS ? lg[j] : -INFINITY;
    m = fmaxf(m, x[k]);
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < 62; ++k) {
    x[k] = expf(x[k] - m);
    s += x[k];
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
  const float inv = 1.0f / s;
  if (p.stats) {
    // the search reads ~35 of the 1,968 probabilities of a row: hand it (max, 1 / sum) and let it evaluate
    // expf(logit - max) * inv -- this kernel's own expression -- for the entries it needs (PolicyView, tree_core.cuh)
    if (lane == 0) {
      p.stats[2 * pos] = m;
      p.stats[2 * pos + 1] = inv;
    }
  } else {
    float* out = p.policy + (long long)pos * CRL_N_LABELS;
#pragma unroll
    for (int k = 0; k < 62; ++k) {
      const int j = lane + 32 * k;
      if (j < CRL_N_LABELS) out[j] = x[k] * inv;
    }
  }
  float v = 0.f;
  for (int j = lane; j < 256; j += 32) v = fmaf(s_hid[warp][j], p.wv2[j], v);
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  if (lane == 0) p.value[pos] = tanhf(v + p.bv2[0]);
}

// fp8 tower input: bf16 planes -> e4m3 (round to nearest even, saturating; the encoder's 0 / 1 planes are exact), 8 per thread
__global__ void __launch_bounds__(256) k_planes_to_e4m3(const uint4* __restrict__ in, uint2* __restrict__ out, long long n8) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n8) return;
  const uint4 v = in[i];
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
  uint32_t pk[2];
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const float2 f0 = make_float2(__uint_as_float(w[2 * h] << 16), __uint_as_float(w[2 * h] & 0xFFFF0000u));
    const float2 f1 = make_float2(__uint_as_float(w[2 * h + 1] << 16), __uint_as_float(w[2 * h + 1] & 0xFFFF0000u));
    pk[h] = (uint32_t)__nv_cvt_float2_to_fp8x2(f0, __NV_SATFINITE, __NV_E4M3) |
            ((uint32_t)__nv_cvt_float2_to_fp8x2(f1, __NV_SATFINITE, __NV_E4M3) << 16);
  }
  out[i] = make_uint2(pk[0], pk[1]);
}

// calibration: *amax = max(*amax, max |x|) over n8 x 8 bf16 values (non-negative floats order as their bit patterns)
__global__ void __launch_bounds__(256) k_absmax_bf16(const uint4* __restrict__ x, long long n8, unsigned* amax) {
  float m = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    const uint4 v = x[i];
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int h = 0; h < 4; ++h) {
      m = fmaxf(m, fabsf(__uint_as_float(w[h] << 16)));
      m = fmaxf(m, fabsf(__uint_as_float(w[h] & 0xFFFF0000u)));
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
  if ((threadIdx.x & 31) == 0) atomicMax(amax, __float_as_uint(m));
}

// ======================================================================================================
// host side: weight pack, tensor maps, forward
// ======================================================================================================
static constexpr int N_CONVS = 21;
static constexpr float BN_EPS = 1e-3f;   // Keras BatchNormalization default

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct NetWeights {
  int slot = 0;                             // network slot (crl_net_select_slot)
  int cap_rows = 0;                         // activation capacity in boards (even)
  void* planes_buf = nullptr;               // where the search encodes this slot's rows (R + 2 bf16 rows; slot 0: e->d_planes)
  float* stats = nullptr;                   // softmax statistics of this slot's search rows (e->d_stats + 2 x slot rows)
  bool loaded = false;
  __nv_bfloat16* w[N_CONVS] = {nullptr};    // [256][9*Cin] K-major
  float* scale[N_CONVS] = {nullptr};
  float* shift[N_CONVS] = {nullptr};
  int cin[N_CONVS] = {0};
  const void* planes_ptr = nullptr;
  int planes_rows = 0;
  float *w1x1 = nullptr, *s1x1 = nullptr, *wv1 = nullptr, *bv1 = nullptr, *wv2 = nullptr, *bv2 = nullptr;
  PFN_encodeTiled encode = nullptr;
  int n_sms = 148;
  CUtensorMap map_w2[N_CONVS];              // weight boxes of 128 filters (one CTA's half)
  __nv_bfloat16* pf = nullptr;              // [cap][128] policy features (bf16)
  float* vf = nullptr;                      // [cap][64] value features
  float* logits = nullptr;                  // [cap + 256][2048] policy logits (slot k: rows k x slot_stride of one buffer)
  __nv_bfloat16* wp_bf16 = nullptr;         // [2048][128] policy dense kernel, K-major, zero padded
  float* bp_pad = nullptr;                  // [2048]
  float* ones = nullptr;                    // [2048]
  CUtensorMap map_pf, map_wp;
  // the tower (k_trunk4)
  __nv_bfloat16* act4[2] = {nullptr, nullptr};  // [n_sms/2 pairs x 8 boards][64][256]: ping-pong scratch by CTA-pair slot
  int act4_rows = 0;
  CUtensorMap map_act4[2];
  CUtensorMap map_planes4;
  CUtensorMap* d_maps4 = nullptr;           // [3 + N_CONVS] device copies: (unused: the planes map is a kernel
                                            // parameter), act4[0], act4[1], weights (128-filter boxes)
  LayerDesc* d_layers4 = nullptr;           // [N_CONVS], out / residual pointing into act4
  // fp8 tower (crl_net_load_fp8_host); buffers are allocated by the first fp8 load
  bool fp8_loaded = false;
  bool fp8 = false;                         // the fp8 tower is selected
  bool planes_fp8 = false;                  // dtype of the cached planes maps
  uint8_t* w8[N_CONVS] = {nullptr};         // [256][9*Cin] e4m3, K-major
  float* scale8[N_CONVS] = {nullptr};       // weight scale x input scale x BatchNorm scale
  float* shift8[N_CONVS] = {nullptr};
  uint8_t* act8[2] = {nullptr, nullptr};    // [act4_rows][64][256] e4m3 scratch by CTA-pair slot
  CUtensorMap* d_maps8 = nullptr;
  LayerDesc8* d_layers8 = nullptr;
};

static int make_act_map(NetWeights* nw, CUtensorMap* map, const void* base, int cin, int rows) {
  cuuint64_t dims[4] = {(cuuint64_t)cin, 8, 8, (cuuint64_t)rows};
  cuuint64_t strides[3] = {(cuuint64_t)cin * 2, (cuuint64_t)cin * 16, (cuuint64_t)cin * 128};
  cuuint32_t box[4] = {BLOCK_K, 8, 8, 2};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = nw->encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(activations) failed: %d", (int)r);
    return CRL_ECUDA;
  }
  return CRL_OK;
}
// v4: the same activations seen as (C, W, B, H), box {64, 10, 2, 10} = the zero-padded image of two boards laid out
// [y][board][x] in shared memory (see k_trunk4)
// fp8: e4m3 elements, box {128, 10, 2, 10} (the same 128 bytes per row)
static int make_act_map4(NetWeights* nw, CUtensorMap* map, const void* base, int cin, int rows, bool fp8 = false) {
  const cuuint64_t es = fp8 ? 1 : 2;
  cuuint64_t dims[4] = {(cuuint64_t)cin, 8, (cuuint64_t)rows, 8};
  cuuint64_t strides[3] = {(cuuint64_t)cin * es, (cuuint64_t)cin * 64 * es, (cuuint64_t)cin * 8 * es};
  cuuint32_t box[4] = {fp8 ? 128u : (cuuint32_t)BLOCK_K, 10, 2, 10};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = nw->encode(map, fp8 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4,
                          const_cast<void*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(activations, padded image) failed: %d", (int)r);
    return CRL_ECUDA;
  }
  return CRL_OK;
}
static int make_w_map(NetWeights* nw, CUtensorMap* map, const void* base, int k_total, int n_rows = TILE_N,
                      int box_n = TILE_N, bool fp8 = false) {
  cuuint64_t dims[2] = {(cuuint64_t)k_total, (cuuint64_t)n_rows};
  cuuint64_t strides[1] = {(cuuint64_t)k_total * (fp8 ? 1 : 2)};
  cuuint32_t box[2] = {fp8 ? 128u : (cuuint32_t)BLOCK_K, (cuuint32_t)box_n};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = nw->encode(map, fp8 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
                          const_cast<void*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(weights) failed: %d", (int)r);
    return CRL_ECUDA;
  }
  return CRL_OK;
}

template <class T>
static int dev_alloc(crl_engine_impl* e, T** p, size_t count) {
  void* q = nullptr;
  cudaError_t err = cudaMalloc(&q, count * sizeof(T));
  if (err != cudaSuccess) {
    set_error("cudaMalloc(%zu bytes) failed: %s", count * sizeof(T), cudaGetErrorString(err));
    return CRL_ENOMEM;
  }
  e->allocs.push_back(q);
  *p = (T*)q;
  return CRL_OK;
}

int net_create(crl_engine_impl* e, int slot) {
  NetWeights* nw = new NetWeights();
  e->nets[slot] = nw;
  if (e->sel_slot == slot) e->net = nw;
  nw->slot = slot;
  nw->cap_rows = (e->R + 2) & ~1;
  nw->stats = e->d_stats + 2 * (long long)slot * e->slot_stride;
  if (slot == 0) {
    nw->planes_buf = e->d_planes;
  } else {
    __nv_bfloat16* pb = nullptr;
    int rc0 = dev_alloc(e, &pb, (size_t)(e->R + 2) * 64 * 128);
    if (rc0) return rc0;
    nw->planes_buf = pb;
  }
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t err = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (err != cudaSuccess || fn == nullptr) {
    set_error("cuTensorMapEncodeTiled is not available from the driver: %s", cudaGetErrorString(err));
    return CRL_ECUDA;
  }
  nw->encode = (PFN_encodeTiled)fn;
  int dev = e->device;
  cudaDeviceGetAttribute(&nw->n_sms, cudaDevAttrMultiProcessorCount, dev);
  int rc;
  for (int i = 0; i < N_CONVS; ++i) {
    nw->cin[i] = i == 0 ? 128 : 256;
    if ((rc = dev_alloc(e, &nw->w[i], (size_t)TILE_N * 9 * nw->cin[i]))) return rc;
    if ((rc = dev_alloc(e, &nw->scale[i], 256))) return rc;
    if ((rc = dev_alloc(e, &nw->shift[i], 256))) return rc;
    if ((rc = make_w_map(nw, &nw->map_w2[i], nw->w[i], 9 * nw->cin[i], TILE_N, 128))) return rc;
  }
  {
    if ((rc = dev_alloc(e, &nw->pf, (size_t)(nw->cap_rows + 256) * 128))) return rc;
    if ((rc = dev_alloc(e, &nw->vf, (size_t)(nw->cap_rows + 256) * 64))) return rc;
    if (slot == 0) {
      if ((rc = dev_alloc(e, &nw->logits, (size_t)(nw->cap_rows + 256) * 2048))) return rc;
    } else {                              // its rows of the two-slot logits buffer (net_two_slot_layout)
      nw->logits = e->nets[0]->logits + (size_t)slot * e->slot_stride * 2048;
    }
    if ((rc = dev_alloc(e, &nw->wp_bf16, (size_t)2048 * 128))) return rc;
    if ((rc = dev_alloc(e, &nw->bp_pad, 2048))) return rc;
    if ((rc = dev_alloc(e, &nw->ones, 2048))) return rc;
    CRL_CUDA(cudaMemsetAsync(nw->pf, 0, (size_t)(nw->cap_rows + 256) * 128 * 2, e->stream));
    if ((rc = make_w_map(nw, &nw->map_pf, nw->pf, 128, nw->cap_rows + 256, 128))) return rc;
    if ((rc = make_w_map(nw, &nw->map_wp, nw->wp_bf16, 128, 2048, 128))) return rc;
  }
  nw->act4_rows = (nw->n_sms / 2) * 8;
  for (int i = 0; i < 2; ++i) {
    if ((rc = dev_alloc(e, &nw->act4[i], (size_t)nw->act4_rows * 64 * 256))) return rc;
    CRL_CUDA(cudaMemsetAsync(nw->act4[i], 0, (size_t)nw->act4_rows * 64 * 256 * 2, e->stream));
    if ((rc = make_act_map4(nw, &nw->map_act4[i], nw->act4[i], 256, nw->act4_rows))) return rc;
  }
  if ((rc = dev_alloc(e, &nw->w1x1, 3 * 256))) return rc;
  if ((rc = dev_alloc(e, &nw->s1x1, 6))) return rc;
  if ((rc = dev_alloc(e, &nw->wv1, 64 * 256))) return rc;
  if ((rc = dev_alloc(e, &nw->bv1, 256))) return rc;
  if ((rc = dev_alloc(e, &nw->wv2, 256))) return rc;
  if ((rc = dev_alloc(e, &nw->bv2, 1))) return rc;
  CRL_CUDA(cudaFuncSetAttribute(k_conv_v2, cudaFuncAttributeMaxDynamicSharedMemorySize, V2_SMEM_BYTES));
  CRL_CUDA(cudaFuncSetAttribute(k_trunk4<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, T4_SMEM_BYTES));
  CRL_CUDA(cudaFuncSetAttribute(k_trunk4<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, T4_SMEM_BYTES));
  CRL_CUDA(cudaFuncSetAttribute(k_trunk4<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, T4_SMEM_BYTES));
  CRL_CUDA(cudaFuncSetAttribute(k_trunk4<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, T4_SMEM_BYTES));
  {
    // tensor-map table + layer table of the tower kernel
    if ((rc = dev_alloc(e, &nw->d_maps4, 3 + N_CONVS))) return rc;
    if ((rc = dev_alloc(e, &nw->d_layers4, N_CONVS))) return rc;
    std::vector<CUtensorMap> hm(3 + N_CONVS);
    memset(hm.data(), 0, hm.size() * sizeof(CUtensorMap));
    hm[1] = nw->map_act4[0];
    hm[2] = nw->map_act4[1];
    for (int i = 0; i < N_CONVS; ++i) hm[3 + i] = nw->map_w2[i];
    CRL_CUDA(cudaMemcpyAsync(nw->d_maps4, hm.data(), hm.size() * sizeof(CUtensorMap), cudaMemcpyHostToDevice, e->stream));
    std::vector<LayerDesc> hl(N_CONVS);
    __nv_bfloat16* const* act = nw->act4;
    for (int L = 0; L < N_CONVS; ++L) {
      LayerDesc& d = hl[L];
      memset(&d, 0, sizeof(d));
      d.map_w = 3 + L;
      d.k_chunks = nw->cin[L] / BLOCK_K;
      d.scale = nw->scale[L];
      d.shift = nw->shift[L];
      if (L == 0) {                      // stem: planes -> act[0], no BN / activation
        d.map_in = 0;
        d.out = act[0];
        d.write_out = 1;
      } else if ((L - 1) % 2 == 0) {     // conv_a: act[0] -> act[1], BN + ReLU
        d.map_in = 1;
        d.out = act[1];
        d.relu = 1;
        d.write_out = 1;
      } else {                           // conv_b: act[1] -> act[0] in place (+ residual act[0]), BN, ReLU
        d.map_in = 2;
        d.out = act[0];
        d.residual = act[0];
        d.relu = 1;
        d.write_out = L != N_CONVS - 1;  // the last layer only feeds the fused heads
        d.fuse_heads = L == N_CONVS - 1;
      }
    }
    CRL_CUDA(cudaMemcpyAsync(nw->d_layers4, hl.data(), hl.size() * sizeof(LayerDesc), cudaMemcpyHostToDevice, e->stream));
    CRL_CUDA(cudaStreamSynchronize(e->stream));   // hm and hl are locals
  }
  return CRL_OK;
}

void net_destroy(crl_engine_impl* e) {
  for (int k = 0; k < CRL_NET_SLOTS; ++k) {
    delete e->nets[k];
    e->nets[k] = nullptr;
  }
  e->net = nullptr;
}

// replaces the device buffer *p (old_count elements, in e->allocs) by one of new_count elements; contents are not kept
template <class T>
static int regrow(crl_engine_impl* e, T** p, size_t new_count) {
  T* q = nullptr;
  int rc = dev_alloc(e, &q, new_count);
  if (rc) return rc;
  for (size_t i = 0; i < e->allocs.size(); ++i)
    if (e->allocs[i] == (void*)*p) {
      cudaFree(*p);
      e->allocs.erase(e->allocs.begin() + i);
      break;
    }
  *p = q;
  return CRL_OK;
}

// The first configuration of slot 1: the row lists, policy, value, statistics and logits buffers grow to two slots of
// slot_stride rows each, so that one PolicyView and one value array serve both slots' rows (DESIGN.md 3.5).  Nothing
// in flight reads them between API calls (every crl_mcts_simulate call finishes its simulations); the captured
// simulation graphs name the old buffers and are dropped.
int net_two_slot_layout(crl_engine_impl* e) {
  if (e->slot_stride) return CRL_OK;
  NetWeights* n0 = e->nets[0];
  const long long S = (long long)n0->cap_rows + 256;     // the rows of one slot's logits
  CRL_CUDA(cudaStreamSynchronize(e->stream));
  int rc;
  for (int i = 0; i < 2; ++i)
    if ((rc = regrow(e, &e->d_list[i], (size_t)(2 * S)))) return rc;
  if ((rc = regrow(e, &e->d_policy, (size_t)(2 * S) * CRL_N_LABELS))) return rc;
  if ((rc = regrow(e, &e->d_value, (size_t)(2 * S)))) return rc;
  if ((rc = regrow(e, &e->d_stats, (size_t)(4 * S)))) return rc;
  if ((rc = regrow(e, &n0->logits, (size_t)(2 * S) * 2048))) return rc;
  CRL_CUDA(cudaMemsetAsync(e->d_list[0], 0, (size_t)(2 * S) * sizeof(int), e->stream));
  CRL_CUDA(cudaMemsetAsync(e->d_list[1], 0, (size_t)(2 * S) * sizeof(int), e->stream));
  e->slot_stride = S;
  e->P.slot_stride = (int)S;
  e->P.eval_list = e->d_list[0];
  n0->stats = e->d_stats;
  if (NetWeights* n1 = e->nets[1]) {
    n1->stats = e->d_stats + 2 * S;
    n1->logits = n0->logits + (size_t)S * 2048;
  }
  e->pview = PolicyView{e->d_policy, CRL_N_LABELS, nullptr};
  for (int i = 0; i < 2; ++i) {
    if (e->sim_graph[i]) cudaGraphExecDestroy(e->sim_graph[i]);
    e->sim_graph[i] = nullptr;
    e->sim_graph_key[i] = 0;
  }
  return CRL_OK;
}

int net_slot_ensure(crl_engine_impl* e, int slot) {
  if (e->nets[slot]) return CRL_OK;
  int rc = net_two_slot_layout(e);
  if (rc) return rc;
  if ((rc = net_create(e, slot))) return rc;
  CRL_CUDA(cudaStreamSynchronize(e->stream));
  return CRL_OK;
}

static inline uint16_t f2bf(float f) {   // round to nearest even
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7FFFFFFFu) > 0x7F800000u) return (uint16_t)((u >> 16) | 0x40);
  u += 0x7FFFu + ((u >> 16) & 1);
  return (uint16_t)(u >> 16);
}

// Weight pack (140 fp32 tensors, Keras layouts), see DESIGN.md:
//   0,1            stem conv kernel [3][3][127][256], bias [256]
//   2+12b .. +11   residual block b: conv_a kernel [3][3][256][256], bias, BN gamma, beta, mean, var,
//                                    conv_b kernel, bias, BN gamma, beta, mean, var
//   122..129       policy head: conv kernel [1][1][256][2], bias[2], BN gamma,beta,mean,var [2],
//                               dense kernel [128][1968], bias [1968]
//   130..139       value head: conv kernel [1][1][256][1], bias[1], BN x4 [1], dense kernel [64][256], bias[256],
//                              dense kernel [256][1], bias[1]
// pack indices of convolution L's kernel, bias and BatchNorm quadruple (-1: the stem has none)
static void conv_tensors(int L, int* ik, int* ib, int* ibn) {
  if (L == 0) {
    *ik = 0;
    *ib = 1;
    *ibn = -1;
  } else {
    const int blk = (L - 1) / 2, second = (L - 1) % 2;
    *ik = 2 + 12 * blk + 6 * second;
    *ib = *ik + 1;
    *ibn = *ik + 2;
  }
}
// bias + BatchNorm folded into a per-filter scale and shift
static void fold_bn(const float* const* w, int ib, int ibn, float* sc, float* sh) {
  for (int o = 0; o < 256; ++o) {
    float s = 1.f, b = w[ib][o];
    if (ibn >= 0) {
      s = w[ibn][o] / sqrtf(w[ibn + 3][o] + BN_EPS);
      b = (b - w[ibn + 2][o]) * s + w[ibn + 1][o];
    }
    sc[o] = s;
    sh[o] = b;
  }
}

int net_load(crl_engine_impl* e, const float* const* w, const int64_t* sizes, int n) {
  NetWeights* nw = e->net;
  if (n != CRL_N_WEIGHT_TENSORS) {
    set_error("crl_net_load_host: expected %d tensors, got %d", CRL_N_WEIGHT_TENSORS, n);
    return CRL_EINVAL;
  }
  auto need = [&](int i, int64_t sz) -> bool {
    if (sizes[i] != sz) {
      set_error("crl_net_load_host: tensor %d has %lld elements, expected %lld", i, (long long)sizes[i], (long long)sz);
      return false;
    }
    return true;
  };
  nw->fp8 = false;            // a bf16 load drops the fp8 tower; crl_net_load_fp8_host builds it again
  nw->fp8_loaded = false;
  std::vector<uint16_t> wt;
  std::vector<float> sc(256), sh(256);
  for (int L = 0; L < N_CONVS; ++L) {
    const int cin_real = L == 0 ? 127 : 256, cin = nw->cin[L];
    int ik, ib, ibn;
    conv_tensors(L, &ik, &ib, &ibn);
    if (!need(ik, (int64_t)9 * cin_real * 256) || !need(ib, 256)) return CRL_EINVAL;
    if (ibn >= 0 && (!need(ibn, 256) || !need(ibn + 1, 256) || !need(ibn + 2, 256) || !need(ibn + 3, 256)))
      return CRL_EINVAL;
    wt.assign((size_t)256 * 9 * cin, 0);
    for (int t = 0; t < 9; ++t)
      for (int c = 0; c < cin_real; ++c)
        for (int o = 0; o < 256; ++o)
          wt[(size_t)o * 9 * cin + t * cin + c] = f2bf(w[ik][((size_t)t * cin_real + c) * 256 + o]);
    fold_bn(w, ib, ibn, sc.data(), sh.data());
    CRL_CUDA(cudaMemcpyAsync(nw->w[L], wt.data(), wt.size() * 2, cudaMemcpyHostToDevice, e->stream));
    CRL_CUDA(cudaMemcpyAsync(nw->scale[L], sc.data(), 1024, cudaMemcpyHostToDevice, e->stream));
    CRL_CUDA(cudaMemcpyAsync(nw->shift[L], sh.data(), 1024, cudaMemcpyHostToDevice, e->stream));
    CRL_CUDA(cudaStreamSynchronize(e->stream));
  }
  // heads
  const int P0 = 122, V0 = 130;
  if (!need(P0, 512) || !need(P0 + 1, 2) || !need(P0 + 6, (int64_t)128 * CRL_N_LABELS) || !need(P0 + 7, CRL_N_LABELS) ||
      !need(V0, 256) || !need(V0 + 1, 1) || !need(V0 + 6, 64 * 256) || !need(V0 + 7, 256) || !need(V0 + 8, 256) ||
      !need(V0 + 9, 1))
    return CRL_EINVAL;
  std::vector<float> w1(3 * 256), s1(6);
  for (int c = 0; c < 256; ++c) {
    w1[c] = w[P0][c * 2 + 0];
    w1[256 + c] = w[P0][c * 2 + 1];
    w1[512 + c] = w[V0][c];
  }
  for (int o = 0; o < 2; ++o) {
    float s = w[P0 + 2][o] / sqrtf(w[P0 + 5][o] + BN_EPS);
    s1[o] = s;
    s1[3 + o] = (w[P0 + 1][o] - w[P0 + 4][o]) * s + w[P0 + 3][o];
  }
  {
    float s = w[V0 + 2][0] / sqrtf(w[V0 + 5][0] + BN_EPS);
    s1[2] = s;
    s1[5] = (w[V0 + 1][0] - w[V0 + 4][0]) * s + w[V0 + 3][0];
  }
  CRL_CUDA(cudaMemcpyAsync(nw->w1x1, w1.data(), w1.size() * 4, cudaMemcpyHostToDevice, e->stream));
  CRL_CUDA(cudaMemcpyAsync(nw->s1x1, s1.data(), s1.size() * 4, cudaMemcpyHostToDevice, e->stream));
  CRL_CUDA(cudaMemcpyAsync(nw->wv1, w[V0 + 6], 64 * 256 * 4, cudaMemcpyHostToDevice, e->stream));
  CRL_CUDA(cudaMemcpyAsync(nw->bv1, w[V0 + 7], 256 * 4, cudaMemcpyHostToDevice, e->stream));
  CRL_CUDA(cudaMemcpyAsync(nw->wv2, w[V0 + 8], 256 * 4, cudaMemcpyHostToDevice, e->stream));
  CRL_CUDA(cudaMemcpyAsync(nw->bv2, w[V0 + 9], 4, cudaMemcpyHostToDevice, e->stream));
  {
    std::vector<uint16_t> wpt((size_t)2048 * 128, 0);
    std::vector<float> bpad(2048, 0.f), one(2048, 1.f);
    for (int j = 0; j < CRL_N_LABELS; ++j) {
      bpad[j] = w[P0 + 7][j];
      for (int i = 0; i < 128; ++i) wpt[(size_t)j * 128 + i] = f2bf(w[P0 + 6][(size_t)i * CRL_N_LABELS + j]);
    }
    CRL_CUDA(cudaMemcpyAsync(nw->wp_bf16, wpt.data(), wpt.size() * 2, cudaMemcpyHostToDevice, e->stream));
    CRL_CUDA(cudaMemcpyAsync(nw->bp_pad, bpad.data(), 2048 * 4, cudaMemcpyHostToDevice, e->stream));
    CRL_CUDA(cudaMemcpyAsync(nw->ones, one.data(), 2048 * 4, cudaMemcpyHostToDevice, e->stream));
    CRL_CUDA(cudaStreamSynchronize(e->stream));
  }
  CRL_CUDA(cudaStreamSynchronize(e->stream));
  nw->loaded = true;
  return CRL_OK;
}

static int launch_conv_v2(crl_engine_impl* e, NetWeights* nw, const CUtensorMap& map_in, int L, const int* n_dev,
                          int n_host, const __nv_bfloat16* residual, __nv_bfloat16* out, int relu) {
  ConvParams2 p;
  memset(&p, 0, sizeof(p));
  p.n_units_dev = n_dev;
  p.n_units_host = n_host;
  p.rows_per_unit = 64;
  p.taps = 9;
  p.k_chunks = nw->cin[L] / BLOCK_K;
  p.n_tiles = 1;
  p.scale = nw->scale[L];
  p.shift = nw->shift[L];
  p.residual = residual;
  p.out = out;
  p.relu = relu;
  int work = (n_host + 3) / 4;
  int pairs = work < nw->n_sms / 2 ? work : nw->n_sms / 2;
  if (pairs < 1) pairs = 1;
  LaunchScope ls(e, KC_CONV);
  k_conv_v2<<<2 * pairs, CONV_THREADS, V2_SMEM_BYTES, e->stream>>>(map_in, nw->map_w2[L], p);
  CRL_CUDA(cudaGetLastError());
  return CRL_OK;
}

// policy dense layer (128 -> 1968, zero padded to 2048) as a tcgen05 GEMM, then softmax + value head
static int launch_heads_v2(crl_engine_impl* e, NetWeights* nw, const int* n_dev, int n_host, float* policy, float* value,
                           PolicyView* view_out) {
  ConvParams2 p;
  memset(&p, 0, sizeof(p));
  p.n_units_dev = n_dev;
  p.n_units_host = n_host;
  p.rows_per_unit = 1;
  p.taps = 1;
  p.k_chunks = 2;
  p.n_tiles = 8;
  p.scale = nw->ones;
  p.shift = nw->bp_pad;
  p.out_f32 = nw->logits;
  p.out_ld = 2048;
  int work = ((n_host + 255) / 256) * 8;
  int pairs = work < nw->n_sms / 2 ? work : nw->n_sms / 2;
  if (pairs < 1) pairs = 1;
  {
    LaunchScope ls(e, KC_HEADS);
    k_conv_v2<<<2 * pairs, CONV_THREADS, V2_SMEM_BYTES, e->stream>>>(nw->map_pf, nw->map_wp, p);
    CRL_CUDA(cudaGetLastError());
  }
  TailParams t;
  t.n_rows_dev = n_dev;
  t.n_rows_host = n_host;
  t.logits = nw->logits;
  t.ld = 2048;
  t.vf = nw->vf;
  t.wv1 = nw->wv1;
  t.bv1 = nw->bv1;
  t.wv2 = nw->wv2;
  t.bv2 = nw->bv2;
  t.policy = policy;
  t.value = value;
  t.stats = nullptr;
  if (view_out) {
    t.stats = nw->stats;
    *view_out = PolicyView{nw->logits, 2048, nw->stats};
  }
  LaunchScope ls(e, KC_HEADS);
  k_softmax_value<<<div_up(n_host, 8), 256, 0, e->stream>>>(t);
  CRL_CUDA(cudaGetLastError());
  return CRL_OK;
}

static int forward_nw(crl_engine_impl* e, NetWeights* nw, const __nv_bfloat16* planes, int n_host, const int* n_dev,
                      float* policy, float* value, __nv_bfloat16* dbg_out, int dbg_layer, PolicyView* view_out) {
  if (view_out) *view_out = PolicyView{policy, CRL_N_LABELS, nullptr};   // unless the heads below switch to statistics
  if (!nw || !nw->loaded) {
    set_error("network weights are not loaded (crl_net_load_host)");
    return CRL_ESTATE;
  }
  if (n_host <= 0) return CRL_OK;
  if (n_host > nw->cap_rows) {
    set_error("crl_net_forward: %d positions exceed the engine capacity %d", n_host, nw->cap_rows);
    return CRL_EINVAL;
  }
  const bool fp8 = nw->fp8;
  __nv_bfloat16* const own = (__nv_bfloat16*)nw->planes_buf;
  if (fp8 && planes != own) {
    // a caller's bf16 planes: converted into the slot's planes buffer, where the search encodes its e4m3 rows
    const long long n8 = (long long)n_host * 64 * 128 / 8;     // groups of 8 values
    LaunchScope ls(e, KC_ENCODE);
    k_planes_to_e4m3<<<(unsigned)div_up(n8, 256), 256, 0, e->stream>>>(reinterpret_cast<const uint4*>(planes),
                                                                         reinterpret_cast<uint2*>(own), n8);
    CRL_CUDA(cudaGetLastError());
    planes = own;
  }
  {
    // the box may start at row n-1 for an odd n: rows beyond the map are zero-filled by the TMA unit.  e4m3 planes in
    // the slot's planes buffer: it holds R + 2 bf16 rows, so every row a caller may convert into it is inside the map; the
    // rows after the batch are then stale buffer contents, not zeros.  That is harmless: an output row of the implicit
    // GEMM depends on its own board's rows only, and the epilogue skips the boards at or after the row count.
    const int rows = fp8 ? e->R + 2 : planes == own ? e->R : n_host;
    if (planes != nw->planes_ptr || rows != nw->planes_rows || fp8 != nw->planes_fp8) {
      const int rc = make_act_map4(nw, &nw->map_planes4, planes, 128, rows, fp8);
      if (rc) return rc;
      nw->planes_ptr = planes;
      nw->planes_rows = rows;
      nw->planes_fp8 = fp8;
    }
  }
  TrunkParams tp;
  tp.n_dev = n_dev;
  tp.n_host = n_host;
  tp.n_layers = N_CONVS;
  tp.head_w = nw->w1x1;
  tp.head_s = nw->s1x1;
  tp.pf_out = nw->pf;
  tp.vf_out = nw->vf;
  tp.dbg_out = dbg_out;
  tp.dbg_layer = dbg_layer;
  tp.hint_planes = L2_EVICT_FIRST;
  tp.hint_weights = L2_EVICT_LAST;
  // small batches (every tile of the batch BOUND gets a CTA pair of its own): the single-tile instantiation, one pair per
  // tile; otherwise groups of two tiles on at most one pair per two SMs
  const int tiles = (n_host + 3) / 4;
  const bool single = tiles <= nw->n_sms / 2;
  const int pairs = single ? tiles : std::min((tiles + 1) / 2, nw->n_sms / 2);
  {
    LaunchScope ls(e, KC_CONV);
    const dim3 grid(2 * pairs), block(CONV_THREADS);
    if (fp8) {
      if (single)
        k_trunk4<true, true><<<grid, block, T4_SMEM_BYTES, e->stream>>>(nw->map_planes4, nw->d_maps8, nw->d_layers8, tp);
      else
        k_trunk4<false, true><<<grid, block, T4_SMEM_BYTES, e->stream>>>(nw->map_planes4, nw->d_maps8, nw->d_layers8, tp);
    } else if (single) {
      k_trunk4<true, false><<<grid, block, T4_SMEM_BYTES, e->stream>>>(nw->map_planes4, nw->d_maps4, nw->d_layers4, tp);
    } else {
      k_trunk4<false, false><<<grid, block, T4_SMEM_BYTES, e->stream>>>(nw->map_planes4, nw->d_maps4, nw->d_layers4, tp);
    }
    CRL_CUDA(cudaGetLastError());
  }
  return launch_heads_v2(e, nw, n_dev, n_host, policy, value, view_out);
}

int net_forward(crl_engine_impl* e, const __nv_bfloat16* planes, int n_host, const int* n_dev, float* policy,
                float* value, __nv_bfloat16* dbg_out, int dbg_layer, PolicyView* view_out) {
  return forward_nw(e, e->net, planes, n_host, n_dev, policy, value, dbg_out, dbg_layer, view_out);
}

int net_forward_slot(crl_engine_impl* e, int slot, const void* planes, int n_host, const int* n_dev, float* policy,
                     float* value, PolicyView* view_out) {
  return forward_nw(e, e->nets[slot], (const __nv_bfloat16*)planes, n_host, n_dev, policy, value, nullptr, -1, view_out);
}

void* net_planes_buf(const crl_engine_impl* e, int slot) { return e->nets[slot] ? e->nets[slot]->planes_buf : nullptr; }

// debug / test hook: one convolution layer on caller-provided activations (see tests/test_gpu_net.py)
int net_debug_conv(crl_engine_impl* e, int layer, const __nv_bfloat16* in, int cin, int n, const __nv_bfloat16* residual,
                   __nv_bfloat16* out, int relu) {
  NetWeights* nw = e->net;
  if (!nw || !nw->loaded) {
    set_error("network weights are not loaded");
    return CRL_ESTATE;
  }
  if (layer < 0 || layer >= N_CONVS || cin != nw->cin[layer]) {
    set_error("crl_debug_conv: bad layer %d / cin %d", layer, cin);
    return CRL_EINVAL;
  }
  CUtensorMap m;
  int rc = make_act_map(nw, &m, in, cin, n);
  if (rc) return rc;
  return launch_conv_v2(e, nw, m, layer, nullptr, n, residual, out, relu);
}


// test hook (crl_debug_tower): the production forward pass -- k_trunk4 + policy GEMM + softmax/value kernel -- with a
// tap on convolution `layer`'s output and copies of the head inputs / policy logits
int net_debug_tower(crl_engine_impl* e, const __nv_bfloat16* planes, int n, int layer, __nv_bfloat16* act_out,
                    float* logits_out, __nv_bfloat16* pf_out, float* vf_out, float* policy, float* value) {
  NetWeights* nw = e->net;
  if (!nw || !nw->loaded) {
    set_error("network weights are not loaded");
    return CRL_ESTATE;
  }
  if (n <= 0 || n > nw->cap_rows || (act_out && (layer < 0 || layer >= N_CONVS))) {
    set_error("crl_debug_tower: bad arguments (n %d of %d, layer %d)", n, nw->cap_rows, layer);
    return CRL_EINVAL;
  }
  int rc = net_forward(e, planes, n, nullptr, policy, value, act_out, layer);
  if (rc) return rc;
  if (logits_out)
    CRL_CUDA(cudaMemcpy2DAsync(logits_out, (size_t)CRL_N_LABELS * 4, nw->logits, 2048 * 4, (size_t)CRL_N_LABELS * 4, n,
                               cudaMemcpyDeviceToDevice, e->stream));
  if (pf_out) CRL_CUDA(cudaMemcpyAsync(pf_out, nw->pf, (size_t)n * 128 * 2, cudaMemcpyDeviceToDevice, e->stream));
  if (vf_out) CRL_CUDA(cudaMemcpyAsync(vf_out, nw->vf, (size_t)n * 64 * 4, cudaMemcpyDeviceToDevice, e->stream));
  return CRL_OK;
}

// ======================================================================================================
// fp8 evaluation: calibration, quantised weight pack, precision switch (DESIGN.md section 3.1, row a7)
// ======================================================================================================
bool net_fp8(const crl_engine_impl* e, int slot) { return e->nets[slot] && e->nets[slot]->fp8; }

// activation scale of one layer: the power of two max(2^ceil(log2(amax / 448)), 2^-126), 1 for amax = 0.  The floor is
// the smallest normal power of two: below it 1 / s overflows to inf and the epilogue's e4m3(a * inf) is NaN for a = 0.
static float act_scale(float amax) {
  if (!(amax > 0.f)) return 1.f;
  if (amax <= 448.f * 0x1p-126f) return 0x1p-126f;   // also where amax / 448 would round to a subnormal or to 0
  const float r = amax / 448.f;
  int ex;
  const float m = frexpf(r, &ex);   // r = m * 2^ex, m in [0.5, 1)
  return ldexpf(1.f, m == 0.5f ? ex - 1 : ex);
}

int net_calibrate(crl_engine_impl* e, const __nv_bfloat16* planes, int n, float* amax_host) {
  NetWeights* nw = e->net;
  if (!nw || !nw->loaded) {
    set_error("crl_net_calibrate_host: network weights are not loaded");
    return CRL_ESTATE;
  }
  if (n <= 0 || n > nw->cap_rows) {
    set_error("crl_net_calibrate_host: %d positions (1..%d)", n, nw->cap_rows);
    return CRL_EINVAL;
  }
  const size_t n_act = (size_t)n * 64 * 256;
  void* buf = nullptr;
  CRL_CUDA(cudaMalloc(&buf, n_act * 2 + (size_t)n * (CRL_N_LABELS + 1) * 4 + N_CONVS * 4));
  __nv_bfloat16* act = (__nv_bfloat16*)buf;
  float* policy = (float*)(act + n_act);
  float* value = policy + (size_t)n * CRL_N_LABELS;
  unsigned* amax = (unsigned*)(value + n);
  const bool was_fp8 = nw->fp8;
  nw->fp8 = false;                    // calibration measures the bf16 tower
  int rc = CRL_OK;
  cudaError_t ce = cudaMemsetAsync(amax, 0, N_CONVS * 4, e->stream);
  for (int L = 0; L < N_CONVS && rc == CRL_OK && ce == cudaSuccess; ++L) {
    rc = net_forward(e, planes, n, nullptr, policy, value, act, L);
    if (rc == CRL_OK) {
      const long long n8 = (long long)n_act / 8;
      k_absmax_bf16<<<(unsigned)std::min<long long>(div_up(n8, 256), 4 * nw->n_sms), 256, 0, e->stream>>>(
          reinterpret_cast<const uint4*>(act), n8, amax + L);
      ce = cudaGetLastError();
    }
  }
  if (rc == CRL_OK && ce == cudaSuccess) ce = cudaMemcpyAsync(amax_host, amax, N_CONVS * 4, cudaMemcpyDeviceToHost, e->stream);
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(e->stream);
  nw->fp8 = was_fp8;
  cudaFree(buf);
  if (rc != CRL_OK) return rc;
  if (ce != cudaSuccess) return cuda_fail(ce, "crl_net_calibrate_host");
  return CRL_OK;
}

int net_load_fp8(crl_engine_impl* e, const float* const* w, const int64_t* sizes, int n, const float* act_amax) {
  NetWeights* nw = e->net;
  nw->fp8 = false;                                     // whatever fails below, the engine is left in bf16
  for (int L = 0; L < N_CONVS; ++L) {
    if (!(act_amax[L] >= 0.f) || !isfinite(act_amax[L])) {
      set_error("crl_net_load_fp8_host: activation amax %d is %g (must be finite and >= 0)", L, (double)act_amax[L]);
      return CRL_EINVAL;
    }
  }
  int rc = net_load(e, w, sizes, n);                   // validates the pack, loads the bf16 tower, drops fp8 state
  if (rc) return rc;
  if (!nw->act8[0]) {
    for (int L = 0; L < N_CONVS; ++L) {
      if ((rc = dev_alloc(e, &nw->w8[L], (size_t)TILE_N * 9 * nw->cin[L]))) return rc;
      if ((rc = dev_alloc(e, &nw->scale8[L], 256))) return rc;
      if ((rc = dev_alloc(e, &nw->shift8[L], 256))) return rc;
    }
    for (int i = 0; i < 2; ++i) {
      if ((rc = dev_alloc(e, &nw->act8[i], (size_t)nw->act4_rows * 64 * 256))) return rc;
      CRL_CUDA(cudaMemsetAsync(nw->act8[i], 0, (size_t)nw->act4_rows * 64 * 256, e->stream));
    }
    if ((rc = dev_alloc(e, &nw->d_maps8, 3 + N_CONVS))) return rc;
    if ((rc = dev_alloc(e, &nw->d_layers8, N_CONVS))) return rc;
    std::vector<CUtensorMap> hm(3 + N_CONVS);
    memset(hm.data(), 0, hm.size() * sizeof(CUtensorMap));
    for (int i = 0; i < 2; ++i)
      if ((rc = make_act_map4(nw, &hm[1 + i], nw->act8[i], 256, nw->act4_rows, true))) return rc;
    for (int L = 0; L < N_CONVS; ++L)
      if ((rc = make_w_map(nw, &hm[3 + L], nw->w8[L], 9 * nw->cin[L], TILE_N, 128, true))) return rc;
    CRL_CUDA(cudaMemcpyAsync(nw->d_maps8, hm.data(), hm.size() * sizeof(CUtensorMap), cudaMemcpyHostToDevice, e->stream));
    CRL_CUDA(cudaStreamSynchronize(e->stream));
  }
  float s_act[N_CONVS];
  for (int L = 0; L < N_CONVS; ++L) s_act[L] = act_scale(act_amax[L]);
  std::vector<uint8_t> wq;
  std::vector<float> sc(256), sh(256), ws(256);
  std::vector<LayerDesc8> hl(N_CONVS);
  for (int L = 0; L < N_CONVS; ++L) {
    const int cin_real = L == 0 ? 127 : 256, cin = nw->cin[L];
    int ik, ib, ibn;
    conv_tensors(L, &ik, &ib, &ibn);
    const float* k = w[ik];
    // per output channel: ws = max_k |W| / 448 (1 for an all-zero column), Wq = e4m3(W / ws)
    for (int o = 0; o < 256; ++o) {
      float m = 0.f;
      for (int t = 0; t < 9 * cin_real; ++t) m = fmaxf(m, fabsf(k[(size_t)t * 256 + o]));
      ws[o] = m > 0.f ? m / 448.f : 1.f;
    }
    wq.assign((size_t)256 * 9 * cin, 0);
    for (int t = 0; t < 9; ++t)
      for (int c = 0; c < cin_real; ++c)
        for (int o = 0; o < 256; ++o)
          wq[(size_t)o * 9 * cin + t * cin + c] =
              __nv_cvt_float_to_fp8(k[((size_t)t * cin_real + c) * 256 + o] / ws[o], __NV_SATFINITE, __NV_E4M3);
    fold_bn(w, ib, ibn, sc.data(), sh.data());
    const float s_in = L == 0 ? 1.f : s_act[L - 1];
    for (int o = 0; o < 256; ++o) sc[o] = ws[o] * s_in * sc[o];
    CRL_CUDA(cudaMemcpyAsync(nw->w8[L], wq.data(), wq.size(), cudaMemcpyHostToDevice, e->stream));
    CRL_CUDA(cudaMemcpyAsync(nw->scale8[L], sc.data(), 1024, cudaMemcpyHostToDevice, e->stream));
    CRL_CUDA(cudaMemcpyAsync(nw->shift8[L], sh.data(), 1024, cudaMemcpyHostToDevice, e->stream));
    CRL_CUDA(cudaStreamSynchronize(e->stream));
    // the same dataflow as the bf16 tower's layer table (net_create), on the e4m3 scratch
    LayerDesc8& d = hl[L];
    memset(&d, 0, sizeof(d));
    d.map_w = 3 + L;
    d.k_chunks = cin / 128;
    d.scale = nw->scale8[L];
    d.shift = nw->shift8[L];
    d.s_out = s_act[L];
    d.inv_out = 1.f / s_act[L];
    if (L == 0) {
      d.map_in = 0;
      d.out = nw->act8[0];
      d.write_out = 1;
    } else if ((L - 1) % 2 == 0) {
      d.map_in = 1;
      d.out = nw->act8[1];
      d.relu = 1;
      d.write_out = 1;
    } else {
      d.map_in = 2;
      d.out = nw->act8[0];
      d.residual = nw->act8[0];
      d.s_res = s_act[L - 2];       // the block input: the stem's or the previous block's output
      d.relu = 1;
      d.write_out = L != N_CONVS - 1;
      d.fuse_heads = L == N_CONVS - 1;
    }
  }
  CRL_CUDA(cudaMemcpyAsync(nw->d_layers8, hl.data(), hl.size() * sizeof(LayerDesc8), cudaMemcpyHostToDevice, e->stream));
  CRL_CUDA(cudaStreamSynchronize(e->stream));
  nw->fp8_loaded = true;
  nw->fp8 = true;
  return CRL_OK;
}

int net_set_precision(crl_engine_impl* e, int precision) {
  NetWeights* nw = e->net;
  if (precision == CRL_NET_BF16) {
    if (nw) nw->fp8 = false;
    return CRL_OK;
  }
  if (precision != CRL_NET_FP8) {
    set_error("crl_net_set_precision: unknown precision %d", precision);
    return CRL_EINVAL;
  }
  if (!nw) {
    set_error("crl_net_set_precision: no fp8 weights in slot %d (crl_net_load_fp8_host)", e->sel_slot);
    return CRL_ESTATE;
  }
  if (!nw->fp8_loaded) {
    set_error("crl_net_set_precision: no fp8 weights (crl_net_load_fp8_host)");
    return CRL_ESTATE;
  }
  nw->fp8 = true;
  return CRL_OK;
}

}  // namespace crl
