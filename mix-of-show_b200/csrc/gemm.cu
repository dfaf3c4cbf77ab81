// gemm.cu — K1/K4: warp-specialised tcgen05 GEMM and implicit-GEMM 3x3 convolution for sm_100a.
//
//   out[m,n] = epilogue( sum_k A[m,k] W[n,k] )        A, W bf16 K-major; fp32 accumulation in TMEM
//
// Persistent kernel: one CTA per SM loops over 128 x 160 output tiles (160 divides every SD1.5 channel count); when the
// problem has an even number of 128-row tiles the CTAs work in PAIRS (2-CTA clusters, tcgen05 cta_group::2) on 256 x 160
// tiles and each CTA fetches only half of the W tile (see the PAIR comment at the kernel).
// Roles (64 + 256 threads):
//   warp 0      TMA producer   cp.async.bulk.tensor -> 128B-swizzled smem ring, mbarrier complete_tx
//   warp 1      TMEM allocator + single-thread tcgen05.mma issuer (UMMA 128|256 x (160|176) x 16), 2 accumulator stages
//   warps 2..9  epilogue       tcgen05.ld (32x32b) -> registers -> fused epilogue -> smem staging -> coalesced stores;
//                              runs concurrently with the next tile's mainloop
// LoRA fusion (edlora.py:244-246): the rank-padded down matrix [16, K] rides along as 16 extra B rows, so the
// same MMA also produces t = x * down^T in TMEM columns 160..175; the epilogue adds t * (alpha*up)^T.
// Convolution: the A tile is a TW x TH x TB pixel patch of the NHWC activation fetched by a 4-D tensor map at
// the tap-shifted coordinate; TMA out-of-bounds zero fill implements the padding.
#include <stdlib.h>

#include "common.h"
#include "tc.cuh"

namespace mos {

constexpr int BM = 128;
constexpr int BN = 160;
constexpr int BK = 64;
constexpr int LORA_N = 16;
constexpr int MAX_STAGES = 8;
constexpr int A_STAGE_BYTES = BM * BK * 2;               // 16384
constexpr int B_STAGE_BYTES = BN * BK * 2;               // 20480
constexpr int L_STAGE_BYTES = LORA_N * BK * 2;           // 2048
constexpr int TMEM_COLS = 512;            // two accumulator stages of 256 columns
constexpr int ACC_STRIDE = 256;
constexpr int STG_PITCH = BN * 2 + 16;    // padded row pitch of the epilogue staging tile (bank-conflict free)
constexpr int STG_BYTES = BM * STG_PITCH;  // 43008
constexpr int EPI_SMEM_BYTES = STG_BYTES + 4 * BN * 4 + BN * 16;
constexpr int EPI_THREADS = 256;           // 8 epilogue warps: 2 per TMEM lane quadrant, each half of the tile columns
constexpr int NUM_THREADS = 64 + EPI_THREADS;
constexpr int MAX_DYN_SMEM = 227 * 1024 - 2048;  // leave room for the static barriers

struct GemmDev {
  int M, N;
  int kb_total;        // number of 64-wide k blocks over the whole reduction (conv: 9 * C/64)
  int kb_per_split;
  int stages;
  int conv, H, W, B, kc_per_tap, TW, TH, TB, lgTW, lgTH, tiles_w, tiles_h;
  int lora;
  int geglu;
  int out_mode;
  int splits;
  int n_tiles, m_tiles, total_super, nbatch;
  int pair;            // work items are 256 x 160 tiles of a 2-CTA cluster (tcgen05 cta_group::2)
  float* partial;
  const float* bias;
  const float* bias_batch;
  long long rows_per_batch;
  long long bias_batch_ld;
  const __nv_bfloat16* residual;
  long long ldr;
  const float* lora_up;
  long long lora_seg;
  void* out;
  long long ldc;
  void* seg_ptr[3];
  int seg_kind[3];
  long long seg_rows_pad[3];
  int heads, head_dim, dpad, dv_pad;
  long long tokens_per_batch;
  int accum;           // MOS_OUT_F32: out += result (Gram accumulation)
  unsigned long long* tl;   // optional timeline buffer (mos_debug_set_timeline)
  int w_static;        // reserved (round-1 weight-prefetch experiment: neutral, removed)
  int* counters;       // split-K with in-kernel finalize: one arrival counter per output tile (zero between launches)
  int stg_alias;       // the epilogue staging tile overlays pipeline stage 0.. (launches with <= 1 work item per CTA)
  const uint8_t* pf;   // optional: bytes to pull into L2 for a LATER launch (the next layer's weights), see mos_gemm_args
  long long pf_bytes;
  int act;             // MOS_ACT_*: applied to acc + bias (+ LoRA) before the residual
};

template <bool F16>
__device__ __forceinline__ void store16x8(__nv_bfloat16* dst, const float* v) {
  uint4 u;
  u.x = pack16x2<F16>(v[0], v[1]);
  u.y = pack16x2<F16>(v[2], v[3]);
  u.z = pack16x2<F16>(v[4], v[5]);
  u.w = pack16x2<F16>(v[6], v[7]);
  *reinterpret_cast<uint4*>(dst) = u;
}

__device__ __forceinline__ void epi_bar() {  // epilogue warps only
  asm volatile("bar.sync 1, %0;" ::"r"((int)blockDim.x - 64) : "memory");
}
__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
  asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}

// ---- optional in-kernel timeline (profiling aid): when a buffer is registered through mos_debug_set_timeline, the
// first 8 CTAs of every gemm launch record %globaltimer stamps (ns) at their phase boundaries.  The pointer travels in
// the kernel parameters (constant bank): a __device__ global would cost an L2 round trip at every stamp site, on the
// critical path of the TMA / MMA threads.
#define stamp(slot)                                                       \
  do {                                                                    \
    if (p.tl != nullptr && blockIdx.x < 8) {                              \
      unsigned long long t_;                                              \
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));              \
      p.tl[blockIdx.x * 8 + (slot)] = t_;                                 \
    }                                                                     \
  } while (0)

struct TileCoord {
  int n0, m0, cb0, ch0, cw0, split;
};
// work item ws (of a CTA, or of a CTA pair) + cluster rank -> this CTA's 128 x 160 tile
__device__ __forceinline__ TileCoord item_coord(const GemmDev& p, int ws, int rank) {
  TileCoord t;
  t.split = ws % p.splits;
  const int tt = ws / p.splits;
  const int tn = tt % p.n_tiles;
  const int tm = p.pair ? 2 * (tt / p.n_tiles) + rank : tt / p.n_tiles;
  t.n0 = tn * BN;
  t.m0 = tm * BM;
  t.cb0 = t.ch0 = t.cw0 = 0;
  if (p.conv) {
    t.cw0 = (tm % p.tiles_w) * p.TW;
    t.ch0 = ((tm / p.tiles_w) % p.tiles_h) * p.TH;
    t.cb0 = (tm / (p.tiles_w * p.tiles_h)) * p.TB;
  }
  return t;
}
// row r of a tile -> global output row m (and validity)
__device__ __forceinline__ bool row_coord(const GemmDev& p, const TileCoord& t, int r, long long& m, int& b) {
  if (p.conv) {
    const int tw = r & (p.TW - 1), th = (r >> p.lgTW) & (p.TH - 1), tb = r >> (p.lgTW + p.lgTH);
    b = t.cb0 + tb;
    const int h = t.ch0 + th, w = t.cw0 + tw;
    m = ((long long)b * p.H + h) * p.W + w;
    return (b < p.B) && (h < p.H);
  }
  m = (long long)t.m0 + r;
  b = (int)(m / p.rows_per_batch);
  return m < p.M;
}

// same without the batch index (no 64-bit division on the copy loops)
__device__ __forceinline__ bool row_m(const GemmDev& p, const TileCoord& t, int r, long long& m) {
  if (p.conv) {
    const int tw = r & (p.TW - 1), th = (r >> p.lgTW) & (p.TH - 1), tb = r >> (p.lgTW + p.lgTH);
    const int b = t.cb0 + tb, h = t.ch0 + th, w = t.cw0 + tw;
    m = ((long long)b * p.H + h) * p.W + w;
    return (b < p.B) && (h < p.H);
  }
  m = (long long)t.m0 + r;
  return m < p.M;
}

// coalesced copy between the padded staging tile and global rows; CPR = 16-byte chunks per row (20 or 10)
template <int CPR, bool TO_GLOBAL>
__device__ __forceinline__ void stage_copy(const GemmDev& p, const TileCoord& t, uint8_t* stg, __nv_bfloat16* gbase,
                                           long long ld, int col0, int et) {
#pragma unroll 4
  const int nthr = (int)blockDim.x - 64;
  for (int i = et; i < BM * CPR; i += nthr) {
    const int rr = i / CPR, ch = i - rr * CPR;
    long long mm;
    if (row_m(p, t, rr, mm)) {
      uint8_t* s = stg + rr * STG_PITCH + ch * 16;
      __nv_bfloat16* g = gbase + mm * ld + col0 + ch * 8;
      if (TO_GLOBAL)
        *reinterpret_cast<uint4*>(g) = *reinterpret_cast<const uint4*>(s);
      else
        cp_async16(s, g);
    }
  }
}

// ---- CTA-pair primitives (tcgen05 cta_group::2): the two CTAs of a cluster sit on the two SMs of one TPC; one MMA of the
// leader (cluster rank 0) multiplies a 256-row A tile (128 rows in each CTA's shared memory) with an N-row W tile of which
// each CTA holds one half, and writes 128 accumulator rows into each CTA's TMEM.  PTX forms as in the CUTLASS headers of
// this image (cute/arch/copy_sm100_tma.hpp SM100_TMA_2SM_LOAD_*, cutlass/arch/barrier.h umma_arrive_multicast_2x1SM,
// cute/arch/tmem_allocator_sm100.hpp Allocator2Sm).
constexpr uint32_t PEER_MASK = 0xFEFFFFFFu;   // shared::cluster address of the same object in cluster rank 0

__device__ __forceinline__ void tma_load_2d_2sm(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  // issued by both CTAs; the transaction bytes count on the LEADER's mbarrier
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & PEER_MASK), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_2sm(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                                int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, "
      "%6}], [%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & PEER_MASK), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void umma_f16_2cta(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_2cta(uint64_t* bar) {   // arrives on this barrier in BOTH CTAs of the pair
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"((uint16_t)3)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_2cta(uint32_t* dst_smem, uint32_t ncols) {   // same warp index in both CTAs
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2cta(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// arrive (release, cluster scope) on the mbarrier at the same shared-memory offset in cluster rank `rank`
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t rank) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t}\n" ::"r"(smem_u32(bar)),
      "r"(rank)
      : "memory");
}

// F16 : 16-bit type of A, of the row / head-split outputs and of the residual (fp16 or bf16).
// PAIR: the grid is made of 2-CTA clusters and a work item is a 256 x 160 output tile computed with cta_group::2 MMAs:
//       every CTA fetches its own 128 A rows but only HALF of the W tile per k-block (26 KB instead of 36 KB for the same
//       MMA work per SM - the mainloop of the 1-CTA kernel sits on the L2 -> SM fabric limit, profiles/README.md), the
//       leader issues the MMAs for both, each CTA drains its own 128 accumulator rows.
template <bool F16, bool PAIR>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
            const __grid_constant__ CUtensorMap tmB1, const __grid_constant__ CUtensorMap tmL, const GemmDev p) {
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment is required by SWIZZLE_128B; the dynamic smem base offset is identical in both CTAs of a pair
  // (same kernel, same static smem), which the cta_group::2 operand addressing relies on.
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  // W rows held by one CTA per k-block: the whole tile (160, + 16 LoRA rows), or in a pair one half of N = 160 / 176
  const int b_rows = PAIR ? (p.lora ? (BN + LORA_N) / 2 : BN / 2) : (p.lora ? BN + LORA_N : BN);
  const int stage_bytes = A_STAGE_BYTES + b_rows * 128;
  // epilogue staging tile [128][STG_PITCH]: behind the pipeline stages, or - when every CTA has at most one work item, so
  // that no load of a following item can be in flight during an epilogue - on top of stage 0.., which buys two more stages
  uint8_t* tables = smem + p.stages * stage_bytes;
  uint8_t* stg = p.stg_alias ? smem : tables;
  float* cb_s = reinterpret_cast<float*>(p.stg_alias ? tables : tables + STG_BYTES);   // [4][BN] bias (+ per-batch bias)
  float4* up_s = reinterpret_cast<float4*>(cb_s + 4 * BN);          // [BN] LoRA up rows (pre-scaled by alpha)

  __shared__ uint64_t full_bar[MAX_STAGES];
  __shared__ uint64_t empty_bar[MAX_STAGES];
  __shared__ uint64_t tmem_full_bar[2];
  __shared__ uint64_t tmem_empty_bar[2];
  __shared__ uint32_t tmem_base_holder;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int epi_warps = ((int)blockDim.x - 64) >> 5;
  const int rank = PAIR ? (int)cluster_ctarank() : 0;      // 0 = leader
  const int unit_id = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;       // CTA (or CTA pair) index
  const int num_units = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  if (threadIdx.x == 0) stamp(0);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(PAIR && rank == 1 && p.lora ? &tmB1 : &tmB);
    if (p.lora) tma_prefetch_desc(&tmL);
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full_bar[s], 1);        // one arrive.expect_tx (pair: by the leader's producer, for the bytes of both)
      mbar_init(&empty_bar[s], 1);       // one tcgen05.commit (pair: multicast to both CTAs)
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full_bar[s], 1);
      mbar_init(&tmem_empty_bar[s], (PAIR ? 2 : 1) * epi_warps);   // one arrival per epilogue warp (of both CTAs)
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    if (PAIR) tmem_alloc_2cta(&tmem_base_holder, TMEM_COLS);
    else tmem_alloc(&tmem_base_holder, TMEM_COLS);
  }
  tc_fence_before();
  if (PAIR) cluster_sync_all();   // the peer must see initialised barriers before any remote complete_tx / commit / arrive
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_holder;

  // Everything above touched no global memory written by the previous kernel in the stream.
  if (threadIdx.x == 0) stamp(1);
  if (p.pf != nullptr && warp == 0 && lane == 1) {
    // L2 staging of a later launch's weights (static data: no dependency on the previous kernel, so ahead of the wait):
    // this CTA's 1/gridDim slice, in 16 KB bulk prefetches.  HBM is idle for most of the step (the step streams 1.7 GB
    // of weights in ~6 ms), the 126 MB L2 holds the next layer's whole weight matrix.
    constexpr long long CH = 16384;
    const long long per = ((p.pf_bytes + gridDim.x - 1) / gridDim.x + CH - 1) / CH * CH;
    const long long lo = (long long)blockIdx.x * per, hi = min(p.pf_bytes, lo + per);
    for (long long off = lo; off < hi; off += CH) {
      const uint32_t n = (uint32_t)min(CH, hi - off) & ~15u;
      if (n) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p.pf + off), "r"(n) : "memory");
    }
  }
  pdl_wait();
  pdl_launch_dependents();

  if (warp == 0) {
    // ===================================================================== TMA producer (every CTA)
    if (lane == 0) {
      stamp(2);
      int stage = 0;
      uint32_t phase = 0;
      for (int ws = unit_id; ws < p.total_super; ws += num_units) {
        const TileCoord t = item_coord(p, ws, rank);
        const int kb_begin = t.split * p.kb_per_split;
        const int kb_end = min(p.kb_total, kb_begin + p.kb_per_split);
        for (int kb = kb_begin; kb < kb_end; ++kb) {
          uint8_t* sa = smem + stage * stage_bytes;
          uint8_t* sb = sa + A_STAGE_BYTES;
          mbar_wait(&empty_bar[stage], phase ^ 1);     // the MMAs that read this slot have retired
          if (!PAIR) mbar_expect_tx(&full_bar[stage], (uint32_t)stage_bytes);
          else if (rank == 0) mbar_expect_tx(&full_bar[stage], 2u * (uint32_t)stage_bytes);
          if (p.conv) {
            const int tap = kb / p.kc_per_tap;
            const int kc = kb - tap * p.kc_per_tap;
            const int kh = tap / 3, kw = tap - kh * 3;
            if (PAIR) tma_load_4d_2sm(sa, &tmA, &full_bar[stage], kc * BK, t.cw0 + kw - 1, t.ch0 + kh - 1, t.cb0);
            else tma_load_4d(sa, &tmA, &full_bar[stage], kc * BK, t.cw0 + kw - 1, t.ch0 + kh - 1, t.cb0);
          } else {
            if (PAIR) tma_load_2d_2sm(sa, &tmA, &full_bar[stage], kb * BK, t.m0);
            else tma_load_2d(sa, &tmA, &full_bar[stage], kb * BK, t.m0);
          }
          if (!PAIR) {
            tma_load_2d(sb, &tmB, &full_bar[stage], kb * BK, t.n0);
            if (p.lora) tma_load_2d(sb + B_STAGE_BYTES, &tmL, &full_bar[stage], kb * BK, 0);
          } else if (!p.lora) {
            tma_load_2d_2sm(sb, &tmB, &full_bar[stage], kb * BK, t.n0 + rank * (BN / 2));
          } else if (rank == 0) {       // N = 176 = [160 W rows | 16 LoRA rows]: leader holds W rows 0..87 ...
            tma_load_2d_2sm(sb, &tmB, &full_bar[stage], kb * BK, t.n0);
          } else {                      // ... the peer W rows 88..159 and the 16 LoRA rows
            constexpr int W1 = BN - (BN + LORA_N) / 2;     // 72
            tma_load_2d_2sm(sb, &tmB1, &full_bar[stage], kb * BK, t.n0 + (BN + LORA_N) / 2);
            tma_load_2d_2sm(sb + W1 * 128, &tmL, &full_bar[stage], kb * BK, 0);
          }
          if (++stage == p.stages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================================================================== MMA issuer (pair: the leader only)
    if (lane == 0 && rank == 0) {
      const uint32_t idesc = make_idesc(PAIR ? 2 * BM : BM, p.lora ? BN + LORA_N : BN, F16 ? 0 : 1);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int ws = unit_id; ws < p.total_super; ws += num_units, ++it) {
        const TileCoord t = item_coord(p, ws, 0);
        const int kb_begin = t.split * p.kb_per_split;
        const int kb_end = min(p.kb_total, kb_begin + p.kb_per_split);
        const int acc = it & 1;
        mbar_wait(&tmem_empty_bar[acc], ((it >> 1) & 1) ^ 1);   // the epilogue (of both CTAs) drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * ACC_STRIDE;
        for (int kb = kb_begin; kb < kb_end; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          if (it == 0 && kb == kb_begin) stamp(3);
          uint8_t* sa = smem + stage * stage_bytes;
          const uint64_t adesc = make_desc_sw128(smem_u32(sa));
          const uint64_t bdesc = make_desc_sw128(smem_u32(sa + A_STAGE_BYTES));
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            // advance 16 elements = 32 B along K inside the 128B swizzle atom: +2 in the (addr >> 4) field
            const uint32_t accf = (kb > kb_begin || k > 0) ? 1u : 0u;
            if (PAIR) umma_f16_2cta(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, accf);
            else umma_bf16(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, accf);
          }
          // frees the smem slot (in both CTAs of a pair) once these MMAs retire
          if (PAIR) umma_commit_2cta(&empty_bar[stage]);
          else umma_commit(&empty_bar[stage]);
          if (++stage == p.stages) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (PAIR) umma_commit_2cta(&tmem_full_bar[acc]);
        else umma_commit(&tmem_full_bar[acc]);
      }
    }
  } else {
    // ===================================================================== epilogue (warps 2..9; every CTA, own 128 rows)
    const int q = warp & 3;                  // TMEM lane quadrant this warp may access
    const int chalf0 = (warp - 2) >> 2;      // first column half this warp handles
    const int chalf_step = epi_warps >> 2;   // 1 (4 epilogue warps: both halves) or 2 (8 warps)
    const int r = q * 32 + lane;             // tile row owned by this thread
    const int et = threadIdx.x - 64;         // 0..255
    const bool staged = (p.splits == 1) && (p.out_mode == MOS_OUT_BF16);
    int it = 0;
    for (int ws = unit_id; ws < p.total_super; ws += num_units, ++it) {
      const TileCoord t = item_coord(p, ws, rank);
      const int acc = it & 1;
      long long m;
      int b;
      const bool valid = row_coord(p, t, r, m, b);
      int b_lo;
      {
        long long m_first;
        row_coord(p, t, 0, m_first, b_lo);
      }
      // ---- 1. residual tile -> staging (coalesced 16-byte cp.async, in flight while the bias tables are staged)
      if (staged && p.residual && !p.stg_alias) {
        __nv_bfloat16* rbase = const_cast<__nv_bfloat16*>(p.residual);
        if (p.geglu) stage_copy<BN / 16, false>(p, t, stg, rbase, p.ldr, t.n0 / 2, et);
        else stage_copy<BN / 8, false>(p, t, stg, rbase, p.ldr, t.n0, et);
      }
      // ---- 2. bias (+ per-batch bias) and LoRA-up rows of this tile's columns
      if (p.splits == 1) {
        for (int i = et; i < 4 * BN; i += (int)blockDim.x - 64) {
          const int j = i / BN, n = i - j * BN;
          float v = p.bias ? __ldg(p.bias + t.n0 + n) : 0.f;
          if (p.bias_batch && (b_lo + j) < p.nbatch)
            v += __ldg(p.bias_batch + (long long)(b_lo + j) * p.bias_batch_ld + t.n0 + n);
          cb_s[i] = v;
        }
        if (p.lora)
          for (int i = et; i < BN; i += (int)blockDim.x - 64)
            up_s[i] = __ldg(reinterpret_cast<const float4*>(p.lora_up) + t.n0 + i);
      }
      cp_async_wait_all();
      epi_bar();
      if (et == 0 && it == 0) stamp(4);
      // ---- 3. accumulators ready?  (one lane per warp polls: 256 spinning threads would steal issue slots from the
      //         single-thread TMA / MMA roles)
      if (lane == 0) mbar_wait(&tmem_full_bar[acc], (it >> 1) & 1);
      __syncwarp();
      tc_fence_after();
      if (et == 0 && it == 0) stamp(5);
      if (staged && p.residual && p.stg_alias) {
        // every MMA of the (only) item has retired, so every TMA load has landed and been consumed: the pipeline stages
        // are free to carry the staging tile
        __nv_bfloat16* rbase = const_cast<__nv_bfloat16*>(p.residual);
        if (p.geglu) stage_copy<BN / 16, false>(p, t, stg, rbase, p.ldr, t.n0 / 2, et);
        else stage_copy<BN / 8, false>(p, t, stg, rbase, p.ldr, t.n0, et);
        cp_async_wait_all();
        epi_bar();
      }
      const uint32_t trow = tmem_base + acc * ACC_STRIDE + (uint32_t(q * 32) << 16);
      const int bsel = min(max(b - b_lo, 0), 3);
      const float* cb = cb_s + bsel * BN;
      uint8_t* srow = stg + r * STG_PITCH;

      for (int chalf = chalf0; chalf < 2; chalf += chalf_step) {
        // this warp's 80 accumulator columns (and the 16 LoRA columns) in ONE round of TMEM loads: a tcgen05.ld costs a few
        // hundred cycles of latency while the tensor pipe is busy, and a load-wait-compute loop pays it once per chunk
        uint32_t vv[5][16];
        float t4[16];
        if (p.geglu) {
          // tile columns [0,80) = a, [80,160) = gate for the same 80 outputs; this warp: outputs [40*chalf, +40)
#pragma unroll
          for (int c = 0; c < 5; ++c) {
            tmem_ld8(trow + (chalf * 5 + c) * 8, *reinterpret_cast<uint32_t(*)[8]>(&vv[c][0]));
            tmem_ld8(trow + BN / 2 + (chalf * 5 + c) * 8, *reinterpret_cast<uint32_t(*)[8]>(&vv[c][8]));
          }
        } else {
#pragma unroll
          for (int c = 0; c < 5; ++c) tmem_ld16(trow + (chalf * 5 + c) * 16, vv[c]);
        }
        if (p.lora && p.splits == 1) {
          uint32_t tv[16];
          tmem_ld16(trow + BN, tv);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; ++j) t4[j] = __uint_as_float(tv[j]);
        } else {
          tmem_ld_wait();
        }
        if (p.splits > 1) {
          if (valid) {
            float* dst = p.partial + ((long long)t.split * p.M + m) * p.N + t.n0 + chalf * 80;
#pragma unroll
            for (int c = 0; c < 5; ++c) {
#pragma unroll
              for (int j = 0; j < 16; j += 4)
                *reinterpret_cast<uint4*>(dst + c * 16 + j) = make_uint4(vv[c][j], vv[c][j + 1], vv[c][j + 2], vv[c][j + 3]);
            }
          }
        } else if (p.geglu) {
#pragma unroll
          for (int cc = 0; cc < 5; ++cc) {
            const int c = chalf * 5 + cc;
            float o[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int na = c * 8 + j, ng = na + BN / 2;
              float a = __uint_as_float(vv[cc][j]) + cb[na];
              float g = __uint_as_float(vv[cc][8 + j]) + cb[ng];
              if (p.lora) {
                const float4 ua = up_s[na], ug = up_s[ng];
                a += t4[0] * ua.x + t4[1] * ua.y + t4[2] * ua.z + t4[3] * ua.w;
                g += t4[0] * ug.x + t4[1] * ug.y + t4[2] * ug.z + t4[3] * ug.w;
              }
              o[j] = a * gelu_erf(g);
            }
            store16x8<F16>(reinterpret_cast<__nv_bfloat16*>(srow + c * 16), o);
          }
        } else {
#pragma unroll
          for (int cc = 0; cc < 5; ++cc) {
            const int c = chalf * 5 + cc;
            const int nl = c * 16;               // column inside the tile
            const int nc = t.n0 + nl;            // global column
            float o[16];
            float tt[4] = {0.f, 0.f, 0.f, 0.f};
            if (p.lora) {
              const int sidx = (int)(nc / p.lora_seg);
#pragma unroll
              for (int i = 0; i < 4; ++i)
                tt[i] = sidx == 0 ? t4[i] : sidx == 1 ? t4[4 + i] : sidx == 2 ? t4[8 + i] : t4[12 + i];
            }
#pragma unroll
            for (int j4 = 0; j4 < 16; j4 += 4) {
              const float4 cbv = *reinterpret_cast<const float4*>(cb + nl + j4);
              o[j4 + 0] = __uint_as_float(vv[cc][j4 + 0]) + cbv.x;
              o[j4 + 1] = __uint_as_float(vv[cc][j4 + 1]) + cbv.y;
              o[j4 + 2] = __uint_as_float(vv[cc][j4 + 2]) + cbv.z;
              o[j4 + 3] = __uint_as_float(vv[cc][j4 + 3]) + cbv.w;
            }
            if (p.lora) {
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                const float4 u = up_s[nl + j];
                o[j] += tt[0] * u.x + tt[1] * u.y + tt[2] * u.z + tt[3] * u.w;
              }
            }
            if (p.act == MOS_ACT_RELU) {
#pragma unroll
              for (int j = 0; j < 16; ++j) o[j] = fmaxf(o[j], 0.f);
            }
            if (p.out_mode == MOS_OUT_BF16) {
              if (p.residual) {
                const uint4 r0 = *reinterpret_cast<const uint4*>(srow + nl * 2);
                const uint4 r1 = *reinterpret_cast<const uint4*>(srow + nl * 2 + 16);
                const uint32_t rr[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  const float2 f = unpack16x2<F16>(rr[j]);
                  o[2 * j] += f.x;
                  o[2 * j + 1] += f.y;
                }
              }
              store16x8<F16>(reinterpret_cast<__nv_bfloat16*>(srow + nl * 2), o);
              store16x8<F16>(reinterpret_cast<__nv_bfloat16*>(srow + nl * 2 + 16), o + 8);
            } else if (p.out_mode == MOS_OUT_F32) {
              if (valid) {
                float* orow = reinterpret_cast<float*>(p.out) + m * p.ldc + nc;
#pragma unroll
                for (int j = 0; j < 16; j += 4) {
                  float4 r4 = make_float4(o[j], o[j + 1], o[j + 2], o[j + 3]);
                  if (p.accum) {
                    const float4 old = *reinterpret_cast<const float4*>(orow + j);
                    r4.x += old.x; r4.y += old.y; r4.z += old.z; r4.w += old.w;
                  }
                  *reinterpret_cast<float4*>(orow + j) = r4;
                }
              }
            } else if (valid) {  // MOS_OUT_HEADS
              const int seg_len = p.heads * p.head_dim;
              const long long bb = m / p.tokens_per_batch;
              const long long tok = m - bb * p.tokens_per_batch;
#pragma unroll
              for (int half = 0; half < 2; ++half) {
                const int n = nc + half * 8;
                const int seg = n / seg_len;
                const int cc2 = n - seg * seg_len;
                const int head = cc2 / p.head_dim;
                const int j0 = cc2 - head * p.head_dim;
                __nv_bfloat16* base = reinterpret_cast<__nv_bfloat16*>(p.seg_ptr[seg]);
                const long long bh = bb * p.heads + head;
                if (p.seg_kind[seg] == MOS_SEG_ROWS) {
                  store16x8<F16>(base + (bh * p.seg_rows_pad[seg] + tok) * p.dpad + j0, o + half * 8);
                } else {
                  __nv_bfloat16* d = base + (bh * p.dv_pad + j0) * p.seg_rows_pad[seg] + tok;
#pragma unroll
                  for (int e = 0; e < 8; ++e)
                    reinterpret_cast<uint16_t*>(d)[(long long)e * p.seg_rows_pad[seg]] = cvt16<F16>(o[half * 8 + e]);
                }
              }
            }
          }
        }
      }  // column halves
      // ---- 4. accumulator drained: hand it back to the MMA thread of the leader (next-but-one tile)
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PAIR) mbar_arrive_cluster(&tmem_empty_bar[acc], 0);
        else mbar_arrive(&tmem_empty_bar[acc]);
      }
      if (et == 0 && it == 0) stamp(6);
      // ---- 5. coalesced write-out of the staged 16-bit tile
      if (staged) {
        epi_bar();
        __nv_bfloat16* obase = reinterpret_cast<__nv_bfloat16*>(p.out);
        if (p.geglu) stage_copy<BN / 16, true>(p, t, stg, obase, p.ldc, t.n0 / 2, et);
        else stage_copy<BN / 8, true>(p, t, stg, obase, p.ldc, t.n0, et);
      }
      epi_bar();   // staging / bias tables are reused by the next item
      if (et == 0 && it == 0) stamp(7);
      if (p.counters != nullptr) {
        // split-K, in-kernel finalize: publish this item's partial tile (bar.sync ordered every epilogue thread's stores
        // before this thread; its gpu-scope fence is cumulative over them - the pattern of a cooperative grid sync)
        if (et == 0) {
          __threadfence();
          atomicAdd(p.counters + ws / p.splits, 1);
        }
      }
    }
    tc_fence_before();
    if (p.counters != nullptr) {
      // ---- phase 2 (split-K only): the `splits` CTAs that hold the partials of one output tile each reduce 1/splits of
      // its rows, in the fixed order split 0..S-1 (bitwise reproducible), and apply bias / per-batch bias / residual.
      // Deadlock-free: the grid has at most one CTA per SM (all resident), and no CTA waits before ALL its own partials are
      // published.  The counter runs 0 -> S (arrivals) -> 2S (slices done) and is reset by the last slice.
      const int nthr = (int)blockDim.x - 64;
      const int S = p.splits;
      const int rows_per = (BM + S - 1) / S;
      for (int ws = unit_id; ws < p.total_super; ws += num_units) {
        const TileCoord t = item_coord(p, ws, rank);
        int* ctr = p.counters + ws / S;
        if (et == 0) {
          int seen;
          do {
            asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(seen) : "l"(ctr) : "memory");
          } while (seen < S);
        }
        epi_bar();
        const int rlo = t.split * rows_per, rhi = min(BM, rlo + rows_per);
        const int total = (rhi - rlo) * (BN / 4);
        const long long MN = (long long)p.M * p.N;
        // two output quads per thread and four splits per round: 8 independent 16-byte L2 loads in flight per thread (the
        // partials were written by other SMs: the reduction is L2-latency bound, not bandwidth bound)
        for (int i0 = et; i0 < total; i0 += 2 * nthr) {
          bool ok[2];
          long long m[2];
          int b[2], n[2];
          const float* src[2];
          float4 acc[2];
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int i = i0 + e * nthr;
            const int rr = rlo + i / (BN / 4), c4 = i % (BN / 4);
            m[e] = 0;
            b[e] = 0;
            ok[e] = (i < total) && row_coord(p, t, rr, m[e], b[e]);
            n[e] = t.n0 + c4 * 4;
            src[e] = p.partial + m[e] * p.N + n[e];
            acc[e] = make_float4(0.f, 0.f, 0.f, 0.f);
          }
          for (int sp = 0; sp < S; sp += 4) {
            float4 v[2][4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
              for (int e = 0; e < 2; ++e)
                if (ok[e] && sp + u < S) v[e][u] = __ldcg(reinterpret_cast<const float4*>(src[e] + (sp + u) * MN));
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
              for (int e = 0; e < 2; ++e)
                if (ok[e] && sp + u < S) {     // split order 0..S-1: the summation order of mos_splitk_finalize
                  acc[e].x += v[e][u].x; acc[e].y += v[e][u].y; acc[e].z += v[e][u].z; acc[e].w += v[e][u].w;
                }
          }
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            if (!ok[e]) continue;
            float4 a4 = acc[e];
            if (p.bias) {
              const float4 bv = __ldg(reinterpret_cast<const float4*>(p.bias + n[e]));
              a4.x += bv.x; a4.y += bv.y; a4.z += bv.z; a4.w += bv.w;
            }
            if (p.bias_batch) {
              const float4 bv = __ldg(reinterpret_cast<const float4*>(p.bias_batch + (long long)b[e] * p.bias_batch_ld + n[e]));
              a4.x += bv.x; a4.y += bv.y; a4.z += bv.z; a4.w += bv.w;
            }
            if (p.residual) {
              const uint2 rv = *reinterpret_cast<const uint2*>(p.residual + m[e] * p.ldr + n[e]);
              const float2 r0 = unpack16x2<F16>(rv.x), r1 = unpack16x2<F16>(rv.y);
              a4.x += r0.x; a4.y += r0.y; a4.z += r1.x; a4.w += r1.y;
            }
            uint2 o;
            o.x = pack16x2<F16>(a4.x, a4.y);
            o.y = pack16x2<F16>(a4.z, a4.w);
            *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(p.out) + m[e] * p.ldc + n[e]) = o;
          }
        }
        epi_bar();
        if (et == 0) {
          const int old = atomicAdd(ctr, 1);
          if (old == 2 * S - 1) atomicExch(ctr, 0);     // every slice of this tile is written: ready for the next launch
        }
      }
    }
  }

  // a CTA of a pair may not exit while its peer can still read its shared memory (MMA operands), complete transactions or
  // arrive on its barriers
  if (PAIR) cluster_sync_all();
  else __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    if (PAIR) tmem_dealloc_2cta(tmem_base, TMEM_COLS);
    else tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ---------------------------------------------------------------------------------------------- split-K finalize
template <bool F16>
__global__ void splitk_finalize_kernel(const float* __restrict__ partial, int splits, long long M, long long N,
                                       const float* __restrict__ bias, const float* __restrict__ bias_batch,
                                       long long rows_per_batch, long long bias_batch_ld,
                                       const __nv_bfloat16* __restrict__ residual, long long ldr,
                                       __nv_bfloat16* __restrict__ out, long long ldc) {
  pdl_wait();
  pdl_launch_dependents();
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // one thread per 4 columns
  long long n4 = N / 4;
  if (idx >= M * n4) return;
  long long m = idx / n4;
  long long n = (idx - m * n4) * 4;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int s = 0; s < splits; ++s) {
    float4 v = __ldg(reinterpret_cast<const float4*>(partial + ((long long)s * M + m) * N + n));
    acc.x += v.x;
    acc.y += v.y;
    acc.z += v.z;
    acc.w += v.w;
  }
  if (bias) {
    float4 b = __ldg(reinterpret_cast<const float4*>(bias + n));
    acc.x += b.x; acc.y += b.y; acc.z += b.z; acc.w += b.w;
  }
  if (bias_batch) {
    float4 b = __ldg(reinterpret_cast<const float4*>(bias_batch + (m / rows_per_batch) * bias_batch_ld + n));
    acc.x += b.x; acc.y += b.y; acc.z += b.z; acc.w += b.w;
  }
  if (residual) {
    uint2 r = __ldg(reinterpret_cast<const uint2*>(residual + m * ldr + n));
    float2 a = unpack16x2<F16>(r.x), b = unpack16x2<F16>(r.y);
    acc.x += a.x; acc.y += a.y; acc.z += b.x; acc.w += b.y;
  }
  uint2 o;
  o.x = pack16x2<F16>(acc.x, acc.y);
  o.y = pack16x2<F16>(acc.z, acc.w);
  *reinterpret_cast<uint2*>(out + m * ldc + n) = o;
}

static unsigned long long* g_timeline_host = nullptr;
static bool is_aligned(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) % a) == 0; }
static int ilog2(int v) {
  int l = 0;
  while ((1 << l) < v) ++l;
  return l;
}

}  // namespace mos

using namespace mos;

extern "C" int mos_gemm_bf16(const mos_gemm_args* a, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  MOS_CHECK_ARG(a != nullptr, "mos_gemm_bf16: args is NULL");
  MOS_CHECK_ARG(a->A && a->W, "mos_gemm_bf16: A/W is NULL");
  MOS_CHECK_ARG(a->M > 0 && a->N > 0 && a->K > 0, "mos_gemm_bf16: bad shape M=%lld N=%lld K=%lld",
                (long long)a->M, (long long)a->N, (long long)a->K);
  MOS_CHECK_ARG(a->N % BN == 0, "mos_gemm_bf16: N=%lld must be a multiple of %d", (long long)a->N, BN);
  MOS_CHECK_ARG(a->K % BK == 0, "mos_gemm_bf16: K=%lld must be a multiple of %d", (long long)a->K, BK);
  MOS_CHECK_ARG(is_aligned(a->A, 16) && is_aligned(a->W, 16), "mos_gemm_bf16: A/W must be 16-byte aligned");
  MOS_CHECK_DTYPE(a->a_dtype, "mos_gemm_bf16 (a_dtype)");
  MOS_CHECK_DTYPE(a->w_dtype, "mos_gemm_bf16 (w_dtype)");
  MOS_CHECK_ARG(a->a_dtype == a->w_dtype,
                "mos_gemm_bf16: A and W must share the 16-bit type (tcgen05 kind::f16 takes one operand format per MMA; a "
                "mixed fp16 x bf16 descriptor raises an illegal-instruction fault on B200)");
  const bool f16 = a->a_dtype == MOS_DT_F16;
  const int splits = a->splits > 0 ? a->splits : 1;
  const bool lora = a->lora_down != nullptr;
  MOS_CHECK_ARG(a->act == MOS_ACT_NONE || a->act == MOS_ACT_RELU, "mos_gemm_bf16: act=%d is not a MOS_ACT_* value", a->act);
  if (a->act != MOS_ACT_NONE)
    MOS_CHECK_ARG(splits == 1 && !lora && !a->geglu && a->out_mode == MOS_OUT_BF16,
                  "mos_gemm_bf16: act needs 16-bit row output without split-K / geglu / LoRA / head-split / fp32 output");
  if (splits > 1) {
    MOS_CHECK_ARG(a->partial != nullptr, "mos_gemm_bf16: split-K needs a partial workspace");
    if (a->tile_counters != nullptr)
      MOS_CHECK_ARG(a->out != nullptr && a->ldc >= a->N && a->ldc % 4 == 0 && a->N % 4 == 0 && a->pair_mode != 1,
                    "mos_gemm_bf16: in-kernel split-K finalize needs `out` (16-bit rows, ldc %% 4 == 0) and the 1-CTA kernel");
    MOS_CHECK_ARG(!lora && !a->geglu && a->out_mode == MOS_OUT_BF16,
                  "mos_gemm_bf16: split-K cannot be combined with lora / geglu / head-split output");
  } else {
    MOS_CHECK_ARG(a->out_mode == MOS_OUT_HEADS || a->out != nullptr, "mos_gemm_bf16: out is NULL");
  }
  if (lora) {
    MOS_CHECK_ARG(a->lora_up != nullptr && a->lora_seg > 0 && a->lora_seg % 16 == 0 && !a->conv,
                  "mos_gemm_bf16: bad LoRA arguments");
    MOS_CHECK_ARG(a->N / a->lora_seg <= 4, "mos_gemm_bf16: at most 4 LoRA segments");
  }
  if (a->out_mode == MOS_OUT_HEADS) {
    MOS_CHECK_ARG(a->heads > 0 && a->head_dim % 8 == 0 && a->N % (a->heads * a->head_dim) == 0 &&
                      a->N / (a->heads * a->head_dim) <= 3 && a->tokens_per_batch > 0,
                  "mos_gemm_bf16: bad head-split arguments");
  }
  if (a->geglu) MOS_CHECK_ARG(a->out_mode == MOS_OUT_BF16, "mos_gemm_bf16: geglu needs bf16 row-major output");

  GemmDev p;
  memset(&p, 0, sizeof(p));
  CUtensorMap tmA, tmB, tmL;
  memset(&tmL, 0, sizeof(tmL));
  p.M = (int)a->M;
  p.N = (int)a->N;
  p.conv = a->conv;
  p.n_tiles = (int)(a->N / BN);
  int m_tiles;
  if (a->conv) {
    MOS_CHECK_ARG(a->B > 0 && a->H > 0 && a->Wd > 0 && a->C == a->K, "mos_gemm_bf16: bad conv geometry");
    MOS_CHECK_ARG((int64_t)a->B * a->H * a->Wd == a->M, "mos_gemm_bf16: conv M != B*H*W");
    int TW = 1;
    while (TW * 2 <= 128 && a->Wd % (TW * 2) == 0) TW *= 2;
    // choose TH (power of two) maximising the fraction of valid rows in the 128-row tile
    int best_th = 1;
    double best_eff = -1;
    for (int TH = 1; TH * TW <= 128; TH *= 2) {
      int TB = 128 / (TW * TH);
      if (TB > 4 && TH * 2 * TW <= 128) continue;   // the epilogue stages per-batch bias for <= 4 batches per tile
      double eff = ((double)a->H / (ceil_div(a->H, TH) * TH)) * ((double)a->B / (ceil_div(a->B, TB) * TB));
      if (eff > best_eff + 1e-9) {
        best_eff = eff;
        best_th = TH;
      }
    }
    p.TW = TW;
    p.TH = best_th;
    p.TB = 128 / (TW * best_th);
    p.lgTW = ilog2(p.TW);
    p.lgTH = ilog2(p.TH);
    p.H = a->H;
    p.W = a->Wd;
    p.B = a->B;
    p.tiles_w = a->Wd / TW;
    p.tiles_h = (int)ceil_div(a->H, p.TH);
    int tiles_b = (int)ceil_div(a->B, p.TB);
    m_tiles = p.tiles_w * p.tiles_h * tiles_b;
    p.kc_per_tap = (int)(a->K / BK);
    p.kb_total = 9 * p.kc_per_tap;
  } else {
    MOS_CHECK_ARG(a->lda >= a->K && a->lda % 8 == 0, "mos_gemm_bf16: lda=%lld invalid", (long long)a->lda);
    m_tiles = (int)ceil_div(a->M, BM);
    p.kb_total = (int)(a->K / BK);
  }
  p.m_tiles = m_tiles;
  // ---- CTA pairs (tcgen05 cta_group::2): a work item is a 256 x 160 tile of a 2-CTA cluster; needs an even number of
  // 128-row tiles.  MOS_GEMM_PAIR=0 forces the 1-CTA kernel (A/B comparison, profiles/README.md).
  static int use_pair = -1, pair_min_kb = 16;
  if (use_pair < 0) {
    const char* e = getenv("MOS_GEMM_PAIR");
    use_pair = (e && e[0] == '1') ? 1 : 0;
    const char* m = getenv("MOS_GEMM_PAIR_MIN_KB");
    if (m) pair_min_kb = atoi(m);
  }
  // Measured on B200 (tools/gemm_shape_bench.py, profiles/README.md "round 2: CTA pairs"): parity-green on every layer shape
  // of the step, but never faster than the 1-CTA kernel - 29.7 vs 31.7 us on the res-64 3x3 conv, 67.6 vs 66.5 us on the
  // longest one, +2 us on every short-K projection (two cluster barriers, remote barrier hops) - i.e. the mainloop is not
  // bound by the bytes a CTA pulls through its own L2 port.  The pair path is therefore OPT-IN (MOS_GEMM_PAIR=1 with at
  // least MOS_GEMM_PAIR_MIN_KB k-blocks per work item, or mos_gemm_args.pair_mode = 1).
  const int kb_per_item = (int)ceil_div(p.kb_total, splits);
  bool pair = use_pair && (m_tiles % 2 == 0) && kb_per_item >= pair_min_kb;
  if (a->pair_mode == 1) pair = (m_tiles % 2 == 0);
  else if (a->pair_mode == 2) pair = false;
  if (splits > 1 && a->tile_counters != nullptr) pair = false;   // the in-kernel finalize is built for 1-CTA work items
  p.pair = pair ? 1 : 0;

  // ---- tensor maps.  W box: the whole tile (160 rows), or a pair's half: 80 rows, with LoRA (N = 176 = 160 W rows + 16
  // LoRA rows) 88 rows for the leader (tmB) and 72 W rows + the 16 LoRA rows for its peer (tmB1, tmL).
  CUtensorMap tmB1;
  memset(&tmB1, 0, sizeof(tmB1));
  const uint32_t wrows0 = pair ? (lora ? (BN + LORA_N) / 2 : BN / 2) : BN;
  const uint32_t wrows1 = BN - (BN + LORA_N) / 2;
  if (a->conv) {
    uint64_t dims[4] = {(uint64_t)a->C, (uint64_t)a->Wd, (uint64_t)a->H, (uint64_t)a->B};
    const uint64_t pitch = (uint64_t)(a->lda > 0 ? a->lda : a->C);
    MOS_CHECK_ARG(pitch >= (uint64_t)a->C && pitch % 8 == 0, "mos_gemm_bf16: conv pixel pitch %llu invalid",
                  (unsigned long long)pitch);
    uint64_t str[3] = {pitch * 2, (uint64_t)a->Wd * pitch * 2, (uint64_t)a->H * a->Wd * pitch * 2};
    uint32_t box[4] = {BK, (uint32_t)p.TW, (uint32_t)p.TH, (uint32_t)p.TB};
    int rc = encode_tmap(&tmA, a->A, 2, 4, dims, str, box, 3);
    if (rc) return rc;
    uint64_t wd[2] = {(uint64_t)a->K * 9, (uint64_t)a->N};
    uint64_t ws[1] = {(uint64_t)a->K * 9 * 2};
    uint32_t wb[2] = {BK, wrows0};
    rc = encode_tmap(&tmB, a->W, 2, 2, wd, ws, wb, 3);
    if (rc) return rc;
  } else {
    uint64_t dims[2] = {(uint64_t)a->K, (uint64_t)a->M};
    uint64_t str[1] = {(uint64_t)a->lda * 2};
    uint32_t box[2] = {BK, (uint32_t)BM};
    int rc = encode_tmap(&tmA, a->A, 2, 2, dims, str, box, 3);
    if (rc) return rc;
    uint64_t wd[2] = {(uint64_t)a->K, (uint64_t)a->N};
    uint64_t ws[1] = {(uint64_t)a->K * 2};
    uint32_t wb[2] = {BK, wrows0};
    rc = encode_tmap(&tmB, a->W, 2, 2, wd, ws, wb, 3);
    if (rc) return rc;
    if (lora) {
      if (pair) {
        uint32_t wb1[2] = {BK, wrows1};
        rc = encode_tmap(&tmB1, a->W, 2, 2, wd, ws, wb1, 3);
        if (rc) return rc;
      }
      uint64_t ld[2] = {(uint64_t)a->K, LORA_N};
      uint64_t ls[1] = {(uint64_t)a->K * 2};
      uint32_t lb[2] = {BK, LORA_N};
      rc = encode_tmap(&tmL, a->lora_down, 2, 2, ld, ls, lb, 3);
      if (rc) return rc;
    }
  }
  MOS_CHECK_ARG(splits <= p.kb_total, "mos_gemm_bf16: splits=%d > k blocks=%d", splits, p.kb_total);
  p.splits = splits;
  p.kb_per_split = (int)ceil_div(p.kb_total, splits);
  MOS_CHECK_ARG((long long)p.kb_per_split * (splits - 1) < p.kb_total, "mos_gemm_bf16: empty split");
  p.lora = lora ? 1 : 0;
  p.geglu = a->geglu;
  p.out_mode = a->out_mode;
  p.partial = a->partial;
  p.bias = a->bias;
  p.bias_batch = a->bias_batch;
  p.rows_per_batch = a->rows_per_batch > 0 ? a->rows_per_batch : 1;
  p.bias_batch_ld = a->bias_batch_ld > 0 ? a->bias_batch_ld : a->N;
  p.residual = reinterpret_cast<const __nv_bfloat16*>(a->residual);
  p.ldr = a->ldr;
  p.lora_up = a->lora_up;
  p.lora_seg = a->lora_seg > 0 ? a->lora_seg : a->N;
  p.out = a->out;
  p.ldc = a->ldc;
  for (int i = 0; i < 3; ++i) {
    p.seg_ptr[i] = a->seg_ptr[i];
    p.seg_kind[i] = a->seg_kind[i];
    p.seg_rows_pad[i] = a->seg_rows_pad[i];
  }
  p.heads = a->heads;
  p.head_dim = a->head_dim;
  p.dpad = a->dpad;
  p.dv_pad = a->dv_pad;
  p.tokens_per_batch = a->tokens_per_batch > 0 ? a->tokens_per_batch : 1;
  p.accum = a->accumulate;
  p.tl = g_timeline_host;
  p.w_static = a->w_static;
  p.pf = nullptr;
  p.pf_bytes = 0;
  p.act = a->act;
  if (a->prefetch_ptr != nullptr && a->prefetch_bytes >= 16) {
    MOS_CHECK_ARG(is_aligned(a->prefetch_ptr, 16), "mos_gemm_bf16: prefetch_ptr must be 16-byte aligned");
    p.pf = reinterpret_cast<const uint8_t*>(a->prefetch_ptr);
    p.pf_bytes = a->prefetch_bytes;
  }
  p.counters = (splits > 1) ? a->tile_counters : nullptr;
  if (p.counters != nullptr) {
    MOS_CHECK_ARG((long long)p.n_tiles * m_tiles <= a->tile_counters_len,
                  "mos_gemm_bf16: tile_counters holds %d counters, the launch needs %lld", (int)a->tile_counters_len,
                  (long long)p.n_tiles * m_tiles);
  }
  if (a->bias_batch && !a->conv)
    MOS_CHECK_ARG(p.rows_per_batch >= 32, "mos_gemm_bf16: bias_batch needs rows_per_batch >= 32 in plain mode");
  p.total_super = p.n_tiles * (pair ? m_tiles / 2 : m_tiles) * splits;
  p.nbatch = a->conv ? a->B : (int)ceil_div(a->M, p.rows_per_batch);

  // MOS_GEMM_STG_ALIAS=1: staging tile on top of the pipeline stages (measured slower: the residual prefetch moves behind the
  // mainloop and more than 3 stages buy nothing, tools/gemm_stage_sweep.py).  MOS_GEMM_STAGES=n: default pipeline depth.
  static int num_sms = 0, stg_alias_env = -1, stages_env = 0;
  if (stg_alias_env < 0) {
    const char* e = getenv("MOS_GEMM_STG_ALIAS");
    stg_alias_env = (e && e[0] == '1') ? 1 : 0;
    const char* st = getenv("MOS_GEMM_STAGES");
    if (st) stages_env = atoi(st);
  }
  if (num_sms == 0) {
    int dev = 0;
    MOS_CHECK_CUDA(cudaGetDevice(&dev));
    MOS_CHECK_CUDA(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
  }
  const int b_rows = pair ? (int)wrows0 : (lora ? BN + LORA_N : BN);
  const int stage_bytes = A_STAGE_BYTES + b_rows * 128;
  // one work item per CTA at most (the common case of the batch-2 step): the staging tile overlays the pipeline stages
  p.stg_alias = (stg_alias_env && !pair && p.total_super <= num_sms && 2 * stage_bytes >= STG_BYTES) ? 1 : 0;
  const int epi_bytes = p.stg_alias ? EPI_SMEM_BYTES - STG_BYTES : EPI_SMEM_BYTES;
  int stages = a->stages > 0 ? a->stages : (stages_env > 0 ? stages_env : MAX_STAGES);
  if (stages > MAX_STAGES) stages = MAX_STAGES;
  while (stages * stage_bytes + epi_bytes + 1024 > MAX_DYN_SMEM) --stages;
  if (stages < 2) stages = 2;
  p.stages = stages;
  const int smem_bytes = stages * stage_bytes + epi_bytes + 1024;

  static bool configured = false;
  if (!configured) {
    configured = true;
    MOS_CHECK_CUDA(cudaFuncSetAttribute(gemm_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, MAX_DYN_SMEM));
    MOS_CHECK_CUDA(cudaFuncSetAttribute(gemm_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, MAX_DYN_SMEM));
    MOS_CHECK_CUDA(cudaFuncSetAttribute(gemm_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, MAX_DYN_SMEM));
    MOS_CHECK_CUDA(cudaFuncSetAttribute(gemm_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, MAX_DYN_SMEM));
  }
  // persistent: one CTA per SM; each CTA (or CTA pair) loops over its share of the (tile, split) work items
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  static int epi_warps = 0;
  if (epi_warps == 0) {
    const char* e = getenv("MOS_GEMM_EPI_WARPS");
    epi_warps = (e && e[0] == '4') ? 4 : 8;
  }
  cfg.blockDim = dim3(64 + 32 * epi_warps);
  cfg.dynamicSmemBytes = (size_t)smem_bytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  attr[1].id = cudaLaunchAttributeClusterDimension;
  attr[1].val.clusterDim.x = 2;
  attr[1].val.clusterDim.y = 1;
  attr[1].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pair ? 2 : 1;   // no cluster attribute at all for unclustered launches
  int units = pair ? num_sms / 2 : num_sms;      // 2-CTA clusters pack the 148 SMs exactly (one pair per TPC)
  if (units > p.total_super) units = p.total_super;
  cfg.gridDim = dim3((unsigned)(pair ? 2 * units : units));
  if (pair) {
    if (f16) MOS_CHECK_CUDA(cudaLaunchKernelEx(&cfg, gemm_kernel<true, true>, tmA, tmB, tmB1, tmL, p));
    else MOS_CHECK_CUDA(cudaLaunchKernelEx(&cfg, gemm_kernel<false, true>, tmA, tmB, tmB1, tmL, p));
  } else {
    if (f16) MOS_CHECK_CUDA(cudaLaunchKernelEx(&cfg, gemm_kernel<true, false>, tmA, tmB, tmB1, tmL, p));
    else MOS_CHECK_CUDA(cudaLaunchKernelEx(&cfg, gemm_kernel<false, false>, tmA, tmB, tmB1, tmL, p));
  }
  return MOS_OK;
}

extern "C" int mos_debug_set_timeline(void* buf) {
  mos::g_timeline_host = reinterpret_cast<unsigned long long*>(buf);
  return MOS_OK;
}

extern "C" int mos_splitk_finalize(const float* partial, int32_t splits, int64_t M, int64_t N, const float* bias,
                                   const float* bias_batch, int64_t rows_per_batch, int64_t bias_batch_ld,
                                   const void* residual, int64_t ldr, void* out, int64_t ldc, int32_t act_dtype,
                                   void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  MOS_CHECK_ARG(partial && out && splits >= 1 && M > 0 && N > 0 && N % 4 == 0, "mos_splitk_finalize: bad arguments");
  MOS_CHECK_DTYPE(act_dtype, "mos_splitk_finalize");
  long long total = M * (N / 4);
  int threads = 256;
  long long blocks = ceil_div(total, threads);
  MOS_CHECK_CUDA(launch_pdl(act_dtype == MOS_DT_F16 ? splitk_finalize_kernel<true> : splitk_finalize_kernel<false>,
                            dim3((unsigned)blocks), dim3(threads), 0, stream, partial,
                            (int)splits, (long long)M, (long long)N, bias, bias_batch,
                            (long long)(rows_per_batch > 0 ? rows_per_batch : 1),
                            (long long)(bias_batch_ld > 0 ? bias_batch_ld : N),
                            reinterpret_cast<const __nv_bfloat16*>(residual), (long long)ldr,
                            reinterpret_cast<__nv_bfloat16*>(out), (long long)ldc));
  return MOS_OK;
}
