// A run of identical ResNet bottlenecks (layer3 of the dilated ResNet-101: 22 blocks of 1x1 1024->256, 3x3 256->256,
// 1x1 256->1024 + residual, Bottleneck.forward, model/modules/backbone/resnet.py:22-42) as ONE persistent kernel.
//
// Same idea as the WASP chain (wasp_chain.cu): the only cross-tile dependency of a bottleneck is the halo of its 3x3
// conv, and that is PER IMAGE, so CTAs synchronise through per-image-group release/acquire counters instead of
// kernel boundaries.  Every CTA owns one 128-pixel tile for the whole run; CTA pairs (cta_group::2, M = 256) take the
// same tile of two consecutive image groups.  Per block b (input X_b [.., 1024], T1_b = conv1(X_b) [.., 256]):
//   P2  conv2 3x3 -> acc[256]: the centre tap first, from this CTA's own t1 tile in the staging set T, then the halo
//       taps chunk-major over the four 64-channel chunks c of T1_b (chunk 0's eight taps, then chunk 1's, ...).  The
//       halo tiles of chunk c are TMA-loaded once counter[b][c] says every tile of the image group stored chunk c of
//       T1_b, so chunk 0's halo MMAs run while the neighbours are still storing chunks 1..3.
//       epilogue: t2 = ReLU(acc + shift2) -> 16-bit -> staging set T (never goes to global memory); accumulator half
//       0 (t2 groups 0-1) is released as soon as it is in registers, so conv3 N-tile 0 starts mid-epilogue
//   P3  conv3 1x1 in eight N-tiles of 128 output channels, ping-pong in TMEM columns [0,128) / [128,256):
//         acc_j = t2 (A operand straight from the staging set T) x W3_j  (+ X_b residual tile x I as identity MMAs)
//         N-tile 0 takes K-chunk c as soon as t2 group c is staged
//         epilogue j (overlaps the MMAs of N-tile j+1): X_{b+1}[:, j] = ReLU(acc_j + shift3) -> staging set O
//           -> TMA store (the next block's residual) AND the A operand of
//         D2 += X_{b+1}[:, j] x W1_{b+1}[:, j]   -> conv1 of the NEXT block accumulates in TMEM columns [256,512)
//       D2 epilogue: T1_{b+1} = ReLU(D2 + shift1) -> staging set T -> TMA store group by group; counter[b+1][c] is
//       released once the bulk store of group c has completed (bulk groups complete in order, so X_{b+1}, stored
//       earlier, is in global memory too before the first of them)
// so a block costs one halo exchange and its 1x1 convolutions never read their input from memory again.
// P1 (once): T1_0 = conv1 of the first block, a plain GEMM over X_0.
//
// Counters: [tiles_n][nblocks + 1][4] (image group, block, 64-channel chunk) + one exit counter; the last CTA to
// leave re-arms them all to zero.  T1_b lives in the parity buffer n0 + (b & 1) * N, so T1_{b+1} overwrites T1_{b-1}.
// That is safe: a tile stores T1_{b+1} only after its own conv2 of block b, whose halo loads (and the conv3 loads
// behind them) the producer issues only after all four counter[b][c] have been acquired; and a neighbour releases ANY
// counter[b][c] only after its D2 epilogue of block b-1, which waits on an MMA commit issued after every conv2 MMA of
// block b-1, i.e. after every halo load of T1_{b-1} it made has landed.  All four counters of a block are acquired
// even when a tile has no halo taps, which keeps this ordering (and the residual loads of X_b behind them) intact.
// The acquiring is done by the counter watcher (warp 3), which hands each counter[b][c] to the producer through a
// shared-memory barrier: a global round trip per chunk inside the producer would stall the ring's feed.
//
// The epilogue reads the BatchNorm shifts from shared memory: at the start of each block the epilogue warps copy that
// block's shift2 / shift3 and the next block's shift1 (6 KB) there while conv2 runs.  Read from global memory, every
// 64-column group began with an L2 round trip for a line no warp of the SM had touched yet.
//
// Warp roles (384 threads): 0 = TMA producer, 1 = MMA issuer (leader CTA), 2 = TMEM alloc + store thread,
// 3 = counter watcher, 4..11 = epilogue.
#include <cuda.h>
#include <stdlib.h>

#include "up_internal.h"
#include "up_ptx.cuh"

namespace up {

constexpr int kBcThreads = 384;
constexpr int kBcEpiWarp0 = 4;
constexpr int kBcEpiThreads = 256;
constexpr int kBcMaxSlots = 4;
constexpr uint32_t kBcABytes = 16384;      // 128 px x 64 ch
constexpr uint32_t kBcBBytes = 16384;      // up to 128 filter rows x 64 ch (this CTA's half of a 256-row tile)
constexpr uint32_t kBcSlotBytes = kBcABytes + kBcBBytes;
constexpr uint32_t kBcBuf = 16384;         // staging buffer: 128 px x 64 ch
constexpr int kBcP = 256;                  // planes
constexpr int kBcC = 1024;                 // 4 * planes
constexpr int kBcNT = 8;                   // conv3 N-tiles of 128
constexpr int kBcShifts = kBcP + kBcC + kBcP;     // shift2[b], shift3[b], shift1[b+1] staged in shared memory
constexpr long long kBcSpinLimit = 6000000000LL;

struct BcParams {
  int N, H, W;
  int bn, bh, bw;
  int tiles_h, tiles_w, tiles_n;
  int nblocks, dil;
  int slots;
  uint32_t idesc256, idesc128, idesc_res;
  const float* shift1;        // [nblocks][256]
  const float* shift2;        // [nblocks][256]
  const float* shift3;        // [nblocks][1024]
  unsigned int* counters;     // [tiles_n][nblocks + 1][4] + exit counter
  int fmt;
  unsigned long long* dbg;
};

#define BC_STAMP(slot)                                                                     \
  do {                                                                                     \
    if (p.dbg) {                                                                           \
      unsigned long long _t;                                                               \
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(_t));                              \
      p.dbg[blockIdx.x * 32 + (slot)] = _t;                                                \
    }                                                                                      \
  } while (0)

__device__ __forceinline__ unsigned int bc_ld_acquire(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void bc_red_release(unsigned int* p, unsigned int v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void bc_fence_async() { asm volatile("fence.proxy.async;" ::: "memory"); }

__device__ __forceinline__ void bc_wait_counter(const unsigned int* ctr, unsigned int target) {
  if (bc_ld_acquire(ctr) >= target) return;
  const long long t0 = clock64();
  while (bc_ld_acquire(ctr) < target) {
    __nanosleep(32);
    if (clock64() - t0 > kBcSpinLimit) {
      printf("up: bottleneck chain counter watchdog: block %d thread %d\n", blockIdx.x, threadIdx.x);
      __trap();
    }
  }
}

__device__ __forceinline__ void bc_taps(int dil, int x0, int ext, int limit, int& lo, int& hi) {
  lo = 3;
  hi = -1;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int c = x0 + (k - 1) * dil;
    if (c + ext > 0 && c < limit) {
      lo = min(lo, k);
      hi = max(hi, k);
    }
  }
}

template <int kFmt>
__device__ __forceinline__ uint32_t bc_pack2_relu(float lo_elem, float hi_elem) {
  uint32_t d;
  if constexpr (kFmt == 0) asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi_elem), "f"(lo_elem));
  else asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi_elem), "f"(lo_elem));
  return d;
}

template <int kFmt>
__global__ void __launch_bounds__(kBcThreads, 1)
    bneck_chain_kernel(const __grid_constant__ CUtensorMap tmXa, const __grid_constant__ CUtensorMap tmXb,
                       const __grid_constant__ CUtensorMap tmT, const __grid_constant__ CUtensorMap tmW1,
                       const __grid_constant__ CUtensorMap tmW2, const __grid_constant__ CUtensorMap tmW3,
                       const BcParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_al = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t stgT = smem_base + p.slots * kBcSlotBytes;       // 4 buffers: t1 / t2 tiles (256 channels)
  const uint32_t stgO = stgT + 4 * kBcBuf;                         // 2 buffers: one 128-channel N-tile of the block output
  const uint32_t ident = stgO + 2 * kBcBuf;                        // identity B tile for the residual MMAs (8 KB)
  const uint32_t shf = ident + 8192u;                              // BatchNorm shifts of one block (6 KB), see stage_shifts
  const uint32_t bars = shf + 4u * kBcShifts;
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto empty_bar = [&](int s) { return bars + 8u * (kBcMaxSlots + s); };
  const uint32_t b0 = bars + 8u * (2 * kBcMaxSlots);
  auto tfull_bar = [&](int h) { return b0 + 8u * h; };             // [2]
  auto tempty_bar = [&](int h) { return b0 + 8u * (2 + h); };      // [2]
  const uint32_t d2full_bar = b0 + 8u * 4, d2empty_bar = b0 + 8u * 5;
  auto availT = [&](int g) { return b0 + 8u * (6 + g); };          // [4]
  auto readyT = [&](int g) { return b0 + 8u * (10 + g); };         // [4]
  auto s2readyT = [&](int g) { return b0 + 8u * (14 + g); };       // [4]
  auto availO = [&](int g) { return b0 + 8u * (18 + g); };         // [2]
  auto readyO = [&](int g) { return b0 + 8u * (20 + g); };         // [2]
  auto s2readyO = [&](int g) { return b0 + 8u * (22 + g); };       // [2]
  auto haloT = [&](int c) { return b0 + 8u * (24 + c); };          // [4] counter[b][c] acquired, one phase per block
  const uint32_t tmem_slot = b0 + 8u * 28;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_al + (tmem_slot - smem_base));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  uint32_t crank;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(crank));
  const int cluster_id = blockIdx.x >> 1;
  const int per = p.tiles_h * p.tiles_w;
  const int pair = cluster_id / per, tt = cluster_id % per;
  const int tn = 2 * pair + static_cast<int>(crank);
  const int n0 = tn * p.bn, h0 = (tt / p.tiles_w) * p.bh, w0 = (tt % p.tiles_w) * p.bw;
  unsigned int* ctr = p.counters + static_cast<size_t>(tn) * (p.nblocks + 1) * 4;     // [block][chunk]
  const int nb = p.nblocks;
  if (threadIdx.x == 0) BC_STAMP(0);

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmXa);
    tma_prefetch_desc(&tmT);
    tma_prefetch_desc(&tmW1);
    tma_prefetch_desc(&tmW2);
    tma_prefetch_desc(&tmW3);
    for (int s = 0; s < p.slots; ++s) {
      mbar_init(full_bar(s), 2);
      mbar_init(empty_bar(s), 1);
    }
    for (int h = 0; h < 2; ++h) {
      mbar_init(tfull_bar(h), 1);
      mbar_init(tempty_bar(h), 2 * (kBcEpiThreads / 32));
    }
    mbar_init(d2full_bar, 1);
    mbar_init(d2empty_bar, 2 * (kBcEpiThreads / 32));
    for (int g = 0; g < 4; ++g) {
      mbar_init(availT(g), 2);
      mbar_init(readyT(g), kBcEpiThreads / 32);
      mbar_init(s2readyT(g), 2 * (kBcEpiThreads / 32));
    }
    for (int g = 0; g < 2; ++g) {
      mbar_init(availO(g), 2);
      mbar_init(readyO(g), kBcEpiThreads / 32);
      mbar_init(s2readyO(g), 2 * (kBcEpiThreads / 32));
    }
    for (int c = 0; c < 4; ++c) mbar_init(haloT(c), 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc_2cta(tmem_slot, 512);
  {
    // K-major, 128B-swizzled identity: this CTA supplies rows [32*rank, 32*rank+32) of the 64x64 identity (its half of B)
    const uint32_t one = kFmt == 1 ? 0x3F80u : 0x3C00u;
    for (uint32_t i = threadIdx.x; i < 8192u / 16u; i += blockDim.x) {
      const uint32_t n = i >> 3, chunk = i & 7u;
      const uint32_t src_chunk = chunk ^ (n & 7u);
      uint32_t w[4] = {0u, 0u, 0u, 0u};
      const uint32_t gn = n + 32u * crank;
      if (n < 32u && src_chunk == (gn >> 3)) {
        const uint32_t e = gn & 7u;
        w[e >> 1] = one << ((e & 1u) * 16u);
      }
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(ident + i * 16u), "r"(w[0]), "r"(w[1]), "r"(w[2]),
                   "r"(w[3])
                   : "memory");
    }
    fence_proxy_async_smem();
  }
  tcgen05_before_thread_sync();
  __syncthreads();
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
  tcgen05_after_thread_sync();
  const uint32_t tmem_base = *tmem_slot_ptr;
  const uint32_t tmem_d2 = tmem_base + 256u;
  asm volatile("griddepcontrol.wait;" ::: "memory");
  if (threadIdx.x == 0) BC_STAMP(1);

  if (warp == 0) {
    // ===================== TMA producer =====================
    uint32_t slot = 0, par = 1;
    auto advance = [&]() {
      if (++slot == static_cast<uint32_t>(p.slots)) {
        slot = 0;
        par ^= 1u;
      }
    };
    // one ring slot (32 KB): up to four TMA boxes under one barrier.  kind 0: activation tile (A half) + 128 filter
    // rows (B half) - a regular k-block; kinds 1..3 are the merged B-only / residual slots of the fused phases.
    auto acquire = [&](uint32_t bytes) -> uint32_t {
      mbar_wait(empty_bar(slot), par, 16000000000LL);
      const uint32_t dst = smem_base + slot * kBcSlotBytes;
      if (elect_one()) {
        if (crank == 0) mbar_arrive_expect_tx(full_bar(slot), 2u * bytes);
        else mbar_arrive_remote(full_bar(slot), 0u);
      }
      return dst;
    };
    auto issue = [&](const CUtensorMap* amap, int ac, int aw, int ah, int an, const CUtensorMap* bmap, int bc, int brow) {
      const uint32_t dst = acquire(kBcSlotBytes);
      if (elect_one()) {
        tma_load_5d_2cta(amap, dst, full_bar(slot), ac, aw, 0, ah, an);
        tma_load_2d_2cta(bmap, dst + kBcABytes, full_bar(slot), bc, brow);
      }
      __syncwarp();
      advance();
    };
    // two 128-row filter chunks (64 channels each) side by side: the B operands of two consecutive B-only k-steps
    auto issue_b2 = [&](const CUtensorMap* bmap, int bc0, int brow) {
      const uint32_t dst = acquire(kBcSlotBytes);
      if (elect_one()) {
        tma_load_2d_2cta(bmap, dst, full_bar(slot), bc0, brow);
        tma_load_2d_2cta(bmap, dst + kBcABytes, full_bar(slot), bc0 + 64, brow);
      }
      __syncwarp();
      advance();
    };
    // P1: conv1 of the first block over X_0
    for (int chunk = 0; chunk < kBcC / 64; ++chunk)
      issue(&tmXa, chunk * 64, w0, h0, n0, &tmW1, chunk * 64, static_cast<int>(crank) * 128);
    for (int b = 0; b < nb; ++b) {
      // P2, centre tap first: its activation tile is this CTA's own t1 tile, still in the staging set T - only the
      // filter chunks are loaded, and nothing here waits for the neighbours
      const int wrow = (b * 9 + 4) * kBcP + static_cast<int>(crank) * 128;
      issue_b2(&tmW2, 0, wrow);
      issue_b2(&tmW2, 128, wrow);
      // then the halo taps, chunk-major: those of chunk c read chunk c of T1_b's halo tiles, which every tile of this
      // image group has stored once the counter watcher passes haloT(c)
      int kh_lo, kh_hi, kw_lo, kw_hi;
      bc_taps(p.dil, h0, p.bh, p.H, kh_lo, kh_hi);
      bc_taps(p.dil, w0, p.bw, p.W, kw_lo, kw_hi);
      const int tnn = n0 + (b & 1) * p.N;
      for (int chunk = 0; chunk < kBcP / 64; ++chunk) {
        mbar_wait(haloT(chunk), static_cast<uint32_t>(b) & 1u);
        bc_fence_async();
        for (int kh = kh_lo; kh <= kh_hi; ++kh)
          for (int kw = kw_lo; kw <= kw_hi; ++kw) {
            if (kh == 1 && kw == 1) continue;
            issue(&tmT, chunk * 64, w0 + (kw - 1) * p.dil, h0 + (kh - 1) * p.dil, tnn, &tmW2, chunk * 64,
                  (b * 9 + kh * 3 + kw) * kBcP + static_cast<int>(crank) * 128);
          }
      }
      // P3: per conv3 N-tile one slot with its four 64-row filter chunks and one slot with the two residual chunks of
      // X_b; per next-conv1 slice one slot with its two filter chunks - in the order the MMA issuer consumes them
      const CUtensorMap* xmap = (b & 1) ? &tmXb : &tmXa;
      const bool next = b + 1 < nb;
      auto c3 = [&](int j) {
        uint32_t dst = acquire(kBcSlotBytes);
        if (elect_one()) {
          const int brow = b * kBcC + j * 128 + static_cast<int>(crank) * 64;
          for (int c = 0; c < 4; ++c) tma_load_2d_2cta(&tmW3, dst + c * 8192u, full_bar(slot), c * 64, brow);
        }
        __syncwarp();
        advance();
        dst = acquire(kBcSlotBytes);
        if (elect_one()) {
          for (int c = 0; c < 2; ++c)
            tma_load_5d_2cta(xmap, dst + c * kBcABytes, full_bar(slot), j * 128 + c * 64, w0, 0, h0, n0);
        }
        __syncwarp();
        advance();
      };
      auto g2 = [&](int j) { issue_b2(&tmW1, j * 128, (b + 1) * kBcP + static_cast<int>(crank) * 128); };
      c3(0);
      for (int j = 1; j < kBcNT; ++j) {
        c3(j);
        if (next) g2(j - 1);
      }
      if (next) g2(kBcNT - 1);
    }
  } else if (warp == 1 && crank == 0) {
    // ===================== MMA issuer (leader CTA) =====================
    uint32_t slot = 0, phase = 0;
    auto advance = [&]() {
      if (++slot == static_cast<uint32_t>(p.slots)) {
        slot = 0;
        phase ^= 1u;
      }
    };
    const uint64_t adesc0 = make_smem_desc_kmajor(smem_base, 128);
    const uint64_t bdesc0 = make_smem_desc_kmajor(smem_base + kBcABytes, 128);
    const uint64_t tdesc0 = make_smem_desc_kmajor(stgT, 128);
    const uint64_t odesc0 = make_smem_desc_kmajor(stgO, 128);
    const uint64_t identdesc = make_smem_desc_kmajor(ident, 128);
    const uint32_t slot_step = kBcSlotBytes >> 4;
    uint32_t use[2] = {0u, 0u};       // uses of the accumulator halves
    auto wait_acc = [&](int h) {
      mbar_wait(tempty_bar(h), (use[h] & 1u) ^ 1u);
      ++use[h];
    };
    // ---- P1 ----
    wait_acc(0);
    wait_acc(1);
    tcgen05_after_thread_sync();
    for (int kb = 0; kb < kBcC / 64; ++kb) {
      mbar_wait(full_bar(slot), phase);
      tcgen05_after_thread_sync();
      if (elect_one()) {
        const uint64_t ad = adesc0 + static_cast<uint64_t>(slot_step * slot);
        const uint64_t bd = bdesc0 + static_cast<uint64_t>(slot_step * slot);
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_f16_2cta(tmem_base, ad + 2u * k, bd + 2u * k, p.idesc256, (kb | k) ? 1u : 0u);
        umma_commit_2cta_mc(empty_bar(slot), 3);
        if (kb == kBcC / 64 - 1) {
          umma_commit_2cta_mc(tfull_bar(0), 3);
          umma_commit_2cta_mc(tfull_bar(1), 3);
        }
      }
      __syncwarp();
      advance();
    }
    for (int b = 0; b < nb; ++b) {
      // ---- P2: conv2 (centre tap from the staged t1 tile, then the halo taps) ----
      int kh_lo, kh_hi, kw_lo, kw_hi;
      bc_taps(p.dil, h0, p.bh, p.H, kh_lo, kh_hi);
      bc_taps(p.dil, w0, p.bw, p.W, kw_lo, kw_hi);
      const int nkb = ((kh_hi - kh_lo + 1) * (kw_hi - kw_lo + 1) - 1) * (kBcP / 64);
      wait_acc(0);
      wait_acc(1);
      tcgen05_after_thread_sync();
      for (int s2 = 0; s2 < 2; ++s2) {
        mbar_wait(s2readyT(2 * s2), 0u);           // t1 chunks (T use 2b: even parity) staged in both CTAs
        mbar_wait(s2readyT(2 * s2 + 1), 0u);
        mbar_wait(full_bar(slot), phase);
        tcgen05_after_thread_sync();
        if (elect_one()) {
          for (int cc = 0; cc < 2; ++cc) {
            const int c = 2 * s2 + cc;
            const uint64_t ad = tdesc0 + static_cast<uint64_t>((kBcBuf >> 4) * c);
            const uint64_t bd = adesc0 + static_cast<uint64_t>(slot_step * slot) + static_cast<uint64_t>((kBcABytes >> 4) * cc);
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_f16_2cta(tmem_base, ad + 2u * k, bd + 2u * k, p.idesc256, (c | k) ? 1u : 0u);
          }
          umma_commit_2cta_mc(empty_bar(slot), 3);
          if (s2 == 0 && b < 3) BC_STAMP(23 + b);
          if (s2 == 1) {
            for (int g = 0; g < 4; ++g) umma_commit_2cta_mc(availT(g), 3);       // t1 tile consumed
            if (nkb == 0) {
              umma_commit_2cta_mc(tfull_bar(0), 3);
              umma_commit_2cta_mc(tfull_bar(1), 3);
            }
          }
        }
        __syncwarp();
        advance();
      }
      // the halo taps, chunk-major (chunk 0's eight taps first): the order the producer loads them in
      for (int kb = 0; kb < nkb; ++kb) {
        mbar_wait(full_bar(slot), phase);
        tcgen05_after_thread_sync();
        if (elect_one()) {
          const uint64_t ad = adesc0 + static_cast<uint64_t>(slot_step * slot);
          const uint64_t bd = bdesc0 + static_cast<uint64_t>(slot_step * slot);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_f16_2cta(tmem_base, ad + 2u * k, bd + 2u * k, p.idesc256, 1u);
          umma_commit_2cta_mc(empty_bar(slot), 3);
          if (kb == 0 && b < 3) BC_STAMP(26 + b);
          if (kb == nkb - 1) {
            umma_commit_2cta_mc(tfull_bar(0), 3);
            umma_commit_2cta_mc(tfull_bar(1), 3);
            if (b < 3) BC_STAMP(5 + b);
          }
        }
        __syncwarp();
        advance();
      }
      // ---- P3 ----
      const bool next = b + 1 < nb;
      auto c3 = [&](int j) {
        const int h = j & 1;
        wait_acc(h);
        tcgen05_after_thread_sync();
        const uint32_t tacc = tmem_base + static_cast<uint32_t>(h) * 128u;
        // slot 1: the four 64-row filter chunks of this N-tile; A = the staged t2 tile
        mbar_wait(full_bar(slot), phase);
        for (int c = 0; c < 4; ++c) {
          // N-tile 0: K-chunk c as soon as t2 group c (T use 2b+1: odd parity) is staged in both CTAs
          if (j == 0) mbar_wait(s2readyT(c), 1u);
          tcgen05_after_thread_sync();
          if (elect_one()) {
            const uint64_t ad = tdesc0 + static_cast<uint64_t>((kBcBuf >> 4) * c);
            const uint64_t bd = adesc0 + static_cast<uint64_t>(slot_step * slot) + static_cast<uint64_t>((8192u >> 4) * c);
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_f16_2cta(tacc, ad + 2u * k, bd + 2u * k, p.idesc128, (c | k) ? 1u : 0u);
            if (c == 3) umma_commit_2cta_mc(empty_bar(slot), 3);
          }
          __syncwarp();
        }
        advance();
        // slot 2: residual  D[:, c*64 .. c*64+63] += X_b tile chunk x I   (exact: products with 1.0)
        mbar_wait(full_bar(slot), phase);
        tcgen05_after_thread_sync();
        if (elect_one()) {
          for (int c = 0; c < 2; ++c) {
            const uint64_t rd = adesc0 + static_cast<uint64_t>(slot_step * slot) + static_cast<uint64_t>((kBcABytes >> 4) * c);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_f16_2cta(tacc + static_cast<uint32_t>(c) * 64u, rd + 2u * k, identdesc + 2u * k, p.idesc_res, 1u);
          }
          umma_commit_2cta_mc(empty_bar(slot), 3);
          umma_commit_2cta_mc(tfull_bar(h), 3);
          if (j == kBcNT - 1)
            for (int g = 0; g < 4; ++g) umma_commit_2cta_mc(availT(g), 3);     // t2 is dead
        }
        __syncwarp();
        advance();
      };
      auto g2 = [&](int j) {
        if (j == 0) {
          mbar_wait(d2empty_bar, (b & 1u) ^ 1u);
          tcgen05_after_thread_sync();
        }
        mbar_wait(full_bar(slot), phase);
        for (int c = 0; c < 2; ++c) {
          // chunk by chunk: the epilogue of the next N-tile may refill a staging buffer as soon as ITS MMAs are done
          mbar_wait(s2readyO(c), j & 1u);
          tcgen05_after_thread_sync();
          if (elect_one()) {
            const uint64_t ad = odesc0 + static_cast<uint64_t>((kBcBuf >> 4) * c);
            const uint64_t bd = adesc0 + static_cast<uint64_t>(slot_step * slot) + static_cast<uint64_t>((kBcABytes >> 4) * c);
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_f16_2cta(tmem_d2, ad + 2u * k, bd + 2u * k, p.idesc256, (j | c | k) ? 1u : 0u);
            umma_commit_2cta_mc(availO(c), 3);
            if (c == 1) {
              umma_commit_2cta_mc(empty_bar(slot), 3);
              if (j == kBcNT - 1) umma_commit_2cta_mc(d2full_bar, 3);
            }
          }
          __syncwarp();
        }
        advance();
      };
      c3(0);
      for (int j = 1; j < kBcNT; ++j) {
        c3(j);
        if (next) g2(j - 1);
      }
      if (next) g2(kBcNT - 1);
      if (b < 3 && lane == 0) BC_STAMP(8 + b);
    }
  } else if (threadIdx.x == 64) {
    // ===================== store thread =====================
    uint32_t nT = 0, nO = 0;
    // group g of T1_{b1} is in global memory: its staging buffer is free (the other arrival: the centre-tap MMAs of
    // conv2) and counter[b1][g] lets the neighbours load its halo
    auto publish = [&](int b1, int g) {
      mbar_arrive(availT(g));
      bc_fence_async();
      __threadfence();
      bc_red_release(ctr + b1 * 4 + g, 1u);
    };
    // T1_{b1} group by group.  Bulk groups complete in order: once the store of group g is complete, so is every
    // store committed before it (the X_{b1} tile among them, which block b1 reads back as its residual)
    auto store_t1 = [&](int b1) {
      for (int g = 0; g < 4; ++g) {
        mbar_wait(readyT(g), nT & 1u);
        tma_store_5d(&tmT, stgT + g * kBcBuf, g * 64, w0, 0, h0, n0 + (b1 & 1) * p.N);
        tma_store_commit();
        if (g > 0) {
          tma_store_wait_all<1>();
          publish(b1, g - 1);
        }
      }
      tma_store_wait_all<0>();
      publish(b1, 3);
      ++nT;
    };
    // P1: T1_0
    store_t1(0);
    for (int b = 0; b < nb; ++b) {
      const bool next = b + 1 < nb;
      // t2 stays on chip: only the bookkeeping arrival (the second one is the MMA commit after the last conv3 tile)
      for (int g = 0; g < 4; ++g) {
        mbar_wait(readyT(g), nT & 1u);
        mbar_arrive(availT(g));
      }
      ++nT;
      const CUtensorMap* omap = (b & 1) ? &tmXa : &tmXb;       // X_{b+1}
      for (int j = 0; j < kBcNT; ++j) {
        for (int g = 0; g < 2; ++g) {
          mbar_wait(readyO(g), nO & 1u);
          tma_store_5d(omap, stgO + g * kBcBuf, j * 128 + g * 64, w0, 0, h0, n0);
          tma_store_commit();
        }
        tma_store_wait_read<0>();
        for (int g = 0; g < 2; ++g) {
          mbar_arrive(availO(g));
          if (!next) mbar_arrive(availO(g));     // no second GEMM reads the last block's output
        }
        ++nO;
      }
      if (next) store_t1(b + 1);
    }
    tma_store_wait_all<0>();
  } else if (threadIdx.x == 96) {
    // ===================== counter watcher =====================
    // acquires counter[b][c] and passes it to the producer through haloT(c), so that the producer's ring feed never
    // waits for a global round trip.  It cannot run a phase ahead: counter[b+1][c] needs this tile's T1_{b+1}, i.e.
    // its conv2 of block b, i.e. the producer past every haloT wait of block b.
    for (int b = 0; b < nb; ++b)
      for (int c = 0; c < 4; ++c) {
        bc_wait_counter(ctr + b * 4 + c, per);
        mbar_arrive(haloT(c));
      }
  } else if (warp >= kBcEpiWarp0) {
    // ===================== epilogue (8 warps) =====================
    const int ew = warp - kBcEpiWarp0;
    const int etid = threadIdx.x - kBcEpiWarp0 * 32;
    const int quarter = ew & 3;
    const int half = ew >> 2;
    const int row = quarter * 32 + lane;
    const uint32_t rowoff = static_cast<uint32_t>(row) * 128u;
    const uint32_t row7 = static_cast<uint32_t>(row) & 7u;
    const uint32_t tlane = static_cast<uint32_t>(quarter * 32) << 16;
    uint32_t nT = 0, nO = 0;
    uint32_t fullpar = 0u;        // bit h: parity of the next tfull_bar(h) phase
    float* const shs = reinterpret_cast<float*>(smem_al + (shf - smem_base));
    auto release = [&](int h) {
      if (lane == 0) {
        if (crank == 0) mbar_arrive(tempty_bar(h));
        else mbar_arrive_remote(tempty_bar(h), 0u);
      }
    };

    // `groups` x 64 accumulator columns from tmem_col0 -> ReLU(acc + shift) -> 16-bit -> staging buffers stg[g].
    // setO: the O set (2 buffers) instead of the T set (4); second: also hand them to the MMA issuer (A operand);
    // release0: hand accumulator half 0 (groups 0-1) back to the MMA issuer as soon as group 1 is in registers.
    // sho: offset of the shifts in the staged table (shared memory: a global load here would put an L2 round trip in
    // front of every 64-column group)
    auto epilogue = [&](uint32_t tmem_col0, int groups, int sho, bool setO, bool second, bool release0) {
      uint32_t r[32];
      const uint32_t taddr = tmem_col0 + tlane + static_cast<uint32_t>(half * 32);
      const uint32_t nuse = setO ? nO : nT;
      tmem_ld_32x32b_x32(taddr, r);
      for (int g = 0; g < groups; ++g) {
        const float4* s4 = reinterpret_cast<const float4*>(shs + sho + g * 64 + half * 32);
        float v[32];
        tmem_ld_wait();
        if (release0 && g == 1) {       // every load of half 0 has completed; the load of group 2 is not issued yet
          tcgen05_before_thread_sync();
          __syncwarp();
          release(0);
        }
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) {
          const float4 h4 = s4[j4];
          v[4 * j4 + 0] = __uint_as_float(r[4 * j4 + 0]) + h4.x;
          v[4 * j4 + 1] = __uint_as_float(r[4 * j4 + 1]) + h4.y;
          v[4 * j4 + 2] = __uint_as_float(r[4 * j4 + 2]) + h4.z;
          v[4 * j4 + 3] = __uint_as_float(r[4 * j4 + 3]) + h4.w;
        }
        if (g + 1 < groups) tmem_ld_32x32b_x32(taddr + (g + 1) * 64, r);
        uint32_t w[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) w[e] = bc_pack2_relu<kFmt>(v[2 * e], v[2 * e + 1]);
        mbar_wait(setO ? availO(g) : availT(g), (nuse & 1u) ^ 1u);
        const uint32_t rowaddr = (setO ? stgO : stgT) + g * kBcBuf + rowoff;
#pragma unroll
        for (int c4 = 0; c4 < 4; ++c4) {
          const uint32_t addr = rowaddr + (((static_cast<uint32_t>(half) * 4u + c4) ^ row7) << 4);
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(w[4 * c4]), "r"(w[4 * c4 + 1]),
                       "r"(w[4 * c4 + 2]), "r"(w[4 * c4 + 3])
                       : "memory");
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(setO ? readyO(g) : readyT(g));
          if (second) {
            const uint32_t sb = setO ? s2readyO(g) : s2readyT(g);
            if (crank == 0) mbar_arrive(sb);
            else mbar_arrive_remote(sb, 0u);
          }
        }
      }
      if (setO) ++nO; else ++nT;
    };
    auto wait_full = [&](int h) {
      mbar_wait(tfull_bar(h), (fullpar >> h) & 1u);
      fullpar ^= 1u << h;
    };
    // The shifts block b's epilogues use: [0,256) shift2[b], [256,1280) shift3[b], [1280,1536) shift1[b+1] (the T1
    // epilogue of the next block); b = -1 stages only shift1[0].  Copied while the epilogue warps wait for conv2, once
    // every epilogue warp is done with the previous block's table.
    auto stage_shifts = [&](int b) {
      asm volatile("bar.sync 1, %0;" ::"n"(kBcEpiThreads) : "memory");
      for (int e = 4 * etid; e < kBcShifts; e += 4 * kBcEpiThreads) {
        const float* src = e < kBcP ? p.shift2 + b * kBcP + e
                           : e < kBcP + kBcC ? p.shift3 + b * kBcC + (e - kBcP)
                                             : p.shift1 + (b + 1) * kBcP + (e - kBcP - kBcC);
        if ((e < kBcP + kBcC && b < 0) || (e >= kBcP + kBcC && b + 1 >= nb)) continue;
        *reinterpret_cast<float4*>(shs + e) = __ldg(reinterpret_cast<const float4*>(src));
      }
      asm volatile("bar.sync 1, %0;" ::"n"(kBcEpiThreads) : "memory");
    };
    // ---- P1: T1_0 = ReLU(bn1(conv1(X_0))) ----
    stage_shifts(-1);
    wait_full(0);
    wait_full(1);
    tcgen05_after_thread_sync();
    epilogue(tmem_base, 4, kBcP + kBcC, false, true, false);
    tcgen05_before_thread_sync();
    __syncwarp();
    release(0);
    release(1);
    for (int b = 0; b < nb; ++b) {
      const bool next = b + 1 < nb;
      stage_shifts(b);
      // ---- P2: t2 (stays on chip); half 0 goes back mid-epilogue, conv3 N-tile 0 writes only there ----
      wait_full(0);
      wait_full(1);
      tcgen05_after_thread_sync();
      epilogue(tmem_base, 4, 0, false, true, true);
      tcgen05_before_thread_sync();
      __syncwarp();
      release(1);
      if (b < 3 && etid == 0) BC_STAMP(11 + b);
      // ---- P3: the block's output, 128 channels at a time ----
      for (int j = 0; j < kBcNT; ++j) {
        const int h = j & 1;
        wait_full(h);
        tcgen05_after_thread_sync();
        epilogue(tmem_base + static_cast<uint32_t>(h) * 128u, 2, kBcP + j * 128, true, next, false);
        tcgen05_before_thread_sync();
        __syncwarp();
        release(h);
      }
      if (b < 3 && etid == 0) BC_STAMP(14 + b);
      if (next) {
        // ---- T1_{b+1} = ReLU(bn1(conv1(X_{b+1}))) from the second accumulator ----
        mbar_wait(d2full_bar, b & 1u);
        tcgen05_after_thread_sync();
        epilogue(tmem_d2, 4, kBcP + kBcC, false, true, false);
        tcgen05_before_thread_sync();
        __syncwarp();
        if (lane == 0) {
          if (crank == 0) mbar_arrive(d2empty_bar);
          else mbar_arrive_remote(d2empty_bar, 0u);
        }
        if (b < 3 && etid == 0) BC_STAMP(17 + b);
      }
    }
  }

  tcgen05_before_thread_sync();
  __syncthreads();
  if (threadIdx.x == 0) BC_STAMP(31);
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
  if (warp == 2) {
    tcgen05_after_thread_sync();
    tmem_dealloc_2cta(tmem_base, 512);
  }
  if (threadIdx.x == 0) {
    const int n_ctr = p.tiles_n * (p.nblocks + 1) * 4;
    __threadfence();
    const unsigned int old = atomicAdd(p.counters + n_ctr, 1u);
    if (old == gridDim.x - 1) {
      for (int i = 0; i <= n_ctr; ++i) p.counters[i] = 0u;
      __threadfence();
    }
  }
}

}  // namespace up
#include "up_conv_host.h"
namespace up {

struct BcPlan {
  int bn, bh, bw, tiles_h, tiles_w, tiles_n, per;
};

static int bc_plan(const UpBneckChainDesc* d, BcPlan& pl) {
  if (!d) return fail(UP_ERR_INVALID, "up_bneck_chain: null descriptor");
  if (d->dtype != UP_FP16 && d->dtype != UP_BF16)
    return fail(UP_ERR_UNSUPPORTED, "up_bneck_chain: fp16 / bf16 only (the fp32-grade split mode runs the layer-wise plan)");
  if (d->n <= 0 || d->h <= 0 || d->w <= 0 || d->nblocks < 1 || d->dil < 1) return fail(UP_ERR_INVALID, "up_bneck_chain: bad dims");
  if (d->planes != kBcP) return fail(UP_ERR_UNSUPPORTED, "up_bneck_chain: planes must be %d (got %d)", kBcP, d->planes);
  pick_tile(d->n, d->h, d->w, pl.bn, pl.bh, pl.bw);
  if (pl.bn > 2) return fail(UP_ERR_UNSUPPORTED, "up_bneck_chain: map %dx%d too small for the fused chain", d->h, d->w);
  pl.tiles_w = (d->w + pl.bw - 1) / pl.bw;
  pl.tiles_h = (d->h + pl.bh - 1) / pl.bh;
  if (d->n % (2 * pl.bn) != 0)
    return fail(UP_ERR_UNSUPPORTED, "up_bneck_chain: batch %d is not a multiple of %d", d->n, 2 * pl.bn);
  pl.tiles_n = d->n / pl.bn;
  pl.per = pl.tiles_h * pl.tiles_w;
  return 0;
}

static unsigned long long* g_bc_dbg = nullptr;

static int bc_max_clusters(DeviceInfo* di) {
  int* cached = di->max_clusters;
  if (cached[1] == 0) {     // slot 1: this kernel
    cudaLaunchConfig_t occ{};
    occ.gridDim = dim3(di->sm_count / 2 * 2);
    occ.blockDim = dim3(kBcThreads);
    occ.dynamicSmemBytes = di->max_smem;
    cudaLaunchAttribute oa[1];
    oa[0].id = cudaLaunchAttributeClusterDimension;
    oa[0].val.clusterDim.x = 2;
    oa[0].val.clusterDim.y = 1;
    oa[0].val.clusterDim.z = 1;
    occ.attrs = oa;
    occ.numAttrs = 1;
    int nc = 0;
    if (cudaOccupancyMaxActiveClusters(&nc, bneck_chain_kernel<0>, &occ) == cudaSuccess && nc > 0) cached[1] = nc;
    else {
      (void)cudaGetLastError();
      cached[1] = di->sm_count / 2;
    }
  }
  return cached[1] < di->sm_count / 2 ? cached[1] : di->sm_count / 2;
}

static int bc_ensure(DeviceInfo*& di) {
  di = device_info();
  if (!di) return UP_ERR_CUDA;
  if (!di->bneck_attr) {
    int rc = check_cuda(cudaFuncSetAttribute(bneck_chain_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             static_cast<int>(di->max_smem)),
                        "cudaFuncSetAttribute(bneck chain)");
    if (rc) return rc;
    rc = check_cuda(cudaFuncSetAttribute(bneck_chain_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         static_cast<int>(di->max_smem)),
                    "cudaFuncSetAttribute(bneck chain bf16)");
    if (rc) return rc;
    di->bneck_attr = true;
  }
  return 0;
}

}  // namespace up

using namespace up;

extern "C" int up_debug_bneck_timing(unsigned long long* h_out) {
  if (!g_bc_dbg) return up::fail(UP_ERR_INVALID, "no timing buffer (set UP_DEBUG_TIMING=1)");
  return up::check_cuda(cudaMemcpy(h_out, g_bc_dbg, 160 * 32 * sizeof(unsigned long long), cudaMemcpyDeviceToHost),
                        "cudaMemcpy(bneck timing)");
}

extern "C" int up_bneck_chain_supported(const UpBneckChainDesc* d) {
  BcPlan pl;
  int rc = bc_plan(d, pl);
  if (rc) return rc;
  DeviceInfo* di = device_info();
  if (di) {
    rc = bc_ensure(di);
    if (rc) return rc;
    if (pl.per * (pl.tiles_n / 2) > bc_max_clusters(di))
      return fail(UP_ERR_UNSUPPORTED, "up_bneck_chain: %d tile pairs exceed the co-resident CTA pairs", pl.per * (pl.tiles_n / 2));
  }
  return 0;
}

extern "C" int64_t up_bneck_chain_workspace_bytes(const UpBneckChainDesc* d) {
  BcPlan pl;
  if (bc_plan(d, pl)) return -1;
  // counters [tiles_n][nblocks + 1][4 chunks] + the exit counter, 4 bytes each
  return ((static_cast<int64_t>(pl.tiles_n) * (d->nblocks + 1) * 4 + 1) * 4 + 255) & ~static_cast<int64_t>(255);
}

extern "C" int up_bneck_chain_fwd(const UpBneckChainDesc* d, const UpBneckChainWeights* w, void* xa, void* xb, void* t1,
                                  void* workspace, int64_t workspace_bytes, void* stream) {
  UP_CHECK_ARG(d && w && xa && xb && t1 && workspace, "up_bneck_chain_fwd: null argument");
  UP_CHECK_ARG(w->w1 && w->w2 && w->w3 && w->shift1 && w->shift2 && w->shift3, "up_bneck_chain_fwd: missing weights");
  BcPlan pl;
  int rc = bc_plan(d, pl);
  if (rc) return rc;
  UP_CHECK_ARG(workspace_bytes >= up_bneck_chain_workspace_bytes(d), "up_bneck_chain_fwd: workspace too small");
  DeviceInfo* di = nullptr;
  rc = bc_ensure(di);
  if (rc) return rc;
  const int clusters = pl.per * (pl.tiles_n / 2);
  UP_CHECK_ARG(clusters <= bc_max_clusters(di), "up_bneck_chain_fwd: %d tile pairs exceed the co-resident CTA pairs", clusters);
  const int fmt = fmt_of_dtype(d->dtype);
  BcParams p{};
  p.N = d->n;
  p.H = d->h;
  p.W = d->w;
  p.bn = pl.bn;
  p.bh = pl.bh;
  p.bw = pl.bw;
  p.tiles_h = pl.tiles_h;
  p.tiles_w = pl.tiles_w;
  p.tiles_n = pl.tiles_n;
  p.nblocks = d->nblocks;
  p.dil = d->dil;
  const size_t fixed = 1024 + 6 * kBcBuf + 8192 + 4 * kBcShifts + 8 * (2 * kBcMaxSlots + 28) + 16;
  int slots = static_cast<int>((di->max_smem - fixed) / kBcSlotBytes);
  if (slots > kBcMaxSlots) slots = kBcMaxSlots;
  UP_CHECK_ARG(slots >= 2, "up_bneck_chain_fwd: not enough shared memory");
  p.slots = slots;
  p.idesc256 = make_idesc_f16(static_cast<uint32_t>(fmt), 256u, 256u);
  p.idesc128 = make_idesc_f16(static_cast<uint32_t>(fmt), 256u, 128u);
  p.idesc_res = make_idesc_f16(static_cast<uint32_t>(fmt), 256u, 64u);
  p.shift1 = w->shift1;
  p.shift2 = w->shift2;
  p.shift3 = w->shift3;
  p.counters = static_cast<unsigned int*>(workspace);
  p.fmt = fmt;
  p.dbg = nullptr;
  if (getenv("UP_DEBUG_TIMING")) {
    if (!g_bc_dbg) cudaMalloc(&g_bc_dbg, 160 * 32 * sizeof(unsigned long long));
    cudaMemsetAsync(g_bc_dbg, 0, 160 * 32 * sizeof(unsigned long long), static_cast<cudaStream_t>(stream));
    p.dbg = g_bc_dbg;
  }
  CUtensorMap tmXa, tmXb, tmT, tmW1, tmW2, tmW3;
  const uint32_t abox[5] = {64u, static_cast<uint32_t>(pl.bw), 1u, static_cast<uint32_t>(pl.bh),
                            static_cast<uint32_t>(pl.bn)};
  rc = encode_act_map(&tmXa, fmt, xa, d->n, d->h, d->w, kBcC, 1, abox, 128, "bneck.xa");
  if (rc) return rc;
  rc = encode_act_map(&tmXb, fmt, xb, d->n, d->h, d->w, kBcC, 1, abox, 128, "bneck.xb");
  if (rc) return rc;
  rc = encode_act_map(&tmT, fmt, t1, 2 * d->n, d->h, d->w, kBcP, 1, abox, 128, "bneck.t1");
  if (rc) return rc;
  {
    const uint64_t dims[2] = {kBcC, static_cast<uint64_t>(d->nblocks) * kBcP};
    const uint64_t st[1] = {kBcC * 2};
    const uint32_t box[2] = {64u, 128u};
    rc = encode_map(&tmW1, fmt, 2, w->w1, dims, st, box, 128, "bneck.w1");
    if (rc) return rc;
  }
  {
    const uint64_t dims[2] = {kBcP, static_cast<uint64_t>(d->nblocks) * 9 * kBcP};
    const uint64_t st[1] = {kBcP * 2};
    const uint32_t box[2] = {64u, 128u};
    rc = encode_map(&tmW2, fmt, 2, w->w2, dims, st, box, 128, "bneck.w2");
    if (rc) return rc;
  }
  {
    const uint64_t dims[2] = {kBcP, static_cast<uint64_t>(d->nblocks) * kBcC};
    const uint64_t st[1] = {kBcP * 2};
    const uint32_t box[2] = {64u, 64u};
    rc = encode_map(&tmW3, fmt, 2, w->w3, dims, st, box, 128, "bneck.w3");
    if (rc) return rc;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(2 * clusters);
  cfg.blockDim = dim3(kBcThreads);
  cfg.dynamicSmemBytes = fixed + static_cast<size_t>(slots) * kBcSlotBytes;
  cfg.stream = static_cast<cudaStream_t>(stream);
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  rc = check_cuda(fmt == 0 ? cudaLaunchKernelEx(&cfg, bneck_chain_kernel<0>, tmXa, tmXb, tmT, tmW1, tmW2, tmW3, p)
                           : cudaLaunchKernelEx(&cfg, bneck_chain_kernel<1>, tmXa, tmXb, tmT, tmW1, tmW2, tmW3, p),
                  "bneck_chain_kernel launch");
  return rc;
}
