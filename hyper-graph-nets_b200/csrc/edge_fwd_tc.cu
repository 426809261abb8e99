// bf16 tcgen05 forward of the projected edge update (HGN_BF16 only):
//     e' = e + LN( W2 relu( W1 relu( We e + Ps[s] + Pr[r] + b0 ) + b1 ) + b2 )          (src/migration/graphnet.py:22-32)
// with Ps = v Ws^T, Pr = v Wr^T precomputed per node (edge_tc.cu).  Also used for the node update in 'sum' mode
// (graphnet.py:34-48) with e := v, Ps := agg Wagg^T gathered through the identity (senders == nullptr) and no Pr.
//
// Persistent, one CTA per SM, two 128-row tiles in flight:
//   warp 17     loader (lane 0 = TMA thread; all lanes: gather indices -> shared-memory ring, table rows -> L2 prefetch): cp.async.bulk.tensor loads of the [128 x 128] bf16 edge tile (two 128B-swizzled panels) into a
//               3-stage ring; after the epilogue has turned a stage into the OUTPUT tile in place (residual add), the same
//               thread stores it with cp.async.bulk.tensor and recycles the stage once the store has read it
//   warp 16     MMA issuer: per tile  GEMM0 = e We^T (A from the stage, SS), GEMM1 = H1 W1^T, GEMM2 = H2 W2^T (A = bf16
//               activations in TMEM, TS); the steps of the two tiles in flight are interleaved so that the tensor pipe works
//               on one tile while the other is in its epilogue
//   warps 0-7 / 8-15  epilogue sets (even / odd tiles): row = TMEM lane, each thread owns 64 of a row's 128 columns.
//               P0: + table rows + b0, ReLU -> bf16 -> TMEM;  P1: + b1, ReLU -> TMEM;  P2: + b2, LayerNorm (row statistics
//               merged between the two half-row threads through shared memory), affine, + e from the stage -> stage.
// TMEM: tile slot s -> accumulator [256 s, +128), bf16 A operand [256 s + 128, +64).
// Shared memory: We, W1, W2 resident (96 KiB) + 3 stages (96 KiB) + parameters + LayerNorm exchange = 203 KiB; the
// remaining ~24 KiB of the SM's unified array serve as L1 for the gathered table rows.
#include <cuda.h>
#include <stdlib.h>

#include "tile_common.cuh"

namespace hgn {

constexpr int kEfSetThreads = 256;
constexpr int kEfThreads = 2 * kEfSetThreads + 64;     // 18 warps (17-20 warps: at most 96 registers per thread)
constexpr int kEfStages = 3;
constexpr uint32_t kEfWe = 0, kEfW1 = kChunkBytes, kEfW2 = 2 * kChunkBytes, kEfStage = 3 * kChunkBytes;
constexpr uint32_t kEfParams = kEfStage + kEfStages * kChunkBytes;     // b0 b1 b2 gamma beta (fp32 x 128 each)
constexpr uint32_t kEfXch = kEfParams + 5 * kD * 4;                    // float2 [set][tile parity][half][128]
constexpr int kEfRing = 8;                             // tiles of gather indices kept in shared memory (> lookahead + tiles in flight)
constexpr uint32_t kEfIdx = kEfXch + 2 * 2 * 2 * kTile * 8;              // int32 [ring][2][128]: table row of every tile row
constexpr uint32_t kEfBars = kEfIdx + kEfRing * 2 * kTile * 4;
constexpr uint32_t kEfSmem = kEfBars + 128;
enum { kEfFull = 0, kEfOut = 3, kEfAcc = 6, kEfEpi = 8, kEfTmem = 10, kEfIdxDone = 12 };

struct EdgeFwdArgs {
  const __nv_bfloat16 *proj_s, *proj_r;     // per-node tables; proj_r may be null
  const int32_t *senders, *receivers;       // null = identity (row i gathers table row i)
  int w0_chunks, w0_chunk0;                 // W0 is [128][128 w0_chunks]; the dense input multiplies chunk w0_chunk0
  long long* timeline;                      // development (HGN_TC_ABLATE bit 64): clock64 stamps of block 0, [tile][32]
};

__global__ void __launch_bounds__(kEfThreads, 1)
edge_fwd_tc_kernel(int64_t rows, int64_t num_tiles, const uint8_t* __restrict__ packed, EdgeFwdArgs a,
                   const __grid_constant__ CUtensorMap tm_in, const __grid_constant__ CUtensorMap tm_out) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  if ((sbase & 1023u) != 0) __trap();
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kEfBars);
  float* prm = reinterpret_cast<float*>(smem + kEfParams);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const PackedTc P(a.w0_chunks);
  {
    const float* pg = reinterpret_cast<const float*>(packed + P.params);
    for (int i = tid; i < 5 * kD; i += kEfThreads) prm[i] = pg[i];
    const __nv_bfloat16* w0g = reinterpret_cast<const __nv_bfloat16*>(packed + P.w0);
    load_weight_block(sbase + kEfWe, w0g + a.w0_chunk0 * kD, int64_t(a.w0_chunks) * kD, tid, kEfThreads);
    load_weight_block(sbase + kEfW1, reinterpret_cast<const __nv_bfloat16*>(packed + P.w1), kD, tid, kEfThreads);
    load_weight_block(sbase + kEfW2, reinterpret_cast<const __nv_bfloat16*>(packed + P.w2), kD, tid, kEfThreads);
    cp_async_commit();
    if (tid == 0) {
      for (int s = 0; s < kEfStages; ++s) mbar_init(&bars[kEfFull + s], 1);
      for (int s = 0; s < 2; ++s) { mbar_init(&bars[kEfAcc + s], 1); mbar_init(&bars[kEfEpi + s], kEfSetThreads); mbar_init(&bars[kEfOut + s], kEfSetThreads); }
      *reinterpret_cast<volatile int*>(&bars[kEfIdxDone]) = 0;
      mbar_init_fence();
    }
    if (warp == 16) tmem_alloc<512>(reinterpret_cast<uint32_t*>(&bars[kEfTmem]));
    if (warp == 17 && lane == 0) { tma_prefetch_desc(&tm_in); tma_prefetch_desc(&tm_out); }
    cp_async_wait<0>();
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
  }
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(&bars[kEfTmem]);
  const int64_t my_tiles = (num_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x;
  auto stage_addr = [&](int64_t it) -> uint32_t { return sbase + kEfStage + uint32_t(it % kEfStages) * kChunkBytes; };
  auto tile_row0 = [&](int64_t it) -> int64_t { return (blockIdx.x + it * gridDim.x) * kTile; };
  auto stamp = [&](int64_t it, int slot) { if (a.timeline != nullptr && blockIdx.x == 0 && it < 12) a.timeline[it * 32 + slot] = clock64(); };

  if (warp == 17) {
    // =============================== loader warp ==========================================================
    // Per tile: (lane 0) TMA load of the edge tile into its ring stage as soon as the stage is free; (all lanes) the tile's
    // gather indices, read one tile ahead, are published in a shared-memory ring for the epilogue threads (an index held in
    // a register across a tile gets spilled, and the spill store waits for the load) and the table rows they name are
    // pulled into L2 with fire-and-forget prefetches, two to three tiles before the epilogue gathers them.
    auto pf = [](const void* p) { asm volatile("prefetch.global.L2 [%0];" :: "l"(p)); };
    int32_t* ring = reinterpret_cast<int32_t*>(smem + kEfIdx);
    int32_t cs[4], cr[4], ns[4], nr[4];
    auto fetch = [&](int64_t i, int32_t (&s4)[4], int32_t (&r4)[4]) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int64_t grow = tile_row0(i) + lane + 32 * j;
        const bool ok = i < my_tiles && grow < rows;
        s4[j] = ok ? (a.senders != nullptr ? __ldg(a.senders + grow) : int32_t(grow)) : 0;
        r4[j] = ok ? (a.receivers != nullptr ? __ldg(a.receivers + grow) : int32_t(grow)) : 0;
      }
    };
    fetch(0, cs, cr);
    for (int64_t i = 0; i < my_tiles + kEfStages; ++i) {
      if (i >= kEfStages) {                       // tile j sits finished in the stage tile i wants: store it, then reuse
        const int64_t j = i - kEfStages;
        mbar_wait(&bars[kEfOut + int(j & 1)], uint32_t(j >> 1) & 1, 30);
        if (lane == 0) {
          stamp(j, 20);
          const uint32_t src = stage_addr(j);
          const int y = int(tile_row0(j));
          tma_store_2d(&tm_out, src, 0, y);
          tma_store_2d(&tm_out, src + kPanel, 64, y);
          tma_store_commit();
          tma_store_wait_read<0>();
          stamp(j, 21);
        }
        __syncwarp();
      }
      if (i >= my_tiles) continue;
      if (lane == 0) {
        const int st = int(i % kEfStages);
        const uint32_t dst = stage_addr(i);
        const int y = int(tile_row0(i));
        stamp(i, 22);
        mbar_expect_tx(&bars[kEfFull + st], kChunkBytes);
        tma_load_2d(dst, &tm_in, 0, y, &bars[kEfFull + st]);
        tma_load_2d(dst + kPanel, &tm_in, 64, y, &bars[kEfFull + st]);
      }
      fetch(i + 1, ns, nr);
      int32_t* slot = ring + int(i % kEfRing) * 2 * kTile;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        slot[lane + 32 * j] = cs[j];
        slot[kTile + lane + 32 * j] = cr[j];
        pf(a.proj_s + int64_t(cs[j]) * kD); pf(a.proj_s + int64_t(cs[j]) * kD + 64);
        if (a.proj_r != nullptr) { pf(a.proj_r + int64_t(cr[j]) * kD); pf(a.proj_r + int64_t(cr[j]) * kD + 64); }
      }
      __syncwarp();
      if (lane == 0) {
        __threadfence_block();
        *reinterpret_cast<volatile int*>(&bars[kEfIdxDone]) = int(i + 1);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) { cs[j] = ns[j]; cr[j] = nr[j]; }
    }
    if (lane == 0) tma_store_wait<0>();
  } else if (warp == 16) {
    // =============================== MMA issuer =========================================================
    if (lane == 0) {
      const uint32_t idesc = make_idesc_bf16(128, 128, 0, 0);
      uint32_t epi_phase[2] = {0, 0};
      auto gemm_ts = [&](int s, uint32_t b_addr) {       // acc_s = A_s (TMEM, bf16) * B^T
        const uint32_t acc = tmem_base + s * 256, aop = acc + 128;
#pragma unroll
        for (int ks = 0; ks < 8; ++ks) mma_ts(acc, aop + ks * 8, sdesc_kmajor(b_addr + (ks >> 2) * kPanel + (ks & 3) * 32), idesc, ks != 0);
        mma_commit(&bars[kEfAcc + s]);
      };
      // Event driven: each slot (tiles s, s + 2, ...) advances through GEMM0 / GEMM1 / GEMM2 as soon as ITS inputs are ready
      // (stage loaded and accumulator drained / previous phase's activations written), so a slot waiting for a tile load
      // never holds the other one back -- a fixed issue order locks the two slots into step and halves the prefetch lead.
      int64_t slot_tile[2] = {0, 1};
      int slot_step[2] = {0, 0};
      uint32_t idle = 0;
      while (slot_tile[0] < my_tiles || slot_tile[1] < my_tiles) {
        bool progressed = false;
#pragma unroll
        for (int s = 0; s < 2; ++s) {
          const int64_t it = slot_tile[s];
          if (it >= my_tiles) continue;
          const int k = slot_step[s];
          const bool need_epi = k > 0 || it >= 2;
          if (need_epi && !mbar_test(&bars[kEfEpi + s], epi_phase[s] & 1)) continue;
          if (k == 0 && !mbar_test(&bars[kEfFull + int(it % kEfStages)], uint32_t(it / kEfStages) & 1)) continue;
          if (need_epi) ++epi_phase[s];
          fence_after_sync();
          if (k == 0) {
            stamp(it, 1);
            const uint32_t acc = tmem_base + s * 256, a_addr = stage_addr(it), b_addr = sbase + kEfWe;
#pragma unroll
            for (int ks = 0; ks < 8; ++ks) {
              const uint32_t koff = (ks >> 2) * kPanel + (ks & 3) * 32;
              mma_ss(acc, sdesc_kmajor(a_addr + koff), sdesc_kmajor(b_addr + koff), idesc, ks != 0);
            }
            mma_commit(&bars[kEfAcc + s]);
          } else {
            stamp(it, 1 + k);
            gemm_ts(s, k == 1 ? sbase + kEfW1 : sbase + kEfW2);
          }
          if (++slot_step[s] == 3) { slot_step[s] = 0; slot_tile[s] += 2; }
          progressed = true;
        }
        if (progressed) idle = 0;
        else if (++idle > (1u << 24)) { debug_record(36, uint32_t(slot_tile[0]), uint32_t(slot_tile[1]), uint32_t(slot_step[0]), uint32_t(slot_step[1]), epi_phase[0], epi_phase[1]); __trap(); }
      }
    }
  } else {
    // =============================== epilogue sets ========================================================
    const int set = warp >> 3, q = warp & 3, hh = (warp >> 2) & 1;
    const int r = q * 32 + lane;
    const uint32_t lane_addr = uint32_t(q * 32) << 16;
    const uint32_t acc = tmem_base + lane_addr + set * 256 + hh * 64;
    const uint32_t aop = tmem_base + lane_addr + set * 256 + 128 + hh * 32;
    const float2 *b0 = reinterpret_cast<const float2*>(prm + hh * 64), *b1 = reinterpret_cast<const float2*>(prm + kD + hh * 64),
                 *b2 = reinterpret_cast<const float2*>(prm + 2 * kD + hh * 64), *gam = reinterpret_cast<const float2*>(prm + 3 * kD + hh * 64),
                 *bet = reinterpret_cast<const float2*>(prm + 4 * kD + hh * 64);
    float2* xch_base = reinterpret_cast<float2*>(smem + kEfXch) + set * 4 * kTile;
    const int pair_bar = 1 + set * 4 + q;                     // named barrier of the two warps that share rows 32 q ..
    uint32_t acc_phase = 0;
    auto wait_acc = [&](int tag) {
      mbar_wait(&bars[kEfAcc + set], acc_phase++ & 1, tag);
      fence_after_sync();
    };
    const int32_t* ring = reinterpret_cast<const int32_t*>(smem + kEfIdx);
    for (int64_t it = set; it < my_tiles; it += 2) {
      // table rows of this tile, in four blocks of 16 columns: two blocks are requested before the accumulator wait, the other
      // two while the first ones are consumed (64 table registers at once would spill); the row indices come from the prefetch warp's ring
      for (uint32_t spin = 0; *reinterpret_cast<volatile int*>(&bars[kEfIdxDone]) <= int(it); ++spin)
        if (spin > (1u << 26)) { debug_record(35, uint32_t(it), 0, 0, 0, 0, 0); __trap(); }
      __threadfence_block();
      const int32_t* slot = ring + int(it % kEfRing) * 2 * kTile;
      const __nv_bfloat16* psrow = a.proj_s + int64_t(slot[r]) * kD + hh * 64;
      const __nv_bfloat16* prrow = a.proj_r != nullptr ? a.proj_r + int64_t(slot[kTile + r]) * kD + hh * 64 : nullptr;
      uint32_t pa[2][8], pb[2][8];              // Ps / Pr words of the blocks in flight (ring of two)
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        ldg256_l1(psrow + 16 * k, pa[k]);
        if (prrow != nullptr) ldg256_l1(prrow + 16 * k, pb[k]);
        else {
#pragma unroll
          for (int j = 0; j < 8; ++j) pb[k][j] = 0u;
        }
      }
      // ---- P0: H1 = relu(e We^T + Ps[s] + Pr[r] + b0) -> TMEM ------------------------------------------------
      if ((tid & 255) == 0) stamp(it, 8);
      wait_acc(100);
      if ((tid & 255) == 0) stamp(it, 9);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        uint32_t v[16], h[8];
        tmem_ld16(acc + k * 16, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float2 x = make_float2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
          x = __fadd2_rn(x, unpack_bf16x2(pa[k & 1][j]));
          x = __fadd2_rn(x, unpack_bf16x2(pb[k & 1][j]));
          x = __fadd2_rn(x, b0[k * 8 + j]);
          h[j] = cvt_relu_bf16x2(x.x, x.y);
        }
        if (k < 2) {                            // refill the ring slot just consumed with block k + 2
          ldg256_l1(psrow + 16 * (k + 2), pa[k & 1]);
          if (prrow != nullptr) ldg256_l1(prrow + 16 * (k + 2), pb[k & 1]);
        }
        tmem_st8(aop + k * 8, h);
      }
      tmem_st_wait();
      fence_before_sync();
      mbar_arrive(&bars[kEfEpi + set]);
      // ---- P1: H2 = relu(H1 W1^T + b1) -> TMEM ------------------------------------------------------------------
      if ((tid & 255) == 0) stamp(it, 10);
      wait_acc(101);
      if ((tid & 255) == 0) stamp(it, 11);
#pragma unroll
      for (int cg = 0; cg < 2; ++cg) {
        uint32_t v[32], h[16];
        tmem_ld32(acc + cg * 32, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const float2 x = __fadd2_rn(make_float2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1])), b1[cg * 16 + j]);
          h[j] = cvt_relu_bf16x2(x.x, x.y);
        }
        tmem_st8(aop + cg * 16, h);
        tmem_st8(aop + cg * 16 + 8, h + 8);
      }
      tmem_st_wait();
      fence_before_sync();
      mbar_arrive(&bars[kEfEpi + set]);
      // ---- P2: y = H2 W2^T + b2 ; e' = e + LN(y) gamma + beta, written over e in the stage ------------------------------
      if ((tid & 255) == 0) stamp(it, 12);
      wait_acc(102);
      if ((tid & 255) == 0) stamp(it, 13);
      float2 y[32];
      {
        uint32_t v[32];
        tmem_ld32(acc, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) y[j] = __fadd2_rn(make_float2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1])), b2[j]);
        tmem_ld32(acc + 32, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) y[16 + j] = __fadd2_rn(make_float2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1])), b2[16 + j]);
      }
      fence_before_sync();
      mbar_arrive(&bars[kEfEpi + set]);                       // accumulator drained: the slot's next tile may start
      // statistics of my 64 columns (shifted by the first value), merged with the other half of the row (Chan's update)
      const float c0 = y[0].x;
      const float2 nc = make_float2(-c0, -c0);
      float2 s1a = make_float2(0.f, 0.f), s1b = s1a, s2a = s1a, s2b = s1a;
#pragma unroll
      for (int j = 0; j < 32; j += 2) {
        const float2 d0 = __fadd2_rn(y[j], nc), d1 = __fadd2_rn(y[j + 1], nc);
        s1a = __fadd2_rn(s1a, d0); s1b = __fadd2_rn(s1b, d1);
        s2a = __ffma2_rn(d0, d0, s2a); s2b = __ffma2_rn(d1, d1, s2b);
      }
      const float s1 = (s1a.x + s1a.y) + (s1b.x + s1b.y), s2 = (s2a.x + s2a.y) + (s2b.x + s2b.y);
      const float mean_h = c0 + s1 * (1.0f / 64.0f);
      const float m2h = s2 - s1 * s1 * (1.0f / 64.0f);
      float2* xch = xch_base + int((it >> 1) & 1) * 2 * kTile;
      xch[hh * kTile + r] = make_float2(mean_h, m2h);
      asm volatile("bar.sync %0, 64;" :: "r"(pair_bar) : "memory");
      const float2 oth = xch[(1 - hh) * kTile + r];
      const float mean = 0.5f * (mean_h + oth.x);
      const float dm = mean_h - oth.x;
      const float rstd = rsqrtf(fmaxf(m2h + oth.y + 32.0f * dm * dm, 0.f) * (1.0f / kD) + kEps);
      const float2 rs2 = make_float2(rstd, rstd), nm2 = make_float2(-mean * rstd, -mean * rstd);
      // the TMA bytes of this tile's stage were observed by the MMA thread; observe the same barrier phase here before
      // the generic-proxy reads of e
      mbar_wait(&bars[kEfFull + int(it % kEfStages)], uint32_t(it / kEfStages) & 1, 103);
      const uint32_t erow = stage_addr(it) + hh * kPanel;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        uint32_t ew[4], ow[4];
        const uint32_t addr = erow + sw128_chunk(r, k);
        ld_shared128(addr, ew);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 yh = __ffma2_rn(y[4 * k + j], rs2, nm2);
          const float2 o = __fadd2_rn(__ffma2_rn(yh, gam[4 * k + j], bet[4 * k + j]), unpack_bf16x2(ew[j]));
          ow[j] = pack_bf16(o.x, o.y);
        }
        st_shared128(addr, ow);
      }
      fence_async_smem();                                     // generic-proxy writes -> visible to the TMA store
      mbar_arrive(&bars[kEfOut + set]);
      if ((tid & 255) == 0) stamp(it, 14);
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 16) tmem_dealloc<512>(tmem_base);
}

// ---- host side -----------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

typedef CUresult (*CtxGetCurrentFn)(CUcontext*);

// cuTensorMapEncodeTiled needs a current context on the calling thread.  The runtime binds the device's primary context to a thread
// lazily, at the thread's first runtime call that needs one; a thread whose first call into the library encodes a map (e.g. the
// autograd engine's device thread starting a backward with a node update) has none yet, and the encode fails with
// CUDA_ERROR_INVALID_CONTEXT.  cudaSetDevice binds the primary context of the thread's current device.
static int ensure_current_context() {
  static CtxGetCurrentFn get = nullptr;
  if (get == nullptr) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    HGN_CUDA_OK(cudaGetDriverEntryPoint("cuCtxGetCurrent", &p, cudaEnableDefault, &qres));
    if (p == nullptr || qres != cudaDriverEntryPointSuccess) { set_error("cuCtxGetCurrent is not available from this driver"); return HGN_ERR_CUDA; }
    get = reinterpret_cast<CtxGetCurrentFn>(p);
  }
  CUcontext ctx = nullptr;
  if (get(&ctx) == CUDA_SUCCESS && ctx != nullptr) return HGN_OK;
  int dev = 0;
  HGN_CUDA_OK(cudaGetDevice(&dev));
  HGN_CUDA_OK(cudaSetDevice(dev));
  return HGN_OK;
}

// [rows][128] bf16 row-major tensor, boxes of 128 rows x 64 columns (one 128B-swizzled operand panel)
int make_rows_tensor_map(CUtensorMap* tm, const void* base, int64_t rows) {
  if (int rc = ensure_current_context()) return rc;
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    HGN_CUDA_OK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres));
    if (p == nullptr || qres != cudaDriverEntryPointSuccess) { set_error("cuTensorMapEncodeTiled is not available from this driver"); return HGN_ERR_CUDA; }
    fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  const cuuint64_t gdim[2] = {cuuint64_t(kD), cuuint64_t(rows)};
  const cuuint64_t gstride[1] = {cuuint64_t(kD) * 2};
  const cuuint32_t box[2] = {64, cuuint32_t(kTile)};
  const cuuint32_t estride[2] = {1, 1};
  const CUresult rc = fn(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estride, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (rc != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed with %d (base %p, rows %lld)", int(rc), base, (long long)rows); return HGN_ERR_CUDA; }
  return HGN_OK;
}

int edge_fwd_tc_launch(int64_t rows, const void* dense, const void* proj_s, const void* proj_r, const int32_t* senders, const int32_t* receivers,
                       const void* packed, int w0_chunks, int w0_chunk0, void* out, const char* name, cudaStream_t st) {
  static bool configured = false;
  if (!configured) {
    uint32_t* dbg = debug_buffer_device();
    HGN_CUDA_OK(cudaMemcpyToSymbol(tc05::g_debug_words, &dbg, sizeof(dbg)));
    HGN_CUDA_OK(cudaFuncSetAttribute(edge_fwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kEfSmem)));
    configured = true;
  }
  if (rows <= 0) return HGN_OK;
  CUtensorMap tm_in, tm_out;
  if (int rc = make_rows_tensor_map(&tm_in, dense, rows)) return rc;
  if (int rc = make_rows_tensor_map(&tm_out, out, rows)) return rc;
  EdgeFwdArgs a{};
  a.proj_s = static_cast<const __nv_bfloat16*>(proj_s);
  a.proj_r = static_cast<const __nv_bfloat16*>(proj_r);
  a.senders = senders;
  a.receivers = receivers;
  a.w0_chunks = w0_chunks;
  a.w0_chunk0 = w0_chunk0;
  const int64_t tiles = ceil_div(rows, kTile);
  const unsigned grid = unsigned(tiles < tc_sm_count() ? tiles : tc_sm_count());
  static long long* tl_dev = nullptr;
  { const char* ab = getenv("HGN_TC_ABLATE"); if (ab != nullptr && (atoi(ab) & 64)) {
      if (tl_dev == nullptr) cudaMalloc(&tl_dev, 12 * 32 * sizeof(long long));
      cudaMemsetAsync(tl_dev, 0, 12 * 32 * sizeof(long long), st);
      a.timeline = tl_dev;
  } }
  {
    HGN_TIMED(name, st);
    edge_fwd_tc_kernel<<<grid, kEfThreads, kEfSmem, st>>>(rows, tiles, static_cast<const uint8_t*>(packed), a, tm_in, tm_out);
  }
  HGN_LAUNCH_OK(name);
  if (a.timeline != nullptr) {
    long long h[12 * 32];
    cudaMemcpyAsync(h, a.timeline, sizeof(h), cudaMemcpyDeviceToHost, st);
    cudaStreamSynchronize(st);
    for (int t = 0; t < 12; ++t) {
      fprintf(stderr, "fwd tile %d:", t);
      for (int k = 0; k < 24; ++k) fprintf(stderr, " %lld", h[t * 32 + k] ? h[t * 32 + k] - h[1] : -1);
      fprintf(stderr, "\n");
    }
  }
  return HGN_OK;
}

}  // namespace hgn
