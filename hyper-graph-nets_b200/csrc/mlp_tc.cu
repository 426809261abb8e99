// bf16 tcgen05 path of the fused "MLP tile" (HGN_BF16): gather + 3-layer MLP + LayerNorm + residual,
// its data-gradient pass (activations recomputed) and the weight-gradient GEMMs.
//
// Tile kernel (forward / backward share one skeleton; persistent, one CTA per SM, 13 warps):
//   warps 8-11  producers  : cp.async gather of 128-row x 128-col bf16 chunks (sender rows, receiver
//                            rows, edge rows / node rows, aggregates) into a 2-stage ring of
//                            128B-swizzled K-major operand panels (+ the matching W0 panel pair when
//                            W0 has more than 3 chunks and is streamed instead of resident)
//   warp 12     MMA issuer : one thread issues tcgen05.mma (M=128, N=128, K=16, cta_group::1);
//                            layer 0 = one K=128 accumulation per chunk, so the [rows,128*n] concat
//                            never exists; every later GEMM takes its A operand (H1, H2, dY, dH2', dH1')
//                            straight from TMEM; the dgrad GEMMs read the SAME resident weight panels
//                            as MN-major B operands (no transposed weight copies)
//   warps 0-3 / 4-7 epilogue groups, one per accumulator slot: tcgen05.ld -> bias + ReLU -> bf16 ->
//                            tcgen05.st (next A operand); LayerNorm forward/backward are thread-local
//                            (row = TMEM lane = thread).
// Two tiles are in flight (TMEM slots 0/1), so the tensor pipe works on one tile while the epilogue
// warps drain the other.  TMEM: slot s -> accumulator [256s, 256s+128), bf16 A operand [256s+128, +64).
// Shared memory: W1, W2 (and W0 when <= 3 chunks) resident as SW128 panels; 2 stages.
//
// Weight-gradient kernel: dW = G^T Z as tcgen05 GEMMs with BOTH operands MN-major, i.e. the row-major
// [rows,128] activation / gradient tiles are consumed exactly as they sit in memory; accumulators stay in
// TMEM over a CTA's whole row range; per-CTA partials are reduced in a fixed order afterwards.
#include <stdlib.h>

#include "tile_common.cuh"

namespace hgn {

__global__ void pack_tc_kernel(int n_chunks, const float* W0, const float* b0, const float* W1, const float* b1, const float* W2,
                               const float* b2, const float* gamma, const float* beta, uint8_t* packed) {
  const PackedTc L(n_chunks);
  const int64_t k0 = int64_t(n_chunks) * kD;
  const int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  __nv_bfloat16* w0 = reinterpret_cast<__nv_bfloat16*>(packed + L.w0);
  __nv_bfloat16* w1 = reinterpret_cast<__nv_bfloat16*>(packed + L.w1);
  __nv_bfloat16* w2 = reinterpret_cast<__nv_bfloat16*>(packed + L.w2);
  float* p = reinterpret_cast<float*>(packed + L.params);
  if (i < k0 * kD) w0[i] = __float2bfloat16_rn(W0[i]);
  if (i < kD * kD) { w1[i] = __float2bfloat16_rn(W1[i]); w2[i] = __float2bfloat16_rn(W2[i]); }
  if (i < kD) { p[i] = b0[i]; p[kD + i] = b1[i]; p[2 * kD + i] = b2[i]; p[3 * kD + i] = gamma[i]; p[4 * kD + i] = beta[i]; }
}

// ---- shared-memory map of the tile kernel ------------------------------------------------------------
struct TileSmem {
  int w0_panels;          // 2*n_chunks when resident else 0
  uint32_t w0, w1, w2, stages, w0b, params, bars, total;
  int stage_bytes;
  __host__ __device__ TileSmem(int n_chunks, bool resident, bool bwd) {
    w0_panels = resident ? 2 * n_chunks : 0;
    stage_bytes = resident ? kChunkBytes : 2 * kChunkBytes;
    uint32_t o = 0;
    w0 = o; o += uint32_t(w0_panels) * kPanel;
    w1 = o; o += 2 * kPanel;
    w2 = o; o += 2 * kPanel;
    stages = o; o += uint32_t(kStages) * stage_bytes;
    w0b = o; o += (!resident && bwd) ? kChunkBytes : 0;     // streamed W0: panel pair for the dX GEMMs
    params = o; o += 5 * kD * 4;
    bars = o; o += 128;
    total = o;
  }
};
// mbarrier slots (uint64 each) inside the 128-byte barrier block
// (16 slots).  kBarAcc + (tile % 6): tile i uses accumulator i%3 and epilogue group i%2, so each of the six
// barriers has ONE waiting group that consumes its phases in program order.  kBarEpi: "step drained, next A
// operand written"; kBarDone: "tile finished, accumulator free" -- split because a group can publish the first
// step of its next tile before the MMA warp has looked at the previous tile's last signal; on one barrier that
// would put it two phases ahead and the parity test could no longer tell them apart.
enum { kBarFull = 0, kBarEmpty = 2, kBarAcc = 4, kBarEpi = 10, kBarDone = 12, kBarTmemPtr = 14, kBarW0b = 15 };
constexpr int kAccSlots = 3;                    // TMEM accumulators [0,128) [128,256) [256,384)
constexpr uint32_t kAopCol = 384;               // bf16 A operands of the two epilogue groups: [384,448) [448,512)

struct BwdArgs {
  const __nv_bfloat16* grad_out;
  __nv_bfloat16* grad_chunk[HGN_MAX_CHUNKS];
  __nv_bfloat16 *H1, *H2, *P, *G2, *G1, *G0;   // slab workspaces [rows,128]
  int resid_chunk;
  int ablate;   // development switches (HGN_TC_ABLATE): 1 skip workspace stores, 2 skip dX stores, 4 skip dO loads
};

// 8 MMAs: acc (+)= A[128 x 128] * B^T with A in TMEM (bf16 pairs) and B = a resident 128x128 weight block
//   b_mn = 0: B K-major   (forward:  out[n] = sum_k A[k] W[n][k])
//   b_mn = 1: B MN-major  (dgrad:    out[n] = sum_k A[k] W[k][n], the same panels read "transposed")
__device__ __forceinline__ void issue_ts_gemm(uint32_t acc, uint32_t a_tmem, uint32_t b_addr, int b_mn) {
  const uint32_t idesc = make_idesc_bf16(128, 128, 0, b_mn);
#pragma unroll
  for (int ks = 0; ks < 8; ++ks) {
    const uint64_t bd = b_mn ? sdesc_mnmajor(b_addr + ks * 2048, kPanel)
                             : sdesc_kmajor(b_addr + (ks >> 2) * kPanel + (ks & 3) * 32);
    mma_ts(acc, a_tmem + ks * 8, bd, idesc, ks != 0);
  }
}

// ---- tile kernel ---------------------------------------------------------------------------------------
// Steps per tile: forward 0:L0 1:L1 2:L2 ; backward adds 3:dH2=dY W2  4:dH1=dH2' W1  5+c: dX_c = dH1' W0[:,c].
// Scheduling: tile i of a CTA uses accumulator i%3 and epilogue group i%2.  The MMA warp is event driven: it
// streams layer 0 of the next tile chunk by chunk as the ring fills, and issues step k+1 of a tile the moment
// its epilogue group reports step k drained -- so gather latency, tensor work and epilogue work overlap.
template <bool kBwd>
__global__ void __launch_bounds__(kTileThreads, 1)
mlp_tile_tc_kernel(int64_t rows, int64_t num_tiles, int64_t slab0, hgn_chunks ch, const uint8_t* __restrict__ packed,
                   int w0_resident, const __nv_bfloat16* __restrict__ resid, int64_t resid_off, __nv_bfloat16* __restrict__ out,
                   BwdArgs bw) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int nch = ch.n_chunks;
  const TileSmem S(nch, w0_resident != 0, kBwd);
  const int w0_chunks = nch;
  const PackedTc P(w0_chunks);
  const uint32_t sbase = smem_u32(smem);
  if ((sbase & 1023u) != 0) __trap();   // SW128 atoms need 1024-byte alignment
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S.bars);
  float* sparams = reinterpret_cast<float*>(smem + S.params);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t k0 = int64_t(w0_chunks) * kD;
  const int n_steps = kBwd ? 5 + nch : 3;

  // ---- prologue: resident weights, parameters, barriers, TMEM ------------------------------------
  {
    const __nv_bfloat16* w0g = reinterpret_cast<const __nv_bfloat16*>(packed + P.w0);
    if (w0_resident)
      for (int c = 0; c < nch; ++c) load_weight_block(sbase + S.w0 + c * kChunkBytes, w0g + c * kD, k0, tid, kTileThreads);
    load_weight_block(sbase + S.w1, reinterpret_cast<const __nv_bfloat16*>(packed + P.w1), kD, tid, kTileThreads);
    load_weight_block(sbase + S.w2, reinterpret_cast<const __nv_bfloat16*>(packed + P.w2), kD, tid, kTileThreads);
    cp_async_commit();
    const float* pg = reinterpret_cast<const float*>(packed + P.params);
    for (int i = tid; i < 5 * kD; i += kTileThreads) sparams[i] = pg[i];
    if (tid == 0) {
      for (int s = 0; s < kStages; ++s) { mbar_init(&bars[kBarFull + s], kProdThreads / kStages); mbar_init(&bars[kBarEmpty + s], 1); }
      for (int s = 0; s < 6; ++s) mbar_init(&bars[kBarAcc + s], 1);
      for (int s = 0; s < 2; ++s) { mbar_init(&bars[kBarEpi + s], kEpiThreads / 2); mbar_init(&bars[kBarDone + s], kEpiThreads / 2); }
      mbar_init(&bars[kBarW0b], 1);
      mbar_init_fence();
    }
    if (warp == 12) tmem_alloc<512>(reinterpret_cast<uint32_t*>(&bars[kBarTmemPtr]));
    cp_async_wait<0>();
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
  }
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(&bars[kBarTmemPtr]);
  const int64_t my_tiles = (num_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x;   // tiles b, b+G, ...

  if (warp >= 8 && warp < 12) {
    // =============================== producers ====================================================
    // ring slot g holds chunk (g % nch) of this CTA's tile (g / nch); group `g & 1` fills it.
    const int ptid = tid - kEpiThreads;          // 0..127
    const int group = ptid >> 6;
    const int gt = ptid & 63;
    if (gt == 0) mbar_arrive(&bars[kBarEmpty + group]);   // the ring starts empty
    const uint32_t stage_addr = sbase + S.stages + group * S.stage_bytes;
    const __nv_bfloat16* w0g = reinterpret_cast<const __nv_bfloat16*>(packed + P.w0);
    const int64_t n_slots = my_tiles * nch;
    const int c16 = gt & 15, rbase = gt >> 4;    // this thread copies 16-byte piece c16 of rows rbase + 4 j
    // all 32 source-row indices of a slot are fetched in one batch, one slot ahead of the copies
    auto fetch_rows = [&](int64_t g, int32_t (&srow)[32]) {
      const int c = int(g % nch);
      const int64_t row0 = slab0 + (blockIdx.x + (g / nch) * gridDim.x) * kTile;
      const int32_t* idx = ch.idx[c];
      const int64_t roff = ch.row_offset[c];
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const int64_t grow = row0 + rbase + 4 * j;
        srow[j] = -1;
        if (grow < rows) srow[j] = idx ? __ldg(idx + grow) : int32_t(grow + roff);
      }
    };
    int32_t cur[32], nxt[32];
    int64_t g = group;
    if (g < n_slots) fetch_rows(g, cur);
    for (; g < n_slots; g += 2) {
      const int c = int(g % nch);
      mbar_wait(&bars[kBarEmpty + group], uint32_t(g >> 1) & 1, 1);
      const __nv_bfloat16* src = static_cast<const __nv_bfloat16*>(ch.src[c]);
      const uint32_t dst0 = stage_addr + (c16 >> 3) * kPanel;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const bool valid = cur[j] >= 0;
        cp_async16_zfill(dst0 + sw128_chunk(rbase + 4 * j, c16 & 7), src + int64_t(valid ? cur[j] : 0) * kD + c16 * 8, valid);
      }
      if (!w0_resident) load_weight_block(stage_addr + kChunkBytes, w0g + c * kD, k0, gt, 64);
      cp_async_commit();
      if (g + 2 < n_slots) fetch_rows(g + 2, nxt);     // index loads overlap the row copies in flight
      cp_async_wait<0>();
      fence_async_smem();
      mbar_arrive(&bars[kBarFull + group]);
#pragma unroll
      for (int j = 0; j < 32; ++j) cur[j] = nxt[j];
    }
  } else if (warp == 12) {
    // =============================== MMA warp (lane 0 issues) =====================================
    const uint32_t idesc_kk = make_idesc_bf16(128, 128, 0, 0);
    int64_t t_l0 = 0, g = 0, done = 0;
    int c_l0 = 0;
    int64_t wg_tile[2] = {0, 1};
    int wg_step[2] = {0, 0};
    uint32_t wg_sig[2] = {0, 0}, wg_fin[2] = {0, 0};
    uint32_t acc_busy = 0, w0b_uses = 0, idle = 0;
    const __nv_bfloat16* w0g = reinterpret_cast<const __nv_bfloat16*>(packed + P.w0);
    while (done < my_tiles) {
      bool progressed = false;
      // lane 0 polls the barriers once per round and broadcasts, so the whole warp takes the same path
      uint32_t ev = 0;
      if (lane == 0) {
#pragma unroll
        for (int w = 0; w < 2; ++w)
          if (wg_tile[w] < t_l0 &&
              (wg_step[w] == n_steps - 1 ? mbar_test(&bars[kBarDone + w], wg_fin[w] & 1) : mbar_test(&bars[kBarEpi + w], wg_sig[w] & 1)))
            ev |= 1u << w;
        if (t_l0 < my_tiles && (c_l0 > 0 || !((acc_busy >> int(t_l0 % kAccSlots)) & 1u)) &&
            mbar_test(&bars[kBarFull + int(g & 1)], uint32_t(g >> 1) & 1)) ev |= 4u;
      }
      ev = __shfl_sync(0xffffffffu, ev, 0);
      // ---- steps 1.. of the tiles whose epilogue group has reported the previous step drained -----
#pragma unroll
      for (int w = 0; w < 2; ++w) {
        const int64_t t = wg_tile[w];
        if ((ev >> w) & 1u) {
          fence_after_sync();
          const int k = wg_step[w]++;
          const int slot = int(t % kAccSlots);
          if (k == n_steps - 1) {                      // tile finished: its accumulator is free again
            ++wg_fin[w];
            acc_busy &= ~(1u << slot);
            wg_tile[w] += 2;
            wg_step[w] = 0;
            ++done;
          } else {
            ++wg_sig[w];
            const int step = k + 1;
            const uint32_t acc = tmem_base + slot * 128;
            const uint32_t aop = tmem_base + kAopCol + w * 64;
            if (step >= 5 && !w0_resident) {
              // streamed W0: fetch the panel pair of chunk c for this dX GEMM (the warp blocks ~1 us; only
              // node MLPs with more than 3 input chunks take this path)
              const int c = step - 5;
              if (w0b_uses > 0) mbar_wait(&bars[kBarW0b], (w0b_uses - 1) & 1);
              load_weight_block(sbase + S.w0b, w0g + c * kD, k0, lane, 32);
              cp_async_commit();
              cp_async_wait<0>();
              fence_async_smem();
              __syncwarp();
              if (lane == 0) { issue_ts_gemm(acc, aop, sbase + S.w0b, 1); mma_commit(&bars[kBarW0b]); }
              ++w0b_uses;
            } else if (lane == 0) {
              if (step == 1) issue_ts_gemm(acc, aop, sbase + S.w1, 0);
              else if (step == 2) issue_ts_gemm(acc, aop, sbase + S.w2, 0);
              else if (step == 3) issue_ts_gemm(acc, aop, sbase + S.w2, 1);
              else if (step == 4) issue_ts_gemm(acc, aop, sbase + S.w1, 1);
              else issue_ts_gemm(acc, aop, sbase + S.w0 + (step - 5) * kChunkBytes, 1);
            }
            if (lane == 0) mma_commit(&bars[kBarAcc + int(t % 6)]);
            __syncwarp();
          }
          progressed = true;
        }
      }
      // ---- layer 0 of the next tile: one chunk per visit, as soon as its ring slot is full --------
      if (ev & 4u) {
        const int slot = int(t_l0 % kAccSlots);
        {
          const int stage = int(g & 1);
          {
            fence_after_sync();
            if (lane == 0) {
              const uint32_t acc = tmem_base + slot * 128;
              const uint32_t a_addr = sbase + S.stages + stage * S.stage_bytes;
              const uint32_t b_addr = w0_resident ? sbase + S.w0 + c_l0 * kChunkBytes : a_addr + kChunkBytes;
#pragma unroll
              for (int ks = 0; ks < 8; ++ks) {
                const uint32_t koff = (ks >> 2) * kPanel + (ks & 3) * 32;
                mma_ss(acc, sdesc_kmajor(a_addr + koff), sdesc_kmajor(b_addr + koff), idesc_kk, (c_l0 | ks) != 0);
              }
              mma_commit(&bars[kBarEmpty + stage]);
              if (c_l0 + 1 == nch) mma_commit(&bars[kBarAcc + int(t_l0 % 6)]);
            }
            __syncwarp();
            acc_busy |= 1u << slot;
            ++g;
            if (++c_l0 == nch) { c_l0 = 0; ++t_l0; }
            progressed = true;
          }
        }
      }
      if (!progressed) {
        if (!(bw.ablate & 8)) __nanosleep(20);
        if (++idle > (1u << 22)) {
          if (lane == 0)
            debug_record(900u + uint32_t(kBwd), uint32_t(t_l0) | (uint32_t(c_l0) << 16), uint32_t(g), uint32_t(done) | (uint32_t(my_tiles) << 16),
                         uint32_t(wg_tile[0]) | (uint32_t(wg_tile[1]) << 16), uint32_t(wg_step[0]) | (uint32_t(wg_step[1]) << 8) | (acc_busy << 16),
                         wg_sig[0] | (wg_sig[1] << 16));
          __trap();
        }
      } else {
        idle = 0;
      }
    }
  } else {
    // =============================== epilogue groups ==============================================
    const int wg = warp >> 2;                         // warps 0-3 -> group 0 (even tiles), 4-7 -> group 1 (odd tiles)
    const int r = (warp & 3) * 32 + lane;             // tile row = TMEM lane
    const uint32_t lane_addr = uint32_t((warp & 3) * 32) << 16;
    const uint32_t aop = tmem_base + kAopCol + wg * 64 + lane_addr;
    const float* b2 = sparams + 2 * kD;
    const float* gam = sparams + 3 * kD;
    const float* bet = sparams + 4 * kD;
    for (int64_t it = wg; it < my_tiles; it += 2) {
      const int slot = int(it % kAccSlots);
      const uint32_t acc = tmem_base + slot * 128 + lane_addr;
      uint32_t acc_phase = uint32_t((it / 6) * n_steps);   // completions of this (group, accumulator) barrier so far
      uint32_t steps_done = 0;
      auto wait_acc = [&]() {
        mbar_wait(&bars[kBarAcc + int(it % 6)], acc_phase & 1, 100 + int(steps_done));
        ++acc_phase;
        fence_after_sync();
      };
      auto signal_done = [&]() {
        fence_before_sync();
        mbar_arrive(&bars[(++steps_done == uint32_t(n_steps) ? kBarDone : kBarEpi) + wg]);
      };
      const int64_t grow = slab0 + (blockIdx.x + it * gridDim.x) * kTile + r;
      const bool valid = grow < rows;
      const int64_t lrow = valid ? grow - slab0 : 0;   // row inside the slab workspaces
      uint32_t mask1[4] = {0, 0, 0, 0}, mask2[4] = {0, 0, 0, 0};   // ReLU masks (backward)
      // ---- hidden layers: bias + ReLU -> bf16 A operand in TMEM -------------------------------
#pragma unroll 1
      for (int layer = 0; layer < 2; ++layer) {
        wait_acc();
        const float* bias = sparams + layer * kD;
        __nv_bfloat16* hws = kBwd ? (layer == 0 ? bw.H1 : bw.H2) + lrow * kD : nullptr;
#pragma unroll 1
        for (int cg = 0; cg < 4; ++cg) {
          uint32_t v[32];
          tmem_ld32(acc + cg * 32, v);
          tmem_ld_wait();
          uint32_t h[16];
          uint32_t m = 0;
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float a = fmaxf(__uint_as_float(v[2 * j]) + bias[cg * 32 + 2 * j], 0.f);
            const float b = fmaxf(__uint_as_float(v[2 * j + 1]) + bias[cg * 32 + 2 * j + 1], 0.f);
            h[j] = pack_bf16(a, b);
            if (kBwd) m |= (a > 0.f ? (1u << (2 * j)) : 0u) | (b > 0.f ? (1u << (2 * j + 1)) : 0u);
          }
          tmem_st8(aop + cg * 16, h);
          tmem_st8(aop + cg * 16 + 8, h + 8);
          if (kBwd) {
            if (layer == 0) mask1[cg] = m; else mask2[cg] = m;
            if (valid && !(bw.ablate & 1)) { stg256(hws + cg * 32, h); stg256(hws + cg * 32 + 16, h + 8); }
          }
        }
        tmem_st_wait();
        signal_done();
      }
      // ---- last layer: bias, LayerNorm statistics -----------------------------------------------
      wait_acc();
      float sum = 0.f;
#pragma unroll 1
      for (int cg = 0; cg < 4; ++cg) {
        uint32_t v[32];
        tmem_ld32(acc + cg * 32, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) sum += __uint_as_float(v[j]) + b2[cg * 32 + j];
      }
      const float mean = sum * (1.0f / kD);
      float sq = 0.f;
#pragma unroll 1
      for (int cg = 0; cg < 4; ++cg) {
        uint32_t v[32];
        tmem_ld32(acc + cg * 32, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) { const float d = __uint_as_float(v[j]) + b2[cg * 32 + j] - mean; sq = fmaf(d, d, sq); }
      }
      const float rstd = rsqrtf(sq * (1.0f / kD) + kEps);
      if (!kBwd) {
        // ---- forward: affine, residual, store (32-byte sectors per lane) ----------------------
        const __nv_bfloat16* rp = resid + (valid ? grow + resid_off : 0) * kD;
        __nv_bfloat16* op = out + (valid ? grow : 0) * kD;
#pragma unroll 1
        for (int cg = 0; cg < 4; ++cg) {
          uint32_t v[32];
          tmem_ld32(acc + cg * 32, v);
          tmem_ld_wait();
          if (valid) {
            uint32_t rw[16], ow[16];
            ldg256(rp + cg * 32, rw);
            ldg256(rp + cg * 32 + 16, rw + 8);
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const int col = cg * 32 + 2 * j;
              const float y0 = (__uint_as_float(v[2 * j]) + b2[col] - mean) * rstd * gam[col] + bet[col];
              const float y1 = (__uint_as_float(v[2 * j + 1]) + b2[col + 1] - mean) * rstd * gam[col + 1] + bet[col + 1];
              ow[j] = pack_bf16(bf16_lo(rw[j]) + y0, bf16_hi(rw[j]) + y1);
            }
            stg256(op + cg * 32, ow);
            stg256(op + cg * 32 + 16, ow + 8);
          }
        }
        signal_done();
      } else {
        // ---- backward: LayerNorm backward -> dY (A operand) ; P = dO * yhat for the gamma gradient --
        const __nv_bfloat16* gop = bw.grad_out + (valid ? grow : 0) * kD;
        __nv_bfloat16* pws = bw.P + lrow * kD;
        float m1 = 0.f, m2 = 0.f;
#pragma unroll 1
        for (int cg = 0; cg < 4; ++cg) {
          uint32_t v[32];
          tmem_ld32(acc + cg * 32, v);
          tmem_ld_wait();
          uint32_t gw[16], pw[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) gw[j] = 0u;
          if (valid && !(bw.ablate & 4)) { ldg256(gop + cg * 32, gw); ldg256(gop + cg * 32 + 16, gw + 8); }
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int col = cg * 32 + 2 * j;
            const float yh0 = (__uint_as_float(v[2 * j]) + b2[col] - mean) * rstd;
            const float yh1 = (__uint_as_float(v[2 * j + 1]) + b2[col + 1] - mean) * rstd;
            const float d0 = bf16_lo(gw[j]), d1 = bf16_hi(gw[j]);
            const float dy0 = d0 * gam[col], dy1 = d1 * gam[col + 1];
            m1 += dy0 + dy1;
            m2 = fmaf(dy0, yh0, fmaf(dy1, yh1, m2));
            pw[j] = pack_bf16(d0 * yh0, d1 * yh1);
          }
          if (valid && !(bw.ablate & 1)) { stg256(pws + cg * 32, pw); stg256(pws + cg * 32 + 16, pw + 8); }
          tmem_st8(aop + cg * 16, gw);           // park dO (bf16) in the free A-operand columns
          tmem_st8(aop + cg * 16 + 8, gw + 8);
        }
        tmem_st_wait();
        m1 *= (1.0f / kD);
        m2 *= (1.0f / kD);
        __nv_bfloat16* g2ws = bw.G2 + lrow * kD;
#pragma unroll 1
        for (int cg = 0; cg < 4; ++cg) {
          uint32_t v[32], dpk[16];
          tmem_ld32(acc + cg * 32, v);
          tmem_ld16(aop + cg * 16, dpk);
          tmem_ld_wait();
          uint32_t o[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int col = cg * 32 + 2 * j;
            const float yh0 = (__uint_as_float(v[2 * j]) + b2[col] - mean) * rstd;
            const float yh1 = (__uint_as_float(v[2 * j + 1]) + b2[col + 1] - mean) * rstd;
            const float dy0 = rstd * (bf16_lo(dpk[j]) * gam[col] - m1 - yh0 * m2);
            const float dy1 = rstd * (bf16_hi(dpk[j]) * gam[col + 1] - m1 - yh1 * m2);
            o[j] = pack_bf16(dy0, dy1);
          }
          tmem_st8(aop + cg * 16, o);
          tmem_st8(aop + cg * 16 + 8, o + 8);
          if (valid && !(bw.ablate & 1)) { stg256(g2ws + cg * 32, o); stg256(g2ws + cg * 32 + 16, o + 8); }
        }
        tmem_st_wait();
        signal_done();
        // ---- dH2' = (dY W2) * [H2 > 0] ; dH1' = (dH2' W1) * [H1 > 0] ------------------------------
#pragma unroll 1
        for (int layer = 1; layer >= 0; --layer) {
          wait_acc();
          __nv_bfloat16* gws = (layer == 1 ? bw.G1 : bw.G0) + lrow * kD;
#pragma unroll 1
          for (int cg = 0; cg < 4; ++cg) {
            uint32_t v[32];
            tmem_ld32(acc + cg * 32, v);
            tmem_ld_wait();
            const uint32_t m = layer == 1 ? mask2[cg] : mask1[cg];
            uint32_t o[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const float a = (m >> (2 * j)) & 1u ? __uint_as_float(v[2 * j]) : 0.f;
              const float b = (m >> (2 * j + 1)) & 1u ? __uint_as_float(v[2 * j + 1]) : 0.f;
              o[j] = pack_bf16(a, b);
            }
            tmem_st8(aop + cg * 16, o);
            tmem_st8(aop + cg * 16 + 8, o + 8);
            if (valid && !(bw.ablate & 1)) { stg256(gws + cg * 32, o); stg256(gws + cg * 32 + 16, o + 8); }
          }
          tmem_st_wait();
          signal_done();
        }
        // ---- dX_c = dH1' W0[:, c]  (+ grad_out for the residual chunk) -------------------------------
        for (int c = 0; c < nch; ++c) {
          wait_acc();
          __nv_bfloat16* dst = bw.grad_chunk[c];
          if (dst != nullptr) {                       // warp-uniform: tcgen05.ld is a warp-collective
            __nv_bfloat16* dp = dst + (valid ? grow : 0) * kD;
            const bool add_resid = (c == bw.resid_chunk);
#pragma unroll 1
            for (int cg = 0; cg < 4; ++cg) {
              uint32_t v[32];
              tmem_ld32(acc + cg * 32, v);
              tmem_ld_wait();
              if (valid) {
                uint32_t gw[16], ow[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) gw[j] = 0u;
                if (add_resid) { ldg256(gop + cg * 32, gw); ldg256(gop + cg * 32 + 16, gw + 8); }
#pragma unroll
                for (int j = 0; j < 16; ++j)
                  ow[j] = pack_bf16(__uint_as_float(v[2 * j]) + bf16_lo(gw[j]), __uint_as_float(v[2 * j + 1]) + bf16_hi(gw[j]));
                if (!(bw.ablate & 2)) { stg256(dp + cg * 32, ow); stg256(dp + cg * 32 + 16, ow + 8); }
              }
            }
          }
          signal_done();
        }
      }
    }
  }
  // ---- teardown ------------------------------------------------------------------------------------
  fence_before_sync();
  __syncthreads();
  if (warp == 12) tmem_dealloc<512>(tmem_base);
}

// ---- weight-gradient kernel --------------------------------------------------------------------------
// grid (parts, groups).  group 0: dW2 = G2^T H2, dW1 = G1^T H1.  group j >= 1: dW0 chunks 3(j-1) .. 3(j-1)+2
// = G0^T X_c (X_c gathered like in the forward).  K (= rows) advances in 64-row stages; every operand tile
// [64 rows][128 cols] bf16 sits in two SW128 panels of 8 KiB and is read MN-major.
constexpr int kWgRows = 64;
constexpr int kWgTileBytes = 2 * 8192;         // one [64][128] operand tile
constexpr int kWgStageTiles = 4;
constexpr int kWgStageBytes = kWgStageTiles * kWgTileBytes;   // 64 KiB
constexpr int kWgStages = 3;
constexpr int kWgThreads = 128 + 32 + 128;     // warps 0-3 producers, warp 4 MMA, warps 5-8 epilogue (final drain)

struct WgradArgs {
  const __nv_bfloat16 *G2, *G1, *G0, *H1, *H2;
  float* partial;       // [parts][n_z][128][128]
  int n_z;
  int accumulate;
};

__global__ void __launch_bounds__(kWgThreads, 1)
mlp_wgrad_tc_kernel(int64_t rows, int64_t slab0, int64_t slab_rows, int64_t rows_per_part, hgn_chunks ch, WgradArgs wa) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  if ((sbase & 1023u) != 0) __trap();
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kWgStages * kWgStageBytes);   // full[3], empty[3], done, tmem ptr
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int part = blockIdx.x, group = blockIdx.y, nch = ch.n_chunks;
  const int c_first = group == 0 ? 0 : 3 * (group - 1);
  const bool single = group == 0 && wa.G1 == nullptr;                // one (G, Z) pair only
  const int n_out = group == 0 ? (single ? 1 : 2) : min(3, nch - c_first);   // accumulators of this CTA
  const int n_tiles = group == 0 ? 4 : 1 + n_out;                    // operand tiles per stage
  const int64_t row_end = min(rows, slab0 + slab_rows);
  const int64_t r_beg = slab0 + int64_t(part) * rows_per_part;
  const int64_t r_end = min(row_end, r_beg + rows_per_part);
  const int64_t n_steps = r_end > r_beg ? (r_end - r_beg + kWgRows - 1) / kWgRows : 0;

  if (tid == 0) {
    for (int s = 0; s < kWgStages; ++s) { mbar_init(&bars[s], 128); mbar_init(&bars[3 + s], 1); }
    mbar_init(&bars[6], 1);
    mbar_init_fence();
  }
  if (warp == 4) tmem_alloc<512>(reinterpret_cast<uint32_t*>(&bars[7]));
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(&bars[7]);

  if (warp < 4) {
    // ---- producers: dense rows (and gathered X chunks) -> MN-major operand tiles ------------------------
    if (tid < kWgStages) mbar_arrive(&bars[3 + tid]);     // ring starts empty
    const int c16 = tid & 15, rbase = tid >> 4;           // this thread copies piece c16 of rows rbase + 8 j
    // source rows of the gathered X tiles, fetched one stage ahead of the copies that use them
    auto fetch_rows = [&](int64_t st, int32_t (&srow)[3][8]) {
      if (group == 0) return;
      const int64_t row0 = r_beg + st * kWgRows;
#pragma unroll
      for (int t = 0; t < 3; ++t) {
        if (t >= n_out) break;
        const int32_t* idx = ch.idx[c_first + t];
        const int64_t roff = ch.row_offset[c_first + t];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int64_t grow = row0 + rbase + 8 * j;
          srow[t][j] = -1;
          if (grow < r_end) srow[t][j] = idx ? __ldg(idx + grow) : int32_t(grow + roff);
        }
      }
    };
    int32_t cur[3][8], nxt[3][8];
    if (n_steps > 0) fetch_rows(0, cur);
    for (int64_t st = 0; st < n_steps; ++st) {
      const int stage = int(st % kWgStages);
      mbar_wait(&bars[3 + stage], uint32_t(st / kWgStages) & 1, 10);
      const int64_t row0 = r_beg + st * kWgRows;
      const uint32_t saddr = sbase + stage * kWgStageBytes + (c16 >> 3) * 8192;
      // dense workspace tiles (slab-local rows)
      const int n_dense = group == 0 ? (single ? 2 : 4) : 1;
      for (int t = 0; t < n_dense; ++t) {
        const __nv_bfloat16* src = group == 0 ? (t == 0 ? wa.G2 : t == 1 ? wa.H2 : t == 2 ? wa.G1 : wa.H1) : wa.G0;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int64_t grow = row0 + rbase + 8 * j;
          const bool valid = grow < r_end;
          cp_async16_zfill(saddr + t * kWgTileBytes + sw128_chunk(rbase + 8 * j, c16 & 7), src + (valid ? grow - slab0 : 0) * kD + c16 * 8, valid);
        }
      }
      if (group != 0) {
#pragma unroll
        for (int t = 0; t < 3; ++t) {
          if (t >= n_out) break;
          const __nv_bfloat16* src = static_cast<const __nv_bfloat16*>(ch.src[c_first + t]);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const bool valid = cur[t][j] >= 0;
            cp_async16_zfill(saddr + (1 + t) * kWgTileBytes + sw128_chunk(rbase + 8 * j, c16 & 7),
                             src + int64_t(valid ? cur[t][j] : 0) * kD + c16 * 8, valid);
          }
        }
      }
      cp_async_commit();
      if (st + 1 < n_steps) fetch_rows(st + 1, nxt);
      // keep up to three stages of loads in flight: publish stage st-2 once its group has landed
      if (st >= 2) {
        cp_async_wait<2>();
        fence_async_smem();
        mbar_arrive(&bars[int((st - 2) % kWgStages)]);
      }
#pragma unroll
      for (int t = 0; t < 3; ++t)
#pragma unroll
        for (int j = 0; j < 8; ++j) cur[t][j] = nxt[t][j];
    }
    cp_async_wait<0>();
    fence_async_smem();
    if (n_steps >= 2) mbar_arrive(&bars[int((n_steps - 2) % kWgStages)]);
    if (n_steps >= 1) mbar_arrive(&bars[int((n_steps - 1) % kWgStages)]);
  } else if (warp == 4) {
    if (lane == 0) {
      const uint32_t idesc = make_idesc_bf16(128, 128, 1, 1);     // both operands MN-major
      for (int64_t st = 0; st < n_steps; ++st) {
        const int stage = int(st % kWgStages);
        mbar_wait(&bars[stage], uint32_t(st / kWgStages) & 1, 11);
        fence_after_sync();
        const uint32_t saddr = sbase + stage * kWgStageBytes;
        for (int o = 0; o < n_out; ++o) {
          const uint32_t a_addr = saddr + (group == 0 ? 2 * o : 0) * kWgTileBytes;            // G tile
          const uint32_t b_addr = saddr + (group == 0 ? 2 * o + 1 : 1 + o) * kWgTileBytes;    // Z tile
#pragma unroll
          for (int ks = 0; ks < kWgRows / 16; ++ks)
            mma_ss(tmem_base + o * 128, sdesc_mnmajor(a_addr + ks * 2048, 8192), sdesc_mnmajor(b_addr + ks * 2048, 8192), idesc,
                   (st | ks) != 0);
        }
        mma_commit(&bars[3 + stage]);
      }
      mma_commit(&bars[6]);
    }
  } else {
    // ---- final drain: TMEM accumulators -> fp32 partials ---------------------------------------------------
    const int ew = warp - 5;                      // 0..3
    const int quarter = warp & 3;                 // TMEM lane quarter this warp may read
    (void)ew;
    if (n_steps > 0) {
      mbar_wait(&bars[6], 0, 12);
      fence_after_sync();
    }
    const int o_row = quarter * 32 + lane;        // output row (= "out" feature of the weight)
    for (int o = 0; o < n_out; ++o) {
      const int z = group == 0 ? (o == 0 ? nch + 1 : nch) : c_first + o;     // partial layout: W0 chunks, W1, W2
      float* dst = wa.partial + ((int64_t(part) * wa.n_z + z) * kD + o_row) * kD;
#pragma unroll 1
      for (int cg = 0; cg < 4; ++cg) {
        uint32_t v[32];
        if (n_steps > 0) {
          tmem_ld32(tmem_base + (uint32_t(quarter * 32) << 16) + o * 128 + cg * 32, v);
          tmem_ld_wait();
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = 0u;
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          float4 val = make_float4(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]), __uint_as_float(v[4 * q + 2]), __uint_as_float(v[4 * q + 3]));
          float4* p = reinterpret_cast<float4*>(dst + cg * 32 + q * 4);
          if (wa.accumulate) { const float4 old = *p; val.x += old.x; val.y += old.y; val.z += old.z; val.w += old.w; }
          *p = val;
        }
      }
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 4) tmem_dealloc<512>(tmem_base);
}

// ---- host side -----------------------------------------------------------------------------------------
size_t mlp_tc_packed_bytes(int n_chunks) { return PackedTc(n_chunks).total; }

int mlp_tc_pack(int n_chunks, const float* W0, const float* b0, const float* W1, const float* b1, const float* W2,
                const float* b2, const float* gamma, const float* beta, void* packed, cudaStream_t st) {
  const int64_t n = int64_t(n_chunks) * kD * kD;
  HGN_TIMED("pack_tc", st);
  pack_tc_kernel<<<unsigned(ceil_div(n, 256)), 256, 0, st>>>(n_chunks, W0, b0, W1, b1, W2, b2, gamma, beta, static_cast<uint8_t*>(packed));
  HGN_LAUNCH_OK("pack_tc");
  return HGN_OK;
}

int tc_sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

static int configure_kernels() {
  static bool configured = false;
  if (!configured) {
    uint32_t* dbg = debug_buffer_device();
    HGN_CUDA_OK(cudaMemcpyToSymbol(tc05::g_debug_words, &dbg, sizeof(dbg)));
    HGN_CUDA_OK(cudaFuncSetAttribute(mlp_tile_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
    HGN_CUDA_OK(cudaFuncSetAttribute(mlp_tile_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
    HGN_CUDA_OK(cudaFuncSetAttribute(mlp_wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
    configured = true;
  }
  return HGN_OK;
}

int mlp_tc_forward(int64_t rows, const hgn_chunks* ch, const void* packed, const void* resid, int64_t resid_off, void* out,
                   cudaStream_t st) {
  const char* name = "mlp_tile_tc_fwd";
  const int nch = ch->n_chunks;
  const bool resident = nch <= kMaxResidentChunks;
  const TileSmem S(nch, resident, false);
  if (int rc = configure_kernels()) return rc;
  const int64_t tiles = ceil_div(rows, kTile);
  const unsigned grid = unsigned(tiles < tc_sm_count() ? tiles : tc_sm_count());
  BwdArgs none{};
  { const char* ab = getenv("HGN_TC_ABLATE"); none.ablate = ab ? atoi(ab) : 0; }
  HGN_TIMED(name, st);
  mlp_tile_tc_kernel<false><<<grid, kTileThreads, S.total, st>>>(rows, tiles, 0, *ch, static_cast<const uint8_t*>(packed), resident ? 1 : 0,
                                                                 static_cast<const __nv_bfloat16*>(resid), resid_off,
                                                                 static_cast<__nv_bfloat16*>(out), none);
  HGN_LAUNCH_OK("mlp_fwd_tc");
  return HGN_OK;
}

// dWa = Ga^T Za and dWb = Gb^T Zb over dense [rows,128] bf16 operands (node-level weight gradients of the projected edge
// update): per-part fp32 partials [parts][2][128][128], z = 1: a, z = 0: b.
int tc_pair_wgrad_parts(int64_t rows) {
  const int64_t r = rows > 0 ? rows : 1;
  return int(r >= int64_t(tc_sm_count()) * 4 * kWgRows ? tc_sm_count() : ceil_div(r, 4 * kWgRows));
}

int tc_pair_wgrad(int64_t rows, const void* Ga, const void* Za, const void* Gb, const void* Zb, float* partial, int parts, cudaStream_t st) {
  if (int rc = configure_kernels()) return rc;
  WgradArgs wa{};
  wa.G2 = static_cast<const __nv_bfloat16*>(Ga); wa.H2 = static_cast<const __nv_bfloat16*>(Za);
  wa.G1 = static_cast<const __nv_bfloat16*>(Gb); wa.H1 = static_cast<const __nv_bfloat16*>(Zb);
  wa.partial = partial; wa.n_z = 2; wa.accumulate = 0;
  hgn_chunks none{};
  const int64_t rpp = ceil_div(ceil_div(rows > 0 ? rows : 1, parts), kWgRows) * kWgRows;
  const size_t wg_smem = size_t(kWgStages) * kWgStageBytes + 64;
  HGN_TIMED("mlp_wgrad_tc", st);
  mlp_wgrad_tc_kernel<<<dim3(unsigned(parts), 1), kWgThreads, wg_smem, st>>>(rows, 0, rows > 0 ? rows : 1, rpp, none, wa);
  HGN_LAUNCH_OK("pair_wgrad_tc");
  return HGN_OK;
}

// dW2 = G2^T H2, dW1 = G1^T H1 and dW0 = G0^T X over one slab of a one-chunk MLP whose data-gradient pass runs elsewhere (the encoder
// and decoder kernels of io_mlp_tc.cu): per-part fp32 partials [parts][3][128][128], z = 0: W0, 1: W1, 2: W2.  X is [*, 128] bf16,
// row r of the slab read from row r + x_row_offset.
int tc_io_wgrad(int64_t rows, int64_t slab0, int64_t slab_rows, int parts, const void* X, int64_t x_row_offset, const void* G2, const void* H2,
                const void* G1, const void* H1, const void* G0, float* partial, int accumulate, cudaStream_t st) {
  if (int rc = configure_kernels()) return rc;
  WgradArgs wa{};
  wa.G2 = static_cast<const __nv_bfloat16*>(G2); wa.H2 = static_cast<const __nv_bfloat16*>(H2);
  wa.G1 = static_cast<const __nv_bfloat16*>(G1); wa.H1 = static_cast<const __nv_bfloat16*>(H1);
  wa.G0 = static_cast<const __nv_bfloat16*>(G0);
  wa.partial = partial; wa.n_z = 3; wa.accumulate = accumulate;
  hgn_chunks ch{};
  ch.n_chunks = 1; ch.src[0] = X; ch.idx[0] = nullptr; ch.row_offset[0] = x_row_offset;
  const int64_t this_rows = rows - slab0 < slab_rows ? rows - slab0 : slab_rows;
  const int64_t rpp = ceil_div(ceil_div(this_rows > 0 ? this_rows : 1, parts), kWgRows) * kWgRows;
  const size_t wg_smem = size_t(kWgStages) * kWgStageBytes + 64;
  HGN_TIMED("mlp_wgrad_tc", st);
  mlp_wgrad_tc_kernel<<<dim3(unsigned(parts), 2), kWgThreads, wg_smem, st>>>(rows, slab0, slab_rows, rpp, ch, wa);
  HGN_LAUNCH_OK("io_wgrad_tc");
  return HGN_OK;
}

struct BwdLayoutTc {
  int64_t slab_rows, parts, rows_per_part;
  int groups, n_z;
  size_t act[6], partial, vec_partial, total;   // act: H1 H2 P G2 G1 G0
};

static BwdLayoutTc bwd_layout_tc(int64_t rows, int n_chunks) {
  BwdLayoutTc L{};
  const int64_t cap = int64_t(1) << 21;                      // <= 2M rows per pass (6 x 512 MiB of bf16 workspace)
  L.slab_rows = rows < cap ? (rows > 0 ? rows : 1) : cap;
  L.slab_rows = ceil_div(L.slab_rows, kTile) * kTile;
  L.parts = L.slab_rows >= int64_t(tc_sm_count()) * 4 * kWgRows ? tc_sm_count() : ceil_div(L.slab_rows, 4 * kWgRows);
  L.rows_per_part = ceil_div(ceil_div(L.slab_rows, L.parts), kWgRows) * kWgRows;
  L.groups = 1 + (n_chunks + 2) / 3;
  L.n_z = n_chunks + 2;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
  for (int i = 0; i < 6; ++i) L.act[i] = take(size_t(L.slab_rows) * kD * 2);
  L.partial = take(size_t(L.parts) * L.n_z * kD * kD * 4);
  L.vec_partial = take(colsum5_workspace_bytes(L.slab_rows));
  L.total = off;
  return L;
}

size_t mlp_tc_backward_workspace_bytes(int64_t rows, int n_chunks) { return bwd_layout_tc(rows, n_chunks).total; }

int mlp_tc_backward(int64_t rows, const hgn_chunks* ch, const void* packed, const void* grad_out, int resid_chunk,
                    void* const* grad_chunk, float* gW0, float* gb0, float* gW1, float* gb1, float* gW2, float* gb2,
                    float* ggamma, float* gbeta, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  const int nch = ch->n_chunks;
  const bool resident = nch <= kMaxResidentChunks;
  const TileSmem S(nch, resident, true);
  const BwdLayoutTc L = bwd_layout_tc(rows, nch);
  if (workspace_bytes < L.total) { set_error("mlp_backward(bf16): workspace %zu < %zu", workspace_bytes, L.total); return HGN_ERR_WORKSPACE; }
  if (int rc = configure_kernels()) return rc;
  char* ws = static_cast<char*>(workspace);
  BwdArgs bw{};
  bw.grad_out = static_cast<const __nv_bfloat16*>(grad_out);
  for (int c = 0; c < nch; ++c) bw.grad_chunk[c] = grad_chunk ? static_cast<__nv_bfloat16*>(grad_chunk[c]) : nullptr;
  bw.H1 = (__nv_bfloat16*)(ws + L.act[0]); bw.H2 = (__nv_bfloat16*)(ws + L.act[1]); bw.P = (__nv_bfloat16*)(ws + L.act[2]);
  bw.G2 = (__nv_bfloat16*)(ws + L.act[3]); bw.G1 = (__nv_bfloat16*)(ws + L.act[4]); bw.G0 = (__nv_bfloat16*)(ws + L.act[5]);
  bw.resid_chunk = resid_chunk;
  { const char* ab = getenv("HGN_TC_ABLATE"); bw.ablate = ab ? atoi(ab) : 0; }
  float* partial = (float*)(ws + L.partial);
  float* vec_ws = (float*)(ws + L.vec_partial);
  const size_t colsum_ws_bytes = colsum5_workspace_bytes(L.slab_rows);
  WgradArgs wa{};
  wa.G2 = bw.G2; wa.G1 = bw.G1; wa.G0 = bw.G0; wa.H1 = bw.H1; wa.H2 = bw.H2;
  wa.partial = partial; wa.n_z = L.n_z;
  const size_t wg_smem = size_t(kWgStages) * kWgStageBytes + 64;
  float* vec_out[5] = {gb2, gb1, gb0, ggamma, gbeta};
  int pass = 0;
  for (int64_t slab0 = 0; slab0 < rows || pass == 0; slab0 += L.slab_rows, ++pass) {
    const int64_t this_rows = rows - slab0 < L.slab_rows ? rows - slab0 : L.slab_rows;
    if (this_rows > 0) {
      const int64_t tiles = ceil_div(this_rows, kTile);
      const unsigned grid = unsigned(tiles < tc_sm_count() ? tiles : tc_sm_count());
      HGN_TIMED("mlp_tile_tc_bwd", st);
      mlp_tile_tc_kernel<true><<<grid, kTileThreads, S.total, st>>>(rows, tiles, slab0, *ch, static_cast<const uint8_t*>(packed),
                                                                    resident ? 1 : 0, nullptr, 0, nullptr, bw);
      HGN_LAUNCH_OK("mlp_bwd_tc");
    }
    wa.accumulate = pass > 0;
    dim3 grid(unsigned(L.parts), unsigned(L.groups));
    { HGN_TIMED("mlp_wgrad_tc", st);
    const int64_t rpp = ceil_div(ceil_div(this_rows > 0 ? this_rows : 1, L.parts), kWgRows) * kWgRows;
    mlp_wgrad_tc_kernel<<<grid, kWgThreads, wg_smem, st>>>(rows, slab0, L.slab_rows, rpp, *ch, wa);
    }
    HGN_LAUNCH_OK("mlp_wgrad_tc");
    // bias / LayerNorm vector gradients: column sums of G2, G1, G0, P and grad_out over this slab
    const void* mats[5] = {bw.G2, bw.G1, bw.G0, bw.P, bw.grad_out ? (const void*)(bw.grad_out + slab0 * kD) : nullptr};
    if (int rc = colsum5_bf16(mats, vec_out, this_rows > 0 ? this_rows : 0, pass > 0, vec_ws, colsum_ws_bytes, st)) return rc;
    if (rows == 0) break;
  }
  launch_reduce_weight_partials(partial, int(L.parts), nch, gW0, gW1, gW2, st);
  HGN_LAUNCH_OK("mlp_bwd_tc reductions");
  return HGN_OK;
}

}  // namespace hgn
