// bf16 tcgen05 encoder and decoder MLPs (HGN_BF16 models, opt-in): the two MLPs on either side of the processor, in the
// reference's _make_mlp shape with num_layers = 2 (meshgraphnet.py:93-108).
//
//   encoder  fp32 X[R,K] (1 <= K <= 128)  -> Linear(K,128) ReLU Linear(128,128) ReLU Linear(128,128) LayerNorm -> bf16 [R,128]
//   decoder  bf16 X[N,128]                -> Linear(128,128) ReLU Linear(128,128) ReLU Linear(128,n_out)      -> fp32 [N,n_out]
//                                            (1 <= n_out <= 16; no LayerNorm, no residual)
//
// The skeleton is the generic tile kernel's (mlp_tc.cu): persistent CTAs of 13 warps, producers (warps 8-11) fill a 2-stage ring
// of SW128 operand panels, one MMA thread (warp 12) issues the GEMMs, two epilogue groups (warps 0-3 / 4-7) alternate over three
// TMEM accumulators, the backward recomputes the activations, and the weight gradients are the tile kernel's wgrad GEMMs
// (mlp_wgrad_tc_kernel through tc_io_wgrad) into per-CTA partials reduced in a fixed order.  What differs:
//   * encoder producers read the K fp32 values of a row (row pitch 4K bytes: no 16-byte alignment), round them to bf16 and
//     zero-fill the panel up to the next multiple of 16 columns; layer 0 issues ceil(K/16) K=16 MMA steps instead of 8;
//   * the encoder has no residual; the decoder has no LayerNorm and its last GEMM is N = 16 (W2 zero-padded to 16 rows), whose
//     epilogue adds b2 in fp32 and writes n_out fp32 values per row;
//   * the decoder backward starts its dgrad chain at dH2 = dY W2 (one K=16 MMA step on the bf16-rounded upstream gradient).
//
// Rounding points (the tests emulate exactly these):
//   encoder  X, W0, W1, W2 -> bf16; H0 = bf16(relu(acc + b0)), H1 = bf16(relu(acc + b1)); LayerNorm in fp32 on acc + b2; the
//            output is rounded once to bf16.
//   decoder  X is bf16; W0, W1, W2 -> bf16; H0, H1 as in the encoder; the output is acc + b2 in fp32.
//   backward the upstream gradient is rounded to bf16 where it becomes an MMA operand (the decoder's dY; the encoder's dO is bf16
//            already); LayerNorm backward in fp32 -> bf16 dY; dH' = bf16(acc * [H > 0]); the encoder's raw-feature gradient is the
//            fp32 accumulator, the decoder's input gradient is rounded to bf16; weight gradients are fp32 sums of bf16 products,
//            bias / gamma / beta gradients fp32 column sums of the bf16 dgrad tiles (the tile kernel's rounding points).
#include "tile_common.cuh"

namespace hgn {

// Packed blob: the tile kernel's one-chunk layout (PackedTc(1)) with zero padding -- W0 [128][128] (encoder: columns >= K zero),
// W1 [128][128], W2 [128][128] (decoder: rows >= n_out zero), fp32 b0 b1 b2 gamma beta (decoder: b2 beyond n_out, gamma, beta zero).
__global__ void io_pack_kernel(int enc, int width, const float* W0, const float* b0, const float* W1, const float* b1, const float* W2,
                               const float* b2, const float* gamma, const float* beta, uint8_t* packed) {
  const PackedTc L(1);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= kD * kD) return;
  const int r = i / kD, c = i % kD;
  __nv_bfloat16* w0 = reinterpret_cast<__nv_bfloat16*>(packed + L.w0);
  __nv_bfloat16* w1 = reinterpret_cast<__nv_bfloat16*>(packed + L.w1);
  __nv_bfloat16* w2 = reinterpret_cast<__nv_bfloat16*>(packed + L.w2);
  float* p = reinterpret_cast<float*>(packed + L.params);
  w0[i] = __float2bfloat16_rn(enc ? (c < width ? W0[r * width + c] : 0.f) : W0[i]);
  w1[i] = __float2bfloat16_rn(W1[i]);
  w2[i] = __float2bfloat16_rn(enc ? W2[i] : (r < width ? W2[i] : 0.f));
  if (i < kD) {
    p[i] = b0[i];
    p[kD + i] = b1[i];
    p[2 * kD + i] = enc ? b2[i] : (i < width ? b2[i] : 0.f);
    p[3 * kD + i] = enc ? gamma[i] : 0.f;
    p[4 * kD + i] = enc ? beta[i] : 0.f;
  }
}

struct IoSmem {
  uint32_t w0, w1, w2, stages, params, bars, total;
  __host__ __device__ IoSmem() {
    uint32_t o = 0;
    w0 = o; o += kChunkBytes;
    w1 = o; o += kChunkBytes;
    w2 = o; o += kChunkBytes;
    stages = o; o += uint32_t(kStages) * kChunkBytes;
    params = o; o += 5 * kD * 4;
    bars = o; o += 128;
    total = o;
  }
};
// the tile kernel's barrier slots and TMEM map (mlp_tc.cu)
enum { kIoBarFull = 0, kIoBarEmpty = 2, kIoBarAcc = 4, kIoBarEpi = 10, kIoBarDone = 12, kIoBarTmemPtr = 14 };
constexpr int kIoAccSlots = 3;
constexpr uint32_t kIoAopCol = 384;

struct IoArgs {
  int width;                       // encoder: K; decoder: n_out
  const float* x;                  // encoder input  [rows, K] fp32
  const __nv_bfloat16* xb;         // decoder input  [rows, 128] bf16
  __nv_bfloat16* out_b;            // encoder output [rows, 128] bf16
  float* out_f;                    // decoder output [rows, n_out] fp32
  // backward
  const __nv_bfloat16* grad_ob;    // encoder upstream gradient [rows, 128] bf16
  const float* grad_of;            // decoder upstream gradient [rows, n_out] fp32
  float* grad_xf;                  // encoder raw-feature gradient [rows, K] fp32 (NULL: not requested)
  __nv_bfloat16* grad_xb;          // decoder input gradient [rows, 128] bf16
  __nv_bfloat16 *H1, *H2, *P, *G2, *G1, *G0, *X;   // slab workspaces [slab, 128] (X: the encoder's bf16 input, first 16 ceil(K/16) cols)
};

// acc (+)= A[128 x 16 ksteps] * B with A in TMEM and B a resident weight block: K-major (forward) or MN-major (dgrad)
__device__ __forceinline__ void io_ts_gemm(uint32_t acc, uint32_t a_tmem, uint32_t b_addr, int b_mn, int ksteps, int n) {
  const uint32_t idesc = make_idesc_bf16(128, n, 0, b_mn);
  for (int ks = 0; ks < ksteps; ++ks) {
    const uint64_t bd = b_mn ? sdesc_mnmajor(b_addr + ks * 2048, kPanel) : sdesc_kmajor(b_addr + (ks >> 2) * kPanel + (ks & 3) * 32);
    mma_ts(acc, a_tmem + ks * 8, bd, idesc, ks != 0);
  }
}

// Steps per tile.  Forward: 0:L0 1:L1 2:L2.  Encoder backward adds 3:dH1=dY W2  4:dH0=dH1' W1  [5:dX=dH0' W0, when requested].
// Decoder backward: 0:L0 1:L1 2:dH1=dY W2 3:dH0=dH1' W1 4:dX=dH0' W0 (its last layer's output is not needed).
template <bool kBwd, bool kEnc>
__global__ void __launch_bounds__(kTileThreads, 1)
io_mlp_tc_kernel(int64_t rows, int64_t num_tiles, int64_t slab0, const uint8_t* __restrict__ packed, IoArgs a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const IoSmem S;
  const PackedTc P(1);
  const uint32_t sbase = smem_u32(smem);
  if ((sbase & 1023u) != 0) __trap();
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S.bars);
  float* sparams = reinterpret_cast<float*>(smem + S.params);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n_steps = !kBwd ? 3 : kEnc ? (a.grad_xf != nullptr ? 6 : 5) : 5;
  const int k_steps0 = kEnc ? (a.width + 15) / 16 : 8;      // K=16 steps of layer 0

  {
    load_weight_block(sbase + S.w0, reinterpret_cast<const __nv_bfloat16*>(packed + P.w0), kD, tid, kTileThreads);
    load_weight_block(sbase + S.w1, reinterpret_cast<const __nv_bfloat16*>(packed + P.w1), kD, tid, kTileThreads);
    load_weight_block(sbase + S.w2, reinterpret_cast<const __nv_bfloat16*>(packed + P.w2), kD, tid, kTileThreads);
    cp_async_commit();
    const float* pg = reinterpret_cast<const float*>(packed + P.params);
    for (int i = tid; i < 5 * kD; i += kTileThreads) sparams[i] = pg[i];
    if (tid == 0) {
      for (int s = 0; s < kStages; ++s) { mbar_init(&bars[kIoBarFull + s], kProdThreads / kStages); mbar_init(&bars[kIoBarEmpty + s], 1); }
      for (int s = 0; s < 6; ++s) mbar_init(&bars[kIoBarAcc + s], 1);
      for (int s = 0; s < 2; ++s) { mbar_init(&bars[kIoBarEpi + s], kEpiThreads / 2); mbar_init(&bars[kIoBarDone + s], kEpiThreads / 2); }
      mbar_init_fence();
    }
    if (warp == 12) tmem_alloc<512>(reinterpret_cast<uint32_t*>(&bars[kIoBarTmemPtr]));
    cp_async_wait<0>();
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
  }
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(&bars[kIoBarTmemPtr]);
  const int64_t my_tiles = (num_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x;

  if (warp >= 8 && warp < 12) {
    // =============================== producers: ring slot g holds tile g of this CTA; group g & 1 fills it =============
    const int ptid = tid - kEpiThreads;
    const int group = ptid >> 6;
    const int gt = ptid & 63;
    if (gt == 0) mbar_arrive(&bars[kIoBarEmpty + group]);
    const uint32_t stage_addr = sbase + S.stages + group * kChunkBytes;
    for (int64_t g = group; g < my_tiles; g += 2) {
      mbar_wait(&bars[kIoBarEmpty + group], uint32_t(g >> 1) & 1, 1);
      const int64_t row0 = slab0 + (blockIdx.x + g * gridDim.x) * kTile;
      if (kEnc) {
        // rows gt and gt + 64: K fp32 values -> bf16, 8 columns per 16-byte piece, pieces up to 16 * ceil(K/16) columns
        const int K = a.width, n_pieces = 2 * k_steps0;
#pragma unroll 1
        for (int h = 0; h < 2; ++h) {
          const int r = gt + 64 * h;
          const int64_t grow = row0 + r;
          const bool valid = grow < rows;
          const float* xr = a.x + (valid ? grow : 0) * K;
          __nv_bfloat16* xw = kBwd && valid ? a.X + (grow - slab0) * kD : nullptr;
#pragma unroll 1
          for (int pc = 0; pc < n_pieces; ++pc) {
            float f[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) { const int col = pc * 8 + j; f[j] = valid && col < K ? __ldg(xr + col) : 0.f; }
            uint32_t w[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) w[j] = pack_bf16(f[2 * j], f[2 * j + 1]);
            st_shared128(stage_addr + (pc >> 3) * kPanel + sw128_chunk(r, pc & 7), w);
            if (xw != nullptr) *reinterpret_cast<uint4*>(xw + pc * 8) = make_uint4(w[0], w[1], w[2], w[3]);
          }
        }
      } else {
        const int c16 = gt & 15, rbase = gt >> 4;   // piece c16 of rows rbase + 4 j
#pragma unroll 4
        for (int j = 0; j < 32; ++j) {
          const int64_t grow = row0 + rbase + 4 * j;
          const bool valid = grow < rows;
          cp_async16_zfill(stage_addr + (c16 >> 3) * kPanel + sw128_chunk(rbase + 4 * j, c16 & 7), a.xb + (valid ? grow : 0) * kD + c16 * 8, valid);
        }
        cp_async_commit();
        cp_async_wait<0>();
      }
      fence_async_smem();
      mbar_arrive(&bars[kIoBarFull + group]);
    }
  } else if (warp == 12) {
    // =============================== MMA warp (lane 0 issues) =====================================
    const uint32_t idesc_kk = make_idesc_bf16(128, 128, 0, 0);
    int64_t t_l0 = 0, done = 0;
    int64_t wg_tile[2] = {0, 1};
    int wg_step[2] = {0, 0};
    uint32_t wg_sig[2] = {0, 0}, wg_fin[2] = {0, 0};
    uint32_t acc_busy = 0, idle = 0;
    while (done < my_tiles) {
      bool progressed = false;
      uint32_t ev = 0;
      if (lane == 0) {
#pragma unroll
        for (int w = 0; w < 2; ++w)
          if (wg_tile[w] < t_l0 &&
              (wg_step[w] == n_steps - 1 ? mbar_test(&bars[kIoBarDone + w], wg_fin[w] & 1) : mbar_test(&bars[kIoBarEpi + w], wg_sig[w] & 1)))
            ev |= 1u << w;
        if (t_l0 < my_tiles && !((acc_busy >> int(t_l0 % kIoAccSlots)) & 1u) &&
            mbar_test(&bars[kIoBarFull + int(t_l0 & 1)], uint32_t(t_l0 >> 1) & 1)) ev |= 4u;
      }
      ev = __shfl_sync(0xffffffffu, ev, 0);
#pragma unroll
      for (int w = 0; w < 2; ++w) {
        const int64_t t = wg_tile[w];
        if ((ev >> w) & 1u) {
          fence_after_sync();
          const int k = wg_step[w]++;
          const int slot = int(t % kIoAccSlots);
          if (k == n_steps - 1) {
            ++wg_fin[w];
            acc_busy &= ~(1u << slot);
            wg_tile[w] += 2;
            wg_step[w] = 0;
            ++done;
          } else {
            ++wg_sig[w];
            const int step = k + 1;
            const uint32_t acc = tmem_base + slot * 128;
            const uint32_t aop = tmem_base + kIoAopCol + w * 64;
            if (lane == 0) {
              if (step == 1) io_ts_gemm(acc, aop, sbase + S.w1, 0, 8, 128);
              else if (!kBwd || kEnc) {
                if (step == 2) io_ts_gemm(acc, aop, sbase + S.w2, 0, 8, kEnc ? 128 : 16);
                else if (step == 3) io_ts_gemm(acc, aop, sbase + S.w2, 1, 8, 128);
                else if (step == 4) io_ts_gemm(acc, aop, sbase + S.w1, 1, 8, 128);
                else io_ts_gemm(acc, aop, sbase + S.w0, 1, 8, 128);
              } else {
                if (step == 2) io_ts_gemm(acc, aop, sbase + S.w2, 1, 1, 128);   // dY [128 x 16] W2[0:16, :]
                else if (step == 3) io_ts_gemm(acc, aop, sbase + S.w1, 1, 8, 128);
                else io_ts_gemm(acc, aop, sbase + S.w0, 1, 8, 128);
              }
              mma_commit(&bars[kIoBarAcc + int(t % 6)]);
            }
            __syncwarp();
          }
          progressed = true;
        }
      }
      if (ev & 4u) {
        const int slot = int(t_l0 % kIoAccSlots);
        const int stage = int(t_l0 & 1);
        fence_after_sync();
        if (lane == 0) {
          const uint32_t acc = tmem_base + slot * 128;
          const uint32_t a_addr = sbase + S.stages + stage * kChunkBytes;
          for (int ks = 0; ks < k_steps0; ++ks) {
            const uint32_t koff = (ks >> 2) * kPanel + (ks & 3) * 32;
            mma_ss(acc, sdesc_kmajor(a_addr + koff), sdesc_kmajor(sbase + S.w0 + koff), idesc_kk, ks != 0);
          }
          mma_commit(&bars[kIoBarEmpty + stage]);
          mma_commit(&bars[kIoBarAcc + int(t_l0 % 6)]);
        }
        __syncwarp();
        acc_busy |= 1u << slot;
        ++t_l0;
        progressed = true;
      }
      if (!progressed) {
        __nanosleep(20);
        if (++idle > (1u << 22)) {
          if (lane == 0)
            debug_record(910u + uint32_t(kBwd) + 2u * uint32_t(kEnc), uint32_t(t_l0), uint32_t(done) | (uint32_t(my_tiles) << 16),
                         uint32_t(wg_tile[0]) | (uint32_t(wg_tile[1]) << 16), uint32_t(wg_step[0]) | (uint32_t(wg_step[1]) << 8) | (acc_busy << 16),
                         wg_sig[0] | (wg_sig[1] << 16), 0);
          __trap();
        }
      } else {
        idle = 0;
      }
    }
  } else {
    // =============================== epilogue groups ==============================================
    const int wg = warp >> 2;
    const int r = (warp & 3) * 32 + lane;
    const uint32_t lane_addr = uint32_t((warp & 3) * 32) << 16;
    const uint32_t aop = tmem_base + kIoAopCol + wg * 64 + lane_addr;
    const float* b2 = sparams + 2 * kD;
    const float* gam = sparams + 3 * kD;
    const float* bet = sparams + 4 * kD;
    for (int64_t it = wg; it < my_tiles; it += 2) {
      const int slot = int(it % kIoAccSlots);
      const uint32_t acc = tmem_base + slot * 128 + lane_addr;
      uint32_t acc_phase = uint32_t((it / 6) * n_steps);
      uint32_t steps_done = 0;
      auto wait_acc = [&]() {
        mbar_wait(&bars[kIoBarAcc + int(it % 6)], acc_phase & 1, 100 + int(steps_done));
        ++acc_phase;
        fence_after_sync();
      };
      auto signal_done = [&]() {
        fence_before_sync();
        mbar_arrive(&bars[(++steps_done == uint32_t(n_steps) ? kIoBarDone : kIoBarEpi) + wg]);
      };
      const int64_t grow = slab0 + (blockIdx.x + it * gridDim.x) * kTile + r;
      const bool valid = grow < rows;
      const int64_t lrow = valid ? grow - slab0 : 0;
      uint32_t mask1[4] = {0, 0, 0, 0}, mask2[4] = {0, 0, 0, 0};
      // ---- hidden layers: bias + ReLU -> bf16 A operand in TMEM ----------------------------------
#pragma unroll 1
      for (int layer = 0; layer < 2; ++layer) {
        wait_acc();
        const float* bias = sparams + layer * kD;
        const bool to_aop = kEnc || !kBwd || layer == 0;   // the decoder backward puts dY there after the last hidden layer
        __nv_bfloat16* hws = kBwd ? (layer == 0 ? a.H1 : a.H2) + lrow * kD : nullptr;
#pragma unroll 1
        for (int cg = 0; cg < 4; ++cg) {
          uint32_t v[32];
          tmem_ld32(acc + cg * 32, v);
          tmem_ld_wait();
          uint32_t h[16];
          uint32_t m = 0;
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float x0 = fmaxf(__uint_as_float(v[2 * j]) + bias[cg * 32 + 2 * j], 0.f);
            const float x1 = fmaxf(__uint_as_float(v[2 * j + 1]) + bias[cg * 32 + 2 * j + 1], 0.f);
            h[j] = pack_bf16(x0, x1);
            if (kBwd) m |= (x0 > 0.f ? (1u << (2 * j)) : 0u) | (x1 > 0.f ? (1u << (2 * j + 1)) : 0u);
          }
          if (to_aop) {
            tmem_st8(aop + cg * 16, h);
            tmem_st8(aop + cg * 16 + 8, h + 8);
          }
          if (kBwd) {
            if (layer == 0) mask1[cg] = m; else mask2[cg] = m;
            if (valid) { stg256(hws + cg * 32, h); stg256(hws + cg * 32 + 16, h + 8); }
          }
        }
        if (!kEnc && kBwd && layer == 1) {
          // decoder upstream gradient: n_out fp32 values -> bf16 A operand [128 x 16]; G2 keeps them for dW2 / db2 (columns >= 16
          // of a G2 row are never written: they only reach the rows of dW2 and entries of db2 beyond n_out, which are dropped)
          uint32_t gw[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float g0 = valid && 2 * j < a.width ? a.grad_of[grow * a.width + 2 * j] : 0.f;
            const float g1 = valid && 2 * j + 1 < a.width ? a.grad_of[grow * a.width + 2 * j + 1] : 0.f;
            gw[j] = pack_bf16(g0, g1);
          }
          tmem_st8(aop, gw);
          if (valid) stg256(a.G2 + lrow * kD, gw);
        }
        tmem_st_wait();
        signal_done();
      }
      if (!kBwd && !kEnc) {
        // ---- decoder output: acc[:, 0:16] + b2 in fp32, n_out values per row -------------------------
        wait_acc();
        uint32_t v[16];
        tmem_ld16(acc, v);
        tmem_ld_wait();
        if (valid) {
          float* op = a.out_f + grow * a.width;
#pragma unroll
          for (int j = 0; j < 16; ++j)
            if (j < a.width) op[j] = __uint_as_float(v[j]) + b2[j];
        }
        signal_done();
        continue;
      }
      if (kEnc) {
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
          __nv_bfloat16* op = a.out_b + (valid ? grow : 0) * kD;
#pragma unroll 1
          for (int cg = 0; cg < 4; ++cg) {
            uint32_t v[32];
            tmem_ld32(acc + cg * 32, v);
            tmem_ld_wait();
            if (valid) {
              uint32_t ow[16];
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                const int col = cg * 32 + 2 * j;
                const float y0 = (__uint_as_float(v[2 * j]) + b2[col] - mean) * rstd * gam[col] + bet[col];
                const float y1 = (__uint_as_float(v[2 * j + 1]) + b2[col + 1] - mean) * rstd * gam[col + 1] + bet[col + 1];
                ow[j] = pack_bf16(y0, y1);
              }
              stg256(op + cg * 32, ow);
              stg256(op + cg * 32 + 16, ow + 8);
            }
          }
          signal_done();
          continue;
        }
        // ---- LayerNorm backward -> dY (A operand); P = dO * yhat for the gamma gradient --------------
        const __nv_bfloat16* gop = a.grad_ob + (valid ? grow : 0) * kD;
        __nv_bfloat16* pws = a.P + lrow * kD;
        float m1 = 0.f, m2 = 0.f;
#pragma unroll 1
        for (int cg = 0; cg < 4; ++cg) {
          uint32_t v[32];
          tmem_ld32(acc + cg * 32, v);
          tmem_ld_wait();
          uint32_t gw[16], pw[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) gw[j] = 0u;
          if (valid) { ldg256(gop + cg * 32, gw); ldg256(gop + cg * 32 + 16, gw + 8); }
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
          if (valid) { stg256(pws + cg * 32, pw); stg256(pws + cg * 32 + 16, pw + 8); }
          tmem_st8(aop + cg * 16, gw);
          tmem_st8(aop + cg * 16 + 8, gw + 8);
        }
        tmem_st_wait();
        m1 *= (1.0f / kD);
        m2 *= (1.0f / kD);
        __nv_bfloat16* g2ws = a.G2 + lrow * kD;
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
          if (valid) { stg256(g2ws + cg * 32, o); stg256(g2ws + cg * 32 + 16, o + 8); }
        }
        tmem_st_wait();
        signal_done();
      }
      // ---- dH1' = (dY W2) * [H1 > 0] ; dH0' = (dH1' W1) * [H0 > 0] ------------------------------------
#pragma unroll 1
      for (int layer = 1; layer >= 0; --layer) {
        wait_acc();
        __nv_bfloat16* gws = (layer == 1 ? a.G1 : a.G0) + lrow * kD;
#pragma unroll 1
        for (int cg = 0; cg < 4; ++cg) {
          uint32_t v[32];
          tmem_ld32(acc + cg * 32, v);
          tmem_ld_wait();
          const uint32_t m = layer == 1 ? mask2[cg] : mask1[cg];
          uint32_t o[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float x0 = (m >> (2 * j)) & 1u ? __uint_as_float(v[2 * j]) : 0.f;
            const float x1 = (m >> (2 * j + 1)) & 1u ? __uint_as_float(v[2 * j + 1]) : 0.f;
            o[j] = pack_bf16(x0, x1);
          }
          tmem_st8(aop + cg * 16, o);
          tmem_st8(aop + cg * 16 + 8, o + 8);
          if (valid) { stg256(gws + cg * 32, o); stg256(gws + cg * 32 + 16, o + 8); }
        }
        tmem_st_wait();
        signal_done();
      }
      // ---- input gradient dX = dH0' W0 ----------------------------------------------------------------
      if (kEnc && a.grad_xf != nullptr) {
        wait_acc();
        const int K = a.width;
#pragma unroll 1
        for (int cg = 0; cg < (K + 31) / 32; ++cg) {    // warp-uniform
          uint32_t v[32];
          tmem_ld32(acc + cg * 32, v);
          tmem_ld_wait();
          if (valid) {
            float* dp = a.grad_xf + grow * K;
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (cg * 32 + j < K) dp[cg * 32 + j] = __uint_as_float(v[j]);
          }
        }
        signal_done();
      } else if (!kEnc) {
        wait_acc();
        __nv_bfloat16* dp = a.grad_xb + (valid ? grow : 0) * kD;
#pragma unroll 1
        for (int cg = 0; cg < 4; ++cg) {
          uint32_t v[32];
          tmem_ld32(acc + cg * 32, v);
          tmem_ld_wait();
          if (valid) {
            uint32_t ow[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) ow[j] = pack_bf16(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
            stg256(dp + cg * 32, ow);
            stg256(dp + cg * 32 + 16, ow + 8);
          }
        }
        signal_done();
      }
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 12) tmem_dealloc<512>(tmem_base);
}

// Fixed-order reduction of the per-CTA weight-gradient partials (z = 0: W0, 1: W1, 2: W2 of tc_io_wgrad) and copy of the column
// sums into the parameter shapes: gW0 [128, K] (encoder) / [128, 128], gW2 [n_out, 128] (decoder) / [128, 128].
__global__ void io_reduce_kernel(const float* __restrict__ partial, int parts, const float* __restrict__ vec, int enc, int width,
                                 float* gW0, float* gW1, float* gW2, float* gb0, float* gb1, float* gb2, float* ggamma, float* gbeta) {
  const int64_t blk = int64_t(kD) * kD;
  const int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  const int z = int(blockIdx.y);
  if (i >= blk) {
    // vector gradients: colsum5 order G2, G1, G0, P, dO -> b2, b1, b0, gamma, beta
    const int64_t j = i - blk;
    if (j >= 5 * kD || z != 0) return;
    const int which = int(j / kD), c = int(j % kD);
    const float v = vec[j];
    if (which == 0) { if (enc || c < width) gb2[c] = v; }
    else if (which == 1) gb1[c] = v;
    else if (which == 2) gb0[c] = v;
    else if (enc && which == 3) ggamma[c] = v;
    else if (enc && which == 4) gbeta[c] = v;
    return;
  }
  const int o = int(i / kD), c = int(i % kD);
  if (z == 0 && enc && c >= width) return;
  if (z == 2 && !enc && o >= width) return;
  const float s = ordered_sum(partial + int64_t(z) * blk + i, parts, 3 * blk);
  if (z == 0) gW0[enc ? o * width + c : i] = s;
  else if (z == 1) gW1[i] = s;
  else gW2[i] = s;
}

// ---- host side -----------------------------------------------------------------------------------------
int tc_io_wgrad(int64_t rows, int64_t slab0, int64_t slab_rows, int parts, const void* X, int64_t x_row_offset, const void* G2, const void* H2,
                const void* G1, const void* H1, const void* G0, float* partial, int accumulate, cudaStream_t st);   // mlp_tc.cu

static int io_configure() {
  static bool configured = false;
  if (!configured) {
    uint32_t* dbg = debug_buffer_device();
    HGN_CUDA_OK(cudaMemcpyToSymbol(tc05::g_debug_words, &dbg, sizeof(dbg)));
    const int smem = int(IoSmem().total);
    HGN_CUDA_OK(cudaFuncSetAttribute(io_mlp_tc_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    HGN_CUDA_OK(cudaFuncSetAttribute(io_mlp_tc_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    HGN_CUDA_OK(cudaFuncSetAttribute(io_mlp_tc_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    HGN_CUDA_OK(cudaFuncSetAttribute(io_mlp_tc_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    configured = true;
  }
  return HGN_OK;
}

struct IoBwdLayout {
  int64_t slab_rows, parts;
  size_t act[7], partial, vec_partial, vec, total;   // act: H1 H2 P G2 G1 G0 X
};

static IoBwdLayout io_bwd_layout(int64_t rows, bool enc) {
  IoBwdLayout L{};
  const int64_t cap = int64_t(1) << 21;                      // <= 2M rows per pass, as the tile kernel
  L.slab_rows = rows < cap ? (rows > 0 ? rows : 1) : cap;
  L.slab_rows = ceil_div(L.slab_rows, kTile) * kTile;
  L.parts = L.slab_rows >= int64_t(tc_sm_count()) * 256 ? tc_sm_count() : ceil_div(L.slab_rows, 256);
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
  for (int i = 0; i < 7; ++i) {
    const bool used = enc || (i != 2 && i != 6);               // the decoder has no LayerNorm (P) and reads its input in place (X)
    L.act[i] = used ? take(size_t(L.slab_rows) * kD * 2) : 0;
  }
  L.partial = take(size_t(L.parts) * 3 * kD * kD * 4);
  L.vec_partial = take(colsum5_workspace_bytes(L.slab_rows));
  L.vec = take(5 * kD * 4);
  L.total = off;
  return L;
}

static int io_backward(bool enc, int64_t rows, int width, const void* x, const void* packed, const void* grad_out, void* grad_x,
                       float* gW0, float* gb0, float* gW1, float* gb1, float* gW2, float* gb2, float* ggamma, float* gbeta,
                       void* workspace, size_t workspace_bytes, cudaStream_t st) {
  const char* who = enc ? "encoder_backward" : "decoder_backward";
  const IoBwdLayout L = io_bwd_layout(rows, enc);
  if (workspace_bytes < L.total) { set_error("%s: workspace %zu < %zu", who, workspace_bytes, L.total); return HGN_ERR_WORKSPACE; }
  if (int rc = io_configure()) return rc;
  char* ws = static_cast<char*>(workspace);
  auto act = [&](int i) { return reinterpret_cast<__nv_bfloat16*>(ws + L.act[i]); };
  IoArgs a{};
  a.width = width;
  if (enc) { a.x = static_cast<const float*>(x); a.grad_ob = static_cast<const __nv_bfloat16*>(grad_out); a.grad_xf = static_cast<float*>(grad_x); }
  else { a.xb = static_cast<const __nv_bfloat16*>(x); a.grad_of = static_cast<const float*>(grad_out); a.grad_xb = static_cast<__nv_bfloat16*>(grad_x); }
  a.H1 = act(0); a.H2 = act(1); a.P = enc ? act(2) : nullptr; a.G2 = act(3); a.G1 = act(4); a.G0 = act(5); a.X = enc ? act(6) : nullptr;
  float* partial = reinterpret_cast<float*>(ws + L.partial);
  float* vec = reinterpret_cast<float*>(ws + L.vec);
  float* vec_out[5] = {vec, vec + kD, vec + 2 * kD, vec + 3 * kD, vec + 4 * kD};
  const IoSmem S;
  int pass = 0;
  for (int64_t slab0 = 0; slab0 < rows || pass == 0; slab0 += L.slab_rows, ++pass) {
    const int64_t this_rows = rows - slab0 < L.slab_rows ? rows - slab0 : L.slab_rows;
    if (this_rows > 0) {
      const int64_t tiles = ceil_div(this_rows, kTile);
      const unsigned grid = unsigned(tiles < tc_sm_count() ? tiles : tc_sm_count());
      HGN_TIMED(enc ? "encoder_tc_bwd" : "decoder_tc_bwd", st);
      if (enc) io_mlp_tc_kernel<true, true><<<grid, kTileThreads, S.total, st>>>(rows, tiles, slab0, static_cast<const uint8_t*>(packed), a);
      else io_mlp_tc_kernel<true, false><<<grid, kTileThreads, S.total, st>>>(rows, tiles, slab0, static_cast<const uint8_t*>(packed), a);
      HGN_LAUNCH_OK(who);
    }
    // dW0 = G0^T X: the encoder's bf16 X rows are slab-local, the decoder reads its input rows in place
    const void* xs = enc ? static_cast<const void*>(a.X) : x;
    if (int rc = tc_io_wgrad(rows, slab0, L.slab_rows, int(L.parts), xs, enc ? -slab0 : 0, a.G2, a.H2, a.G1, a.H1, a.G0, partial, pass > 0, st))
      return rc;
    const void* mats[5] = {a.G2, a.G1, a.G0, a.P, enc && grad_out ? static_cast<const void*>(a.grad_ob + slab0 * kD) : nullptr};
    if (int rc = colsum5_bf16(mats, vec_out, this_rows > 0 ? this_rows : 0, pass > 0, ws + L.vec_partial, colsum5_workspace_bytes(L.slab_rows), st))
      return rc;
    if (rows == 0) break;
  }
  const int64_t blk = int64_t(kD) * kD;
  HGN_TIMED("io_reduce", st);
  io_reduce_kernel<<<dim3(unsigned(ceil_div(blk + 5 * kD, 256)), 3), 256, 0, st>>>(partial, int(L.parts), vec, enc ? 1 : 0, width, gW0, gW1,
                                                                                 gW2, gb0, gb1, gb2, ggamma, gbeta);
  HGN_LAUNCH_OK("io_reduce");
  return HGN_OK;
}

}  // namespace hgn

using namespace hgn;

extern "C" size_t hgn_io_mlp_packed_bytes(void) { return PackedTc(1).total; }

extern "C" int hgn_io_mlp_pack(int32_t kind, int32_t width, const float* W0, const float* b0, const float* W1, const float* b1, const float* W2,
                               const float* b2, const float* gamma, const float* beta, void* packed, void* stream) {
  HGN_CHECK_ARG(kind == HGN_IO_ENCODER || kind == HGN_IO_DECODER, "io_mlp_pack: kind=%d", kind);
  const bool enc = kind == HGN_IO_ENCODER;
  HGN_CHECK_ARG(width >= 1 && width <= (enc ? kD : HGN_IO_MAX_OUT), "io_mlp_pack: %s=%d outside [1,%d]", enc ? "K" : "n_out", width,
                enc ? kD : HGN_IO_MAX_OUT);
  HGN_CHECK_ARG(W0 && b0 && W1 && b1 && W2 && b2 && packed && (!enc || (gamma && beta)), "io_mlp_pack: null pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  HGN_TIMED("io_pack_tc", st);
  io_pack_kernel<<<kD * kD / 256, 256, 0, st>>>(enc ? 1 : 0, width, W0, b0, W1, b1, W2, b2, gamma, beta, static_cast<uint8_t*>(packed));
  HGN_LAUNCH_OK("io_pack_tc");
  return HGN_OK;
}

extern "C" int hgn_encoder_forward(int64_t rows, int32_t k_in, const float* x, const void* packed, void* out, void* stream) {
  HGN_CHECK_ARG(rows >= 0 && rows < (int64_t(1) << 31), "encoder_forward: rows=%lld", (long long)rows);
  HGN_CHECK_ARG(k_in >= 1 && k_in <= kD, "encoder_forward: K=%d outside [1,%d]", k_in, kD);
  if (rows == 0) return HGN_OK;
  HGN_CHECK_ARG(x && packed && out, "encoder_forward: null pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int rc = io_configure()) return rc;
  IoArgs a{};
  a.width = k_in; a.x = x; a.out_b = static_cast<__nv_bfloat16*>(out);
  const int64_t tiles = ceil_div(rows, kTile);
  const unsigned grid = unsigned(tiles < tc_sm_count() ? tiles : tc_sm_count());
  HGN_TIMED("encoder_tc_fwd", st);
  io_mlp_tc_kernel<false, true><<<grid, kTileThreads, IoSmem().total, st>>>(rows, tiles, 0, static_cast<const uint8_t*>(packed), a);
  HGN_LAUNCH_OK("encoder_tc_fwd");
  return HGN_OK;
}

extern "C" int hgn_decoder_forward(int64_t rows, int32_t n_out, const void* x, const void* packed, float* out, void* stream) {
  HGN_CHECK_ARG(rows >= 0 && rows < (int64_t(1) << 31), "decoder_forward: rows=%lld", (long long)rows);
  HGN_CHECK_ARG(n_out >= 1 && n_out <= HGN_IO_MAX_OUT, "decoder_forward: n_out=%d outside [1,%d]", n_out, HGN_IO_MAX_OUT);
  if (rows == 0) return HGN_OK;
  HGN_CHECK_ARG(x && packed && out, "decoder_forward: null pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int rc = io_configure()) return rc;
  IoArgs a{};
  a.width = n_out; a.xb = static_cast<const __nv_bfloat16*>(x); a.out_f = out;
  const int64_t tiles = ceil_div(rows, kTile);
  const unsigned grid = unsigned(tiles < tc_sm_count() ? tiles : tc_sm_count());
  HGN_TIMED("decoder_tc_fwd", st);
  io_mlp_tc_kernel<false, false><<<grid, kTileThreads, IoSmem().total, st>>>(rows, tiles, 0, static_cast<const uint8_t*>(packed), a);
  HGN_LAUNCH_OK("decoder_tc_fwd");
  return HGN_OK;
}

extern "C" size_t hgn_encoder_backward_workspace_bytes(int64_t rows, int32_t k_in) {
  if (rows < 0 || k_in < 1 || k_in > kD) return 0;
  return io_bwd_layout(rows, true).total;
}

extern "C" size_t hgn_decoder_backward_workspace_bytes(int64_t rows, int32_t n_out) {
  if (rows < 0 || n_out < 1 || n_out > HGN_IO_MAX_OUT) return 0;
  return io_bwd_layout(rows, false).total;
}

extern "C" int hgn_encoder_backward(int64_t rows, int32_t k_in, const float* x, const void* packed, const void* grad_out, float* grad_x,
                                    float* grad_W0, float* grad_b0, float* grad_W1, float* grad_b1, float* grad_W2, float* grad_b2,
                                    float* grad_gamma, float* grad_beta, void* workspace, size_t workspace_bytes, void* stream) {
  HGN_CHECK_ARG(rows >= 0 && rows < (int64_t(1) << 31), "encoder_backward: rows=%lld", (long long)rows);
  HGN_CHECK_ARG(k_in >= 1 && k_in <= kD, "encoder_backward: K=%d outside [1,%d]", k_in, kD);
  HGN_CHECK_ARG(packed && workspace && grad_W0 && grad_b0 && grad_W1 && grad_b1 && grad_W2 && grad_b2 && grad_gamma && grad_beta,
                "encoder_backward: null pointer");
  HGN_CHECK_ARG(rows == 0 || (x && grad_out), "encoder_backward: null pointer");
  return io_backward(true, rows, k_in, x, packed, grad_out, grad_x, grad_W0, grad_b0, grad_W1, grad_b1, grad_W2, grad_b2, grad_gamma,
                     grad_beta, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

extern "C" int hgn_decoder_backward(int64_t rows, int32_t n_out, const void* x, const void* packed, const float* grad_out, void* grad_x,
                                    float* grad_W0, float* grad_b0, float* grad_W1, float* grad_b1, float* grad_W2, float* grad_b2,
                                    void* workspace, size_t workspace_bytes, void* stream) {
  HGN_CHECK_ARG(rows >= 0 && rows < (int64_t(1) << 31), "decoder_backward: rows=%lld", (long long)rows);
  HGN_CHECK_ARG(n_out >= 1 && n_out <= HGN_IO_MAX_OUT, "decoder_backward: n_out=%d outside [1,%d]", n_out, HGN_IO_MAX_OUT);
  HGN_CHECK_ARG(packed && workspace && grad_W0 && grad_b0 && grad_W1 && grad_b1 && grad_W2 && grad_b2, "decoder_backward: null pointer");
  HGN_CHECK_ARG(rows == 0 || (x && grad_out && grad_x), "decoder_backward: null pointer");
  return io_backward(false, rows, n_out, x, packed, grad_out, grad_x, grad_W0, grad_b0, grad_W1, grad_b1, grad_W2, grad_b2, nullptr, nullptr,
                     workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}
