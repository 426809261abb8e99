// Long segments (HyperGraphNet cluster pooling and broadcast at mesh scale): a segment of more than HGN_SEGMENT_SPLIT_THRESHOLD
// elements is cut into pieces of HGN_SEGMENT_SPLIT_PIECE consecutive perm positions, and every piece of a call gets its own half
// warp, so a call keeps all of its pieces' row loads in flight together instead of walking each cluster one round at a time.
// The short segments still run through the kernels of segment.cu, unchanged, on the split's short CSR.  bf16 rows of width 128.
//
// Arithmetic (see include/hgn_b200.h): piece partials are fp32 sums from +0 in perm order, combined in ascending piece order; max /
// min winners keep the sequential first-in-order result (strict comparisons at both stages); backward terms are per element, with
// the arithmetic of segment_bwd_bf16_128_kernel (g_mean * inv contracted into the g_sum term with a fused multiply-add, as that
// kernel compiles) and segment_layer_grad_bf16_128_kernel (no contraction).  No floating-point atomics.
#include <cub/device/device_scan.cuh>

#include "common.cuh"

namespace hgn {

constexpr int kSplitT = HGN_SEGMENT_SPLIT_THRESHOLD;
constexpr int kSplitP = HGN_SEGMENT_SPLIT_PIECE;
static_assert(kSplitT >= kSplitP, "a long segment has at least two pieces");

// ------------------------------------------------------------------------------------------------
// split build
// ------------------------------------------------------------------------------------------------
// per segment (and a zero at index S, so that the exclusive scans end with the totals): is it long, its piece count, its short length
__global__ void split_count_kernel(const int32_t* __restrict__ rowptr, int64_t S, int32_t* __restrict__ c_long,
                                   int32_t* __restrict__ c_pieces, int32_t* __restrict__ c_short) {
  const int64_t s = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (s > S) return;
  const int len = s < S ? rowptr[s + 1] - rowptr[s] : 0;
  const bool lng = len > kSplitT;
  c_long[s] = lng;
  c_pieces[s] = lng ? (len + kSplitP - 1) / kSplitP : 0;
  c_short[s] = lng ? 0 : len;
}

__global__ void split_totals_kernel(const int32_t* __restrict__ o_long, const int32_t* __restrict__ o_pieces,
                                    const int32_t* __restrict__ rowptr_short, int64_t S, int32_t* __restrict__ piece_ptr,
                                    int32_t* __restrict__ totals) {
  totals[0] = o_long[S];
  totals[1] = o_pieces[S];
  totals[2] = rowptr_short[S];
  piece_ptr[o_long[S]] = o_pieces[S];
}

// one warp per segment: a long one writes its id, its first piece and its pieces; a short one copies its elements
__global__ void __launch_bounds__(256)
split_fill_kernel(const int32_t* __restrict__ perm, const int32_t* __restrict__ rowptr, int64_t S, const int32_t* __restrict__ o_long,
                  const int32_t* __restrict__ o_pieces, const int32_t* __restrict__ rowptr_short, int32_t* __restrict__ long_ids,
                  int32_t* __restrict__ piece_ptr, int32_t* __restrict__ pieces, int32_t* __restrict__ perm_short) {
  const int lane = threadIdx.x & 31;
  const int64_t s = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
  if (s >= S) return;
  const int beg = rowptr[s], end = rowptr[s + 1], len = end - beg;
  if (len > kSplitT) {
    const int i = o_long[s], p0 = o_pieces[s], np = (len + kSplitP - 1) / kSplitP;
    if (lane == 0) { long_ids[i] = int32_t(s); piece_ptr[i] = p0; }
    for (int k = lane; k < np; k += 32) {
      pieces[3 * int64_t(p0 + k)] = int32_t(s);
      pieces[3 * int64_t(p0 + k) + 1] = beg + k * kSplitP;
      pieces[3 * int64_t(p0 + k) + 2] = min(beg + (k + 1) * kSplitP, end);
    }
  } else {
    const int o = rowptr_short[s];
    for (int j = lane; j < len; j += 32) perm_short[o + j] = perm[beg + j];
  }
}

struct SplitLayout {
  size_t c_long, c_pieces, c_short, o_long, o_pieces, totals, cub, total;
  size_t cub_bytes;
};

static SplitLayout split_layout(int64_t S) {
  SplitLayout L{};
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
  const size_t n = size_t(S + 1) * 4;
  L.c_long = take(n);
  L.c_pieces = take(n);
  L.c_short = take(n);
  L.o_long = take(n);
  L.o_pieces = take(n);
  L.totals = take(16);
  cub::DeviceScan::ExclusiveSum(nullptr, L.cub_bytes, (const int32_t*)nullptr, (int32_t*)nullptr, int(S + 1));
  L.cub = take(L.cub_bytes);
  L.total = off;
  return L;
}

// ------------------------------------------------------------------------------------------------
// forward: per piece fp32 partials, then per long segment a combine in ascending piece order
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void unpack8(const uint4& p, float (&f)[8]) {
  const uint32_t w[4] = {p.x, p.y, p.z, p.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) { f[2 * i] = __uint_as_float(w[i] << 16); f[2 * i + 1] = __uint_as_float(w[i] & 0xFFFF0000u); }
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  uint32_t w[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    __nv_bfloat162 t = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
    w[i] = *reinterpret_cast<uint32_t*>(&t);
  }
  return make_uint4(w[0], w[1], w[2], w[3]);
}
__device__ __forceinline__ void store8f(float* p, const float (&f)[8]) {
  reinterpret_cast<float4*>(p)[0] = make_float4(f[0], f[1], f[2], f[3]);
  reinterpret_cast<float4*>(p)[1] = make_float4(f[4], f[5], f[6], f[7]);
}
__device__ __forceinline__ void store8i(int32_t* p, const int (&a)[8]) {
  reinterpret_cast<int4*>(p)[0] = make_int4(a[0], a[1], a[2], a[3]);
  reinterpret_cast<int4*>(p)[1] = make_int4(a[4], a[5], a[6], a[7]);
}

// Half a warp per piece, 16 bytes (8 features) per lane and row, sixteen rows in flight per lane (eight with max / min): the up-pooling shape (10^6 rows in
// 16 segments) is ~3900 pieces, ~16 MB of loads in flight.  Piece rows are summed from +0 in perm order; a zero row stands in for
// the positions past the piece's end (adding +0 to a sum from +0 changes no bit), the max / min skip them.
template <bool MINMAX>
__global__ void __launch_bounds__(256)
segment_long_partial_kernel(const __nv_bfloat16* __restrict__ data, const int32_t* __restrict__ perm, const int32_t* __restrict__ pieces,
                            int64_t n_pieces, float* __restrict__ p_sum, float* __restrict__ p_max, float* __restrict__ p_min,
                            int32_t* __restrict__ p_amx, int32_t* __restrict__ p_amn, const __nv_bfloat16* prior,
                            __nv_bfloat16* __restrict__ prior_save) {
  const int l16 = threadIdx.x & 15;
  const uint32_t hmask = 0xFFFFu << (threadIdx.x & 16);
  const int64_t k = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 4;
  if (k >= n_pieces) return;                                // whole half-warps leave together
  const int seg = __ldg(pieces + 3 * k), beg = __ldg(pieces + 3 * k + 1), end = __ldg(pieces + 3 * k + 2);
  if (prior_save && (k == 0 || __ldg(pieces + 3 * (k - 1)) != seg))   // a segment's first piece keeps the caller's prior row
    reinterpret_cast<uint4*>(prior_save + k * 128)[l16] = reinterpret_cast<const uint4*>(prior + int64_t(seg) * 128)[l16];
  float s[8], mx[8], mn[8];
  int ax[8], an[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { s[i] = 0.f; mx[i] = -INFINITY; mn[i] = INFINITY; ax[i] = -1; an[i] = -1; }
  constexpr int R = MINMAX ? 8 : 16;                        // rows in flight per lane (the winners need the registers)
  for (int j = beg; j < end; j += R) {
    const int mine = l16 < R && j + l16 < end ? __ldg(perm + j + l16) : -1;
    int e[R];
    uint4 v[R];
#pragma unroll
    for (int q = 0; q < R; ++q) {
      e[q] = __shfl_sync(hmask, mine, q, 16);
      v[q] = make_uint4(0u, 0u, 0u, 0u);
      if (e[q] >= 0) v[q] = __ldg(reinterpret_cast<const uint4*>(data + int64_t(e[q]) * 128) + l16);
    }
#pragma unroll
    for (int q = 0; q < R; ++q) {
      float f[8];
      unpack8(v[q], f);
#pragma unroll
      for (int i = 0; i < 8; ++i) s[i] = __fadd_rn(s[i], f[i]);
      if (MINMAX && e[q] >= 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          if (f[i] > mx[i]) { mx[i] = f[i]; ax[i] = e[q]; }
          if (f[i] < mn[i]) { mn[i] = f[i]; an[i] = e[q]; }
        }
      }
    }
  }
  const int64_t o = k * 128 + l16 * 8;
  store8f(p_sum + o, s);
  if (MINMAX) { store8f(p_max + o, mx); store8f(p_min + o, mn); store8i(p_amx + o, ax); store8i(p_amn + o, an); }
}

// One 128-thread block per long segment, thread = feature: the partials are combined in ascending piece order (sum from +0, strict
// comparisons for max / min), sixteen pieces' loads in flight ahead of the additions, then the requested outputs of the segment's row
// are written.  With accumulate_sum the prior is the row the partial kernel saved before the short-CSR call wrote the row.
template <bool MINMAX>
__global__ void __launch_bounds__(128)
segment_long_combine_kernel(const int32_t* __restrict__ long_ids, const int32_t* __restrict__ piece_ptr, const int32_t* __restrict__ rowptr,
                            const float* __restrict__ p_sum, const float* __restrict__ p_max, const float* __restrict__ p_min,
                            const int32_t* __restrict__ p_amx, const int32_t* __restrict__ p_amn,
                            const __nv_bfloat16* __restrict__ prior_save, __nv_bfloat16* __restrict__ out_sum,
                            __nv_bfloat16* __restrict__ out_mean, __nv_bfloat16* __restrict__ out_max, __nv_bfloat16* __restrict__ out_min,
                            int32_t* __restrict__ argmax, int32_t* __restrict__ argmin) {
  const int c = threadIdx.x;
  const int seg = __ldg(long_ids + blockIdx.x);
  const int k0 = __ldg(piece_ptr + blockIdx.x), k1 = __ldg(piece_ptr + blockIdx.x + 1);
  float t = 0.f, mx = -INFINITY, mn = INFINITY;
  int ax = -1, an = -1;
  for (int k = k0; k < k1; k += 16) {
    float v[16], a[16], b[16];
#pragma unroll
    for (int q = 0; q < 16; ++q) {
      const bool in = k + q < k1;
      v[q] = in ? __ldg(p_sum + int64_t(k + q) * 128 + c) : 0.f;
      if (MINMAX) {
        a[q] = in ? __ldg(p_max + int64_t(k + q) * 128 + c) : -INFINITY;
        b[q] = in ? __ldg(p_min + int64_t(k + q) * 128 + c) : INFINITY;
      }
    }
#pragma unroll
    for (int q = 0; q < 16; ++q) {
      if (k + q < k1) t = __fadd_rn(t, v[q]);
      if (MINMAX) {
        if (a[q] > mx) { mx = a[q]; ax = __ldg(p_amx + int64_t(k + q) * 128 + c); }
        if (b[q] < mn) { mn = b[q]; an = __ldg(p_amn + int64_t(k + q) * 128 + c); }
      }
    }
  }
  const int64_t o = int64_t(seg) * 128 + c;
  if (out_sum) out_sum[o] = __float2bfloat16_rn(prior_save ? __fadd_rn(t, __bfloat162float(prior_save[int64_t(k0) * 128 + c])) : t);
  if (out_mean) {
    const float inv = 1.0f / float(__ldg(rowptr + seg + 1) - __ldg(rowptr + seg));
    out_mean[o] = __float2bfloat16_rn(__fmul_rn(t, inv));
  }
  if (MINMAX) {
    if (out_max) out_max[o] = __float2bfloat16_rn(mx);
    if (out_min) out_min[o] = __float2bfloat16_rn(mn);
    if (argmax) argmax[o] = ax;
    if (argmin) argmin[o] = an;
  }
}

// ------------------------------------------------------------------------------------------------
// backward: half a warp per piece, per element
// ------------------------------------------------------------------------------------------------
// grad[e] = ((0 + g_sum) fma g_mean * inv) + [argmax == e] g_max + [argmin == e] g_min: segment_bwd_bf16_128_kernel's arithmetic
template <bool LAYER>
__global__ void __launch_bounds__(256)
segment_long_bwd_kernel(const int32_t* __restrict__ perm, const int32_t* __restrict__ rowptr, const int32_t* __restrict__ pieces,
                        int64_t n_pieces, const __nv_bfloat16* __restrict__ g_sum, const __nv_bfloat16* __restrict__ g_mean,
                        const __nv_bfloat16* __restrict__ g_max, const __nv_bfloat16* __restrict__ g_min,
                        const int32_t* __restrict__ argmax, const int32_t* __restrict__ argmin, const __nv_bfloat16* __restrict__ base,
                        __nv_bfloat16* __restrict__ agg_grad, __nv_bfloat16* __restrict__ grad) {
  const int l16 = threadIdx.x & 15;
  const uint32_t hmask = 0xFFFFu << (threadIdx.x & 16);
  const int64_t k = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 4;
  if (k >= n_pieces) return;                                // whole half-warps leave together
  const int seg = __ldg(pieces + 3 * k), beg = __ldg(pieces + 3 * k + 1), end = __ldg(pieces + 3 * k + 2);
  const int cnt = __ldg(rowptr + seg + 1) - __ldg(rowptr + seg);
  const int64_t o = int64_t(seg) * 128 + l16 * 8;
  float pre[8], gx[8], gn[8];
  int ax[8], an[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { pre[i] = 0.f; gx[i] = 0.f; gn[i] = 0.f; ax[i] = -1; an[i] = -1; }
  if (g_max) {
    unpack8(__ldg(reinterpret_cast<const uint4*>(g_max + o)), gx);
    const int4 a0 = __ldg(reinterpret_cast<const int4*>(argmax + o)), a1 = __ldg(reinterpret_cast<const int4*>(argmax + o + 4));
    ax[0] = a0.x; ax[1] = a0.y; ax[2] = a0.z; ax[3] = a0.w; ax[4] = a1.x; ax[5] = a1.y; ax[6] = a1.z; ax[7] = a1.w;
  }
  if (g_min) {
    unpack8(__ldg(reinterpret_cast<const uint4*>(g_min + o)), gn);
    const int4 a0 = __ldg(reinterpret_cast<const int4*>(argmin + o)), a1 = __ldg(reinterpret_cast<const int4*>(argmin + o + 4));
    an[0] = a0.x; an[1] = a0.y; an[2] = a0.z; an[3] = a0.w; an[4] = a1.x; an[5] = a1.y; an[6] = a1.z; an[7] = a1.w;
  }
  if (!LAYER) {
    float f[8];
    if (g_sum) { unpack8(__ldg(reinterpret_cast<const uint4*>(g_sum + o)), f);
#pragma unroll
      for (int i = 0; i < 8; ++i) pre[i] = __fadd_rn(pre[i], f[i]); }
    if (g_mean) { unpack8(__ldg(reinterpret_cast<const uint4*>(g_mean + o)), f);
      const float inv = 1.0f / float(cnt);
#pragma unroll
      for (int i = 0; i < 8; ++i) pre[i] = __fmaf_rn(f[i], inv, pre[i]); }
  } else if (agg_grad && beg == __ldg(rowptr + seg)) {     // the segment's first piece writes its agg_grad row
    float a[8], f[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = 0.f;
    if (g_sum) { unpack8(__ldg(reinterpret_cast<const uint4*>(g_sum + o)), f);
#pragma unroll
      for (int i = 0; i < 8; ++i) a[i] = __fadd_rn(a[i], f[i]); }
    if (g_mean) { unpack8(__ldg(reinterpret_cast<const uint4*>(g_mean + o)), f);
      const float inv = 1.0f / float(max(cnt, 1));
#pragma unroll
      for (int i = 0; i < 8; ++i) a[i] = __fadd_rn(a[i], __fmul_rn(f[i], inv)); }
    *reinterpret_cast<uint4*>(agg_grad + o) = pack8(a);
  }
  if (grad == nullptr) return;
  for (int j = beg; j < end; j += 16) {
    const int mine = j + l16 < end ? __ldg(perm + j + l16) : -1;
    int e[16];
    uint4 b[16];
#pragma unroll
    for (int q = 0; q < 16; ++q) {
      e[q] = __shfl_sync(hmask, mine, q, 16);
      b[q] = make_uint4(0u, 0u, 0u, 0u);
      if (LAYER && base && e[q] >= 0) b[q] = __ldg(reinterpret_cast<const uint4*>(base + int64_t(e[q]) * 128) + l16);
    }
#pragma unroll
    for (int q = 0; q < 16; ++q) {
      if (e[q] < 0) break;
      float g[8];
      if (LAYER) {
        unpack8(b[q], g);
#pragma unroll
        for (int i = 0; i < 8; ++i) g[i] = __fadd_rn(0.f, g[i]);
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) g[i] = pre[i];
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (ax[i] == e[q]) g[i] = __fadd_rn(g[i], gx[i]);
        if (an[i] == e[q]) g[i] = __fadd_rn(g[i], gn[i]);
      }
      *(reinterpret_cast<uint4*>(grad + int64_t(e[q]) * 128) + l16) = pack8(g);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// fp32 partials (hgn_segment_partials): the value each segment's result is rounded from, left unrounded
// ------------------------------------------------------------------------------------------------
constexpr int kPartialW = HGN_SEGMENT_PARTIAL_WIDTH;
static_assert(kPartialW == 3 * 128 + 4 && (kPartialW * 4) % 16 == 0, "partial row: sum | max | min | count + padding, 16-byte rows");

// One warp per segment of the (short) CSR, four features per lane: the sum from +0 in perm order (the order of
// segment_sum_bf16_128_kernel and segment_reduce_vec_kernel), max / min with strict comparisons and their first-in-order winners,
// and the element count.  An empty segment leaves 0, -inf, +inf, winners -1 and count 0.
__global__ void __launch_bounds__(256)
segment_partial_short_kernel(const __nv_bfloat16* __restrict__ data, const int32_t* __restrict__ perm, const int32_t* __restrict__ rowptr,
                             int64_t S, int minmax, float* __restrict__ out, int32_t* __restrict__ argmax, int32_t* __restrict__ argmin) {
  const int lane = threadIdx.x & 31;
  const int64_t seg = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
  if (seg >= S) return;
  const int beg = rowptr[seg], end = rowptr[seg + 1];
  const int c = lane * 4;
  float s[4] = {0.f, 0.f, 0.f, 0.f}, mx[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY}, mn[4] = {INFINITY, INFINITY, INFINITY, INFINITY};
  int ax[4] = {-1, -1, -1, -1}, an[4] = {-1, -1, -1, -1};
  for (int j = beg; j < end; ++j) {
    const int e = __ldg(perm + j);
    const uint2 p = __ldg(reinterpret_cast<const uint2*>(data + int64_t(e) * 128 + c));
    const float f[4] = {__uint_as_float(p.x << 16), __uint_as_float(p.x & 0xFFFF0000u), __uint_as_float(p.y << 16),
                        __uint_as_float(p.y & 0xFFFF0000u)};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      s[i] = __fadd_rn(s[i], f[i]);
      if (minmax) {
        if (f[i] > mx[i]) { mx[i] = f[i]; ax[i] = e; }
        if (f[i] < mn[i]) { mn[i] = f[i]; an[i] = e; }
      }
    }
  }
  float* row = out + seg * kPartialW;
  *reinterpret_cast<float4*>(row + c) = make_float4(s[0], s[1], s[2], s[3]);
  if (minmax) {
    *reinterpret_cast<float4*>(row + 128 + c) = make_float4(mx[0], mx[1], mx[2], mx[3]);
    *reinterpret_cast<float4*>(row + 256 + c) = make_float4(mn[0], mn[1], mn[2], mn[3]);
    if (argmax) *reinterpret_cast<int4*>(argmax + seg * 128 + c) = make_int4(ax[0], ax[1], ax[2], ax[3]);
    if (argmin) *reinterpret_cast<int4*>(argmin + seg * 128 + c) = make_int4(an[0], an[1], an[2], an[3]);
  }
  if (lane == 0) *reinterpret_cast<int4*>(row + 384) = make_int4(end - beg, 0, 0, 0);
}

// segment_long_combine_kernel's combine (ascending piece order, sum from +0, strict comparisons), written unrounded with the count
template <bool MINMAX>
__global__ void __launch_bounds__(128)
segment_long_partial_combine_kernel(const int32_t* __restrict__ long_ids, const int32_t* __restrict__ piece_ptr, const int32_t* __restrict__ rowptr,
                                    const float* __restrict__ p_sum, const float* __restrict__ p_max, const float* __restrict__ p_min,
                                    const int32_t* __restrict__ p_amx, const int32_t* __restrict__ p_amn, float* __restrict__ out,
                                    int32_t* __restrict__ argmax, int32_t* __restrict__ argmin) {
  const int c = threadIdx.x;
  const int seg = __ldg(long_ids + blockIdx.x);
  const int k0 = __ldg(piece_ptr + blockIdx.x), k1 = __ldg(piece_ptr + blockIdx.x + 1);
  float t = 0.f, mx = -INFINITY, mn = INFINITY;
  int ax = -1, an = -1;
  for (int k = k0; k < k1; ++k) {
    t = __fadd_rn(t, __ldg(p_sum + int64_t(k) * 128 + c));
    if (MINMAX) {
      const float a = __ldg(p_max + int64_t(k) * 128 + c), b = __ldg(p_min + int64_t(k) * 128 + c);
      if (a > mx) { mx = a; ax = __ldg(p_amx + int64_t(k) * 128 + c); }
      if (b < mn) { mn = b; an = __ldg(p_amn + int64_t(k) * 128 + c); }
    }
  }
  float* row = out + int64_t(seg) * kPartialW;
  row[c] = t;
  if (MINMAX) {
    row[128 + c] = mx;
    row[256 + c] = mn;
    if (argmax) argmax[int64_t(seg) * 128 + c] = ax;
    if (argmin) argmin[int64_t(seg) * 128 + c] = an;
  }
  if (c == 0) reinterpret_cast<int32_t*>(row)[384] = __ldg(rowptr + seg + 1) - __ldg(rowptr + seg);
}

// fp32 sum, max, min and int32 winners per piece and feature, plus a bf16 prior row per piece
static size_t split_reduce_bytes(const hgn_segment_split* sp) { return sp ? size_t(sp->n_pieces) * 128 * (4 * 5 + 2) : 0; }

static int check_split(const hgn_segment_split* sp, int64_t E, int64_t S, const char* what) {
  HGN_CHECK_ARG(sp != nullptr, "%s: null split", what);
  HGN_CHECK_ARG(sp->num_segments == S && sp->num_elements == E,
                "%s: split built for S=%lld E=%lld, called with S=%lld E=%lld", what, (long long)sp->num_segments,
                (long long)sp->num_elements, (long long)S, (long long)E);
  HGN_CHECK_ARG(sp->n_long >= 0 && sp->n_pieces >= 0 && sp->n_short >= 0 && sp->rowptr_short && sp->perm_short &&
                    (sp->n_long == 0 || (sp->long_ids && sp->piece_ptr && sp->pieces)),
                "%s: malformed split", what);
  return HGN_OK;
}

// The long segments' forward of one side in two launches around the caller's short-CSR call: `partial` before it (it reads the
// caller's prior rows before that call writes them), `combine` after it (it overwrites the long rows that call wrote as empty).
struct LongReduce {
  const hgn_segment_split* sp;
  const int32_t* rowptr;
  __nv_bfloat16 *out_sum, *out_mean, *out_max, *out_min;
  int32_t *argmax, *argmin;
  bool accumulate;
  float *p_sum, *p_max, *p_min;
  int32_t *p_amx, *p_amn;
  __nv_bfloat16* prior_save;

  LongReduce(const hgn_segment_split* sp_, const int32_t* rowptr_, void* s, void* m, void* x, void* n, int32_t* am, int32_t* an, int acc,
             void* workspace)
      : sp(sp_), rowptr(rowptr_), out_sum(static_cast<__nv_bfloat16*>(s)), out_mean(static_cast<__nv_bfloat16*>(m)),
        out_max(static_cast<__nv_bfloat16*>(x)), out_min(static_cast<__nv_bfloat16*>(n)), argmax(am), argmin(an),
        accumulate(acc != 0 && s != nullptr) {
    const int64_t n4 = sp->n_pieces * 128;
    p_sum = static_cast<float*>(workspace);
    p_max = p_sum + n4;
    p_min = p_max + n4;
    p_amx = reinterpret_cast<int32_t*>(p_min + n4);
    p_amn = p_amx + n4;
    prior_save = reinterpret_cast<__nv_bfloat16*>(p_amn + n4);
  }
  bool minmax() const { return out_max || out_min; }

  int partial(const __nv_bfloat16* data, const int32_t* perm, cudaStream_t st) const {
    if (sp->n_long == 0) return HGN_OK;
    const unsigned blocks = unsigned(ceil_div(sp->n_pieces * 16, 256));
    __nv_bfloat16* save = accumulate ? prior_save : nullptr;
    HGN_TIMED("segment_long_partial", st);
    if (minmax())
      segment_long_partial_kernel<true><<<blocks, 256, 0, st>>>(data, perm, sp->pieces, sp->n_pieces, p_sum, p_max, p_min, p_amx, p_amn, out_sum, save);
    else
      segment_long_partial_kernel<false><<<blocks, 256, 0, st>>>(data, perm, sp->pieces, sp->n_pieces, p_sum, p_max, p_min, p_amx, p_amn, out_sum, save);
    HGN_LAUNCH_OK("segment_long_partial");
    return HGN_OK;
  }

  int combine(cudaStream_t st) const {
    if (sp->n_long == 0) return HGN_OK;
    const __nv_bfloat16* save = accumulate ? prior_save : nullptr;
    HGN_TIMED("segment_long_combine", st);
    if (minmax())
      segment_long_combine_kernel<true><<<unsigned(sp->n_long), 128, 0, st>>>(sp->long_ids, sp->piece_ptr, rowptr, p_sum, p_max, p_min, p_amx,
                                                                                p_amn, save, out_sum, out_mean, out_max, out_min, argmax, argmin);
    else
      segment_long_combine_kernel<false><<<unsigned(sp->n_long), 128, 0, st>>>(sp->long_ids, sp->piece_ptr, rowptr, p_sum, p_max, p_min, p_amx,
                                                                                 p_amn, save, out_sum, out_mean, out_max, out_min, argmax, argmin);
    HGN_LAUNCH_OK("segment_long_combine");
    return HGN_OK;
  }
};

}  // namespace hgn

using namespace hgn;

extern "C" int32_t hgn_segment_split_threshold(void) { return kSplitT; }
extern "C" int32_t hgn_segment_split_piece(void) { return kSplitP; }

extern "C" int64_t hgn_segment_split_max_long(int64_t E, int64_t S) {
  const int64_t n = E > 0 ? E / (kSplitT + 1) : 0;
  return n < S ? n : (S > 0 ? S : 0);
}
// a long segment of L elements has ceil(L / P) <= L / P + 1 pieces, and there are at most E / (T + 1) of them
extern "C" int64_t hgn_segment_split_max_pieces(int64_t E) { return E > 0 ? E / kSplitP + E / (kSplitT + 1) : 0; }

extern "C" size_t hgn_segment_split_build_workspace_bytes(int64_t E, int64_t S) {
  (void)E;
  return split_layout(S > 0 ? S : 0).total;
}

extern "C" int hgn_segment_split_build(const int32_t* perm, const int32_t* rowptr, int64_t E, int64_t S, int32_t* long_ids,
                                       int32_t* piece_ptr, int32_t* pieces, int32_t* perm_short, int32_t* rowptr_short,
                                       int64_t* host_counts, void* workspace, size_t workspace_bytes, void* stream) {
  HGN_CHECK_ARG(E >= 0 && S >= 0 && E < (int64_t(1) << 31) && S < (int64_t(1) << 31) - 1, "segment_split_build: E=%lld S=%lld out of int32 range",
                (long long)E, (long long)S);
  HGN_CHECK_ARG(rowptr && rowptr_short && piece_ptr && host_counts && workspace && (E == 0 || (perm && perm_short)),
                "segment_split_build: null input/output");
  HGN_CHECK_ARG(hgn_segment_split_max_long(E, S) == 0 || (long_ids && pieces), "segment_split_build: null long-segment output");
  const SplitLayout L = split_layout(S);
  if (workspace_bytes < L.total) { set_error("segment_split_build: workspace %zu < %zu", workspace_bytes, L.total); return HGN_ERR_WORKSPACE; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  char* ws = static_cast<char*>(workspace);
  int32_t* c_long = reinterpret_cast<int32_t*>(ws + L.c_long);
  int32_t* c_pieces = reinterpret_cast<int32_t*>(ws + L.c_pieces);
  int32_t* c_short = reinterpret_cast<int32_t*>(ws + L.c_short);
  int32_t* o_long = reinterpret_cast<int32_t*>(ws + L.o_long);
  int32_t* o_pieces = reinterpret_cast<int32_t*>(ws + L.o_pieces);
  int32_t* totals = reinterpret_cast<int32_t*>(ws + L.totals);
  split_count_kernel<<<unsigned(ceil_div(S + 1, 256)), 256, 0, st>>>(rowptr, S, c_long, c_pieces, c_short);
  HGN_LAUNCH_OK("split_count");
  size_t cub_bytes = L.cub_bytes;
  HGN_CUDA_OK(cub::DeviceScan::ExclusiveSum(ws + L.cub, cub_bytes, c_long, o_long, int(S + 1), st));
  cub_bytes = L.cub_bytes;
  HGN_CUDA_OK(cub::DeviceScan::ExclusiveSum(ws + L.cub, cub_bytes, c_pieces, o_pieces, int(S + 1), st));
  cub_bytes = L.cub_bytes;
  HGN_CUDA_OK(cub::DeviceScan::ExclusiveSum(ws + L.cub, cub_bytes, c_short, rowptr_short, int(S + 1), st));
  split_totals_kernel<<<1, 1, 0, st>>>(o_long, o_pieces, rowptr_short, S, piece_ptr, totals);
  HGN_LAUNCH_OK("split_totals");
  if (S > 0) {
    split_fill_kernel<<<unsigned(ceil_div(S * 32, 256)), 256, 0, st>>>(perm, rowptr, S, o_long, o_pieces, rowptr_short, long_ids, piece_ptr,
                                                                      pieces, perm_short);
    HGN_LAUNCH_OK("split_fill");
  }
  int32_t t[3] = {0, 0, 0};
  HGN_CUDA_OK(cudaMemcpyAsync(t, totals, sizeof(t), cudaMemcpyDeviceToHost, st));
  HGN_CUDA_OK(cudaStreamSynchronize(st));
  host_counts[0] = t[0];
  host_counts[1] = t[1];
  host_counts[2] = t[2];
  return HGN_OK;
}

extern "C" size_t hgn_segment_split_reduce_workspace_bytes(const hgn_segment_split* split) { return split_reduce_bytes(split); }

#define HGN_SPLIT_BF16_128(what)                                                                          \
  HGN_CHECK_ARG(dtype == HGN_BF16, what ": dtype %d, only bf16 (%d) is supported", dtype, int(HGN_BF16)); \
  HGN_CHECK_ARG(D == 128, what ": D=%d, only 128 is supported", D)

extern "C" int hgn_segment_reduce_split(int dtype, const void* data, int64_t E, int32_t D, const int32_t* perm, const int32_t* rowptr,
                                        int64_t S, const hgn_segment_split* split, void* out_sum, void* out_mean, void* out_max,
                                        void* out_min, int32_t* argmax, int32_t* argmin, int accumulate_sum, void* workspace,
                                        size_t workspace_bytes, void* stream) {
  HGN_SPLIT_BF16_128("segment_reduce_split");
  if (int rc = check_split(split, E, S, "segment_reduce_split")) return rc;
  HGN_CHECK_ARG(rowptr && (E == 0 || (data && perm)), "segment_reduce_split: null input");
  if (workspace_bytes < split_reduce_bytes(split) || (split->n_pieces > 0 && !workspace)) {
    set_error("segment_reduce_split: workspace %zu < %zu", workspace_bytes, split_reduce_bytes(split));
    return HGN_ERR_WORKSPACE;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const LongReduce lr(split, rowptr, out_sum, out_mean, out_max, out_min, argmax, argmin, accumulate_sum, workspace);
  if (int rc = lr.partial(static_cast<const __nv_bfloat16*>(data), perm, st)) return rc;
  // the short segments; this call also writes every long segment's row, as an empty segment's (0, -1, or +0 + prior)
  if (int rc = hgn_segment_reduce(dtype, data, E, D, split->perm_short, split->rowptr_short, S, out_sum, out_mean, out_max, out_min, argmax,
                                  argmin, accumulate_sum, stream))
    return rc;
  return lr.combine(st);
}

extern "C" int hgn_segment_sum_pair_split(int dtype, const void* data, int64_t E, int32_t D, const int32_t* perm_a, const int32_t* rowptr_a,
                                          int64_t S_a, const hgn_segment_split* split_a, void* out_a, const int32_t* perm_b,
                                          const int32_t* rowptr_b, int64_t S_b, const hgn_segment_split* split_b, void* out_b,
                                          void* workspace, size_t workspace_bytes, void* stream) {
  HGN_SPLIT_BF16_128("segment_sum_pair_split");
  if (split_a) if (int rc = check_split(split_a, E, S_a, "segment_sum_pair_split")) return rc;
  if (split_b) if (int rc = check_split(split_b, E, S_b, "segment_sum_pair_split")) return rc;
  const size_t need = split_reduce_bytes(split_a) > split_reduce_bytes(split_b) ? split_reduce_bytes(split_a) : split_reduce_bytes(split_b);
  if (workspace_bytes < need || (need > 0 && !workspace)) {
    set_error("segment_sum_pair_split: workspace %zu < %zu", workspace_bytes, need);
    return HGN_ERR_WORKSPACE;
  }
  if (int rc = hgn_segment_sum_pair(dtype, data, E, D, split_a ? split_a->perm_short : perm_a, split_a ? split_a->rowptr_short : rowptr_a, S_a,
                                    out_a, split_b ? split_b->perm_short : perm_b, split_b ? split_b->rowptr_short : rowptr_b, S_b, out_b, stream))
    return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const __nv_bfloat16* x = static_cast<const __nv_bfloat16*>(data);
  for (int side = 0; side < 2; ++side) {       // one workspace, used by the two sides in turn on the stream
    const hgn_segment_split* sp = side ? split_b : split_a;
    if (!sp) continue;
    const LongReduce lr(sp, side ? rowptr_b : rowptr_a, side ? out_b : out_a, nullptr, nullptr, nullptr, nullptr, nullptr, 0, workspace);
    if (int rc = lr.partial(x, side ? perm_b : perm_a, st)) return rc;
    if (int rc = lr.combine(st)) return rc;
  }
  return HGN_OK;
}

extern "C" int hgn_segment_reduce_bwd_split(int dtype, int64_t E, int32_t D, const int32_t* ids32, const int32_t* perm, const int32_t* rowptr,
                                            int64_t S, const hgn_segment_split* split, const void* g_sum, const void* g_mean,
                                            const void* g_max, const void* g_min, const int32_t* argmax, const int32_t* argmin,
                                            void* grad_data, void* stream) {
  HGN_SPLIT_BF16_128("segment_reduce_bwd_split");
  if (int rc = check_split(split, E, S, "segment_reduce_bwd_split")) return rc;
  HGN_CHECK_ARG(E == 0 || (ids32 && perm && rowptr && grad_data), "segment_reduce_bwd_split: null input");
  HGN_CHECK_ARG((!g_max || argmax) && (!g_min || argmin), "segment_reduce_bwd_split: max/min gradients need their arg indices");
  if (int rc = hgn_segment_reduce_bwd(dtype, E, D, ids32, split->perm_short, split->rowptr_short, S, g_sum, g_mean, g_max, g_min, argmax,
                                      argmin, grad_data, 0, stream))
    return rc;
  if (split->n_pieces == 0) return HGN_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  HGN_TIMED("segment_long_bwd", st);
  segment_long_bwd_kernel<false><<<unsigned(ceil_div(split->n_pieces * 16, 256)), 256, 0, st>>>(
      perm, rowptr, split->pieces, split->n_pieces, (const __nv_bfloat16*)g_sum, (const __nv_bfloat16*)g_mean, (const __nv_bfloat16*)g_max,
      (const __nv_bfloat16*)g_min, argmax, argmin, nullptr, nullptr, (__nv_bfloat16*)grad_data);
  HGN_LAUNCH_OK("segment_long_bwd");
  return HGN_OK;
}

extern "C" int hgn_segment_layer_grad_split(int dtype, int64_t E, int32_t D, const int32_t* perm, const int32_t* rowptr, int64_t S,
                                            const hgn_segment_split* split, const void* g_sum, const void* g_mean, const void* g_max,
                                            const void* g_min, const int32_t* argmax, const int32_t* argmin, const void* base,
                                            void* agg_grad, void* edge_grad, void* stream) {
  HGN_SPLIT_BF16_128("segment_layer_grad_split");
  if (int rc = check_split(split, E, S, "segment_layer_grad_split")) return rc;
  HGN_CHECK_ARG(S == 0 || rowptr, "segment_layer_grad_split: null rowptr");
  HGN_CHECK_ARG(!edge_grad || E == 0 || perm, "segment_layer_grad_split: edge_grad needs perm");
  // the short-CSR call checks the remaining arguments and writes the long segments' agg_grad rows as if empty: they are rewritten below
  if (int rc = hgn_segment_layer_grad(dtype, E, D, split->perm_short, split->rowptr_short, S, g_sum, g_mean, g_max, g_min, argmax, argmin, base,
                                      agg_grad, edge_grad, stream))
    return rc;
  if (split->n_pieces == 0 || (!agg_grad && !edge_grad)) return HGN_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  HGN_TIMED("segment_long_layer_grad", st);
  segment_long_bwd_kernel<true><<<unsigned(ceil_div(split->n_pieces * 16, 256)), 256, 0, st>>>(
      perm, rowptr, split->pieces, split->n_pieces, (const __nv_bfloat16*)g_sum, (const __nv_bfloat16*)g_mean, (const __nv_bfloat16*)g_max,
      (const __nv_bfloat16*)g_min, argmax, argmin, (const __nv_bfloat16*)base, (__nv_bfloat16*)agg_grad, (__nv_bfloat16*)edge_grad);
  HGN_LAUNCH_OK("segment_long_layer_grad");
  return HGN_OK;
}

extern "C" int hgn_segment_partials(int dtype, const void* data, int64_t E, int32_t D, const int32_t* perm, const int32_t* rowptr, int64_t S,
                                    const hgn_segment_split* split, int minmax, float* out, int32_t* argmax, int32_t* argmin, void* workspace,
                                    size_t workspace_bytes, void* stream) {
  HGN_SPLIT_BF16_128("segment_partials");
  if (split) if (int rc = check_split(split, E, S, "segment_partials")) return rc;
  HGN_CHECK_ARG(S >= 0 && E >= 0 && (S == 0 || (rowptr && out)) && (E == 0 || (data && perm)), "segment_partials: null input/output");
  HGN_CHECK_ARG(minmax || (!argmax && !argmin), "segment_partials: winners need minmax");
  if (workspace_bytes < split_reduce_bytes(split) || (split && split->n_pieces > 0 && !workspace)) {
    set_error("segment_partials: workspace %zu < %zu", workspace_bytes, split_reduce_bytes(split));
    return HGN_ERR_WORKSPACE;
  }
  if (S == 0) return HGN_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const __nv_bfloat16* x = static_cast<const __nv_bfloat16*>(data);
  {
    HGN_TIMED("segment_partials", st);
    segment_partial_short_kernel<<<unsigned(ceil_div(S * 32, 256)), 256, 0, st>>>(x, split ? split->perm_short : perm, split ? split->rowptr_short : rowptr,
                                                                                   S, minmax, out, argmax, argmin);
    HGN_LAUNCH_OK("segment_partials");
  }
  if (!split || split->n_long == 0) return HGN_OK;
  // the long segments: the pieces of segment_long_partial_kernel, then their combine (it overwrites the rows the short call wrote as
  // empty).  LongReduce only lays out the workspace and picks the piece kernel here: its out_max slot stands for "max / min wanted".
  const LongReduce lr(split, rowptr, nullptr, nullptr, minmax ? out : nullptr, nullptr, nullptr, nullptr, 0, workspace);
  if (int rc = lr.partial(x, perm, st)) return rc;
  HGN_TIMED("segment_partials_long", st);
  if (minmax)
    segment_long_partial_combine_kernel<true><<<unsigned(split->n_long), 128, 0, st>>>(split->long_ids, split->piece_ptr, rowptr, lr.p_sum, lr.p_max,
                                                                                      lr.p_min, lr.p_amx, lr.p_amn, out, argmax, argmin);
  else
    segment_long_partial_combine_kernel<false><<<unsigned(split->n_long), 128, 0, st>>>(split->long_ids, split->piece_ptr, rowptr, lr.p_sum, lr.p_max,
                                                                                       lr.p_min, lr.p_amx, lr.p_amn, out, argmax, argmin);
  HGN_LAUNCH_OK("segment_partials_long");
  return HGN_OK;
}
