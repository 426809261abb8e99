// Receiver-sorted CSR plan + deterministic segmented reductions (no floating-point atomics).
//
// HBM-bound kernels.  Layout: edge rows [E, D] row-major, one warp per segment row; a lane owns 4
// consecutive features so every row access is one coalesced 512-byte (fp32) / 256-byte (bf16)
// request, stores are 128-bit (fp32) / 64-bit (bf16) vectors.  The edges of a segment are visited in
// ascending edge id (stable sort), so sums have a fixed association order and max/min ties resolve
// to the first edge, like torch_scatter's CPU reducer (src/util.py:117-127 call sites).
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <type_traits>

#include "common.cuh"

namespace hgn {

// ------------------------------------------------------------------------------------------------
// plan
// ------------------------------------------------------------------------------------------------
__global__ void csr_prepare_kernel(const int64_t* __restrict__ ids, int64_t E, int64_t S, int32_t* __restrict__ ids32,
                                   int32_t* __restrict__ iota, int32_t* __restrict__ counts, int32_t* __restrict__ bad) {
  int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (i >= E) return;
  int64_t v = ids[i];
  if (v < 0 || v >= S) {
    atomicExch(bad, 1);
    v = 0;
  }
  ids32[i] = int32_t(v);
  iota[i] = int32_t(i);
  atomicAdd(&counts[v], 1);   // integer atomics: the result does not depend on the order
}

static int sort_bits(int64_t S) {
  int bits = 1;
  while ((int64_t(1) << bits) < S) ++bits;
  return bits;
}

struct CsrLayout {
  size_t ids32, keys_out, iota, counts, bad, cub, total;
  size_t cub_bytes;
};

static CsrLayout csr_layout(int64_t E, int64_t S) {
  CsrLayout L{};
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
  size_t e = size_t(E > 0 ? E : 1);
  L.ids32 = take(e * 4);
  L.keys_out = take(e * 4);
  L.iota = take(e * 4);
  L.counts = take(size_t(S + 1) * 4);
  L.bad = take(4);
  size_t sort_bytes = 0, scan_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (const int32_t*)nullptr, (int32_t*)nullptr,
                                  (const int32_t*)nullptr, (int32_t*)nullptr, int(e), 0, sort_bits(S));
  cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (const int32_t*)nullptr, (int32_t*)nullptr, int(S + 1));
  L.cub_bytes = sort_bytes > scan_bytes ? sort_bytes : scan_bytes;
  L.cub = take(L.cub_bytes);
  L.total = off;
  return L;
}

// ------------------------------------------------------------------------------------------------
// forward: sum / mean / max / min (+ arg) in one pass
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
segment_reduce_vec_kernel(const T* __restrict__ data, int32_t D, const int32_t* __restrict__ perm,
                          const int32_t* __restrict__ rowptr, int64_t S, T* __restrict__ out_sum, T* __restrict__ out_mean,
                          T* __restrict__ out_max, T* __restrict__ out_min, int32_t* __restrict__ argmax,
                          int32_t* __restrict__ argmin, int accumulate_sum) {
  const int lane = threadIdx.x & 31;
  const int64_t seg = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
  if (seg >= S) return;
  const int beg = rowptr[seg], end = rowptr[seg + 1];
  const bool want_minmax = (out_max != nullptr) || (out_min != nullptr);
  for (int c = lane * 4; c < D; c += 128) {
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 mx = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    float4 mn = make_float4(INFINITY, INFINITY, INFINITY, INFINITY);
    int4 amx = make_int4(-1, -1, -1, -1), amn = make_int4(-1, -1, -1, -1);
    int j = beg;
    // two rows in flight per lane: the segment (mean in-degree ~6 on triangle meshes) is short, so
    // memory-level parallelism comes from many warps plus this 2-way unroll
    for (; j + 1 < end; j += 2) {
      const int e0 = perm[j], e1 = perm[j + 1];
      const float4 a = load4(data + int64_t(e0) * D + c);
      const float4 b = load4(data + int64_t(e1) * D + c);
      s.x += a.x; s.y += a.y; s.z += a.z; s.w += a.w;
      s.x += b.x; s.y += b.y; s.z += b.z; s.w += b.w;
      if (want_minmax) {
#define HGN_MINMAX(v, e)                                              \
        if (v.x > mx.x) { mx.x = v.x; amx.x = e; } if (v.y > mx.y) { mx.y = v.y; amx.y = e; } \
        if (v.z > mx.z) { mx.z = v.z; amx.z = e; } if (v.w > mx.w) { mx.w = v.w; amx.w = e; } \
        if (v.x < mn.x) { mn.x = v.x; amn.x = e; } if (v.y < mn.y) { mn.y = v.y; amn.y = e; } \
        if (v.z < mn.z) { mn.z = v.z; amn.z = e; } if (v.w < mn.w) { mn.w = v.w; amn.w = e; }
        HGN_MINMAX(a, e0)
        HGN_MINMAX(b, e1)
      }
    }
    if (j < end) {
      const int e0 = perm[j];
      const float4 a = load4(data + int64_t(e0) * D + c);
      s.x += a.x; s.y += a.y; s.z += a.z; s.w += a.w;
      if (want_minmax) { HGN_MINMAX(a, e0) }
    }
#undef HGN_MINMAX
    const int64_t o = seg * D + c;
    if (out_sum) {
      float4 r = s;
      if (accumulate_sum) { float4 p = load4(out_sum + o); r.x += p.x; r.y += p.y; r.z += p.z; r.w += p.w; }
      store4(out_sum + o, r);
    }
    if (out_mean) {
      const float inv = 1.0f / float(max(end - beg, 1));
      store4(out_mean + o, make_float4(s.x * inv, s.y * inv, s.z * inv, s.w * inv));
    }
    if (end == beg) { mx = make_float4(0.f, 0.f, 0.f, 0.f); mn = mx; }   // empty segment -> 0
    if (out_max) store4(out_max + o, mx);
    if (out_min) store4(out_min + o, mn);
    if (argmax) *reinterpret_cast<int4*>(argmax + o) = amx;
    if (argmin) *reinterpret_cast<int4*>(argmin + o) = amn;
  }
}

template <typename T>
__global__ void segment_reduce_scalar_kernel(const T* __restrict__ data, int32_t D, const int32_t* __restrict__ perm,
                                             const int32_t* __restrict__ rowptr, int64_t S, T* out_sum, T* out_mean,
                                             T* out_max, T* out_min, int32_t* argmax, int32_t* argmin, int accumulate_sum) {
  const int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (i >= S * D) return;
  const int64_t seg = i / D;
  const int c = int(i - seg * D);
  const int beg = rowptr[seg], end = rowptr[seg + 1];
  float s = 0.f, mx = -INFINITY, mn = INFINITY;
  int amx = -1, amn = -1;
  for (int j = beg; j < end; ++j) {
    const int e = perm[j];
    const float v = to_f(data[int64_t(e) * D + c]);
    s += v;
    if (v > mx) { mx = v; amx = e; }
    if (v < mn) { mn = v; amn = e; }
  }
  if (end == beg) { mx = 0.f; mn = 0.f; }
  if (out_sum) out_sum[i] = from_f<T>(accumulate_sum ? s + to_f(out_sum[i]) : s);
  if (out_mean) out_mean[i] = from_f<T>(s / float(max(end - beg, 1)));
  if (out_max) out_max[i] = from_f<T>(mx);
  if (out_min) out_min[i] = from_f<T>(mn);
  if (argmax) argmax[i] = amx;
  if (argmin) argmin[i] = amn;
}

// ------------------------------------------------------------------------------------------------
// backward: one warp per edge row, gathers the receiver's gradient rows
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
segment_reduce_bwd_vec_kernel(int64_t E, int32_t D, const int32_t* __restrict__ ids, const int32_t* __restrict__ rowptr,
                              const T* __restrict__ g_sum, const T* __restrict__ g_mean, const T* __restrict__ g_max,
                              const T* __restrict__ g_min, const int32_t* __restrict__ argmax,
                              const int32_t* __restrict__ argmin, T* __restrict__ grad, int accumulate) {
  const int lane = threadIdx.x & 31;
  const int64_t e = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
  if (e >= E) return;
  const int r = ids[e];
  const float inv = g_mean ? 1.0f / float(max(rowptr[r + 1] - rowptr[r], 1)) : 0.f;
  for (int c = lane * 4; c < D; c += 128) {
    const int64_t o = int64_t(r) * D + c;
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
    if (g_sum) { const float4 a = load4(g_sum + o); g.x += a.x; g.y += a.y; g.z += a.z; g.w += a.w; }
    if (g_mean) { const float4 a = load4(g_mean + o); g.x += a.x * inv; g.y += a.y * inv; g.z += a.z * inv; g.w += a.w * inv; }
    if (g_max) {
      const float4 a = load4(g_max + o);
      const int4 w = *reinterpret_cast<const int4*>(argmax + o);
      if (w.x == e) g.x += a.x; if (w.y == e) g.y += a.y; if (w.z == e) g.z += a.z; if (w.w == e) g.w += a.w;
    }
    if (g_min) {
      const float4 a = load4(g_min + o);
      const int4 w = *reinterpret_cast<const int4*>(argmin + o);
      if (w.x == e) g.x += a.x; if (w.y == e) g.y += a.y; if (w.z == e) g.z += a.z; if (w.w == e) g.w += a.w;
    }
    const int64_t q = e * D + c;
    if (accumulate) { const float4 p = load4(grad + q); g.x += p.x; g.y += p.y; g.z += p.z; g.w += p.w; }
    store4(grad + q, g);
  }
}

template <typename T>
__global__ void segment_reduce_bwd_scalar_kernel(int64_t E, int32_t D, const int32_t* ids, const int32_t* rowptr,
                                                 const T* g_sum, const T* g_mean, const T* g_max, const T* g_min,
                                                 const int32_t* argmax, const int32_t* argmin, T* grad, int accumulate) {
  const int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (i >= E * D) return;
  const int64_t e = i / D;
  const int c = int(i - e * D);
  const int r = ids[e];
  const int64_t o = int64_t(r) * D + c;
  float g = 0.f;
  if (g_sum) g += to_f(g_sum[o]);
  if (g_mean) g += to_f(g_mean[o]) / float(max(rowptr[r + 1] - rowptr[r], 1));
  if (g_max && argmax[o] == e) g += to_f(g_max[o]);
  if (g_min && argmin[o] == e) g += to_f(g_min[o]);
  if (accumulate) g += to_f(grad[i]);
  grad[i] = from_f<T>(g);
}

// ------------------------------------------------------------------------------------------------
// halo rows
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void rows_gather_kernel(const T* __restrict__ src, const int32_t* __restrict__ idx, int64_t n, int32_t D, T* __restrict__ dst) {
  const int lane = threadIdx.x & 31;
  const int64_t i = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
  if (i >= n) return;
  const int64_t r = idx[i];
  for (int c = lane * 4; c < D; c += 128) store4(dst + i * D + c, load4(src + r * D + c));
}
template <typename T>
__global__ void rows_scatter_kernel(const T* __restrict__ src, const int32_t* __restrict__ idx, int64_t n, int32_t D, T* __restrict__ dst, int accumulate) {
  const int lane = threadIdx.x & 31;
  const int64_t i = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
  if (i >= n) return;
  const int64_t r = idx[i];
  for (int c = lane * 4; c < D; c += 128) {
    float4 v = load4(src + i * D + c);
    if (accumulate) { const float4 p = load4(dst + r * D + c); v.x += p.x; v.y += p.y; v.z += p.z; v.w += p.w; }
    store4(dst + r * D + c, v);
  }
}

// 'sum' over 128-wide bf16 rows (the per-layer edge -> node aggregation and the sender / receiver keyed sums of the
// projected edge backward): half a warp per segment, 16 bytes per lane and row, the segment's element ids fetched with one
// coalesced load and up to eight row loads in flight per lane (mean in-degree ~6 on triangle meshes, so most segments are a
// single round).  Summation order = ascending position in `perm` (= ascending element id), like the generic kernel.
__device__ __forceinline__ void
segment_sum_bf16_128_body(const __nv_bfloat16* __restrict__ data, const int32_t* __restrict__ perm, const int32_t* __restrict__ rowptr,
                          int64_t S, __nv_bfloat16* __restrict__ out_sum, int accumulate_sum, int64_t seg) {
  const int l16 = threadIdx.x & 15;
  const uint32_t hmask = 0xFFFFu << (threadIdx.x & 16);     // the two halves of a warp run different trip counts
  const bool live = seg < S;
  const int beg = live ? rowptr[seg] : 0, end = live ? rowptr[seg + 1] : 0;
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.f;
  for (int j = beg; j < end; j += 8) {
    const int mine = (l16 < 8 && j + l16 < end) ? __ldg(perm + j + l16) : -1;
    uint4 v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int e = __shfl_sync(hmask, mine, k, 16);
      v[k] = make_uint4(0u, 0u, 0u, 0u);
      if (e >= 0) v[k] = __ldg(reinterpret_cast<const uint4*>(data + int64_t(e) * 128) + l16);
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const uint32_t w[4] = {v[k].x, v[k].y, v[k].z, v[k].w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        acc[2 * i] += __uint_as_float(w[i] << 16);
        acc[2 * i + 1] += __uint_as_float(w[i] & 0xFFFF0000u);
      }
    }
  }
  if (!live) return;
  uint4* op = reinterpret_cast<uint4*>(out_sum + seg * 128) + l16;
  if (accumulate_sum) {
    const uint4 p = *op;
    const uint32_t w[4] = {p.x, p.y, p.z, p.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) { acc[2 * i] += __uint_as_float(w[i] << 16); acc[2 * i + 1] += __uint_as_float(w[i] & 0xFFFF0000u); }
  }
  uint32_t o[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    __nv_bfloat162 t = __floats2bfloat162_rn(acc[2 * i], acc[2 * i + 1]);
    o[i] = *reinterpret_cast<uint32_t*>(&t);
  }
  *op = make_uint4(o[0], o[1], o[2], o[3]);
}

__global__ void __launch_bounds__(256)
segment_sum_bf16_128_kernel(const __nv_bfloat16* __restrict__ data, const int32_t* __restrict__ perm, const int32_t* __restrict__ rowptr,
                            int64_t S, __nv_bfloat16* __restrict__ out_sum, int accumulate_sum) {
  segment_sum_bf16_128_body(data, perm, rowptr, S, out_sum, accumulate_sum, (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 4);
}

// Two sums of the SAME rows under two groupings (the sender-keyed and the receiver-keyed sum of G0 in the projected edge backward):
// even blocks take grouping A, odd blocks grouping B, over the same range of segments, so the two reads of a row fall close together in
// time.  On a mesh whose node numbering is local (an edge's endpoints are near each other in the numbering) the second read of each row
// is an L2 hit: the pair moves E*256 B from HBM once instead of twice.  Arithmetic and order per segment are those of the single kernel.
__global__ void __launch_bounds__(256)
segment_sum_pair_bf16_128_kernel(const __nv_bfloat16* __restrict__ data, const int32_t* __restrict__ perm_a, const int32_t* __restrict__ rowptr_a,
                                 int64_t S_a, __nv_bfloat16* __restrict__ out_a, const int32_t* __restrict__ perm_b,
                                 const int32_t* __restrict__ rowptr_b, int64_t S_b, __nv_bfloat16* __restrict__ out_b) {
  const int64_t seg = ((blockIdx.x >> 1) * int64_t(blockDim.x) + threadIdx.x) >> 4;
  if (blockIdx.x & 1) segment_sum_bf16_128_body(data, perm_b, rowptr_b, S_b, out_b, 0, seg);
  else segment_sum_bf16_128_body(data, perm_a, rowptr_a, S_a, out_a, 0, seg);
}

template <typename T>
static int segment_reduce_impl(const T* data, int64_t E, int32_t D, const int32_t* perm, const int32_t* rowptr, int64_t S,
                               T* out_sum, T* out_mean, T* out_max, T* out_min, int32_t* argmax, int32_t* argmin,
                               int accumulate_sum, cudaStream_t st) {
  if (S == 0) return HGN_OK;
  if (std::is_same<T, __nv_bfloat16>::value && D == 128 && out_sum && !out_mean && !out_max && !out_min) {
    HGN_TIMED("segment_reduce", st);
    segment_sum_bf16_128_kernel<<<unsigned(ceil_div(S * 16, 256)), 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(data), perm, rowptr, S,
                                                                              reinterpret_cast<__nv_bfloat16*>(out_sum), accumulate_sum);
  } else if (D % 4 == 0) {
    const int64_t blocks = ceil_div(S * 32, 256);
    HGN_TIMED("segment_reduce", st);
    segment_reduce_vec_kernel<T><<<unsigned(blocks), 256, 0, st>>>(data, D, perm, rowptr, S, out_sum, out_mean, out_max,
                                                                out_min, argmax, argmin, accumulate_sum);
  } else {
    const int64_t blocks = ceil_div(S * D, 256);
    segment_reduce_scalar_kernel<T><<<unsigned(blocks), 256, 0, st>>>(data, D, perm, rowptr, S, out_sum, out_mean, out_max,
                                                                   out_min, argmax, argmin, accumulate_sum);
  }
  HGN_LAUNCH_OK("segment_reduce");
  return HGN_OK;
}

// Backward of sum / mean / max / min over 128-wide bf16 rows, organised by SEGMENT: half a warp loads the segment's gradient rows
// (and arg rows) once and writes the gradient row of each of its elements (256 B, fully coalesced per element).  The per-element
// kernel above re-reads 2 KB of per-segment data for every element; on a triangle mesh (6 elements per segment) that is 6x the traffic.
// segment_long_bwd_kernel<false> (segment_long.cu) restates this per-element arithmetic for long segments with explicit intrinsics,
// including the fused multiply-add nvcc makes of `base[i] += f[i] * inv`: a change here, or to that contraction, changes both.
__global__ void __launch_bounds__(256)
segment_bwd_bf16_128_kernel(const int32_t* __restrict__ perm, const int32_t* __restrict__ rowptr, int64_t S,
                            const __nv_bfloat16* __restrict__ g_sum, const __nv_bfloat16* __restrict__ g_mean,
                            const __nv_bfloat16* __restrict__ g_max, const __nv_bfloat16* __restrict__ g_min,
                            const int32_t* __restrict__ argmax, const int32_t* __restrict__ argmin, __nv_bfloat16* __restrict__ grad) {
  const int l16 = threadIdx.x & 15;
  const uint32_t hmask = 0xFFFFu << (threadIdx.x & 16);
  const int64_t seg = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 4;
  if (seg >= S) return;                                     // whole half-warps leave together (the shuffles below use hmask)
  const int beg = rowptr[seg], end = rowptr[seg + 1];
  if (end == beg) return;
  const int64_t o = seg * 128 + l16 * 8;
  auto unpack8 = [](const uint4& p, float (&f)[8]) {
    const uint32_t w[4] = {p.x, p.y, p.z, p.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) { f[2 * i] = __uint_as_float(w[i] << 16); f[2 * i + 1] = __uint_as_float(w[i] & 0xFFFF0000u); }
  };
  float base[8], gx[8], gn[8];
  int ax[8], an[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { base[i] = 0.f; gx[i] = 0.f; gn[i] = 0.f; ax[i] = -1; an[i] = -1; }
  if (g_sum) { float f[8]; unpack8(__ldg(reinterpret_cast<const uint4*>(g_sum + o)), f);
#pragma unroll
    for (int i = 0; i < 8; ++i) base[i] += f[i]; }
  if (g_mean) { float f[8]; unpack8(__ldg(reinterpret_cast<const uint4*>(g_mean + o)), f);
    const float inv = 1.0f / float(end - beg);
#pragma unroll
    for (int i = 0; i < 8; ++i) base[i] += f[i] * inv; }
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
  for (int j = beg; j < end; j += 16) {
    const int mine = j + l16 < end ? __ldg(perm + j + l16) : -1;
    const int n = min(16, end - j);
    for (int k = 0; k < n; ++k) {
      const int e = __shfl_sync(hmask, mine, k, 16);
      uint32_t w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float lo = base[2 * i], hi = base[2 * i + 1];
        if (ax[2 * i] == e) lo += gx[2 * i];
        if (ax[2 * i + 1] == e) hi += gx[2 * i + 1];
        if (an[2 * i] == e) lo += gn[2 * i];
        if (an[2 * i + 1] == e) hi += gn[2 * i + 1];
        __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
        w[i] = *reinterpret_cast<uint32_t*>(&t);
      }
      *(reinterpret_cast<uint4*>(grad + int64_t(e) * 128) + l16) = make_uint4(w[0], w[1], w[2], w[3]);
    }
  }
}

// Incoming gradient of e' in a fused non-'sum' GraphNet layer, over the receiver CSR, half a warp per segment (like the kernel above):
//   agg_grad[r]  = g_sum[r] + g_mean[r] * (1 / max(cnt_r, 1))           one row per segment, empty ones included; the edge backward
//                                                                       gathers it through the receivers, so 'sum' / 'mean' need no per-edge pass
//   edge_grad[e] = base[e] + [argmax[r] == e] g_max[r] + [argmin[r] == e] g_min[r]     every element of a non-empty segment
// fp32 from +0 in that term order (absent terms skipped), the product without contraction, one bf16 rounding per output.  Up to eight
// base rows in flight per lane: most segments (in-degree ~6 on triangle meshes) are one round.
__global__ void __launch_bounds__(256)
segment_layer_grad_bf16_128_kernel(const int32_t* __restrict__ perm, const int32_t* __restrict__ rowptr, int64_t S,
                                   const __nv_bfloat16* __restrict__ g_sum, const __nv_bfloat16* __restrict__ g_mean,
                                   const __nv_bfloat16* __restrict__ g_max, const __nv_bfloat16* __restrict__ g_min,
                                   const int32_t* __restrict__ argmax, const int32_t* __restrict__ argmin,
                                   const __nv_bfloat16* __restrict__ base, __nv_bfloat16* __restrict__ agg_grad,
                                   __nv_bfloat16* __restrict__ edge_grad) {
  const int l16 = threadIdx.x & 15;
  const uint32_t hmask = 0xFFFFu << (threadIdx.x & 16);
  const int64_t seg = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 4;
  if (seg >= S) return;                                     // whole half-warps leave together (the shuffles below use hmask)
  const int beg = rowptr[seg], end = rowptr[seg + 1];
  const int64_t o = seg * 128 + l16 * 8;
  auto unpack8 = [](const uint4& p, float (&f)[8]) {
    const uint32_t w[4] = {p.x, p.y, p.z, p.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) { f[2 * i] = __uint_as_float(w[i] << 16); f[2 * i + 1] = __uint_as_float(w[i] & 0xFFFF0000u); }
  };
  auto pack8 = [](const float (&f)[8]) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __nv_bfloat162 t = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
      w[i] = *reinterpret_cast<uint32_t*>(&t);
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
  };
  // Every load that depends only on the segment is issued first (the first eight element ids, the gradient rows, the winners), so a
  // segment costs three dependent memory round trips: rowptr, then these, then the base rows.  agg_grad is stored last.
  const bool edges = edge_grad != nullptr && end > beg;
  const uint4 z4 = make_uint4(0u, 0u, 0u, 0u);
  const int4 none = make_int4(-1, -1, -1, -1);
  int mine = (edges && l16 < 8 && beg + l16 < end) ? __ldg(perm + beg + l16) : -1;
  const uint4 ps = agg_grad && g_sum ? __ldg(reinterpret_cast<const uint4*>(g_sum + o)) : z4;
  const uint4 pm = agg_grad && g_mean ? __ldg(reinterpret_cast<const uint4*>(g_mean + o)) : z4;
  const uint4 px = edges && g_max ? __ldg(reinterpret_cast<const uint4*>(g_max + o)) : z4;
  const uint4 pn = edges && g_min ? __ldg(reinterpret_cast<const uint4*>(g_min + o)) : z4;
  const int4 ax0 = edges && g_max ? __ldg(reinterpret_cast<const int4*>(argmax + o)) : none;
  const int4 ax1 = edges && g_max ? __ldg(reinterpret_cast<const int4*>(argmax + o + 4)) : none;
  const int4 an0 = edges && g_min ? __ldg(reinterpret_cast<const int4*>(argmin + o)) : none;
  const int4 an1 = edges && g_min ? __ldg(reinterpret_cast<const int4*>(argmin + o + 4)) : none;
  if (edges) {
    float gx[8], gn[8];
    unpack8(px, gx);
    unpack8(pn, gn);
    const int ax[8] = {ax0.x, ax0.y, ax0.z, ax0.w, ax1.x, ax1.y, ax1.z, ax1.w};
    const int an[8] = {an0.x, an0.y, an0.z, an0.w, an1.x, an1.y, an1.z, an1.w};
    for (int j = beg; j < end; j += 8) {
      if (j > beg) mine = (l16 < 8 && j + l16 < end) ? __ldg(perm + j + l16) : -1;
      int e[8];
      uint4 b[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        e[k] = __shfl_sync(hmask, mine, k, 16);
        b[k] = z4;
        if (base && e[k] >= 0) b[k] = __ldg(reinterpret_cast<const uint4*>(base + int64_t(e[k]) * 128) + l16);
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        if (e[k] < 0) break;
        float g[8];
        unpack8(b[k], g);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          g[i] = __fadd_rn(0.f, g[i]);
          if (ax[i] == e[k]) g[i] = __fadd_rn(g[i], gx[i]);
          if (an[i] == e[k]) g[i] = __fadd_rn(g[i], gn[i]);
        }
        *(reinterpret_cast<uint4*>(edge_grad + int64_t(e[k]) * 128) + l16) = pack8(g);
      }
    }
  }
  if (agg_grad) {
    float a[8], f[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = 0.f;
    if (g_sum) { unpack8(ps, f);
#pragma unroll
      for (int i = 0; i < 8; ++i) a[i] = __fadd_rn(a[i], f[i]); }
    if (g_mean) { unpack8(pm, f);
      const float inv = 1.0f / float(max(end - beg, 1));
#pragma unroll
      for (int i = 0; i < 8; ++i) a[i] = __fadd_rn(a[i], __fmul_rn(f[i], inv)); }
    *reinterpret_cast<uint4*>(agg_grad + o) = pack8(a);
  }
}

template <typename T>
static int segment_reduce_bwd_impl(int64_t E, int32_t D, const int32_t* ids, const int32_t* perm, const int32_t* rowptr, int64_t S,
                                   const T* g_sum, const T* g_mean, const T* g_max, const T* g_min, const int32_t* argmax,
                                   const int32_t* argmin, T* grad, int accumulate, cudaStream_t st) {
  if (E == 0) return HGN_OK;
  if (std::is_same<T, __nv_bfloat16>::value && D == 128 && perm != nullptr && !accumulate && S > 0) {
    HGN_TIMED("segment_reduce_bwd", st);
    segment_bwd_bf16_128_kernel<<<unsigned(ceil_div(S * 16, 256)), 256, 0, st>>>(
        perm, rowptr, S, reinterpret_cast<const __nv_bfloat16*>(g_sum), reinterpret_cast<const __nv_bfloat16*>(g_mean),
        reinterpret_cast<const __nv_bfloat16*>(g_max), reinterpret_cast<const __nv_bfloat16*>(g_min), argmax, argmin,
        reinterpret_cast<__nv_bfloat16*>(grad));
  } else if (D % 4 == 0) {
    HGN_TIMED("segment_reduce_bwd", st);
    segment_reduce_bwd_vec_kernel<T><<<unsigned(ceil_div(E * 32, 256)), 256, 0, st>>>(E, D, ids, rowptr, g_sum, g_mean, g_max,
                                                                                   g_min, argmax, argmin, grad, accumulate);
  } else {
    segment_reduce_bwd_scalar_kernel<T><<<unsigned(ceil_div(E * D, 256)), 256, 0, st>>>(E, D, ids, rowptr, g_sum, g_mean, g_max,
                                                                                     g_min, argmax, argmin, grad, accumulate);
  }
  HGN_LAUNCH_OK("segment_reduce_bwd");
  return HGN_OK;
}

}  // namespace hgn

using namespace hgn;

extern "C" size_t hgn_csr_workspace_bytes(int64_t E, int64_t S) { return csr_layout(E, S).total; }

extern "C" int hgn_csr_build(const int64_t* segment_ids, int64_t E, int64_t S, int32_t* perm, int32_t* rowptr, int32_t* ids32,
                             void* workspace, size_t workspace_bytes, void* stream) {
  HGN_CHECK_ARG(E >= 0 && S >= 0 && E < (int64_t(1) << 31) && S < (int64_t(1) << 31) - 1, "csr_build: E=%lld S=%lld out of int32 range", (long long)E, (long long)S);
  HGN_CHECK_ARG(perm && rowptr && workspace, "csr_build: null output/workspace");
  const CsrLayout L = csr_layout(E, S);
  if (workspace_bytes < L.total) { set_error("csr_build: workspace %zu < %zu", workspace_bytes, L.total); return HGN_ERR_WORKSPACE; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  char* ws = static_cast<char*>(workspace);
  int32_t* w_ids = reinterpret_cast<int32_t*>(ws + L.ids32);
  int32_t* w_keys = reinterpret_cast<int32_t*>(ws + L.keys_out);
  int32_t* w_iota = reinterpret_cast<int32_t*>(ws + L.iota);
  int32_t* w_counts = reinterpret_cast<int32_t*>(ws + L.counts);
  int32_t* w_bad = reinterpret_cast<int32_t*>(ws + L.bad);
  HGN_CUDA_OK(cudaMemsetAsync(w_counts, 0, size_t(S + 1) * 4 + 0, st));
  HGN_CUDA_OK(cudaMemsetAsync(w_bad, 0, 4, st));
  if (E > 0) {
    csr_prepare_kernel<<<unsigned(ceil_div(E, 256)), 256, 0, st>>>(segment_ids, E, S, w_ids, w_iota, w_counts, w_bad);
    HGN_LAUNCH_OK("csr_prepare");
  }
  size_t cub_bytes = L.cub_bytes;
  HGN_CUDA_OK(cub::DeviceScan::ExclusiveSum(ws + L.cub, cub_bytes, w_counts, rowptr, int(S + 1), st));
  if (E > 0) {
    cub_bytes = L.cub_bytes;
    HGN_CUDA_OK(cub::DeviceRadixSort::SortPairs(ws + L.cub, cub_bytes, (const int32_t*)w_ids, w_keys, (const int32_t*)w_iota, perm,
                                                int(E), 0, sort_bits(S), st));
    if (ids32) HGN_CUDA_OK(cudaMemcpyAsync(ids32, w_ids, size_t(E) * 4, cudaMemcpyDeviceToDevice, st));
  }
  int32_t bad = 0;
  HGN_CUDA_OK(cudaMemcpyAsync(&bad, w_bad, 4, cudaMemcpyDeviceToHost, st));
  HGN_CUDA_OK(cudaStreamSynchronize(st));
  HGN_CHECK_ARG(bad == 0, "csr_build: segment id outside [0, %lld)", (long long)S);
  return HGN_OK;
}

extern "C" int hgn_segment_reduce(int dtype, const void* data, int64_t E, int32_t D, const int32_t* perm, const int32_t* rowptr,
                                  int64_t S, void* out_sum, void* out_mean, void* out_max, void* out_min, int32_t* argmax,
                                  int32_t* argmin, int accumulate_sum, void* stream) {
  HGN_CHECK_ARG(D >= 1 && E >= 0 && S >= 0, "segment_reduce: bad sizes");
  HGN_CHECK_ARG(rowptr && (E == 0 || (data && perm)), "segment_reduce: null input");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == HGN_F32)
    return segment_reduce_impl<float>((const float*)data, E, D, perm, rowptr, S, (float*)out_sum, (float*)out_mean, (float*)out_max,
                                      (float*)out_min, argmax, argmin, accumulate_sum, st);
  if (dtype == HGN_BF16)
    return segment_reduce_impl<__nv_bfloat16>((const __nv_bfloat16*)data, E, D, perm, rowptr, S, (__nv_bfloat16*)out_sum,
                                              (__nv_bfloat16*)out_mean, (__nv_bfloat16*)out_max, (__nv_bfloat16*)out_min, argmax,
                                              argmin, accumulate_sum, st);
  set_error("segment_reduce: unknown dtype %d", dtype);
  return HGN_ERR_INVALID_ARGUMENT;
}

extern "C" int hgn_segment_sum_pair(int dtype, const void* data, int64_t E, int32_t D, const int32_t* perm_a, const int32_t* rowptr_a, int64_t S_a,
                                    void* out_a, const int32_t* perm_b, const int32_t* rowptr_b, int64_t S_b, void* out_b, void* stream) {
  HGN_CHECK_ARG(D >= 1 && E >= 0 && S_a >= 0 && S_b >= 0, "segment_sum_pair: bad sizes");
  HGN_CHECK_ARG(rowptr_a && rowptr_b && (S_a == 0 || out_a) && (S_b == 0 || out_b) && (E == 0 || (data && perm_a && perm_b)),
                "segment_sum_pair: null input");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == HGN_BF16 && D == 128 && S_a > 0 && S_b > 0) {
    const int64_t blocks = ceil_div((S_a > S_b ? S_a : S_b) * 16, 256);
    HGN_TIMED("segment_reduce", st);
    segment_sum_pair_bf16_128_kernel<<<unsigned(2 * blocks), 256, 0, st>>>((const __nv_bfloat16*)data, perm_a, rowptr_a, S_a, (__nv_bfloat16*)out_a,
                                                                        perm_b, rowptr_b, S_b, (__nv_bfloat16*)out_b);
    HGN_LAUNCH_OK("segment_sum_pair");
    return HGN_OK;
  }
  if (int rc = hgn_segment_reduce(dtype, data, E, D, perm_a, rowptr_a, S_a, out_a, nullptr, nullptr, nullptr, nullptr, nullptr, 0, stream)) return rc;
  return hgn_segment_reduce(dtype, data, E, D, perm_b, rowptr_b, S_b, out_b, nullptr, nullptr, nullptr, nullptr, nullptr, 0, stream);
}

extern "C" int hgn_segment_reduce_bwd(int dtype, int64_t E, int32_t D, const int32_t* ids32, const int32_t* perm, const int32_t* rowptr, int64_t S,
                                      const void* g_sum, const void* g_mean, const void* g_max, const void* g_min,
                                      const int32_t* argmax, const int32_t* argmin, void* grad_data, int accumulate, void* stream) {
  HGN_CHECK_ARG(D >= 1 && E >= 0, "segment_reduce_bwd: bad sizes");
  HGN_CHECK_ARG(E == 0 || (ids32 && rowptr && grad_data), "segment_reduce_bwd: null input");
  HGN_CHECK_ARG((!g_max || argmax) && (!g_min || argmin), "segment_reduce_bwd: max/min gradients need their arg indices");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == HGN_F32)
    return segment_reduce_bwd_impl<float>(E, D, ids32, perm, rowptr, S, (const float*)g_sum, (const float*)g_mean, (const float*)g_max,
                                          (const float*)g_min, argmax, argmin, (float*)grad_data, accumulate, st);
  if (dtype == HGN_BF16)
    return segment_reduce_bwd_impl<__nv_bfloat16>(E, D, ids32, perm, rowptr, S, (const __nv_bfloat16*)g_sum, (const __nv_bfloat16*)g_mean,
                                                  (const __nv_bfloat16*)g_max, (const __nv_bfloat16*)g_min, argmax, argmin,
                                                  (__nv_bfloat16*)grad_data, accumulate, st);
  set_error("segment_reduce_bwd: unknown dtype %d", dtype);
  return HGN_ERR_INVALID_ARGUMENT;
}

extern "C" int hgn_segment_layer_grad(int dtype, int64_t E, int32_t D, const int32_t* perm, const int32_t* rowptr, int64_t S,
                                      const void* g_sum, const void* g_mean, const void* g_max, const void* g_min,
                                      const int32_t* argmax, const int32_t* argmin, const void* base, void* agg_grad, void* edge_grad,
                                      void* stream) {
  if (dtype == HGN_F32) { set_error("segment_layer_grad: bf16 only"); return HGN_ERR_UNSUPPORTED; }
  HGN_CHECK_ARG(dtype == HGN_BF16, "segment_layer_grad: unknown dtype %d", dtype);
  HGN_CHECK_ARG(D == 128, "segment_layer_grad: D=%d, only 128 is supported", D);
  HGN_CHECK_ARG(E >= 0 && S >= 0 && E < (int64_t(1) << 31) && S < (int64_t(1) << 31) - 1, "segment_layer_grad: bad sizes");
  HGN_CHECK_ARG((!g_max || argmax) && (!g_min || argmin), "segment_layer_grad: max/min gradients need their arg indices");
  HGN_CHECK_ARG((!g_sum && !g_mean) || agg_grad, "segment_layer_grad: sum/mean gradients need agg_grad");
  HGN_CHECK_ARG((!g_max && !g_min && !base) || edge_grad, "segment_layer_grad: max/min gradients and base need edge_grad");
  HGN_CHECK_ARG(S == 0 || rowptr, "segment_layer_grad: null rowptr");
  HGN_CHECK_ARG(!edge_grad || E == 0 || perm, "segment_layer_grad: edge_grad needs perm");
  HGN_CHECK_ARG(!edge_grad || edge_grad != base, "segment_layer_grad: edge_grad must not alias base");
  HGN_CHECK_ARG(!agg_grad || (agg_grad != g_sum && agg_grad != g_mean && agg_grad != g_max && agg_grad != g_min),
                "segment_layer_grad: agg_grad must not alias a gradient input");
  if (S == 0 || (!agg_grad && !edge_grad)) return HGN_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  HGN_TIMED("segment_layer_grad", st);
  segment_layer_grad_bf16_128_kernel<<<unsigned(ceil_div(S * 16, 256)), 256, 0, st>>>(
      perm, rowptr, S, (const __nv_bfloat16*)g_sum, (const __nv_bfloat16*)g_mean, (const __nv_bfloat16*)g_max, (const __nv_bfloat16*)g_min,
      argmax, argmin, (const __nv_bfloat16*)base, (__nv_bfloat16*)agg_grad, (__nv_bfloat16*)edge_grad);
  HGN_LAUNCH_OK("segment_layer_grad");
  return HGN_OK;
}

extern "C" int hgn_rows_gather(int dtype, const void* src, const int32_t* idx, int64_t n, int32_t D, void* dst, void* stream) {
  HGN_CHECK_ARG(D % 4 == 0 && n >= 0, "rows_gather: D must be a multiple of 4");
  if (n == 0) return HGN_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == HGN_F32) rows_gather_kernel<float><<<unsigned(ceil_div(n * 32, 256)), 256, 0, st>>>((const float*)src, idx, n, D, (float*)dst);
  else rows_gather_kernel<__nv_bfloat16><<<unsigned(ceil_div(n * 32, 256)), 256, 0, st>>>((const __nv_bfloat16*)src, idx, n, D, (__nv_bfloat16*)dst);
  HGN_LAUNCH_OK("rows_gather");
  return HGN_OK;
}

extern "C" int hgn_rows_scatter(int dtype, const void* src, const int32_t* idx, int64_t n, int32_t D, void* dst, int accumulate, void* stream) {
  HGN_CHECK_ARG(D % 4 == 0 && n >= 0, "rows_scatter: D must be a multiple of 4");
  if (n == 0) return HGN_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == HGN_F32) rows_scatter_kernel<float><<<unsigned(ceil_div(n * 32, 256)), 256, 0, st>>>((const float*)src, idx, n, D, (float*)dst, accumulate);
  else rows_scatter_kernel<__nv_bfloat16><<<unsigned(ceil_div(n * 32, 256)), 256, 0, st>>>((const __nv_bfloat16*)src, idx, n, D, (__nv_bfloat16*)dst, accumulate);
  HGN_LAUNCH_OK("rows_scatter");
  return HGN_OK;
}

// ------------------------------------------------------------------------------------------------
// column sums (LayerNorm beta / bias gradients): per-block partials, then a fixed-order second stage
// ------------------------------------------------------------------------------------------------
namespace hgn {
constexpr int kColsumRowsPerBlock = 2048;

template <typename T>
__global__ void __launch_bounds__(256)
colsum_partial_kernel(const T* __restrict__ x, int64_t rows, int32_t D, float* __restrict__ partial) {
  // thread (cx, ry): column group cx (4 columns), row lane ry; D/4 column groups x (256/(D/4)) row lanes
  __shared__ float red[256 * 4];
  const int groups = D / 4;
  const int lanes = 256 / groups;
  const int cx = threadIdx.x % groups, ry = threadIdx.x / groups;
  const int64_t r0 = int64_t(blockIdx.x) * kColsumRowsPerBlock;
  const int64_t r1 = min(rows, r0 + kColsumRowsPerBlock);
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  if (ry < lanes)
    for (int64_t r = r0 + ry; r < r1; r += lanes) {
      const float4 v = load4(x + r * D + cx * 4);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
  red[threadIdx.x * 4 + 0] = s.x; red[threadIdx.x * 4 + 1] = s.y; red[threadIdx.x * 4 + 2] = s.z; red[threadIdx.x * 4 + 3] = s.w;
  __syncthreads();
  if (threadIdx.x < D) {
    const int g = threadIdx.x / 4, k = threadIdx.x % 4;
    float t = 0.f;
    for (int l = 0; l < lanes; ++l) t += red[(l * groups + g) * 4 + k];
    partial[int64_t(blockIdx.x) * D + threadIdx.x] = t;
  }
}
__global__ void colsum_final_kernel(const float* __restrict__ partial, int64_t blocks, int32_t D, float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= D) return;
  float t = 0.f;
  for (int64_t b = 0; b < blocks; ++b) t += partial[b * D + c];
  out[c] = t;
}
}  // namespace hgn

// ---- the five vector gradients of one generic bf16 MLP backward (column sums of G2, G1, G0, P, grad_out: [rows,128] bf16 each) in
// two launches instead of ten: grid (row blocks, matrix); 16 threads per row (8 columns = 16 bytes each), 16 row lanes, four row
// loads in flight per thread; fixed-order shared-memory combine, then a fixed-order sum over the row blocks (ordered_sum_block8).
namespace hgn {
constexpr int kColsum5Rows = 512;
struct Colsum5Args { const __nv_bfloat16* x[5]; float* out[5]; };

__global__ void __launch_bounds__(256)
colsum5_partial_kernel(Colsum5Args a, int64_t rows, float* __restrict__ partial) {
  __shared__ float red[16][128];
  const __nv_bfloat16* x = a.x[blockIdx.y];
  const int cx = threadIdx.x & 15, ry = threadIdx.x >> 4;
  const int64_t r0 = int64_t(blockIdx.x) * kColsum5Rows, r1 = min(rows, r0 + kColsum5Rows);
  float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (x != nullptr) {
    for (int64_t r = r0 + ry; r < r1; r += 64) {
      uint4 w[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) w[k] = r + 16 * k < r1 ? __ldg(reinterpret_cast<const uint4*>(x + (r + 16 * k) * 128 + cx * 8)) : make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const uint32_t u[4] = {w[k].x, w[k].y, w[k].z, w[k].w};
#pragma unroll
        for (int j = 0; j < 4; ++j) { s[2 * j] += __uint_as_float(u[j] << 16); s[2 * j + 1] += __uint_as_float(u[j] & 0xFFFF0000u); }
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) red[ry][cx * 8 + j] = s[j];
  __syncthreads();
  if (threadIdx.x < 128) {
    float t = 0.f;
#pragma unroll
    for (int l = 0; l < 16; ++l) t += red[l][threadIdx.x];
    partial[(int64_t(blockIdx.y) * gridDim.x + blockIdx.x) * 128 + threadIdx.x] = t;
  }
}
__global__ void __launch_bounds__(256)
colsum5_final_kernel(Colsum5Args a, const float* __restrict__ partial, int blocks, int accumulate) {
  __shared__ float sm[256];
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  const float t = ordered_sum_block8(partial + int64_t(blockIdx.y) * blocks * 128 + c, blocks, 128, sm);
  if (threadIdx.x < 32) { float* o = a.out[blockIdx.y]; o[c] = accumulate ? o[c] + t : t; }
}

size_t colsum5_workspace_bytes(int64_t rows) { return size_t(ceil_div(rows > 0 ? rows : 1, kColsum5Rows)) * 5 * 128 * 4; }

int colsum5_bf16(const void* const* mats, float* const* outs, int64_t rows, int accumulate, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  const int64_t blocks = ceil_div(rows > 0 ? rows : 1, kColsum5Rows);
  if (workspace_bytes < size_t(blocks) * 5 * 128 * 4 || !workspace) { set_error("colsum5: workspace too small"); return HGN_ERR_WORKSPACE; }
  Colsum5Args a{};
  for (int i = 0; i < 5; ++i) { a.x[i] = rows > 0 ? static_cast<const __nv_bfloat16*>(mats[i]) : nullptr; a.out[i] = outs[i]; }
  HGN_TIMED("colsum", st);
  colsum5_partial_kernel<<<dim3(unsigned(blocks), 5), 256, 0, st>>>(a, rows, static_cast<float*>(workspace));
  colsum5_final_kernel<<<dim3(4, 5), 256, 0, st>>>(a, static_cast<const float*>(workspace), int(blocks), accumulate);
  HGN_LAUNCH_OK("colsum5");
  return HGN_OK;
}
}  // namespace hgn

extern "C" size_t hgn_colsum_workspace_bytes(int64_t rows, int32_t D) {
  return size_t(hgn::ceil_div(rows > 0 ? rows : 1, hgn::kColsumRowsPerBlock)) * size_t(D) * 4;
}

extern "C" int hgn_colsum(int dtype, const void* x, int64_t rows, int32_t D, float* out, void* workspace, size_t workspace_bytes,
                          void* stream) {
  HGN_CHECK_ARG(D >= 4 && D % 4 == 0 && D <= 256 && 256 % (D / 4) == 0, "colsum: D=%d must divide 1024 and be <= 256", D);
  HGN_CHECK_ARG(out && rows >= 0, "colsum: bad arguments");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (rows == 0) { HGN_CUDA_OK(cudaMemsetAsync(out, 0, size_t(D) * 4, st)); return HGN_OK; }
  const int64_t blocks = hgn::ceil_div(rows, hgn::kColsumRowsPerBlock);
  if (workspace_bytes < size_t(blocks) * D * 4 || !workspace) { hgn::set_error("colsum: workspace too small"); return HGN_ERR_WORKSPACE; }
  float* partial = static_cast<float*>(workspace);
  HGN_TIMED("colsum", st);
  if (dtype == HGN_F32) hgn::colsum_partial_kernel<float><<<unsigned(blocks), 256, 0, st>>>((const float*)x, rows, D, partial);
  else if (dtype == HGN_BF16) hgn::colsum_partial_kernel<__nv_bfloat16><<<unsigned(blocks), 256, 0, st>>>((const __nv_bfloat16*)x, rows, D, partial);
  else { hgn::set_error("colsum: unknown dtype %d", dtype); return HGN_ERR_INVALID_ARGUMENT; }
  hgn::colsum_final_kernel<<<(D + 127) / 128, 128, 0, st>>>(partial, blocks, D, out);
  HGN_LAUNCH_OK("colsum");
  return HGN_OK;
}

// ------------------------------------------------------------------------------------------------
// multi-source segment sum (gather backward): one rounding, fixed order
// ------------------------------------------------------------------------------------------------
namespace hgn {
// base and out are not __restrict__: the header lets out alias base (ops._FusedMLP chains calls with base = out).
template <typename T>
__global__ void __launch_bounds__(256)
multi_segment_sum_kernel(hgn_segment_sources ms, int64_t S, int32_t D, const T* base, T* out) {
  const int lane = threadIdx.x & 31;
  const int64_t seg = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
  if (seg >= S) return;
  for (int c = lane * 4; c < D; c += 128) {
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    if (base) s = load4(base + seg * D + c);
    for (int k = 0; k < ms.n_sources; ++k) {
      const T* data = static_cast<const T*>(ms.data[k]);
      const int32_t* perm = ms.perm[k];
      const int beg = ms.rowptr[k][seg], end = ms.rowptr[k][seg + 1];
      int j = beg;
      for (; j + 1 < end; j += 2) {
        const float4 a = load4(data + int64_t(perm[j]) * D + c);
        const float4 b = load4(data + int64_t(perm[j + 1]) * D + c);
        s.x += a.x; s.y += a.y; s.z += a.z; s.w += a.w;
        s.x += b.x; s.y += b.y; s.z += b.z; s.w += b.w;
      }
      if (j < end) {
        const float4 a = load4(data + int64_t(perm[j]) * D + c);
        s.x += a.x; s.y += a.y; s.z += a.z; s.w += a.w;
      }
    }
    store4(out + seg * D + c, s);
  }
}
}  // namespace hgn

extern "C" int hgn_multi_segment_sum(int dtype, const hgn_segment_sources* sources, int64_t S, int32_t D, const void* base,
                                     void* out, void* stream) {
  HGN_CHECK_ARG(sources && sources->n_sources >= 0 && sources->n_sources <= 4, "multi_segment_sum: bad sources");
  HGN_CHECK_ARG(D >= 4 && D % 4 == 0 && S >= 0 && out, "multi_segment_sum: D must be a multiple of 4");
  if (S == 0) return HGN_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const unsigned blocks = unsigned(hgn::ceil_div(S * 32, 256));
  HGN_TIMED("multi_segment_sum", st);
  if (dtype == HGN_F32) hgn::multi_segment_sum_kernel<float><<<blocks, 256, 0, st>>>(*sources, S, D, (const float*)base, (float*)out);
  else if (dtype == HGN_BF16) hgn::multi_segment_sum_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>(*sources, S, D, (const __nv_bfloat16*)base, (__nv_bfloat16*)out);
  else { hgn::set_error("multi_segment_sum: unknown dtype %d", dtype); return HGN_ERR_INVALID_ARGUMENT; }
  HGN_LAUNCH_OK("multi_segment_sum");
  return HGN_OK;
}
