// Halo exchange over NVLink peer memory (edge-cut partitioning, SURVEY.md s8e; no reference counterpart: the reference is single
// device).  One process per GPU; every rank allocates its exchange pool with cudaMalloc, exports it with cudaIpcGetMemHandle and
// maps its peers' pools with cudaIpcOpenMemHandle (the 64-byte handles travel over torch.distributed).  A push is then ONE small
// kernel of this rank: it copies the boundary rows its peers need straight into their pools (ordinary stores through the NVLink
// mapping), fences, and the last CTA to finish raises a 4-byte flag in each peer's pool; the consumer's stream runs a one-warp
// kernel that spins on its own flags before the kernel that reads the rows.  No NCCL kernel, no host round trip, nothing that
// needs an SM of the receiving GPU while its persistent compute kernels hold all of them.
//
// Flags carry a monotonically increasing exchange number chosen by the (identical) host programs of all ranks, so they are never
// reset: a waiter proceeds as soon as flag >= its exchange number.
#include <cuda_runtime.h>
#include <string.h>

#include "common.cuh"

namespace hgn {

__global__ void halo_push_kernel(const uint4* __restrict__ table, const int32_t* __restrict__ send_index, hgn_halo_peers peers, int n_peers,
                                 int64_t total_rows, int row_u4, uint32_t epoch, unsigned int* done_counter) {
  // one warp per row: D * elem_size bytes = row_u4 16-byte pieces (128 bf16 = 16 pieces: half a warp)
  const int warps_per_block = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int64_t i = int64_t(blockIdx.x) * warps_per_block + warp; i < total_rows; i += int64_t(gridDim.x) * warps_per_block) {
    int q = 0;
    while (q + 1 < n_peers && i >= peers.row_begin[q + 1]) ++q;
    const int64_t local = i - peers.row_begin[q];
    const uint4* src = table + int64_t(__ldg(send_index + i)) * row_u4;
    uint4* dst = reinterpret_cast<uint4*>(peers.dst[q]) + local * row_u4;
    for (int c = lane; c < row_u4; c += 32) dst[c] = __ldg(src + c);
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int prev = atomicAdd(done_counter, 1u);
    if (prev == gridDim.x - 1) {                 // every CTA's rows are fenced: raise the flags, re-arm the counter
      *done_counter = 0u;
      __threadfence_system();
      for (int q = 0; q < n_peers; ++q)
        if (peers.flag[q] != nullptr) *reinterpret_cast<volatile uint32_t*>(peers.flag[q]) = epoch;
    }
  }
}

__global__ void halo_wait_kernel(hgn_halo_flags flags, int n_flags, uint32_t epoch, uint32_t* timeout_word) {
  const int q = threadIdx.x;
  if (q < n_flags && flags.flag[q] != nullptr) {
    const volatile uint32_t* f = reinterpret_cast<const volatile uint32_t*>(flags.flag[q]);
    unsigned long long spins = 0;
    while (int32_t(*f - epoch) < 0) {            // wrap-safe "flag < epoch"
      if (++spins > (1ull << 31)) {              // seconds: a peer that never pushes must end in an error, not in a hung GPU
        if (timeout_word != nullptr) *timeout_word = 0xDEAD0000u | uint32_t(q);
        __trap();
      }
    }
  }
  __threadfence_system();
}

// Cluster pooling across ranks: one 128-thread block per cluster, thread = feature; the ranks' rows are read in rank order.
__global__ void __launch_bounds__(128)
cluster_combine_kernel(const float* __restrict__ slots, int world, int rank, int64_t C, __nv_bfloat16* __restrict__ out_sum,
                       __nv_bfloat16* __restrict__ out_mean, __nv_bfloat16* __restrict__ out_max, __nv_bfloat16* __restrict__ out_min,
                       int32_t* __restrict__ argmax, int32_t* __restrict__ argmin, int32_t* __restrict__ count) {
  constexpr int W = HGN_SEGMENT_PARTIAL_WIDTH;
  const int c = threadIdx.x;
  const int64_t k = blockIdx.x;
  float t = 0.f, mx = 0.f, mn = 0.f;
  int cnt = 0, wx = -1, wn = -1;
  for (int r = 0; r < world; ++r) {
    const float* row = slots + (int64_t(r) * C + k) * W;
    const int n = __float_as_int(row[384]);
    t = __fadd_rn(t, row[c]);
    if (n == 0) continue;                       // a rank without a member of this cluster: its max / min are not values
    cnt += n;
    if (out_max || argmax) { const float a = row[128 + c]; if (wx < 0 || a > mx) { mx = a; wx = r; } }
    if (out_min || argmin) { const float b = row[256 + c]; if (wn < 0 || b < mn) { mn = b; wn = r; } }
  }
  const int64_t o = k * 128 + c;
  if (out_sum) out_sum[o] = __float2bfloat16_rn(t);
  if (out_mean) out_mean[o] = __float2bfloat16_rn(__fmul_rn(t, 1.0f / float(max(cnt, 1))));
  if (out_max) out_max[o] = __float2bfloat16_rn(mx);
  if (out_min) out_min[o] = __float2bfloat16_rn(mn);
  if (argmax && wx != rank) argmax[o] = -1;
  if (argmin && wn != rank) argmin[o] = -1;
  if (count && c == 0) count[k] = cnt;
}

__global__ void cluster_grad_sum_kernel(const __nv_bfloat16* __restrict__ slots, int world, int64_t n, __nv_bfloat16* __restrict__ out) {
  const int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  float t = 0.f;
  for (int r = 0; r < world; ++r) t = __fadd_rn(t, __bfloat162float(slots[int64_t(r) * n + i]));
  out[i] = __float2bfloat16_rn(t);
}

__global__ void cluster_mean_grad_kernel(const __nv_bfloat16* __restrict__ g_sum, const __nv_bfloat16* __restrict__ g_mean,
                                         const int32_t* __restrict__ count, int64_t C, __nv_bfloat16* __restrict__ out) {
  const int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (i >= C * 128) return;
  const float inv = 1.0f / float(max(count[i / 128], 1));
  const float pre = __fadd_rn(0.f, g_sum ? __bfloat162float(g_sum[i]) : 0.f);
  out[i] = __float2bfloat16_rn(__fmaf_rn(__bfloat162float(g_mean[i]), inv, pre));
}

}  // namespace hgn

using namespace hgn;

extern "C" int hgn_peer_alloc(size_t bytes, void** ptr, unsigned char* handle64) {
  HGN_CHECK_ARG(ptr != nullptr && handle64 != nullptr && bytes > 0, "peer_alloc: bad arguments");
  HGN_CUDA_OK(cudaMalloc(ptr, bytes));
  HGN_CUDA_OK(cudaMemset(*ptr, 0, bytes));
  cudaIpcMemHandle_t h;
  HGN_CUDA_OK(cudaIpcGetMemHandle(&h, *ptr));
  static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
  memcpy(handle64, &h, 64);
  HGN_CUDA_OK(cudaDeviceSynchronize());
  return HGN_OK;
}

extern "C" int hgn_peer_open(const unsigned char* handle64, void** ptr) {
  HGN_CHECK_ARG(ptr != nullptr && handle64 != nullptr, "peer_open: bad arguments");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  HGN_CUDA_OK(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return HGN_OK;
}

extern "C" int hgn_peer_close(void* ptr) {
  if (ptr != nullptr) HGN_CUDA_OK(cudaIpcCloseMemHandle(ptr));
  return HGN_OK;
}

extern "C" int hgn_peer_free(void* ptr) {
  if (ptr != nullptr) HGN_CUDA_OK(cudaFree(ptr));
  return HGN_OK;
}

extern "C" int hgn_halo_push(int dtype, const void* table, const int32_t* send_index, int32_t D, const hgn_halo_peers* peers, int32_t n_peers,
                             uint32_t epoch, void* counter, void* stream) {
  HGN_CHECK_ARG(peers != nullptr && n_peers >= 0 && n_peers <= HGN_MAX_PEERS, "halo_push: n_peers=%d outside [0,%d]", n_peers, HGN_MAX_PEERS);
  HGN_CHECK_ARG(counter != nullptr, "halo_push: counter is NULL");
  const size_t elem = dtype == HGN_BF16 ? 2 : 4;
  HGN_CHECK_ARG((size_t(D) * elem) % 16 == 0, "halo_push: rows must be a multiple of 16 bytes");
  if (n_peers == 0) return HGN_OK;
  const int64_t total = peers->row_begin[n_peers];
  HGN_CHECK_ARG(total >= 0 && (total == 0 || (table != nullptr && send_index != nullptr)), "halo_push: null pointer");
  for (int q = 0; q < n_peers; ++q)
    HGN_CHECK_ARG(peers->row_begin[q] <= peers->row_begin[q + 1] && (peers->row_begin[q] == peers->row_begin[q + 1] || peers->dst[q] != nullptr),
                  "halo_push: peer %d has rows but no destination", q);
  const int warps = 8;
  int64_t blocks = (total + warps - 1) / warps;
  if (blocks < 1) blocks = 1;                    // flags are raised even when there is nothing to send (the peer still waits for them)
  if (blocks > 64) blocks = 64;                  // a few CTAs saturate one NVLink direction for these sizes; they slot in beside persistent kernels
  HGN_TIMED("halo_push", static_cast<cudaStream_t>(stream));
  halo_push_kernel<<<unsigned(blocks), warps * 32, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint4*>(table), send_index, *peers, n_peers, total, int(size_t(D) * elem / 16), epoch, static_cast<unsigned int*>(counter));
  HGN_LAUNCH_OK("halo_push");
  return HGN_OK;
}

extern "C" int hgn_halo_wait(const hgn_halo_flags* flags, int32_t n_flags, uint32_t epoch, void* stream) {
  HGN_CHECK_ARG(flags != nullptr && n_flags >= 0 && n_flags <= HGN_MAX_PEERS, "halo_wait: n_flags=%d outside [0,%d]", n_flags, HGN_MAX_PEERS);
  if (n_flags == 0) return HGN_OK;
  HGN_TIMED("halo_wait", static_cast<cudaStream_t>(stream));
  halo_wait_kernel<<<1, 32, 0, static_cast<cudaStream_t>(stream)>>>(*flags, n_flags, epoch, nullptr);
  HGN_LAUNCH_OK("halo_wait");
  return HGN_OK;
}

extern "C" int hgn_cluster_combine(const float* slots, int32_t world, int32_t rank, int64_t C, void* out_sum, void* out_mean, void* out_max,
                                   void* out_min, int32_t* argmax, int32_t* argmin, int32_t* count, void* stream) {
  HGN_CHECK_ARG(world >= 1 && world <= HGN_MAX_PEERS && rank >= 0 && rank < world && C >= 0, "cluster_combine: world=%d rank=%d C=%lld",
                world, rank, (long long)C);
  HGN_CHECK_ARG(C == 0 || slots != nullptr, "cluster_combine: null slots");
  if (C == 0) return HGN_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  HGN_TIMED("cluster_combine", st);
  cluster_combine_kernel<<<unsigned(C), 128, 0, st>>>(slots, world, rank, C, static_cast<__nv_bfloat16*>(out_sum), static_cast<__nv_bfloat16*>(out_mean),
                                                      static_cast<__nv_bfloat16*>(out_max), static_cast<__nv_bfloat16*>(out_min), argmax, argmin, count);
  HGN_LAUNCH_OK("cluster_combine");
  return HGN_OK;
}

extern "C" int hgn_cluster_grad_sum(int dtype, const void* slots, int32_t world, int64_t C, int32_t D, void* out, void* stream) {
  HGN_CHECK_ARG(dtype == HGN_BF16, "cluster_grad_sum: dtype %d, only bf16 (%d) is supported", dtype, int(HGN_BF16));
  HGN_CHECK_ARG(world >= 1 && world <= HGN_MAX_PEERS && C >= 0 && D > 0, "cluster_grad_sum: world=%d C=%lld D=%d", world, (long long)C, D);
  HGN_CHECK_ARG(C == 0 || (slots && out), "cluster_grad_sum: null pointer");
  const int64_t n = C * D;
  if (n == 0) return HGN_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  HGN_TIMED("cluster_grad_sum", st);
  cluster_grad_sum_kernel<<<unsigned(ceil_div(n, 256)), 256, 0, st>>>(static_cast<const __nv_bfloat16*>(slots), world, n, static_cast<__nv_bfloat16*>(out));
  HGN_LAUNCH_OK("cluster_grad_sum");
  return HGN_OK;
}

extern "C" int hgn_cluster_mean_grad(const void* g_sum, const void* g_mean, const int32_t* count, int64_t C, void* out, void* stream) {
  HGN_CHECK_ARG(C >= 0 && (C == 0 || (g_mean && count && out)), "cluster_mean_grad: null pointer");
  if (C == 0) return HGN_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  HGN_TIMED("cluster_mean_grad", st);
  cluster_mean_grad_kernel<<<unsigned(ceil_div(C * 128, 256)), 256, 0, st>>>(static_cast<const __nv_bfloat16*>(g_sum), static_cast<const __nv_bfloat16*>(g_mean),
                                                                           count, C, static_cast<__nv_bfloat16*>(out));
  HGN_LAUNCH_OK("cluster_mean_grad");
  return HGN_OK;
}
