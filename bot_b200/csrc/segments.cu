// Row splitting for heavy-tailed degree distributions (SURVEY.md section 7 "Degree skew": Reddit's largest
// in-degree is ~21 K, products' ~17 K; a power-law synthetic graph is far worse).  A CSR whose longest row
// exceeds the segment length gets a table of work items = row segments; the gather kernels then spread a heavy
// row over several warps, write (max, sum, unnormalised accumulator) / (partial gradient) per segment into
// scratch slots, and a combine kernel merges them in slot order — still no atomics, still deterministic.
#include <cub/cub.cuh>


#include "common.cuh"
#include "params.cuh"

namespace botgat {

int segment_length() {
  const int v = (int)env_int("BOTGAT_SEG", 2048);
  return v < 32 ? 32 : v;
}

__global__ void k_seg_count(int n_rows, const int32_t* __restrict__ deg, int L, int32_t* __restrict__ nseg,
                            int32_t* __restrict__ pcnt, int32_t* __restrict__ flag) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r > n_rows) return;
  int n = 0;
  if (r < n_rows) n = max(1, (deg[r] + L - 1) / L);
  nseg[r] = n;                 // entry n_rows is the 0 sentinel the exclusive scans turn into totals
  pcnt[r] = n > 1 ? n : 0;
  flag[r] = n > 1 ? 1 : 0;
}

__global__ void k_seg_fill(int n_rows, const int32_t* __restrict__ indptr, int L, const int32_t* __restrict__ seg_off,
                           const int32_t* __restrict__ slot_off, const int32_t* __restrict__ split_off,
                           int32_t* __restrict__ row, int32_t* __restrict__ beg, int32_t* __restrict__ end,
                           int32_t* __restrict__ slot, int32_t* __restrict__ split_rows,
                           int32_t* __restrict__ split_first) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r > n_rows) return;
  if (r == n_rows) {
    split_first[split_off[n_rows]] = slot_off[n_rows];  // sentinel: total number of slots
    return;
  }
  const int n = seg_off[r + 1] - seg_off[r];
  const int b = indptr[r], e = indptr[r + 1];
  for (int s = 0; s < n; ++s) {
    const int i = seg_off[r] + s;
    row[i] = r;
    beg[i] = b + s * L;
    end[i] = min(e, b + (s + 1) * L);
    slot[i] = n > 1 ? slot_off[r] + s : -1;
  }
  if (n > 1) {
    split_rows[split_off[r]] = r;
    split_first[split_off[r]] = slot_off[r];
  }
}

void free_segments(botgat_graph::SegTable* t, bool async, cudaStream_t st) {
  void* ptrs[] = {t->row, t->beg, t->end, t->slot, t->split_rows, t->split_first};
  for (void* q : ptrs) {
    if (!q) continue;
    if (!async || cudaFreeAsync(q, st) != cudaSuccess) { cudaGetLastError(); cudaFree(q); }
  }
  *t = botgat_graph::SegTable();
}

int build_segments(int n_rows, const int32_t* indptr, const int32_t* deg, int64_t max_deg, botgat_graph::SegTable* t,
                   cudaStream_t st) {
  const int L = segment_length();
  if (n_rows == 0 || max_deg <= L) return 0;
  int32_t *nseg, *pcnt, *flag, *seg_off, *slot_off, *split_off;
  const size_t nb = sizeof(int32_t) * (n_rows + 1);
  BG_CHECK(cudaMallocAsync(&nseg, nb, st)); BG_CHECK(cudaMallocAsync(&pcnt, nb, st)); BG_CHECK(cudaMallocAsync(&flag, nb, st));
  BG_CHECK(cudaMallocAsync(&seg_off, nb, st)); BG_CHECK(cudaMallocAsync(&slot_off, nb, st));
  BG_CHECK(cudaMallocAsync(&split_off, nb, st));
  k_seg_count<<<(n_rows + 1 + 255) / 256, 256, 0, st>>>(n_rows, deg, L, nseg, pcnt, flag);
  BG_LAUNCHED(1);
  size_t tb = 0;
  BG_CHECK(cub::DeviceScan::ExclusiveSum(nullptr, tb, nseg, seg_off, n_rows + 1, st));
  void* tmp = nullptr;
  BG_CHECK(cudaMallocAsync(&tmp, tb, st));
  BG_CHECK(cub::DeviceScan::ExclusiveSum(tmp, tb, nseg, seg_off, n_rows + 1, st));
  BG_CHECK(cub::DeviceScan::ExclusiveSum(tmp, tb, pcnt, slot_off, n_rows + 1, st));
  BG_CHECK(cub::DeviceScan::ExclusiveSum(tmp, tb, flag, split_off, n_rows + 1, st));
  BG_LAUNCHED(3);
  int32_t tot[3];
  BG_CHECK(cudaMemcpyAsync(&tot[0], seg_off + n_rows, 4, cudaMemcpyDeviceToHost, st));
  BG_CHECK(cudaMemcpyAsync(&tot[1], slot_off + n_rows, 4, cudaMemcpyDeviceToHost, st));
  BG_CHECK(cudaMemcpyAsync(&tot[2], split_off + n_rows, 4, cudaMemcpyDeviceToHost, st));
  BG_CHECK(cudaStreamSynchronize(st));
  t->n_items = tot[0]; t->n_slots = tot[1]; t->n_split = tot[2];
  BG_CHECK(cudaMallocAsync(&t->row, 4 * (size_t)t->n_items, st)); BG_CHECK(cudaMallocAsync(&t->beg, 4 * (size_t)t->n_items, st));
  BG_CHECK(cudaMallocAsync(&t->end, 4 * (size_t)t->n_items, st)); BG_CHECK(cudaMallocAsync(&t->slot, 4 * (size_t)t->n_items, st));
  BG_CHECK(cudaMallocAsync(&t->split_rows, 4 * (size_t)(t->n_split + 1), st));
  BG_CHECK(cudaMallocAsync(&t->split_first, 4 * (size_t)(t->n_split + 1), st));
  k_seg_fill<<<(n_rows + 1 + 255) / 256, 256, 0, st>>>(n_rows, indptr, L, seg_off, slot_off, split_off, t->row, t->beg,
                                                       t->end, t->slot, t->split_rows, t->split_first);
  BG_LAUNCHED(1);
  BG_CHECK(cudaGetLastError());
  BG_CHECK(cudaFreeAsync(tmp, st));
  BG_CHECK(cudaFreeAsync(nseg, st)); BG_CHECK(cudaFreeAsync(pcnt, st)); BG_CHECK(cudaFreeAsync(flag, st));
  BG_CHECK(cudaFreeAsync(seg_off, st)); BG_CHECK(cudaFreeAsync(slot_off, st)); BG_CHECK(cudaFreeAsync(split_off, st));
  BG_CHECK(cudaStreamSynchronize(st));
  return 0;
}

// ---------------------------------------------------------------------------
// combine kernels: one warp per (split row, head)
// ---------------------------------------------------------------------------
// forward scratch slot layout (floats): [H][D] unnormalised accumulators, then [H][2] (max, sum); slot stride
// rounded up to 4 floats so that vector stores into a slot stay 16-byte aligned
__global__ void __launch_bounds__(256)
k_fwd_combine(int n_split, int H, int D, int64_t ld_out, const int32_t* __restrict__ split_rows,
              const int32_t* __restrict__ split_first, const float* __restrict__ scratch,
              const float* __restrict__ ds, float* __restrict__ out, float* __restrict__ row_max,
              float* __restrict__ row_sum, const Epilogue ep) {
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (w >= n_split * H) return;
  const int i = w / H, h = w - i * H;
  const int row = split_rows[i], s0 = split_first[i], s1 = split_first[i + 1];
  const int64_t stride = fwd_slot_floats(H, D);
  const int64_t ml = (int64_t)H * D + h * 2;  // offset of (max, sum) of head h inside a slot
  float M = -INFINITY;
  for (int s = s0; s < s1; ++s) M = fmaxf(M, scratch[s * stride + ml]);
  float L = 0.f;
  for (int s = s0; s < s1; ++s) {
    const float m = scratch[s * stride + ml];
    if (m != -INFINITY) L += scratch[s * stride + ml + 1] * __expf(m - M);
  }
  float scale = L > 0.f ? 1.f / L : 0.f;
  if (ds) scale *= ds[row];
  for (int d = lane; d < D; d += 32) {
    float a = 0.f;
    for (int s = s0; s < s1; ++s) {
      const float m = scratch[s * stride + ml];
      if (m != -INFINITY) a = fmaf(scratch[s * stride + (int64_t)h * D + d], __expf(m - M), a);
    }
    Vec<1> o;
    o.v = a * scale;
    ep.apply(o, row, (int64_t)h * D + d);
    out[(int64_t)row * ld_out + h * D + d] = o.v;
  }
  if (lane == 0) {
    row_max[(int64_t)row * H + h] = M;
    row_sum[(int64_t)row * H + h] = L;
  }
}

// backward scratch slot layout (floats): [H][D] partial grad_ft (before the src scale), then [H] partial grad_el
__global__ void __launch_bounds__(256)
k_bwd_combine(int n_split, int H, int D, int64_t ld_gft, const int32_t* __restrict__ split_rows,
              const int32_t* __restrict__ split_first, const float* __restrict__ scratch,
              const float* __restrict__ cs, float* __restrict__ grad_ft, float* __restrict__ grad_el) {
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (w >= n_split * H) return;
  const int i = w / H, h = w - i * H;
  const int row = split_rows[i], s0 = split_first[i], s1 = split_first[i + 1];
  const int64_t stride = bwd_slot_floats(H, D);
  const float c = cs ? cs[row] : 1.f;
  for (int d = lane; d < D; d += 32) {
    float a = 0.f;
    for (int s = s0; s < s1; ++s) a += scratch[s * stride + (int64_t)h * D + d];
    grad_ft[(int64_t)row * ld_gft + h * D + d] = a * c;
  }
  if (lane == 0) {
    float gsum = 0.f;
    for (int s = s0; s < s1; ++s) gsum += scratch[s * stride + (int64_t)H * D + h];
    grad_el[(int64_t)row * H + h] = gsum;
  }
}

int launch_fwd_combine(const botgat_graph::SegTable& t, int H, int D, int64_t ld_out, const float* scratch,
                       const float* ds, float* out, float* row_max, float* row_sum, const Epilogue& ep, cudaStream_t st) {
  if (t.n_split == 0) return 0;
  const int64_t warps = (int64_t)t.n_split * H;
  k_fwd_combine<<<(unsigned)((warps + 7) / 8), 256, 0, st>>>(t.n_split, H, D, ld_out, t.split_rows, t.split_first,
                                                           scratch, ds, out, row_max, row_sum, ep);
  BG_LAUNCHED(1);
  BG_CHECK(cudaGetLastError());
  return 0;
}

int launch_bwd_combine(const botgat_graph::SegTable& t, int H, int D, int64_t ld_gft, const float* scratch,
                       const float* cs, float* grad_ft, float* grad_el, cudaStream_t st) {
  if (t.n_split == 0) return 0;
  const int64_t warps = (int64_t)t.n_split * H;
  k_bwd_combine<<<(unsigned)((warps + 7) / 8), 256, 0, st>>>(t.n_split, H, D, ld_gft, t.split_rows, t.split_first,
                                                           scratch, cs, grad_ft, grad_el);
  BG_LAUNCHED(1);
  BG_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace botgat
