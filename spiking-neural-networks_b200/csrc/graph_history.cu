// graph_history.cu — Graph::update_history on the device (graph/mod.rs:278-284): one record per timestep holding every edge
// weight of the sliced-ELL table in the canonical CSR order of snn_lattice_get_graph_csr (rows ascending, in-edges of a row in
// ascending presynaptic node order).
//
// Layout facts used here (sell_from_csr_kernel / sell_grid_kernel in kernels.cu): a slice is 32 rows, a k-row is 32 consecutive
// words (lane = row inside the slice), and the valid entries of a row come first, in canonical order.  So the entries of slice s
// are the contiguous output range [row_off[32 s], row_off[32 s + 32]), and the weights of a record are read without `col`.
#include "common.h"

namespace snn {

// per-row number of valid (non-pad) entries, written to row_off[r + 1]; rows are the 32 * n_slices table rows (those past the
// last neuron are all padding and count 0)
__global__ void __launch_bounds__(256) graph_row_count_kernel(const uint32_t *__restrict__ col, const uint32_t *__restrict__ slice_off,
                                                              uint32_t n_slices, uint32_t *__restrict__ row_off) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= (uint64_t)n_slices * 32u) return;
    const uint32_t s = (uint32_t)(r >> 5), lane = (uint32_t)(r & 31u);
    const uint32_t k0 = slice_off[s], k1 = slice_off[s + 1];
    uint32_t c = 0;
    for (uint32_t k = k0; k < k1; ++k) {
        if (col[(size_t)k * 32u + lane] == kColPad) break;   // valid entries first
        ++c;
    }
    row_off[r + 1] = c;
    if (r == 0) row_off[0] = 0;
}

// inclusive prefix sum of v[0, n) in place, one CTA (once per graph build, and once per drained chunk of spike events)
__global__ void __launch_bounds__(1024) graph_row_scan_kernel(uint32_t *v, uint64_t n) {
    __shared__ uint32_t part[1024];
    const uint32_t t = threadIdx.x;
    const uint64_t per = (n + 1023u) / 1024u, b = (uint64_t)t * per, e = b + per < n ? b + per : n;
    uint32_t sum = 0;
    for (uint64_t i = b; i < e; ++i) sum += v[i];
    part[t] = sum;
    __syncthreads();
    for (uint32_t off = 1; off < 1024u; off <<= 1) {
        const uint32_t add = t >= off ? part[t - off] : 0u;
        __syncthreads();
        part[t] += add;
        __syncthreads();
    }
    uint32_t run = part[t] - sum;
    for (uint64_t i = b; i < e; ++i) { run += v[i]; v[i] = run; }
}

constexpr uint32_t kRecWarps = 8;

// one record: out[row_off[r] + k] = wgt of entry k of row r.  Work item = one tile of 32 k-rows of one slice, one warp each,
// staged through shared memory so that the loads are whole k-rows (128 B) and the stores are contiguous: a slice no wider than
// one tile is written as its compacted output range, a tile of a wider slice row by row (each row's part one 128 B store).
// Narrow tables (every slice <= 32 k-rows) put 8 slices in a CTA; wide ones (`tiled`) put 8 tiles of one slice in a CTA, so that
// a table of a few very wide slices (all-to-all input) still spreads over the whole GPU.
__global__ void __launch_bounds__(kRecWarps * 32) graph_record_kernel(const float *__restrict__ wgt, const uint32_t *__restrict__ slice_off,
                                                                      const uint32_t *__restrict__ row_off, uint32_t n_slices,
                                                                      uint32_t tiled, float *__restrict__ out) {
    pdl_wait();   // the weights are those the previous kernel in the stream left
    __shared__ float tile[kRecWarps][32][33];
    __shared__ uint32_t offs[kRecWarps][33];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint32_t s = tiled ? blockIdx.x : blockIdx.x * kRecWarps + warp;
    const uint32_t kt = tiled ? (blockIdx.y * kRecWarps + warp) * 32u : 0u;
    if (s >= n_slices) return;
    const uint32_t k0 = slice_off[s], width = slice_off[s + 1] - k0;
    if (kt >= width) return;
    const uint32_t my_off = row_off[(size_t)s * 32u + lane], my_end = row_off[(size_t)s * 32u + lane + 1];
    const uint32_t base = __shfl_sync(0xFFFFFFFFu, my_off, 0), end = __shfl_sync(0xFFFFFFFFu, my_end, 31);
    offs[warp][lane] = my_off - base;
    if (lane == 31) offs[warp][32] = end - base;
    float (*t)[33] = tile[warp];
    const uint32_t tk = min(32u, width - kt);
    const float *src = wgt + ((size_t)k0 + kt) * 32u + lane;
    for (uint32_t i = 0; i < tk; ++i) t[i][lane] = __ldg(src + (size_t)i * 32u);
    __syncwarp();
    if (width <= 32u) {
        // the whole slice is in the tile: its output range is contiguous
        const uint32_t n = end - base;
        for (uint32_t o = lane; o < n; o += 32u) {
            uint32_t r = 0;   // last row whose range starts at or before o (rows without entries share the next start)
            for (uint32_t step = 16; step; step >>= 1)
                if (offs[warp][r + step] <= o) r += step;
            out[base + o] = t[o - offs[warp][r]][r];
        }
    } else {
        for (uint32_t r = 0; r < 32u; ++r) {
            const uint32_t ro = base + offs[warp][r], rc = offs[warp][r + 1] - offs[warp][r];
            if (lane < tk && kt + lane < rc) out[ro + kt + lane] = t[lane][r];
        }
    }
}

cudaError_t launch_graph_row_offsets(const uint32_t *col, const uint32_t *slice_off, uint32_t n_slices, uint32_t *row_off,
                                     cudaStream_t s) {
    if (n_slices == 0) return cudaMemsetAsync(row_off, 0, 4, s);
    const uint64_t rows = (uint64_t)n_slices * 32u;
    graph_row_count_kernel<<<(unsigned)((rows + 255u) / 256u), 256, 0, s>>>(col, slice_off, n_slices, row_off);
    cudaError_t e = cudaGetLastError();
    return e != cudaSuccess ? e : launch_scan_u32(row_off + 1, rows, s);
}

cudaError_t launch_scan_u32(uint32_t *v, uint64_t n, cudaStream_t s) {
    graph_row_scan_kernel<<<1, 1024, 0, s>>>(v, n);
    return cudaGetLastError();
}

cudaError_t launch_graph_record(const float *wgt, const uint32_t *slice_off, const uint32_t *row_off, uint32_t n_slices,
                                uint32_t max_width, float *out, cudaStream_t s) {
    if (n_slices == 0) return cudaSuccess;
    const uint32_t tiles = (max_width + 31u) / 32u;
    const dim3 grid = tiles > 1 ? dim3(n_slices, (tiles + kRecWarps - 1) / kRecWarps) : dim3((n_slices + kRecWarps - 1) / kRecWarps);
    graph_record_kernel<<<grid, kRecWarps * 32, 0, s>>>(wgt, slice_off, row_off, n_slices, tiles > 1 ? 1u : 0u, out);
    return cudaGetLastError();
}

}  // namespace snn
