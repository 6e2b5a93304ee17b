// spike_events.cu — spike event lists from the staged spike raster (SNN_OPT_UPDATE_SPIKE_EVENTS): per lattice and staged record,
// the indices of the cells that spiked, ascending, records in step order.
//
// The raster holds one bit per node and record (the step kernels' spike_hist words).  The event order is fixed by an item order:
// an item is one raster word of one lattice in one record, lattice-major, then record, then word.  A tile is kEvRounds rounds of
// kEvThreads consecutive items.  Three launches per drained chunk:
//   1. spike_event_count_kernel: set bits per tile (popcount of every masked word) -> tile_off[t + 1];
//   2. the exclusive scan of the tile counts (launch_scan_u32) -> tile_off[t] = events before tile t, tile_off[n_tiles] = total;
//   3. spike_event_scatter_kernel: the tile is read again, scanned inside the CTA round by round, and every set bit's index is
//      written at its final position.  No atomics: positions follow from the scan alone, so the lists come out in canonical order.
// The host reads the total between 2 and 3 to size the event buffer.
#include "common.h"

namespace snn {

constexpr uint32_t kEvThreads = 256, kEvRounds = 16, kEvTile = kEvThreads * kEvRounds;

struct EvItem {
    uint32_t word;   // the raster word with the bits outside the lattice cleared
    uint32_t seg, rec;
    bool first;      // first word of the record (rec_off is written there)
};

// item `it` of the chunk; `k` is a segment at or before the item's own (items of one thread ascend, so k only moves forward)
__device__ __forceinline__ EvItem ev_item(const EvParams &p, uint32_t it, uint32_t &k) {
    while (k + 1 < p.n_seg && it >= p.seg[k + 1].item0) ++k;
    const EvSeg &g = p.seg[k];
    const uint32_t rel = it - g.item0, rec = rel / g.nw, w = g.w0 + (rel - rec * g.nw);
    uint32_t word = __ldg(g.raster + (size_t)rec * g.stride + w);
    const uint32_t b0 = w * 32u;
    const uint32_t lo = g.bit0 > b0 ? g.bit0 - b0 : 0u, hi = g.bit1 - b0 < 32u ? g.bit1 - b0 : 32u;
    const uint32_t mask = (hi == 32u ? 0xFFFFFFFFu : ((1u << hi) - 1u)) & ~((1u << lo) - 1u);
    return EvItem{word & mask, k, rec, w == g.w0};
}

// tile_off[t + 1] = set bits of tile t; tile_off[0] = 0
__global__ void __launch_bounds__(kEvThreads) spike_event_count_kernel(const EvParams p, uint32_t *__restrict__ tile_off) {
    __shared__ uint32_t warp_sum[kEvThreads / 32];
    const uint32_t t0 = blockIdx.x * kEvTile;
    uint32_t k = 0, c = 0;
    for (uint32_t r = 0; r < kEvRounds; ++r) {
        const uint32_t it = t0 + r * kEvThreads + threadIdx.x;
        if (it < p.n_items) c += __popc(ev_item(p, it, k).word);
    }
    for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(0xFFFFFFFFu, c, o);
    if ((threadIdx.x & 31u) == 0) warp_sum[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t s = 0;
        for (uint32_t w = 0; w < kEvThreads / 32; ++w) s += warp_sum[w];
        tile_off[blockIdx.x + 1] = s;
        if (blockIdx.x == 0) tile_off[0] = 0;
    }
}

// events[pos ..] = indices of the set bits of every item, pos = events before the item in item order; rec_off[seg * steps + rec]
// = events before the record's first item
__global__ void __launch_bounds__(kEvThreads) spike_event_scatter_kernel(const EvParams p, const uint32_t *__restrict__ tile_off,
                                                                         uint32_t *__restrict__ events, uint32_t *__restrict__ rec_off) {
    __shared__ uint32_t warp_sum[kEvThreads / 32];
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t t0 = blockIdx.x * kEvTile;
    uint32_t base = tile_off[blockIdx.x];
    uint32_t k = 0;
    for (uint32_t r = 0; r < kEvRounds; ++r) {
        const uint32_t it = t0 + r * kEvThreads + threadIdx.x;
        if (t0 + r * kEvThreads >= p.n_items) break;   // uniform across the CTA
        EvItem e{0u, 0u, 0u, false};
        if (it < p.n_items) e = ev_item(p, it, k);
        const uint32_t c = __popc(e.word);
        uint32_t incl = c;   // inclusive scan inside the warp, then across the warps
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= (uint32_t)o) incl += v;
        }
        if (lane == 31) warp_sum[warp] = incl;
        __syncthreads();
        uint32_t before = 0, round_sum = 0;
        for (uint32_t w = 0; w < kEvThreads / 32; ++w) {
            const uint32_t s = warp_sum[w];
            if (w < warp) before += s;
            round_sum += s;
        }
        __syncthreads();   // warp_sum is rewritten by the next round
        uint32_t pos = base + before + incl - c;
        if (it < p.n_items) {
            const EvSeg &g = p.seg[e.seg];
            if (e.first) rec_off[e.seg * p.steps + e.rec] = pos;
            const uint32_t w = g.w0 + (it - g.item0 - e.rec * g.nw);
            uint32_t word = e.word;
            while (word) {
                const uint32_t b = __ffs(word) - 1u;
                events[pos++] = w * 32u + b - g.bit0 + g.add;
                word &= word - 1u;
            }
        }
        base += round_sum;
    }
}

cudaError_t launch_spike_event_count(const EvParams &p, uint32_t *tile_off, cudaStream_t s) {
    const uint32_t tiles = ev_tiles(p.n_items);
    if (tiles == 0) return cudaMemsetAsync(tile_off, 0, 4, s);
    spike_event_count_kernel<<<tiles, kEvThreads, 0, s>>>(p, tile_off);
    cudaError_t e = cudaGetLastError();
    return e != cudaSuccess ? e : launch_scan_u32(tile_off + 1, tiles, s);
}

cudaError_t launch_spike_event_scatter(const EvParams &p, const uint32_t *tile_off, uint32_t *events, uint32_t *rec_off, cudaStream_t s) {
    const uint32_t tiles = ev_tiles(p.n_items);
    if (tiles == 0) return cudaSuccess;
    spike_event_scatter_kernel<<<tiles, kEvThreads, 0, s>>>(p, tile_off, events, rec_off);
    return cudaGetLastError();
}

uint32_t ev_tiles(uint32_t n_items) { return (n_items + kEvTile - 1) / kEvTile; }

}  // namespace snn
