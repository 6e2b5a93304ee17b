// step_wide.cu — the general step kernel for graphs with wide rows (hundreds of in-edges per neuron): one CTA per 32-row
// slice, all of its warps share the per-edge work of the slice (gather_edges_wide, step_body.cuh), the leader warp does the
// ordered accumulation and the neuron update.  Same arithmetic, bit-identical results; used for single-GPU handles whose
// mean slice width is >= kWideMinWidth (BASELINE.json configs[3]: 784 spike trains -> 400 excitatory <-> 400 inhibitory).
#include "step_body.cuh"
#include "train_body.cuh"

#include <cstdlib>

namespace snn {

struct WideSplit {   // very wide slices: terms pass over all SMs, then the ordered sums (WideSrc::mode, step_body.cuh)
    uint32_t mode;            // 0 single pass, 1 terms pass (grid.y = chunk), 2 sum pass (grid.y = accumulator)
    unsigned char *scratch;
    uint32_t chunks_cap, n_slices;
};

template <int MODEL, int CHEMG, bool NTREL, bool STDP, bool NET>
__global__ void __launch_bounds__(kWideWarps * 32) step_wide_kernel(const __grid_constant__ StepParams p, uint32_t stage_on, const __grid_constant__ WideSplit sp,
                                                                    const __grid_constant__ TrainParams tp) {
    extern __shared__ __align__(16) unsigned char wide_sm[];   // 2 x wide_buf_bytes(CHEMG): double-buffered chunk terms, then the node stage
    const uint32_t warp_global = blockIdx.x;   // one CTA per slice (terms pass: per slice and chunk)
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    pdl_wait();   // launch_pdl: the CTAs were scheduled while the previous pass / timestep was still draining
    if (blockIdx.x >= sp.n_slices) {
        // sum pass with fused spike trains: the CTAs past the last slice step 16 warps of trains each (accumulator row 0 only)
        if (NET && blockIdx.y == 0u) {
            const uint32_t tw = (blockIdx.x - sp.n_slices) * kWideWarps + warp;
            if (tw * 32u < tp.n_trains) train_step(tp, tw, lane);
        }
        return;
    }
    const uint32_t ln = warp_global * 32u + lane;
    const bool valid = ln < p.n_neurons;
    const uint32_t lnc = valid ? ln : p.n_neurons - 1;
    const uint32_t k0 = p.uniform_width ? warp_global * p.uniform_width : __ldg(p.slice_off + warp_global);
    const uint32_t k1 = p.uniform_width ? k0 + p.uniform_width : __ldg(p.slice_off + warp_global + 1);
    if (sp.mode == 1u && blockIdx.y * kWideChunk >= k1 - k0) return;   // this slice has no such chunk (CTA-uniform)
    const float *t0 = nullptr;
    if (CHEMG == 1) t0 = p.t_in + (size_t)(__ffs((int)p.nt_used) - 1) * p.t_stride;
    const WideStage stage = wide_stage_fill<NET>(p, wide_sm + 2u * wide_buf_bytes(CHEMG), stage_on != 0u);
    const WideSrc src{{p, lnc, p.own0 + lnc, lane, k0, k1, t0}, warp, (uint32_t)kWideWarps, wide_sm, stage, sp.mode, blockIdx.y, sp.scratch, sp.chunks_cap, sp.n_slices};
    neuron_step<MODEL, CHEMG, NTREL, STDP, NET>(p, src, warp_global, lane, ln, lnc, valid, false, false);
}

uint32_t wide_chunk_bytes(int chemg) { return wide_buf_bytes(chemg); }
uint32_t wide_chunk_krows() { return kWideChunk; }
size_t wide_part_bytes() { return wide_part_bytes_per_slice(); }

cudaError_t launch_step_wide(const StepParams &p, const StepSpec &spec, unsigned char *scratch, uint32_t chunks_cap, const TrainParams *trains,
                             cudaStream_t s) {
    if (p.n_neurons == 0) return cudaSuccess;
    const unsigned grid = (p.n_neurons + 31u) / 32u;
    static const TrainParams no_trains{};
    return dispatch_step(spec, cudaErrorInvalidValue, [&](auto k) {
        using K = decltype(k);
        auto launch = [&](dim3 g, size_t smem, uint32_t stage, WideSplit sp) -> cudaError_t {
            auto kern = step_wide_kernel<K::MODEL, K::CHEMG, K::NTREL, K::STDP, K::NET>;
            if (smem > 48u * 1024u) { cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); if (e != cudaSuccess) return e; }
            return launch_pdl(pdl_ok(p), kern, g, dim3(kWideWarps * 32), smem, s, p, stage, sp, (sp.mode == 2u && trains) ? *trains : no_trains);
        };
        if (scratch && chunks_cap) {
            // the per-edge work of every (slice, chunk) pair on its own CTA — all SMs — then one CTA per slice for the ordered additions
            // and the neuron update; the terms travel through L2
            cudaError_t e = launch(dim3(grid, chunks_cap), 0, 0u, WideSplit{1u, scratch, chunks_cap, grid});
            if (e != cudaSuccess) return e;
            constexpr uint32_t n_acc = 1u + (K::CHEMG == 3 ? (uint32_t)kNT : (K::CHEMG == 1 ? 1u : 0u));
            const unsigned train_ctas = (K::NET && trains) ? ((trains->n_trains + 31u) / 32u + kWideWarps - 1u) / kWideWarps : 0u;
            return launch(dim3(grid + train_ctas, n_acc), kWideSumBufs * (kWideChunk * 32u * 4u + 128u), 0u, WideSplit{2u, scratch, chunks_cap, grid});
        }
        // small networks: the node state rides in shared memory next to the chunk buffers (WideStage, step_body.cuh)
        const uint32_t sb = wide_stage_bytes(p.n_nodes, K::NET ? p.n_trains : 0u);
        const bool stage = p.n_nodes <= kWideStageMaxNodes && 2u * wide_buf_bytes(K::CHEMG) + sb <= 200u * 1024u;
        return launch(dim3(grid), 2u * wide_buf_bytes(K::CHEMG) + (stage ? sb : 0u), stage ? 1u : 0u, WideSplit{0u, nullptr, 0u, grid});
    });
}

}  // namespace snn
