// step_multi.cu — K timesteps per launch for lattices and networks that live in L2 (BASELINE.json configs[0], [2], [3]).
//
// The reference's accelerator loop costs 4 launches + 4 host waits per timestep (gpu_lattices/mod.rs:809-881); the one-launch-
// per-timestep kernels of this library (kernels.cu, step_wide.cu) still sit on the launch-to-launch floor for small lattices:
// a 100 x 100 Izhikevich lattice steps in 4.1 us of which ~1 us is work.  Here the whole chunk of timesteps runs inside ONE
// cooperative launch: every CTA keeps a private copy of the step parameters in shared memory, rewrites the few fields that
// change from step to step (clock, ping-pong buffers, history record) and meets the other CTAs at a grid-wide barrier between
// timesteps — and, in networks whose neurons read the spike trains' previous last_firing_time (lazy STDP), once more between the
// neurons and the spike trains of a step.  The per-neuron step is the shared neuron_step (step_body.cuh) and the spike-train
// step the shared train_step (train_body.cuh): same arithmetic in the same order, bit-identical to the per-launch path.
//
// Coherence: data written in step s is read in step s + 1 by other SMs.  The barrier is release (fence + atomic) on arrival and
// acquire (ld.acquire.gpu, which also drops the SM's stale L1 lines) on departure; nothing that changes during the launch is read
// through the non-coherent path (__ldg).
#include "step_body.cuh"
#include "train_body.cuh"

#include <cstdio>
#include <cstdlib>

namespace snn {

__device__ __forceinline__ unsigned int ld_acquire_gpu_u32(const unsigned int *p) {
    unsigned int v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// grid-wide barrier on a monotonically increasing counter (zeroed by the host before the launch); every CTA of the cooperative
// launch is resident, so spinning is safe
__device__ __forceinline__ void grid_barrier(unsigned int *counter, unsigned int target) {
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(counter, 1u);
        while (ld_acquire_gpu_u32(counter) < target) {}
    }
    __syncthreads();
}

// lattices of up to ~10^4 neurons fit ONE thread-block cluster (16 CTAs of 640 threads): the hardware cluster barrier (release /
// acquire at cluster scope) replaces the atomic + poll round trips through L2 of the grid barrier — 1.3 us -> 0.3 us per timestep
constexpr int kClusterThreads = 640;
constexpr unsigned kClusterCtas = 16;
__device__ __forceinline__ void cluster_barrier() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// A launch that gives every slice its own warp for all of its timesteps can keep what never changes in registers: the eight col /
// weight words of a radius-1 stencil row and the model parameters.  What remains on the critical path of a timestep is ONE L2
// round trip (the neighbour voltages), the arithmetic, and the barrier — every barrier drops the SM's L1, so without this each
// step paid a second round trip for words it had already read a thousand times.  Same values, same arithmetic.
template <int MODEL, bool NTREL>
struct CachedSrc : GlobalSrc {
    static constexpr uint32_t kWidth = 8;   // neuron_step takes the fixed-width gather (compile-time edge indices)
    uint32_t cc[8];
    float cw[8];
    float fc[F_NA_CUR];
    template <int SLOT> __device__ __forceinline__ float f() const { return fc[SLOT]; }
    __device__ __forceinline__ uint32_t col(uint32_t kk) const { return cc[kk]; }
    __device__ __forceinline__ float wgt(uint32_t kk) const { return cw[kk]; }
    __device__ __forceinline__ Handle gh_row(int, uint32_t j) const { return j; }
    __device__ __forceinline__ void wgt_update(uint32_t, float) const {}   // plasticity never takes this source
    __device__ __forceinline__ void wgt_updates_done() const {}
};

template <int MODEL, int CHEMG, bool NTREL, bool STDP, bool NET, bool WIDE, bool CLUSTER>
__global__ void __launch_bounds__(WIDE ? kWideWarps * 32 : (CLUSTER ? kClusterThreads : 256))
step_multi_kernel(const __grid_constant__ StepParams p0, const __grid_constant__ TrainParams t0, const __grid_constant__ MultiParams m) {
    extern __shared__ __align__(16) unsigned char multi_sm[];   // WIDE: 2 x wide_buf_bytes(CHEMG)
    // per-thread copies of the launch parameters: after inlining every access has a constant offset, so the compiler splits the
    // structs into scalars — the step-invariant fields stay operands from the constant bank (as in the one-launch-per-step
    // kernels), the few fields that change per timestep live in registers
    StepParams p = p0;
    TrainParams tp = t0;
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint32_t warps_per_cta = blockDim.x >> 5;
    const uint32_t n_slices = (p0.n_neurons + 31u) >> 5, n_twarps = (t0.n_trains + 31u) >> 5;
    unsigned int arrivals = 0;
    if constexpr (!WIDE && !NET && !STDP) {
        if (p0.uniform_width == 8u && n_slices <= gridDim.x * warps_per_cta && m.cache_rows) {
            // one slice per warp, radius-1 stencil rows, no plasticity: the register-cached source (CachedSrc)
            const uint32_t slice = blockIdx.x * warps_per_cta + warp;
            const bool active = slice < n_slices;
            const uint32_t ln = slice * 32u + lane;
            const bool valid = active && ln < p.n_neurons;
            const uint32_t lnc = valid ? ln : p.n_neurons - 1;
            CachedSrc<MODEL, NTREL> cs{GlobalSrc{p, lnc, p.own0 + lnc, lane, slice * 8u, slice * 8u + 8u, nullptr}, {}, {}, {}};
            if (active) {
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    cs.cc[u] = __ldg(p.col + (size_t)(slice * 8u + u) * 32u + lane);
                    cs.cw[u] = __ldg(p.wgt + (size_t)(slice * 8u + u) * 32u + lane);
                }
#pragma unroll
                for (int sl = 0; sl < F_NA_CUR; ++sl) cs.fc[sl] = win_field_read(MODEL, NTREL, sl) ? __ldg(p.f[sl] + lnc) : 0.f;
            }
            for (uint32_t s = 0; s < m.steps; ++s) {
                const uint32_t in = (m.cur ^ s) & 1u, out = in ^ 1u;
                p.clock = p0.clock + s;
                p.apply_pending = 0u;
                p.v_in = m.v[in]; p.v_out = m.v[out];
                p.spk_in = m.spk[in]; p.spk_out = m.spk[out];
                p.t_in = m.t[in]; p.t_out = m.t[out];
                const uint32_t li = m.lft_pp ? ((m.lft_loc ^ s) & 1u) : m.lft_loc;
                p.lft_in = m.lft[li]; p.lft_out = m.lft[m.lft_pp ? li ^ 1u : li];
                p.grid_hist = m.grid_hist ? m.grid_hist + (size_t)s * m.n_neurons : nullptr;
                p.spike_hist = m.spike_hist ? m.spike_hist + (size_t)s * m.n_words : nullptr;
                p.out_par = out;
                if (CHEMG == 1) cs.t0 = p.t_in + (size_t)(__ffs((int)p.nt_used) - 1) * p.t_stride;
                if (active) neuron_step<MODEL, CHEMG, NTREL, STDP, NET>(p, cs, slice, lane, ln, lnc, valid, false, false);
                if (s + 1u < m.steps) {
                    if constexpr (CLUSTER) cluster_barrier();
                    else { arrivals += gridDim.x; grid_barrier(m.barrier, arrivals); }
                }
            }
            return;
        }
    }
    for (uint32_t s = 0; s < m.steps; ++s) {
        {
            const uint32_t in = (m.cur ^ s) & 1u, out = in ^ 1u;
            p.clock = p0.clock + s;
            p.apply_pending = (STDP && (s > 0u || m.first_pending)) ? 1u : 0u;
            p.v_in = m.v[in]; p.v_out = m.v[out];
            p.spk_in = m.spk[in]; p.spk_out = m.spk[out];
            p.t_in = m.t[in]; p.t_out = m.t[out];
            const uint32_t li = m.lft_pp ? ((m.lft_loc ^ s) & 1u) : m.lft_loc;
            p.lft_in = m.lft[li]; p.lft_out = m.lft[m.lft_pp ? li ^ 1u : li];
            p.grid_hist = m.grid_hist ? m.grid_hist + (size_t)s * m.n_neurons : nullptr;
            p.spike_hist = m.spike_hist ? m.spike_hist + (size_t)s * m.n_words : nullptr;
            p.out_par = out;
            if (t0.n_trains) {
                tp.v_in = p.v_in; tp.v_out = p.v_out; tp.spk_in = p.spk_in; tp.spk_out = p.spk_out;
                tp.t_in = p.t_in; tp.t_out = p.t_out; tp.lft_in = p.lft_in; tp.lft_out = p.lft_out;
                for (int l = 0; l < t0.n_tl; ++l) tp.tl_clock[l] = t0.tl_clock[l] + s;
                tp.draw = t0.draw + s;
                tp.grid_hist = m.tgrid_hist ? m.tgrid_hist + (size_t)s * m.n_trains : nullptr;
                tp.spike_hist = m.tspike_hist ? m.tspike_hist + (size_t)s * m.t_words : nullptr;
            }
        }
        // ---- the neurons of this timestep
        if constexpr (WIDE) {
            // the node state of this timestep into shared memory, once per CTA and step (WideStage, step_body.cuh)
            const WideStage stage = wide_stage_fill<NET>(p, multi_sm + 2u * wide_buf_bytes(CHEMG), m.wide_stage != 0u && blockIdx.x < n_slices);
            for (uint32_t slice = blockIdx.x; slice < n_slices; slice += gridDim.x) {   // uniform per CTA: gather_edges_wide syncs the CTA
                const uint32_t ln = slice * 32u + lane;
                const bool valid = ln < p.n_neurons;
                const uint32_t lnc = valid ? ln : p.n_neurons - 1;
                const uint32_t k0 = p.uniform_width ? slice * p.uniform_width : __ldg(p.slice_off + slice);
                const uint32_t k1 = p.uniform_width ? k0 + p.uniform_width : __ldg(p.slice_off + slice + 1);
                const float *tt0 = nullptr;
                if (CHEMG == 1) tt0 = p.t_in + (size_t)(__ffs((int)p.nt_used) - 1) * p.t_stride;
                const WideSrc src{{p, lnc, p.own0 + lnc, lane, k0, k1, tt0}, warp, (uint32_t)kWideWarps, multi_sm, stage, 0u, 0u, nullptr, 0u, 0u};
                neuron_step<MODEL, CHEMG, NTREL, STDP, NET>(p, src, slice, lane, ln, lnc, valid, false, false);
                __syncthreads();   // the chunk buffers are reused by the CTA's next slice
            }
        } else {
            for (uint32_t slice = blockIdx.x * warps_per_cta + warp; slice < n_slices; slice += gridDim.x * warps_per_cta) {
                const uint32_t ln = slice * 32u + lane;
                const bool valid = ln < p.n_neurons;
                const uint32_t lnc = valid ? ln : p.n_neurons - 1;
                const uint32_t k0 = p.uniform_width ? slice * p.uniform_width : __ldg(p.slice_off + slice);
                const uint32_t k1 = p.uniform_width ? k0 + p.uniform_width : __ldg(p.slice_off + slice + 1);
                const float *tt0 = nullptr;
                if (CHEMG == 1) tt0 = p.t_in + (size_t)(__ffs((int)p.nt_used) - 1) * p.t_stride;
                const GlobalSrc src{p, lnc, p.own0 + lnc, lane, k0, k1, tt0};
                neuron_step<MODEL, CHEMG, NTREL, STDP, NET>(p, src, slice, lane, ln, lnc, valid, false, false);
            }
        }
        // ---- the spike trains of this timestep (they step after the neurons, neuron/mod.rs:2582-2591).  The lazy STDP of the neurons
        // reads the trains' last_firing_time from before this step out of lft_out, which the trains overwrite now: wait for every
        // neuron first
        if (NET && t0.n_trains) {
            if (m.train_sync) {
                if constexpr (CLUSTER) cluster_barrier();
                else { arrivals += gridDim.x; grid_barrier(m.barrier, arrivals); }
            }
            for (uint32_t tw = blockIdx.x * warps_per_cta + warp; tw < n_twarps; tw += gridDim.x * warps_per_cta) train_step(tp, tw, lane);
        }
        if (s + 1u < m.steps) {
            if constexpr (CLUSTER) cluster_barrier();
            else { arrivals += gridDim.x; grid_barrier(m.barrier, arrivals); }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// launcher
// ------------------------------------------------------------------------------------------------
template <class K, bool WIDE>
static cudaError_t launch_multi(const StepParams &p, const TrainParams &t, const MultiParams &m, int device, bool dry, cudaStream_t s) {
    const uint32_t n_slices = (p.n_neurons + 31u) / 32u, n_twarps = (t.n_trains + 31u) / 32u;
    cudaError_t e;
    if constexpr (!WIDE) {
        // small enough for one cluster: every slice (and spike-train warp) gets its own warp in 16 CTAs of 640 threads
        const uint32_t warps = kClusterCtas * (kClusterThreads / 32);
        if (n_slices <= warps && n_twarps <= warps) {
            auto kc = step_multi_kernel<K::MODEL, K::CHEMG, K::NTREL, K::STDP, K::NET, false, true>;
            static thread_local int cluster_ok = -1;   // per instantiation
            if (cluster_ok < 0) {
                cluster_ok = 0;
                if (cudaFuncSetAttribute(kc, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess) {
                    cudaLaunchConfig_t cfg{};
                    cfg.gridDim = dim3(kClusterCtas); cfg.blockDim = dim3(kClusterThreads);
                    cudaLaunchAttribute at{};
                    at.id = cudaLaunchAttributeClusterDimension; at.val.clusterDim.x = kClusterCtas; at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
                    cfg.attrs = &at; cfg.numAttrs = 1;
                    int n_clusters = 0;
                    if (cudaOccupancyMaxActiveClusters(&n_clusters, kc, &cfg) == cudaSuccess && n_clusters >= 1) cluster_ok = 1;
                }
                cudaGetLastError();
            }
            if (cluster_ok == 1) {
                if (dry) return cudaSuccess;
                cudaLaunchConfig_t cfg{};
                cfg.gridDim = dim3(kClusterCtas); cfg.blockDim = dim3(kClusterThreads); cfg.stream = s;
                cudaLaunchAttribute at{};
                at.id = cudaLaunchAttributeClusterDimension; at.val.clusterDim.x = kClusterCtas; at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
                cfg.attrs = &at; cfg.numAttrs = 1;
                return cudaLaunchKernelEx(&cfg, kc, p, t, m);
            }
        }
    }
    auto k = step_multi_kernel<K::MODEL, K::CHEMG, K::NTREL, K::STDP, K::NET, WIDE, false>;
    const int threads = WIDE ? kWideWarps * 32 : 256;
    const size_t smem = WIDE ? 2u * wide_buf_bytes(K::CHEMG) + (m.wide_stage ? wide_stage_bytes(p.n_nodes, K::NET ? p.n_trains : 0u) : 0u) : 0u;
    if (smem > 40u * 1024u) { e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); if (e != cudaSuccess) return e; }
    int per_sm = 0, sms = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, threads, smem);
    if (e != cudaSuccess) return e;
    e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    if (e != cudaSuccess) return e;
    const uint32_t want_n = WIDE ? n_slices : (n_slices + 7u) / 8u, want_t = WIDE ? (n_twarps + kWideWarps - 1u) / kWideWarps : (n_twarps + 7u) / 8u;
    const uint32_t want = want_n > want_t ? want_n : want_t;
    const uint32_t cap = (uint32_t)per_sm * (uint32_t)sms;
    if (cap == 0) return cudaErrorLaunchOutOfResources;
    // more than a few slices per warp and timestep: the launch-per-step kernels fill the machine better
    if (want > 4u * cap) return cudaErrorLaunchOutOfResources;
    if (dry) return cudaSuccess;
    const unsigned grid = want < cap ? (want ? want : 1u) : cap;
    void *args[] = {(void *)&p, (void *)&t, (void *)&m};
    return cudaLaunchCooperativeKernel((const void *)k, dim3(grid), dim3(threads), args, smem, s);
}

cudaError_t launch_step_multi(const StepParams &p, const TrainParams &t, const MultiParams &m, const StepSpec &spec, bool wide, int device,
                              bool dry, cudaStream_t s) {
    return dispatch_step(spec, cudaErrorInvalidValue, [&](auto k) {
        using K = decltype(k);
        return wide ? launch_multi<K, true>(p, t, m, device, dry, s) : launch_multi<K, false>(p, t, m, device, dry, s);
    });
}

}  // namespace snn
