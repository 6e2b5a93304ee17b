// step_tma.cu — the step kernel for stencil lattices: persistent CTAs, TMA-staged operands.
//
// The general step_kernel (kernels.cu) issues ~60 dependent per-thread loads per neuron and is latency-bound
// (ncu: 42 % issue slots, 33 % DRAM, profiles/).  Every operand that is read exactly once per neuron per step —
// own state, the per-neuron parameters, the slice's col/weight rows — is a contiguous byte range per tile of 256
// neurons, so here one producer lane moves them with TMA bulk copies (cp.async.bulk.shared::cluster.global with
// mbarrier complete_tx) into a multi-stage shared-memory ring, a whole tile (or more) ahead of the 8 consumer warps.
// Consumers read their operands from shared memory (conflict-free: one float per lane), do the neighbour gathers
// through L1/L2, and store results straight to HBM.  The arithmetic is the shared neuron_step (step_body.cuh), so
// results are bit-identical to the general kernel.
//
// Grid = resident CTAs (SM count x CTAs/SM), tiles are taken round-robin; 288 threads = 8 consumer warps + 1 producer.
#include "step_body.cuh"
#include "tma_util.cuh"

namespace snn {

struct SmemSrc {
    static constexpr bool kEarlyLoads = false;  // operands sit in shared memory: read them where they are used
    static constexpr bool kCheapEdges = true;
    static constexpr bool kWide = false;
    const StepParams &p;
    const TmaParams &tp;
    const unsigned char *st;  // this stage
    uint32_t tid;             // neuron within the tile
    uint32_t lane, warp;
    uint32_t w;               // uniform slice width
    uint32_t k0g;             // first k-row of this warp's slice in the global edge arrays
    __device__ __forceinline__ float ld(uint32_t off) const { return *reinterpret_cast<const float *>(st + off + tid * 4u); }
    static constexpr uint32_t kWidth = 0;
    const float *t0;          // CHEMG == 1: row of the single neurotransmitter type in t_in
    template <int SLOT> __device__ __forceinline__ float f() const { return ld(tp.o_f[SLOT]); }
    template <int SLOT> __device__ __forceinline__ float state() const { return ld(tp.o_f[SLOT]); }
    __device__ __forceinline__ uint32_t spk_prev_word(uint32_t warp_global) const { return __ldg(p.spk_in + (p.own0 >> 5) + warp_global); }
    typedef uint32_t Handle;
    __device__ __forceinline__ Handle gh(uint32_t j) const { return j; }
    __device__ __forceinline__ float gv(Handle h) const { return p.v_in[h]; }
    __device__ __forceinline__ int glft(Handle h) const { return p.lft_in[h]; }
    __device__ __forceinline__ float gt0(Handle h) const { return t0[h]; }
    __device__ __forceinline__ float gt(Handle h, int ty) const { return p.t_in[(size_t)ty * p.t_stride + h]; }
    __device__ __forceinline__ float v() const { return ld(tp.o_v); }
    __device__ __forceinline__ int lft() const { return *reinterpret_cast<const int *>(st + tp.o_lft + tid * 4u); }
    __device__ __forceinline__ uint32_t flags() const { return st[tp.o_flags + tid]; }
    __device__ __forceinline__ float t_own(int ty) const { return ld(tp.o_t[ty]); }
    __device__ __forceinline__ float nt(int slot, int ty) const { return ld(tp.o_nt[slot][ty]); }
    __device__ __forceinline__ float rc(int slot, int ty) const { return ld(tp.o_rc[slot][ty]); }
    __device__ __forceinline__ float rc_state(int slot, int ty) const { return ld(tp.o_rc[slot][ty]); }
    __device__ __forceinline__ uint32_t width() const { return w; }
    __device__ __forceinline__ uint32_t col(uint32_t kk) const {
        return *reinterpret_cast<const uint32_t *>(st + tp.o_col + ((warp * w + kk) * 32u + lane) * 4u);
    }
    __device__ __forceinline__ float wgt(uint32_t kk) const {
        return *reinterpret_cast<const float *>(st + tp.o_wgt + ((warp * w + kk) * 32u + lane) * 4u);
    }
    __device__ __forceinline__ float *wgt_ptr(uint32_t kk) const { return p.wgt + (size_t)(k0g + kk) * 32u + lane; }
};

// Register budget: three resident CTAs per SM (<= 75 registers) for the light configurations, two for the ones whose
// live state does not fit (Hodgkin-Huxley, general per-edge neurotransmitter masks) — measured: 3 CTAs/SM is worth
// +15 % on the Izhikevich + AMPA + STDP workload, but costs 150 B of spills on HH with three receptor types.
template <int MODEL, int CHEMG>
constexpr int tma_min_ctas() { return (MODEL == SNN_MODEL_HODGKIN_HUXLEY || CHEMG == 3) ? 2 : 3; }

// row strips: the tiles whose slices import ghosts / export boundary rows are stepped first (see win_tile_of, step_win.cu)
__device__ __forceinline__ uint32_t tma_tile_of(const StepParams &p, uint32_t n_tiles, uint32_t seq) {
    if (!(p.halo[0].active | p.halo[1].active)) return seq;
    const uint32_t n_lo = p.halo[0].active ? (p.halo[0].count + kTmaTile - 1u) / kTmaTile : 0u;
    const uint32_t n_hi = p.halo[1].active ? n_tiles - p.halo[1].first / kTmaTile : 0u;
    if (n_lo + n_hi > n_tiles) return seq;
    if (seq < n_lo) return seq;
    if (seq < n_lo + n_hi) return n_tiles - 1u - (seq - n_lo);
    return seq - n_hi;
}

template <int MODEL, int CHEMG, bool NTREL, bool STDP>
__global__ void __launch_bounds__(kTmaThreads, tma_min_ctas<MODEL, CHEMG>()) step_tma_kernel(const __grid_constant__ StepParams p, const __grid_constant__ TmaParams tp) {
    extern __shared__ __align__(128) unsigned char smem[];
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + (size_t)tp.stages * tp.stage_bytes);
    uint64_t *empty = full + tp.stages;
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    pdl_wait();   // launch_pdl
    if (halo_failed(p)) return;
    if (threadIdx.x == 0) {
        for (uint32_t s = 0; s < tp.stages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], kTmaConsumerWarps);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (warp == kTmaConsumerWarps) {
        // ---- producer: one lane streams whole tiles ahead of the consumers ---------------------------
        if (lane == 0) {
            uint32_t s = 0, ph = 0;
            for (uint32_t seq = blockIdx.x; seq < tp.n_tiles; seq += gridDim.x) {
                const uint32_t tile = tma_tile_of(p, tp.n_tiles, seq);
                mbar_wait_backoff(&empty[s], ph ^ 1u);
                mbar_arrive_expect_tx(&full[s], tp.tx_bytes);
                unsigned char *dst = smem + (size_t)s * tp.stage_bytes;
                for (uint32_t k = 0; k < tp.n_streams; ++k)
                    tma_bulk_g2s(dst + tp.st[k].smem_off, tp.st[k].src + (size_t)tile * tp.st[k].bytes_per_tile,
                                 tp.st[k].bytes_per_tile, &full[s]);
                if (++s == tp.stages) { s = 0; ph ^= 1u; }
            }
        }
        return;
    }
    // ---- consumers: 8 warps x 32 neurons per tile --------------------------------------------------
    uint32_t s = 0, ph = 0;
    for (uint32_t seq = blockIdx.x; seq < tp.n_tiles; seq += gridDim.x) {
        const uint32_t tile = tma_tile_of(p, tp.n_tiles, seq);
        const uint32_t warp_global = tile * kTmaConsumerWarps + warp;
        const uint32_t ln = warp_global * 32u + lane;
        const bool active = warp_global * 32u < p.n_neurons;
        const bool valid = ln < p.n_neurons;
        const uint32_t lnc = valid ? ln : p.n_neurons - 1;
        bool export_lo = false, export_hi = false;
        if (active) halo_import(p, warp_global, lane, ln, valid, export_lo, export_hi);
        mbar_wait(&full[s], ph);
        if (active) {
            const float *t0 = nullptr;
            if (CHEMG == 1) t0 = p.t_in + (size_t)(__ffs((int)p.nt_used) - 1) * p.t_stride;
            const SmemSrc src{p, tp, smem + (size_t)s * tp.stage_bytes, threadIdx.x, lane, warp, p.uniform_width,
                              warp_global * p.uniform_width, t0};
            neuron_step<MODEL, CHEMG, NTREL, STDP, false>(p, src, warp_global, lane, ln, lnc, valid, export_lo, export_hi);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[s]);
        if (active) halo_publish(p, warp_global, lane);
        if (++s == tp.stages) { s = 0; ph ^= 1u; }
    }
}

// ------------------------------------------------------------------------------------------------
// launcher
// ------------------------------------------------------------------------------------------------
cudaError_t launch_step_tma(const StepParams &p, const TmaParams &tp, const StepSpec &spec, unsigned grid, cudaStream_t s) {
    if (p.n_neurons == 0) return cudaSuccess;
    const size_t smem = (size_t)tp.stages * tp.stage_bytes + 2 * tp.stages * sizeof(uint64_t);
    return dispatch_step(spec, cudaErrorInvalidValue, [&](auto k) {
        using K = decltype(k);
        if constexpr (K::NET) {
            return cudaErrorInvalidValue;   // single lattices only
        } else {
            auto kern = step_tma_kernel<K::MODEL, K::CHEMG, K::NTREL, K::STDP>;
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
            return launch_pdl(pdl_ok(p), kern, dim3(grid), dim3(kTmaThreads), smem, s, p, tp);
        }
    });
}

}  // namespace snn
