// kernels.cu — hand-written sm_100a kernels of the lattice stepping path.
//
// One fused kernel per timestep replaces the reference's per-step sequence
//   get_internal_electrical_inputs / get_internal_neurotransmitter_inputs   (neuron/mod.rs:757-826)
//   iterate / iterate_with_neurotransmission / iterate_chemical_synapses_only (neuron/mod.rs:884-982)
//   update_weights_from_neurons (STDP)                                      (neuron/mod.rs:849-881)
// and the OpenCL twin's four launches per step (gpu_lattices/mod.rs:809-881).
//
// Compiled with -fmad=false: Rust never contracts a*b+c, and the deterministic models
// (Izhikevich, LIF, QIF, ...) must reproduce the oracle's spike raster bit for bit.  Every
// expression below is written in the reference's evaluation order (SURVEY.md appendix B).
//
// Layout: structure-of-arrays in HBM, one thread per postsynaptic neuron, one warp per 32-row
// slice of the sliced-ELL in-edge table so that every per-edge load (col, weight) is one coalesced
// 128-byte line per warp; neighbour V / t / last_firing_time are gathered through L1/L2.
// The path is HBM-bound elementwise + sparse gather: no tensor cores.
#include "step_body.cuh"
#include "train_body.cuh"

#include <cfloat>
#include <cstdlib>

namespace snn {


// ------------------------------------------------------------------------------------------------
// the fused step kernel, general form: every operand straight from HBM (any graph, networks, spike trains)
// ------------------------------------------------------------------------------------------------
template <int MODEL, int CHEMG, bool NTREL, bool STDP, bool NET>
__device__ __forceinline__ void step_kernel_body(const StepParams &p) {
    pdl_wait();   // launch_pdl
    if (!NET && halo_failed(p)) return;
    uint32_t block = blockIdx.x;
    if (!NET && (p.halo[0].active | p.halo[1].active)) {
        // row strips: the CTAs whose slices import ghosts / export boundary rows run first (see win_tile_of, step_win.cu)
        const uint32_t n_lo = p.halo[0].active ? (p.halo[0].count + 255u) >> 8 : 0u;
        const uint32_t n_hi = p.halo[1].active ? gridDim.x - (p.halo[1].first >> 8) : 0u;
        if (n_lo + n_hi <= gridDim.x) {
            if (block >= n_lo + n_hi) block -= n_hi;
            else if (block >= n_lo) block = gridDim.x - 1u - (block - n_lo);
        }
    }
    const uint32_t warp_global = (block * blockDim.x + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31u;
    if (warp_global * 32u >= p.n_neurons) return;
    const uint32_t ln = warp_global * 32u + lane;  // local neuron number
    const bool valid = ln < p.n_neurons;
    const uint32_t lnc = valid ? ln : p.n_neurons - 1;  // clamped for loads
    bool export_lo = false, export_hi = false;
    if (!NET) halo_import(p, warp_global, lane, ln, valid, export_lo, export_hi);
    if (!NET) gpart_wait(p, warp_global, lane);
    // uniform slice width (stencil graphs): no dependent load for the slice bounds
    const uint32_t k0 = p.uniform_width ? warp_global * p.uniform_width : __ldg(p.slice_off + warp_global);
    const uint32_t k1 = p.uniform_width ? k0 + p.uniform_width : __ldg(p.slice_off + warp_global + 1);
    const float *t0 = nullptr;
    if (CHEMG == 1) t0 = p.t_in + (size_t)(__ffs((int)p.nt_used) - 1) * p.t_stride;
    const GlobalSrc src{p, lnc, p.own0 + lnc, lane, k0, k1, t0};
    neuron_step<MODEL, CHEMG, NTREL, STDP, NET>(p, src, warp_global, lane, ln, lnc, valid, export_lo, export_hi);
    if (!NET) halo_publish(p, warp_global, lane);
    if (!NET) gpart_export_publish<MODEL == SNN_MODEL_BCM_IZHIKEVICH>(p, warp_global, lane, ln, valid);
}

// (single lattices keep the compiler's choice of 64 registers: bounded to five / six resident CTAs the general-graph lattices of
// tools/bench_general_graph.py got 10 % / 25 % slower — spills on the gather path)
template <int MODEL, int CHEMG, bool NTREL, bool STDP, bool NET>
__global__ void __launch_bounds__(256) step_kernel(const __grid_constant__ StepParams p) {
    step_kernel_body<MODEL, CHEMG, NTREL, STDP, NET>(p);
}
// Networks without chemistry (rows of tens of in-edges from several lattices and spike trains): the kernel is latency-bound at the
// four CTAs per SM that 64 registers allow (ncu, profiles/r2_step_kernel_net_full.txt: 47 % occupancy, 54 % long-scoreboard); five
// resident CTAs (51 registers) measured 97 -> 89 us per step on the 1.1 M-neuron / 25 M-edge network of
// tools/bench_reward_network.py, six were slower again (101 us).
template <int MODEL, int CHEMG, bool NTREL, bool STDP>
__global__ void __launch_bounds__(256, 5) step_net5_kernel(const __grid_constant__ StepParams p) {
    step_kernel_body<MODEL, CHEMG, NTREL, STDP, true>(p);
}

// ------------------------------------------------------------------------------------------------
// multi-GPU: push the current boundary state into the neighbours' ghost slots (start of every run)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) halo_push_kernel(const __grid_constant__ StepParams p) {
    // here *_in are the CURRENT state buffers and out_par their parity
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
#pragma unroll
    for (int d = 0; d < 2; ++d) {
        const HaloDir &H = p.halo[d];
        if (!H.active) continue;
        if (t < H.count) {
            const uint32_t i = p.own0 + H.first + t, dst = H.peer_node0 + t;
            H.peer_v[p.out_par][dst] = p.v_in[i];
            H.peer_lft[p.out_par][dst] = p.lft_in[i];
            for (int ty = 0; ty < kNT; ++ty)
                if (p.nt_used & (1u << ty))
                    H.peer_t[p.out_par][(size_t)ty * H.peer_t_stride + dst] = p.t_in[(size_t)ty * p.t_stride + i];
        }
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int done = atomicAdd(&p.halo_done[0], 1u) + 1u;
        if (done == gridDim.x) {
            p.halo_done[0] = 0u;
            __threadfence_system();
            for (int d = 0; d < 2; ++d)
                if (p.halo[d].active) {
                    st_release_sys(p.halo[d].peer_flag, p.halo_epoch + 1ull);
                    st_release_sys(p.halo[d].peer_flag2, p.halo_epoch + 1ull);   // nothing of an earlier run is still being read
                }
        }
    }
}

// general-graph partition: the same push through the per-neuron export lists (here *_in are the CURRENT buffers, out_par their parity)
__global__ void __launch_bounds__(256) gpart_push_kernel(const __grid_constant__ StepParams p) {
    const uint32_t ln = blockIdx.x * blockDim.x + threadIdx.x;
    if (ln < p.n_neurons) {
        const uint32_t i = p.own0 + ln;
        for (uint32_t e = p.gexp_off[ln]; e < p.gexp_off[ln + 1]; ++e) {
            const uint32_t ent = p.gexp_ent[e], dst = ent & kColIdxMask;
            const GPeer &G = p.gpeers[ent >> 28];
            G.v[p.out_par][dst] = p.v_in[i];
            G.lft[p.out_par][dst] = p.lft_in[i];
            for (int ty = 0; ty < kNT; ++ty)
                if (p.nt_used & (1u << ty)) G.t[p.out_par][(size_t)ty * G.t_stride + dst] = p.t_in[(size_t)ty * p.t_stride + i];
        }
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int done = atomicAdd(&p.halo_done[6], 1u) + 1u;
        if (done == gridDim.x) {
            p.halo_done[6] = 0u;
            __threadfence_system();
            for (uint32_t q = 0; q < p.n_gpeers; ++q) st_release_sys(p.gpeers[q].peer_flag, p.halo_epoch + 1ull);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// end-of-run flush of the lazily applied STDP (the last step's updates are still pending)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) flush_stdp_kernel(const __grid_constant__ StepParams p) {
    if (halo_failed(p)) return;
    const uint32_t warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31u;
    if (warp_global * 32u >= p.n_neurons) return;
    const uint32_t ln = warp_global * 32u + lane;
    // partitioned handles: the neighbours' last step must have landed in the ghost slots before they are read
    if (p.n_gpeers) {
        if (lane == 0)
            for (uint32_t q = 0; q < p.n_gpeers; ++q) halo_wait(p.gpeers[q].my_flag, p.halo_epoch, p.halo_done + 2, p.halo_timeout_ns);
        __syncwarp();
    }
    if (p.halo[0].active | p.halo[1].active) {
        if (lane == 0) {
            if (p.halo[0].active) halo_wait(p.halo[0].my_flag, p.halo_epoch, p.halo_done + 2, p.halo_timeout_ns);
            if (p.halo[1].active) halo_wait(p.halo[1].my_flag, p.halo_epoch, p.halo_done + 2, p.halo_timeout_ns);
        }
        __syncwarp();
    }
    if (ln >= p.n_neurons) return;
    const uint32_t i = p.own0 + ln;
    const int lft_me = p.lft_in[i];
    const int li = lat_index(p, ln);
    const bool post_trig = p.lat[li].do_plasticity && lft_me == (int)p.clock - 1;
    const uint32_t k0 = p.slice_off[warp_global], k1 = p.slice_off[warp_global + 1];
    for (uint32_t k = k0; k < k1; ++k) {
        const size_t e = (size_t)k * 32u + lane;
        const uint32_t c = __ldg(p.col + e);
        if (c == kColPad) continue;
        const uint32_t j = c & kColIdxMask;
        // spike trains: last_firing_time from before their last iterate (see gather_edges); lft_out is that buffer here
        const int lft_pre = (c & kColTrainBit) ? p.lft_out[j] : p.lft_in[j];
        bool pre_trig = !(c & kColTrainBit) && lft_pre == (int)p.clock - 1;
        if (pre_trig) pre_trig = p.lat[p.n_lat > 1 ? lat_index(p, j - p.own0) : 0].do_plasticity != 0;
        if (post_trig | pre_trig) {
            float w = p.wgt[e];
            const float d = stdp_delta(p.lat[li], lft_pre, lft_me);
            w = w + d;
            if (post_trig & pre_trig) w = w + d;
            p.wgt[e] = w;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// BCM plasticity (plasticity/mod.rs:99-111) for lattices of BCM Izhikevich neurons
// ------------------------------------------------------------------------------------------------
// Lattice::update_weights_from_neurons (neuron/mod.rs:849-881) with Plasticity = BCM: every in-edge and every out-edge of a neuron
// that spiked is updated with the same function of (weight, presynaptic activity, postsynaptic activity / average), so an edge
// whose two ends both spiked is simply updated twice.  Runs after the step kernel (deferred, canonicalisation (3)): the raster
// word of the step tells who spiked, the activities are the ones the step just wrote.
//
// PART: row strips and general-graph partitions.  The rank that owns an edge's postsynaptic row applies both of its updates, so an
// out-edge of a neuron on another rank is updated here as an in-edge whose presynaptic node is a ghost.  A ghost has no raster bit
// in this rank's spk_out; it spiked in this step iff its last_firing_time (ping-ponged on every partitioned handle, exported each
// step into the ghost slot of parity out_par) equals the step's clock.  Its current_activity comes from the node-indexed ghost
// buffer tf[TFB_ACT_GHOST], exported next to it.  A warp whose slice reads ghosts first waits until every neighbour / peer has published
// this step (p.halo_epoch).  No second handshake is needed: the neighbour overwrites this parity of the ghost slots in its step
// s + 2, whose boundary warps first wait for this rank's step s + 1, and that kernel starts only after this one has finished
// (same stream, plain launches on partitioned handles).
template <bool PART>
__device__ __forceinline__ void bcm_edge_body(const StepParams &p, const BcmParams &b) {
    pdl_wait();   // launch_pdl
    if (PART && halo_failed(p)) return;
    const uint32_t warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t ln = warp_global * 32u + lane;
    if (warp_global * 32u >= p.n_neurons) return;
    if constexpr (PART) {
        // slices that read ghosts: the first / last halo rows of a strip (the predicates of halo_import), bit 0 of gslice on a
        // general-graph partition; interior slices start at once
        const uint32_t w0 = warp_global * 32u, w1 = min(w0 + 32u, p.n_neurons);
        const bool near_lo = p.halo[0].active && w0 < p.halo[0].first + p.halo[0].count;
        const bool near_hi = p.halo[1].active && w1 > p.halo[1].first;
        const bool gwait = p.n_gpeers && (p.gslice[warp_global] & 1u);
        if (near_lo | near_hi | gwait) {
            if (lane == 0) {
                if (near_lo) halo_wait(p.halo[0].my_flag, p.halo_epoch, p.halo_done + 2, p.halo_timeout_ns);
                if (near_hi) halo_wait(p.halo[1].my_flag, p.halo_epoch, p.halo_done + 2, p.halo_timeout_ns);
                if (gwait)
                    for (uint32_t q = 0; q < p.n_gpeers; ++q)
                        if (!halo_wait(p.gpeers[q].my_flag, p.halo_epoch, p.halo_done + 2, p.halo_timeout_ns)) break;
            }
            __syncwarp();
        }
    }
    const uint32_t k0 = p.uniform_width ? warp_global * p.uniform_width : __ldg(p.slice_off + warp_global);
    const uint32_t k1 = p.uniform_width ? k0 + p.uniform_width : __ldg(p.slice_off + warp_global + 1);
    const uint32_t word0 = p.own0 >> 5;
    const bool valid = ln < p.n_neurons;
    const bool post_spk = valid && ((p.spk_out[word0 + warp_global] >> lane) & 1u);
    for (uint32_t k = k0; k < k1; ++k) {
        const uint32_t e = k * 32u + lane;
        const uint32_t c = valid ? __ldg(p.col + e) : kColPad;
        if (c == kColPad) continue;
        const uint32_t j = c & kColIdxMask;
        bool ghost = false, pre_spk;
        if constexpr (PART) {
            ghost = j - p.own0 >= p.n_neurons;   // below or above this rank's own nodes
            pre_spk = ghost ? p.lft_out[j] == (int)p.clock : ((p.spk_out[j >> 5] >> (j & 31u)) & 1u);
        } else {
            pre_spk = (p.spk_out[j >> 5] >> (j & 31u)) & 1u;
        }
        const int n_upd = (post_spk ? 1 : 0) + (pre_spk ? 1 : 0);
        if (n_upd == 0) continue;
        const uint32_t jl = j - p.own0;
        const float act_post = p.f[F_CUR_ACT][ln], avg_post = p.f[F_AVG_ACT][ln], act_pre = ghost ? p.tf[TFB_ACT_GHOST][j] : p.f[F_CUR_ACT][jl];
        const float sliding_threshold = avg_post / b.average_scalar;
        const float activity_term = act_post * (act_post - sliding_threshold);
        float w = p.wgt[e];
        for (int r = 0; r < n_upd; ++r) {
            const float weight_decay = b.decay * w;
            w = w + (activity_term * act_pre - weight_decay) * b.dt;
        }
        p.wgt[e] = w;
    }
}

__global__ void __launch_bounds__(256) bcm_edge_kernel(const __grid_constant__ StepParams p, const __grid_constant__ BcmParams b) {
    bcm_edge_body<false>(p, b);
}
__global__ void __launch_bounds__(256) bcm_part_edge_kernel(const __grid_constant__ StepParams p, const __grid_constant__ BcmParams b) {
    bcm_edge_body<true>(p, b);
}

// ------------------------------------------------------------------------------------------------
// RewardModulatedLattice: RewardModulatedSTDP::update_weight on every edge (plasticity/mod.rs:197-233)
// ------------------------------------------------------------------------------------------------
// The reference calls the modulator inside the node loop (RewardModulatedLattice::iterate, neuron/mod.rs:3127-3156): when node
// p has been stepped, every in-edge and every out-edge of p is updated, so each edge a -> b is updated twice per timestep —
// first when the lower-indexed end is visited (that end already carries this step's last_firing_time, the other end still
// the previous one), then when the other end is visited (both new).  Per edge this is a closed recurrence over
// {counter, dw, weight, c} driven by four integers, so one thread per (row, k) applies both calls from the ping-ponged
// last_firing_time buffers: no atomics, no ordering between edges.  An edge whose trace is at rest (dw = c = 0, counter = 0)
// and whose ends produce no STDP term is an exact no-op and is not written back.
// the STDP term of RewardModulatedSTDP::update_weight (plasticity/mod.rs:200-214): same expression as stdp_delta
__device__ __forceinline__ float rstdp_delta(const RstdpParams &r, int t_pre_i, int t_post_i) {
    const float t_pre = (float)t_pre_i, t_post = (float)t_post_i;
    if (t_pre < t_post) return r.a_plus * expf((-1.f * fabsf((t_pre - t_post) * r.dt)) / r.tau_plus);
    return (-1.f * r.a_minus) * expf((-1.f * fabsf((t_post - t_pre) * r.dt)) / r.tau_minus);   // callers exclude None and t_pre == t_post
}

// the same term through the difference table (see RstdpParams::tab); spike times below 2^24 are exact in f32, so the term is a
// function of the integer difference alone
__device__ __forceinline__ float rstdp_delta_tab(const RstdpParams &r, int t_pre_i, int t_post_i) {
    const int d = t_post_i - t_pre_i;
    const uint32_t k = min((uint32_t)abs(d), r.tab_n - 1u);
    return __ldg(r.tab + (d > 0 ? 0u : r.tab_n) + k);
}

__global__ void rstdp_table_kernel(const __grid_constant__ RstdpParams r, float *tab, uint32_t tab_n) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= tab_n) return;
    // spike times 0 and k: exactly representable, the difference is what matters
    tab[k] = k ? rstdp_delta(r, 0, (int)k) : 0.f;
    tab[tab_n + k] = k ? rstdp_delta(r, (int)k, 0) : 0.f;
}

cudaError_t launch_rstdp_table(const RstdpParams &r, float *tab, uint32_t tab_n, cudaStream_t s) {
    rstdp_table_kernel<<<(tab_n + 255u) / 256u, 256, 0, s>>>(r, tab, tab_n);
    return cudaGetLastError();
}

__device__ __forceinline__ void rstdp_call(const RstdpParams &r, float delta_w, float decay_c, uint32_t &counter, float &dw, float &c, float &w) {
    dw = dw + delta_w;
    if (counter == 0u) {
        counter = 1u;
    } else {
        c = c * decay_c + r.tau_c * dw;   // TraceRSTDP::update_trace, plasticity/mod.rs:140-142
        counter = 0u;
        dw = 0.f;
    }
    w = w + c * r.dopamine;
}

// One CTA per kRsSlices 32-row slices; its 8 warps stride over the k-rows of each slice (a radius-1 stencil: one k-row per
// warp and slice) and every thread works on one edge of each of the kRsSlices slices at a time: all col / trace loads first,
// then the last_firing_time gathers they address, then the arithmetic — kRsSlices independent chains per thread, ~1000
// resident threads per SM, so that two dependent memory round trips per edge still keep HBM busy.
#ifndef SNN_RS_SLICES
#define SNN_RS_SLICES 4
#endif
#ifndef SNN_RS_CTAS
#define SNN_RS_CTAS 3   // resident CTAs per SM of the persistent variant (register budget 65536 / (256 * CTAS))
#endif
constexpr int kRsSlices = SNN_RS_SLICES;

// CANON: every edge enters the timestep with counter == 0 and dw == 0.  That is the state TraceRSTDP::default starts in and
// the state two calls per timestep always return to, so until a caller stores other values through
// snn_lattice_set_connection_traces the counter / dw arrays hold zeros and need neither be read nor written:
// dw = 0 + d1, then (0 + d1) + d2 — the same additions in the same order.
template <bool CANON, bool TAB>
__global__ void __launch_bounds__(256, 4) rstdp_edge_kernel(const __grid_constant__ StepParams p, const __grid_constant__ RstdpParams r) {
    pdl_wait();   // launch_pdl
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint32_t n_slices = (p.n_neurons + 31u) >> 5;
    const bool part = (p.halo[0].active | p.halo[1].active) != 0;
    if (halo_failed(p)) return;
    if (part) {
        // row strips: the neighbours' last_firing_time of THIS step must have landed in the ghost slots (p.halo_epoch is the value
        // their step kernels publish); my_flag is the step-arrival counter here
        if (threadIdx.x == 0) {
            if (p.halo[0].active) halo_wait(p.halo[0].my_flag, p.halo_epoch, p.halo_done + 2, p.halo_timeout_ns);
            if (p.halo[1].active) halo_wait(p.halo[1].my_flag, p.halo_epoch, p.halo_done + 2, p.halo_timeout_ns);
        }
        __syncthreads();
    }
    uint32_t k0[kRsSlices], k1[kRsSlices], node[kRsSlices];
    int old_post[kRsSlices], new_post[kRsSlices];
    uint32_t rounds = 0;
#pragma unroll
    for (int u = 0; u < kRsSlices; ++u) {
        const uint32_t slice = blockIdx.x * kRsSlices + u;
        const uint32_t ln = slice * 32u + lane;
        const bool ok = slice < n_slices && ln < p.n_neurons;
        node[u] = p.own0 + (ok ? ln : 0u);
        k0[u] = k1[u] = 0u;
        if (ok) {
            k0[u] = p.uniform_width ? slice * p.uniform_width : __ldg(p.slice_off + slice);
            k1[u] = p.uniform_width ? k0[u] + p.uniform_width : __ldg(p.slice_off + slice + 1);
        }
        old_post[u] = p.lft_in[node[u]]; new_post[u] = p.lft_out[node[u]];
        rounds = max(rounds, (k1[u] - k0[u] + 7u) >> 3);
    }
    rounds = __reduce_max_sync(0xffffffffu, rounds);   // lanes of a warp share the slices; keep the loop warp-uniform
    const float decay_c = expf(-r.dt / r.tau_c);
    for (uint32_t t = 0; t < rounds; ++t) {
        uint32_t e[kRsSlices];   // element index in the sliced-ELL arrays (< 2^32, finalize_graph)
        uint32_t cw[kRsSlices], cnt[kRsSlices];
        float dw[kRsSlices], cc[kRsSlices], w[kRsSlices];
        int old_pre[kRsSlices], new_pre[kRsSlices];
#pragma unroll
        for (int u = 0; u < kRsSlices; ++u) {
            const uint32_t k = k0[u] + warp + 8u * t;
            e[u] = k * 32u + lane;
            cw[u] = k < k1[u] ? __ldg(p.col + e[u]) : kColPad;
        }
#pragma unroll
        for (int u = 0; u < kRsSlices; ++u) {
            cnt[u] = 0u; dw[u] = 0.f;
            if (cw[u] != kColPad) {
                if (!CANON) { cnt[u] = r.counter[e[u]]; dw[u] = r.dw[e[u]]; }
                cc[u] = r.c[e[u]]; w[u] = p.wgt[e[u]];
                const uint32_t j = cw[u] & kColIdxMask;
                old_pre[u] = p.lft_in[j]; new_pre[u] = p.lft_out[j];
            }
        }
#pragma unroll
        for (int u = 0; u < kRsSlices; ++u) {
            if (cw[u] == kColPad) continue;
            const uint32_t j = cw[u] & kColIdxMask, i = node[u];
            // first call: the end with the lower node index has been stepped, the other has not (a self-loop sees both new)
            const int t_pre1 = (j <= i) ? new_pre[u] : old_pre[u];
            const int t_post1 = (i <= j) ? new_post[u] : old_post[u];
            const bool first_live = (t_pre1 >= 0 && t_post1 >= 0 && t_pre1 != t_post1);
            const bool second_live = (new_pre[u] >= 0 && new_post[u] >= 0 && new_pre[u] != new_post[u]);
            if (!first_live && !second_live && dw[u] == 0.f && cc[u] == 0.f && cnt[u] == 0u) continue;
            const float d2 = second_live ? (TAB ? rstdp_delta_tab(r, new_pre[u], new_post[u]) : rstdp_delta(r, new_pre[u], new_post[u])) : 0.f;
            // the two calls see the same pair of spike times unless an end of the edge spiked in this very step
            const float d1 = (t_pre1 == new_pre[u] && t_post1 == new_post[u]) ? d2
                             : (first_live ? (TAB ? rstdp_delta_tab(r, t_pre1, t_post1) : rstdp_delta(r, t_pre1, t_post1)) : 0.f);
            rstdp_call(r, d1, decay_c, cnt[u], dw[u], cc[u], w[u]);
            rstdp_call(r, d2, decay_c, cnt[u], dw[u], cc[u], w[u]);
            if (!CANON) { r.counter[e[u]] = (uint8_t)cnt[u]; r.dw[e[u]] = dw[u]; }
            r.c[e[u]] = cc[u]; p.wgt[e[u]] = w[u];
        }
    }
    if (part) {
        // the last CTA tells both neighbours that this rank no longer reads the ghost values of the previous step: their next
        // step kernel may overwrite them
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();
            const unsigned int done = atomicAdd(&p.halo_done[3], 1u) + 1u;
            if (done == gridDim.x) {
                p.halo_done[3] = 0u;
                __threadfence_system();
                for (int d = 0; d < 2; ++d)
                    if (p.halo[d].active) st_release_sys(p.halo[d].peer_flag2, p.halo_epoch);
            }
        }
    }
}

// The same update for radius-1 stencil tables (uniform slice width 8) of whole lattices, as a persistent, software-pipelined
// kernel.  The short-lived CTAs above spend 53 % of their samples on the long scoreboard (profiles/r2_rstdp_edge_full.txt): four
// edges per thread behind TWO dependent memory levels (col -> last_firing_time gathers) and ~35 instructions of per-thread set-up
// amortised over those four edges.  Here a CTA walks many groups of kRsSlices slices; while the gathers of group g are in flight
// the independent loads (col, c, weight, the rows' own spike times) of group g + 1 are already issued, so one of the two round
// trips is hidden, and the set-up is paid once.  Warp w of the CTA owns k-row w of every slice (8 warps = 8 k-rows).
template <bool CANON, bool TAB>
__global__ void __launch_bounds__(256, SNN_RS_CTAS) rstdp_edge8_kernel(const __grid_constant__ StepParams p, const __grid_constant__ RstdpParams r) {
    pdl_wait();   // launch_pdl
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint32_t n_slices = (p.n_neurons + 31u) >> 5;
    const uint32_t n_groups = (n_slices + kRsSlices - 1u) / kRsSlices;
    const float decay_c = expf(-r.dt / r.tau_c);
    struct L1 { uint32_t e, cw, cnt; float cc, w, dw; int old_post, new_post; uint32_t node; };
    auto load1 = [&](uint32_t g, L1 (&x)[kRsSlices]) {
#pragma unroll
        for (int u = 0; u < kRsSlices; ++u) {
            const uint32_t slice = g * kRsSlices + u, ln = slice * 32u + lane;
            const bool ok = slice < n_slices && ln < p.n_neurons;
            x[u].node = p.own0 + (ok ? ln : 0u);
            x[u].e = (slice * 8u + warp) * 32u + lane;
            x[u].cw = ok ? __ldg(p.col + x[u].e) : kColPad;
            x[u].cnt = 0u; x[u].dw = 0.f; x[u].cc = 0.f; x[u].w = 0.f;
            if (ok) {
                if (!CANON) { x[u].cnt = r.counter[x[u].e]; x[u].dw = r.dw[x[u].e]; }
                x[u].cc = r.c[x[u].e]; x[u].w = p.wgt[x[u].e];
            }
            x[u].old_post = p.lft_in[x[u].node]; x[u].new_post = p.lft_out[x[u].node];
        }
    };
    L1 cur[kRsSlices], nxt[kRsSlices];
    uint32_t g = blockIdx.x;
    if (g < n_groups) load1(g, cur);
    for (; g < n_groups; g += gridDim.x) {
        // level 2 of this group (needs its col words) ...
        int old_pre[kRsSlices], new_pre[kRsSlices];
#pragma unroll
        for (int u = 0; u < kRsSlices; ++u) {
            const uint32_t j = cur[u].cw == kColPad ? cur[u].node : (cur[u].cw & kColIdxMask);
            old_pre[u] = p.lft_in[j]; new_pre[u] = p.lft_out[j];
        }
        // ... and level 1 of the next one, in flight together
        const uint32_t gn = g + gridDim.x;
        if (gn < n_groups) load1(gn, nxt);
#pragma unroll
        for (int u = 0; u < kRsSlices; ++u) {
            if (cur[u].cw == kColPad) continue;
            const uint32_t j = cur[u].cw & kColIdxMask, i = cur[u].node;
            const int t_pre1 = (j <= i) ? new_pre[u] : old_pre[u];
            const int t_post1 = (i <= j) ? cur[u].new_post : cur[u].old_post;
            const bool first_live = (t_pre1 >= 0 && t_post1 >= 0 && t_pre1 != t_post1);
            const bool second_live = (new_pre[u] >= 0 && cur[u].new_post >= 0 && new_pre[u] != cur[u].new_post);
            if (!first_live && !second_live && cur[u].dw == 0.f && cur[u].cc == 0.f && cur[u].cnt == 0u) continue;
            const float d2 = second_live ? (TAB ? rstdp_delta_tab(r, new_pre[u], cur[u].new_post) : rstdp_delta(r, new_pre[u], cur[u].new_post)) : 0.f;
            const float d1 = (t_pre1 == new_pre[u] && t_post1 == cur[u].new_post) ? d2
                             : (first_live ? (TAB ? rstdp_delta_tab(r, t_pre1, t_post1) : rstdp_delta(r, t_pre1, t_post1)) : 0.f);
            uint32_t cnt = cur[u].cnt; float dw = cur[u].dw, cc = cur[u].cc, w = cur[u].w;
            rstdp_call(r, d1, decay_c, cnt, dw, cc, w);
            rstdp_call(r, d2, decay_c, cnt, dw, cc, w);
            if (!CANON) { r.counter[cur[u].e] = (uint8_t)cnt; r.dw[cur[u].e] = dw; }
            r.c[cur[u].e] = cc; p.wgt[cur[u].e] = w;
        }
#pragma unroll
        for (int u = 0; u < kRsSlices; ++u) cur[u] = nxt[u];
    }
}

// ------------------------------------------------------------------------------------------------
// derived fields (currents, gate rates): recomputed once after a run from the retained pre-update V
// ------------------------------------------------------------------------------------------------
template <int MODEL>
__global__ void __launch_bounds__(256) finalize_kernel(const __grid_constant__ StepParams p, const float *v_prev) {
    const uint32_t ln = blockIdx.x * blockDim.x + threadIdx.x;
    if (ln >= p.n_neurons) return;
    const uint32_t i = p.own0 + ln;
    const float v = v_prev[i];
    if (p.chemical) {
        const uint32_t rcm = p.node_flags[i] >> 4;
        for (int ty = 0; ty < kNT; ++ty) {
            if (!(rcm & (1u << ty))) continue;
            const size_t o = (size_t)ty * p.rc_stride + ln;
            const float mg = (ty == SNN_NT_NMDA) ? p.rc[RCF_MG][o] : 0.f;
            p.rc[RCF_CUR][o] = receptor_current(ty, p.rc[RCF_G][o], p.rc[RCF_E][o], mg, p.rc[RCF_R][o], v);
        }
    }
    if constexpr (MODEL == SNN_MODEL_HODGKIN_HUXLEY) {
        const float m = p.f[F_M][ln], h = p.f[F_H][ln], n = p.f[F_N][ln];
        p.f[F_M_ALPHA][ln] = 0.1f * ((v + 40.f) / (1.f - expf(-(v + 40.f) / 10.f)));
        p.f[F_M_BETA][ln] = 4.f * expf(-(v + 65.f) / 18.f);
        p.f[F_H_ALPHA][ln] = 0.07f * expf(-(v + 65.f) / 20.f);
        p.f[F_H_BETA][ln] = 1.f / (expf(-(v + 35.f) / 10.f) + 1.f);
        p.f[F_NA_CUR][ln] = ((pow3f(m) * h) * p.f[F_GNA][ln]) * (v - p.f[F_ENA][ln]);
        p.f[F_N_ALPHA][ln] = (0.01f * (v + 55.f)) / (1.f - expf(-(v + 55.f) / 10.f));
        p.f[F_N_BETA][ln] = 0.125f * expf(-(v + 65.f) / 80.f);
        p.f[F_K_CUR][ln] = (pow4f(n) * p.f[F_GK][ln]) * (v - p.f[F_EK][ln]);
        p.f[F_KL_CUR][ln] = p.f[F_GKL][ln] * (v - p.f[F_EKL][ln]);
    }
}

// ------------------------------------------------------------------------------------------------
// spike trains (SpikeTrainLattice::iterate, neuron/mod.rs:1377-1393): train_body.cuh
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) train_kernel(const __grid_constant__ TrainParams p) {
    pdl_wait();   // launch_pdl
    const uint32_t warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31u;
    if (warp_global * 32u >= p.n_trains) return;
    train_step(p, warp_global, lane);
}

// ------------------------------------------------------------------------------------------------
// graph construction on the device
// ------------------------------------------------------------------------------------------------
// CSR (by post, pre ascending) -> sliced ELL, one warp per slice
__global__ void sell_from_csr_kernel(const uint64_t *row_ptr, const uint32_t *pre, const float *w,
                                     const uint8_t *node_flags, uint32_t train0, uint32_t n_rows,
                                     const uint32_t *slice_off, uint32_t *col, float *wgt) {
    const uint32_t warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31u;
    if (warp_global * 32u >= n_rows) return;
    const uint32_t r = warp_global * 32u + lane;
    uint64_t b = 0, len = 0;
    if (r < n_rows) { b = row_ptr[r]; len = row_ptr[r + 1] - b; }
    const uint32_t k0 = slice_off[warp_global], k1 = slice_off[warp_global + 1];
    for (uint32_t k = k0; k < k1; ++k) {
        const size_t e = (size_t)k * 32u + lane;
        const uint32_t kk = k - k0;
        if (kk < len) {
            const uint32_t j = pre[b + kk];
            uint32_t c = j | ((uint32_t)(node_flags[j] & 0x7u) << kColNtShift);
            if (j >= train0) c |= kColTrainBit;
            col[e] = c;
            wgt[e] = w[b + kk];
        } else {
            col[e] = kColPad;
            wgt[e] = 0.f;
        }
    }
}

// Moore-neighbourhood stencil written straight into sliced-ELL form (uniform slice width)
__global__ void sell_grid_kernel(uint32_t rows_local, uint32_t cols, uint32_t row0_global, uint32_t rows_global,
                                 uint32_t radius, float weight, uint32_t own0, const uint8_t *node_flags,
                                 uint32_t width, uint32_t *slice_off, uint32_t *col, float *wgt) {
    const uint32_t warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t n = (uint64_t)rows_local * cols;
    if ((uint64_t)warp_global * 32u >= n) return;
    if (lane == 0) {
        slice_off[warp_global] = warp_global * width;
        if ((uint64_t)(warp_global + 1) * 32u >= n) slice_off[warp_global + 1] = (warp_global + 1) * width;
    }
    const uint64_t ln = (uint64_t)warp_global * 32u + lane;
    const size_t base = (size_t)warp_global * width * 32u + lane;
    if (radius == 1u) {
        // the window step kernel checks its tiles against the same function (tile_params_kernel)
        uint32_t c[8];
        stencil_cols((uint32_t)ln, (uint32_t)n, cols, row0_global, rows_global, own0, 0u, c);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const bool pad = c[k] == kColPad;
            col[base + (size_t)k * 32u] = pad ? kColPad : c[k] | ((uint32_t)(node_flags[c[k]] & 0x7u) << kColNtShift);
            wgt[base + (size_t)k * 32u] = pad ? 0.f : weight;
        }
        return;
    }
    const bool valid = ln < n;
    const int64_t r = valid ? (int64_t)(ln / cols) + row0_global : 0, c0 = valid ? (int64_t)(ln % cols) : 0;
    const int R = (int)radius;
    uint32_t k = 0;
    if (valid) {
        for (int dr = -R; dr <= R; ++dr)
            for (int dc = -R; dc <= R; ++dc) {
                const int64_t a = r + dr, b = c0 + dc;
                if ((dr == 0 && dc == 0) || a < 0 || b < 0 || a >= (int64_t)rows_global || b >= (int64_t)cols) continue;
                // node index of (a, b): the first owned neuron sits at own0; rows above/below the strip are ghosts
                const int64_t j = (int64_t)own0 + (a - (int64_t)row0_global) * (int64_t)cols + b;
                col[base + (size_t)k * 32u] = (uint32_t)j | ((uint32_t)(node_flags[j] & 0x7u) << kColNtShift);
                wgt[base + (size_t)k * 32u] = weight;
                ++k;
            }
    }
    for (; k < width; ++k) {
        col[base + (size_t)k * 32u] = kColPad;
        wgt[base + (size_t)k * 32u] = 0.f;
    }
}

__global__ void fill_u32_kernel(uint32_t *p, uint32_t v, uint64_t n) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

// u32 bools (reference buffer dtype for is_spiking) <-> 1 bit per node
__global__ void bits_from_u32_kernel(const uint32_t *src, uint32_t *words, uint64_t n, uint64_t bit0) {
    // arbitrary bit offset (a lattice segment need not start on a word boundary): one atomic per bit,
    // used only by set_field
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const uint64_t b = bit0 + t;
    if (src[t] != 0u) atomicOr(&words[b >> 5], 1u << (b & 31u));
    else atomicAnd(&words[b >> 5], ~(1u << (b & 31u)));
}
__global__ void u32_from_bits_kernel(const uint32_t *words, uint32_t *dst, uint64_t n, uint64_t bit0) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) dst[t] = (words[(bit0 + t) >> 5] >> ((bit0 + t) & 31u)) & 1u;
}

// neuron-major [n][3] (reference layout) <-> type-major [3][stride] (device layout)
__global__ void transpose_in_kernel(const float *src_nm, float *dst_tm, uint64_t n, uint64_t stride) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n * kNT) dst_tm[(t % kNT) * stride + t / kNT] = src_nm[t];
}
__global__ void transpose_out_kernel(const float *src_tm, float *dst_nm, uint64_t n, uint64_t stride) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n * kNT) dst_nm[t] = src_tm[(t % kNT) * stride + t / kNT];
}

// ------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------
static inline unsigned blocks_for(uint64_t n, unsigned bs) { return (unsigned)((n + bs - 1) / bs); }

cudaError_t launch_step(const StepParams &p, const StepSpec &spec, cudaStream_t s) {
    if (p.n_neurons == 0) return cudaSuccess;
    const unsigned grid = blocks_for((uint64_t)((p.n_neurons + 31u) / 32u) * 32u, 256);
    return dispatch_step(spec, cudaErrorInvalidValue, [&](auto k) {
        using K = decltype(k);
        if constexpr (K::NET && !K::NTREL && K::MODEL != SNN_MODEL_HODGKIN_HUXLEY)
            return launch_pdl(pdl_ok(p), step_net5_kernel<K::MODEL, K::CHEMG, K::NTREL, K::STDP>, dim3(grid), dim3(256), 0, s, p);
        else
            return launch_pdl(pdl_ok(p), step_kernel<K::MODEL, K::CHEMG, K::NTREL, K::STDP, K::NET>, dim3(grid), dim3(256), 0, s, p);
    });
}

cudaError_t launch_trains(const TrainParams &p, cudaStream_t s) {
    if (p.n_trains == 0) return cudaSuccess;
    return launch_pdl(pdl_ok(p), train_kernel, dim3(blocks_for((uint64_t)((p.n_trains + 31u) / 32u) * 32u, 256)), dim3(256), 0, s, p);
}

cudaError_t launch_halo_push(const StepParams &p, cudaStream_t s) {
    const uint32_t cnt = max(p.halo[0].active ? p.halo[0].count : 0u, p.halo[1].active ? p.halo[1].count : 0u);
    if (cnt == 0) return cudaSuccess;
    halo_push_kernel<<<blocks_for(cnt, 256), 256, 0, s>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_gpart_push(const StepParams &p, cudaStream_t s) {
    if (p.n_neurons == 0 || p.n_gpeers == 0) return cudaSuccess;
    gpart_push_kernel<<<blocks_for(p.n_neurons, 256), 256, 0, s>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_bcm_edges(const StepParams &p, const BcmParams &b, cudaStream_t s) {
    if (p.n_neurons == 0) return cudaSuccess;
    const bool part = (p.halo[0].active | p.halo[1].active) || p.n_gpeers;
    return launch_pdl(false, part ? bcm_part_edge_kernel : bcm_edge_kernel, dim3(blocks_for((uint64_t)((p.n_neurons + 31u) / 32u) * 32u, 256)),
                      dim3(256), 0, s, p, b);
}

cudaError_t launch_rstdp_edges(const StepParams &p, const RstdpParams &r, cudaStream_t s) {
    if (p.n_neurons == 0) return cudaSuccess;
    const unsigned n_slices = (p.n_neurons + 31u) / 32u;
    const unsigned grid = (n_slices + kRsSlices - 1) / kRsSlices;
    // the table stands for the formula while every spike time is exact in f32 (clock < 2^24)
    const bool tab = r.tab != nullptr && p.clock < (1u << 24);
    if (p.uniform_width == 8u && !(p.halo[0].active | p.halo[1].active) && grid > 512u) {
        // whole lattices with radius-1 stencil tables, large enough to fill the persistent grid
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        const unsigned pg = (unsigned)sms * (unsigned)SNN_RS_CTAS;
        if (r.canonical) return tab ? launch_pdl(false, rstdp_edge8_kernel<true, true>, dim3(pg), dim3(256), 0, s, p, r) : launch_pdl(false, rstdp_edge8_kernel<true, false>, dim3(pg), dim3(256), 0, s, p, r);
        return tab ? launch_pdl(false, rstdp_edge8_kernel<false, true>, dim3(pg), dim3(256), 0, s, p, r) : launch_pdl(false, rstdp_edge8_kernel<false, false>, dim3(pg), dim3(256), 0, s, p, r);
    }
    if (r.canonical) return tab ? launch_pdl(false, rstdp_edge_kernel<true, true>, dim3(grid), dim3(256), 0, s, p, r) : launch_pdl(false, rstdp_edge_kernel<true, false>, dim3(grid), dim3(256), 0, s, p, r);
    return tab ? launch_pdl(false, rstdp_edge_kernel<false, true>, dim3(grid), dim3(256), 0, s, p, r) : launch_pdl(false, rstdp_edge_kernel<false, false>, dim3(grid), dim3(256), 0, s, p, r);
}

// ------------------------------------------------------------------------------------------------
// RewardModulatedLatticeNetwork::post_neuron_update_step (neuron/mod.rs:5030-5062), the reward-modulated half
// ------------------------------------------------------------------------------------------------
// Runs after the step kernel and before the spike trains step: every neuron of a reward-modulated lattice with do_modulation
// visits its in-edges (update_weights_from_neurons_across_reward_lattices :4855-4929, _within_reward_lattices :4979-5003) and
// the out-edges of its own graph (:5005-5025), with both ends already carrying this step's last_firing_time.  Per edge that is
//  - own graph: two RewardModulatedSTDP::update_weight calls with identical arguments (as in-edge of the post end and as
//    out-edge of the pre end);
//  - connecting edge, RewardModulatedWeight: one call with the post lattice's modulator, whatever the input is;
//  - connecting edge, Weight: STDP::update_weight with the INPUT lattice's plasticity, only when the input is a plain Lattice.
// Connecting edges OUT of such a lattice are refused by Engine::run (the reference looks them up with swapped end points and
// panics).  One CTA per 32-row slice, one thread per edge, no ordering between edges.
// U k-rows per thread and round: all col words first, then the spike-time gathers and trace loads they address, then the
// arithmetic — U independent chains per thread hide the dependent round trips per edge.  Only U = 1 is launched: more k-rows per
// thread lose more in occupancy than they gain in memory-level parallelism (DESIGN.md, 144 / 162 / 199 us for 1 / 2 / 4).  The pass is instruction-bound before it
// is bandwidth-bound (ncu, profiles/r2_rstdp_net_edge_v2_full.txt: 186 warp instructions per k-row with the exponentials
// evaluated in place), hence:
//  - TAB: the STDP term through per-lattice difference tables (RnetParams::tab, filled by rstdp_table_kernel with the very
//    function the formula path calls — bit-identical while spike times are exact in f32);
//  - the edge kind from a 2-bit-per-class mask per post lattice, lattice bounds from the kernel parameters (constant bank);
//  - CANON: the edges of the lattices' own graphs enter every timestep with counter == 0 and dw == 0 (two calls per step return to
//    that state; TraceRSTDP::default starts there), so neither array is read or written for them.
template <bool CANON, bool TAB, int U>
__global__ void __launch_bounds__(256) rstdp_net_edge_kernel(const __grid_constant__ StepParams p, const __grid_constant__ RnetParams r) {
    pdl_wait();   // launch_pdl
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint32_t slice = blockIdx.x;
    const uint32_t ln = slice * 32u + lane;
    if (ln >= p.n_neurons) return;
    int lp = 0;
#pragma unroll 1
    for (uint32_t q = 1; q < r.n_lat; ++q) if (ln >= r.nbase[q]) lp = (int)q;
    const RnetLat &P = r.lat[lp];
    if ((P.flags & 3u) != 3u) return;
    const uint32_t k0 = p.uniform_width ? slice * p.uniform_width : __ldg(p.slice_off + slice);
    const uint32_t k1 = p.uniform_width ? k0 + p.uniform_width : __ldg(p.slice_off + slice + 1);
    const int t_post = p.lft_out[p.own0 + ln];
    const float decay_c = expf(-P.dt / P.tau_c);
    const uint64_t kinds = r.kinds[lp];
    RstdpParams m;
    m.dopamine = P.dopamine; m.tau_c = P.tau_c; m.a_plus = P.a_plus; m.a_minus = P.a_minus;
    m.tau_plus = P.tau_plus; m.tau_minus = P.tau_minus; m.dt = P.dt;
    m.tab = r.tab + (size_t)lp * 2u * r.tab_n; m.tab_n = r.tab_n;
    // round trip 1 of a round: the col words together with the weights and the traces they will most likely need (these do not
    // depend on the col word).  The loads of round t + 1 are issued before the stores of round t — the compiler cannot hoist them
    // itself (the stores may alias) — so a thread always has the next round's first trip in flight.
    uint32_t cw_n[U];
    float c_n[U], w_n[U];
    auto fetch = [&](uint32_t kb) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint32_t k = kb + 8u * u;
            const size_t e = (size_t)k * 32u + lane;
            const bool in = k < k1;
            cw_n[u] = in ? __ldg(p.col + e) : kColPad;
            w_n[u] = in ? p.wgt[e] : 0.f;
            c_n[u] = in ? r.c[e] : 0.f;
        }
    };
    fetch(k0 + warp);
    for (uint32_t kb = k0 + warp; kb < k1; kb += 8u * U) {
        uint32_t cw[U];
        float c[U], w[U];
#pragma unroll
        for (int u = 0; u < U; ++u) { cw[u] = cw_n[u]; c[u] = c_n[u]; w[u] = w_n[u]; }
        if (kb + 8u * U < k1) fetch(kb + 8u * U);
        // round trip 2: the presynaptic spike time the col word addresses, counter / dw where the edge kind needs them
        int t_pre[U], cls[U];
        uint32_t kind[U];   // 0 nothing, 1 own graph (two calls), 2 RewardModulatedWeight (one call), 3 Weight fed by a plain lattice
        uint32_t cnt[U];
        float dw[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            kind[u] = 0u; cnt[u] = 0u; dw[u] = 0.f; t_pre[u] = -1; cls[u] = 0;
            if (cw[u] == kColPad) continue;
            const size_t e = (size_t)(kb + 8u * u) * 32u + lane;
            const uint32_t j = cw[u] & kColIdxMask;
            int q0 = 0;
            if (cw[u] & kColTrainBit) {
                t_pre[u] = p.lft_in[j];   // the trains step after this pass: their current value is still in the input buffer
                const uint32_t tj = j - r.train0;
#pragma unroll 1
                for (uint32_t q = 1; q < r.n_tl; ++q) if (tj >= r.tl_base[q]) q0 = (int)q;
                q0 += kMaxLattices;
            } else {
                t_pre[u] = p.lft_out[j];
                const uint32_t nj = j - p.own0;
#pragma unroll 1
                for (uint32_t q = 1; q < r.n_lat; ++q) if (nj >= r.nbase[q]) q0 = (int)q;
            }
            cls[u] = q0;
            kind[u] = (uint32_t)(kinds >> (2 * q0)) & 3u;
            if (kind[u] == 2u || (!CANON && kind[u] == 1u)) { cnt[u] = r.counter[e]; dw[u] = r.dw[e]; }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (!kind[u]) continue;
            const size_t e = (size_t)(kb + 8u * u) * 32u + lane;
            const bool timed = t_pre[u] >= 0 && t_post >= 0 && t_pre[u] != t_post;
            if (kind[u] == 3u) {
                // STDP::update_weight with the INPUT lattice's parameters
                float d = 0.f;
                if (timed) {
                    if (TAB) { RstdpParams s = m; s.tab = r.tab + (size_t)cls[u] * 2u * r.tab_n; d = rstdp_delta_tab(s, t_pre[u], t_post); }
                    else d = stdp_delta(p.lat[cls[u]], t_pre[u], t_post);
                }
                if (d != 0.f) p.wgt[e] = w[u] + d;
                continue;
            }
            float delta_w = 0.f;
            if (timed) delta_w = TAB ? rstdp_delta_tab(m, t_pre[u], t_post) : rstdp_delta(m, t_pre[u], t_post);
            rstdp_call(m, delta_w, decay_c, cnt[u], dw[u], c[u], w[u]);
            if (kind[u] == 1u) rstdp_call(m, delta_w, decay_c, cnt[u], dw[u], c[u], w[u]);
            if (!(CANON && kind[u] == 1u)) { r.counter[e] = (uint8_t)cnt[u]; r.dw[e] = dw[u]; }
            r.c[e] = c[u]; p.wgt[e] = w[u];
        }
    }
}

template <bool CANON, bool TAB>
static cudaError_t launch_rnet_2(const StepParams &p, const RnetParams &r, cudaStream_t s) {
    return launch_pdl(false, rstdp_net_edge_kernel<CANON, TAB, 1>, dim3((p.n_neurons + 31u) / 32u), dim3(256), 0, s, p, r);
}

cudaError_t launch_rstdp_net_edges(const StepParams &p, const RnetParams &r, cudaStream_t s) {
    if (p.n_neurons == 0) return cudaSuccess;
    // the tables stand for the formula while every spike time is exact in f32 (clock < 2^24)
    const bool tab = r.tab != nullptr && p.clock < (1u << 24);
    if (r.canonical) return tab ? launch_rnet_2<true, true>(p, r, s) : launch_rnet_2<true, false>(p, r, s);
    return tab ? launch_rnet_2<false, true>(p, r, s) : launch_rnet_2<false, false>(p, r, s);
}

cudaError_t launch_flush_stdp(const StepParams &p, cudaStream_t s) {
    if (p.n_neurons == 0) return cudaSuccess;
    flush_stdp_kernel<<<blocks_for((uint64_t)((p.n_neurons + 31u) / 32u) * 32u, 256), 256, 0, s>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_finalize(const StepParams &p, int model, const float *v_prev, cudaStream_t s) {
    if (p.n_neurons == 0) return cudaSuccess;
    const unsigned grid = blocks_for(p.n_neurons, 256);
    if (model == SNN_MODEL_HODGKIN_HUXLEY) finalize_kernel<SNN_MODEL_HODGKIN_HUXLEY><<<grid, 256, 0, s>>>(p, v_prev);
    else finalize_kernel<SNN_MODEL_IZHIKEVICH><<<grid, 256, 0, s>>>(p, v_prev);
    return cudaGetLastError();
}

cudaError_t launch_sell_from_csr(const uint64_t *row_ptr, const uint32_t *pre, const float *w, const uint8_t *node_flags,
                                 uint32_t train0, uint32_t n_rows, const uint32_t *slice_off, uint32_t *col, float *wgt,
                                 cudaStream_t s) {
    if (n_rows == 0) return cudaSuccess;
    sell_from_csr_kernel<<<blocks_for((uint64_t)((n_rows + 31u) / 32u) * 32u, 256), 256, 0, s>>>(
        row_ptr, pre, w, node_flags, train0, n_rows, slice_off, col, wgt);
    return cudaGetLastError();
}

cudaError_t launch_sell_grid(uint32_t rows_local, uint32_t cols, uint32_t row0_global, uint32_t rows_global,
                             uint32_t radius, float weight, uint32_t own0, const uint8_t *node_flags, uint32_t width,
                             uint32_t *slice_off, uint32_t *col, float *wgt, cudaStream_t s) {
    const uint64_t n = (uint64_t)rows_local * cols;
    if (n == 0) return cudaSuccess;
    sell_grid_kernel<<<blocks_for(((n + 31u) / 32u) * 32u, 256), 256, 0, s>>>(
        rows_local, cols, row0_global, rows_global, radius, weight, own0, node_flags, width, slice_off, col, wgt);
    return cudaGetLastError();
}

// AverageVoltageHistory / EEGHistory (neuron/mod.rs:231-322): block (step, lattice) sums the staged grid record in f64 in a
// fixed order (thread-strided partial sums, then a shared-memory tree), so repeated runs give identical values
__global__ void history_reduce_kernel(const float *grid, uint64_t n_neurons, const uint32_t *lat_base, const uint32_t *lat_n,
                                      const float *lat_ref, int n_lat, double *out) {
    __shared__ double sh[2][256];
    const uint32_t step = blockIdx.x, k = blockIdx.y;
    const float *row = grid + (size_t)step * n_neurons + lat_base[k];
    const uint32_t n = lat_n[k];
    const float ref = lat_ref[k];
    double a = 0.0, b = 0.0;
    for (uint32_t i = threadIdx.x; i < n; i += 256u) {
        const float v = row[i];
        a += (double)v;
        b += (double)(v - ref);   // value - self.reference_voltage in f32, neuron/mod.rs:272
    }
    sh[0][threadIdx.x] = a; sh[1][threadIdx.x] = b;
    __syncthreads();
    for (uint32_t w = 128u; w > 0u; w >>= 1) {
        if (threadIdx.x < w) { sh[0][threadIdx.x] += sh[0][threadIdx.x + w]; sh[1][threadIdx.x] += sh[1][threadIdx.x + w]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { out[((size_t)step * n_lat + k) * 2] = sh[0][0]; out[((size_t)step * n_lat + k) * 2 + 1] = sh[1][0]; }
}

cudaError_t launch_history_reduce(const float *grid, uint64_t n_neurons, uint32_t steps, const uint32_t *lat_base, const uint32_t *lat_n,
                                  const float *lat_ref, int n_lat, double *out, cudaStream_t s) {
    if (steps == 0 || n_lat == 0) return cudaSuccess;
    history_reduce_kernel<<<dim3(steps, (unsigned)n_lat), 256, 0, s>>>(grid, n_neurons, lat_base, lat_n, lat_ref, n_lat, out);
    return cudaGetLastError();
}

__global__ void pack_flags_kernel(const uint32_t *src, uint8_t *node_flags, uint64_t n, int shift, unsigned int *changed) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool ch = false;
    if (i < n) {
        uint32_t m = 0;
        for (int ty = 0; ty < kNT; ++ty) if (src[i * kNT + ty]) m |= 1u << ty;
        const uint8_t f = node_flags[i];
        const uint8_t nf = (uint8_t)((f & ~(0xFu << shift)) | (m << shift));
        ch = nf != f;
        if (ch) node_flags[i] = nf;
    }
    if (__any_sync(0xffffffffu, ch) && (threadIdx.x & 31u) == 0) atomicOr(changed, 1u);
}

__global__ void spike_count_kernel(const uint32_t *words, uint32_t steps, uint64_t n_words, uint64_t n, uint32_t *counts) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t *w = words + (i >> 5);
    const uint32_t b = (uint32_t)(i & 31u);
    uint32_t c = 0;
    for (uint32_t s = 0; s < steps; ++s) c += (w[(size_t)s * n_words] >> b) & 1u;
    counts[i] = c;
}

cudaError_t launch_spike_count(const uint32_t *words, uint32_t steps, uint64_t n_words, uint64_t n, uint32_t *counts, cudaStream_t s) {
    if (n == 0) return cudaSuccess;
    spike_count_kernel<<<blocks_for(n, 256), 256, 0, s>>>(words, steps, n_words, n, counts);
    return cudaGetLastError();
}

cudaError_t launch_pack_flags(const uint32_t *src, uint8_t *node_flags, uint64_t n, int shift, unsigned int *changed, cudaStream_t s) {
    if (n == 0) return cudaSuccess;
    pack_flags_kernel<<<blocks_for(n, 256), 256, 0, s>>>(src, node_flags, n, shift, changed);
    return cudaGetLastError();
}

cudaError_t launch_fill_u32(uint32_t *p, uint32_t v, uint64_t n, cudaStream_t s) {
    if (n == 0) return cudaSuccess;
    fill_u32_kernel<<<blocks_for(n, 256), 256, 0, s>>>(p, v, n);
    return cudaGetLastError();
}
cudaError_t launch_bits_from_u32(const uint32_t *src, uint32_t *words, uint64_t n, uint64_t bit0, cudaStream_t s) {
    if (n == 0) return cudaSuccess;
    bits_from_u32_kernel<<<blocks_for(n, 256), 256, 0, s>>>(src, words, n, bit0);
    return cudaGetLastError();
}
cudaError_t launch_u32_from_bits(const uint32_t *words, uint32_t *dst, uint64_t n, uint64_t bit0, cudaStream_t s) {
    if (n == 0) return cudaSuccess;
    u32_from_bits_kernel<<<blocks_for(n, 256), 256, 0, s>>>(words, dst, n, bit0);
    return cudaGetLastError();
}
cudaError_t launch_transpose_in(const float *src_nm, float *dst_tm, uint64_t n, uint64_t stride, cudaStream_t s) {
    if (n == 0) return cudaSuccess;
    transpose_in_kernel<<<blocks_for(n * kNT, 256), 256, 0, s>>>(src_nm, dst_tm, n, stride);
    return cudaGetLastError();
}
cudaError_t launch_transpose_out(const float *src_tm, float *dst_nm, uint64_t n, uint64_t stride, cudaStream_t s) {
    if (n == 0) return cudaSuccess;
    transpose_out_kernel<<<blocks_for(n * kNT, 256), 256, 0, s>>>(src_tm, dst_nm, n, stride);
    return cudaGetLastError();
}

}  // namespace snn
