// step_body.cuh — the per-neuron step shared by the two step kernels.
//
// `neuron_step` is the whole timestep of one postsynaptic neuron: in-edge gather, receptors, model update,
// neurotransmitter release, spike ballot, stores and halo export.  It is parameterised on a *source policy* that says
// where the once-per-neuron streamed operands (own state, parameters, the slice's col/weight rows) come from:
//   GlobalSrc — straight from HBM with per-thread loads            (step_kernel, kernels.cu: general graphs, networks)
//   SmemSrc   — from a shared-memory stage filled by TMA bulk copies (step_tma_kernel, step_tma.cu: stencil lattices)
// Neighbour gathers (V, last_firing_time, t) always go through L1/L2, results are always stored to HBM directly.
#pragma once
#include "common.h"

namespace snn {

// ------------------------------------------------------------------------------------------------
// small helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int lat_index(const StepParams &p, uint32_t ln) {
    if (p.n_lat <= 1) return 0;
    int l = 0;
#pragma unroll 1
    for (int k = 1; k < p.n_lat; ++k)
        if (ln >= p.lat[k].base) l = k;
    return l;
}

// STDP::update_weight, plasticity/mod.rs:46-65
static __device__ __noinline__ float stdp_delta(const LatInfo &L, int t_pre_i, int t_post_i) {
    float delta_w = 0.f;
    if (t_pre_i >= 0 && t_post_i >= 0) {
        const float t_pre = (float)t_pre_i, t_post = (float)t_post_i;
        if (t_pre < t_post) {
            delta_w = L.a_plus * expf((-1.f * fabsf((t_pre - t_post) * L.dt)) / L.tau_plus);
        } else if (t_pre > t_post) {
            delta_w = (-1.f * L.a_minus) * expf((-1.f * fabsf((t_post - t_pre) * L.dt)) / L.tau_minus);
        }
    }
    return delta_w;
}

// NeurotransmitterKinetics::apply_t_change, iterate_and_spike/mod.rs:147-150, 192-196, 301-304, 352-357
__device__ __forceinline__ float nt_apply(int kind, float t, float t_max, float p1, float p2, float voltage,
                                          bool is_spiking, float dt) {
    const float flag = is_spiking ? 1.f : 0.f;
    switch (kind) {
    case SNN_NT_APPROXIMATE: {
        const float a = dt * -p1;
        const float b = a * t;
        const float c = flag * t_max;
        t = t + (b + c);
        return fminf(t_max, fmaxf(t, 0.f));
    }
    case SNN_NT_DESTEXHE:
        return t_max / (1.f + expf(-(voltage - p1) / p2));
    case SNN_NT_DISCRETE_SPIKE:
        return t_max * flag;
    default: {  // SNN_NT_EXPONENTIAL_DECAY
        const float t_change = -t * expf(dt / -p1);
        t = t + (t_change + flag * t_max);
        return fminf(t_max, fmaxf(t, 0.f));
    }
    }
}

// ReceptorKinetics::apply_r_change, iterate_and_spike/mod.rs:403-406, 434-437, 510-514
__device__ __forceinline__ float rc_apply(int kind, float r, float k1, float k2, float t, float dt) {
    switch (kind) {
    case SNN_RC_APPROXIMATE:
        return t;
    case SNN_RC_DESTEXHE: {
        const float a = k1 * t;
        const float b = a * (1.f - r);
        const float c = k2 * r;
        return r + (b - c) * dt;
    }
    default: {  // SNN_RC_EXPONENTIAL_DECAY: k1 = r_max, k2 = decay_constant
        const float dec = -r * expf(dt / -k2);
        r = r + (dec + t);
        return fminf(k1, fmaxf(r, 0.f));
    }
    }
}

// AMPA / NMDA / GABA ::iterate, iterate_and_spike/mod.rs:1101-1103, 1132-1137, 1164-1166
__device__ __forceinline__ float receptor_current(int type, float g, float e, float mg, float r, float v) {
    if (type == SNN_NT_NMDA) {
        const float ex = expf(-0.062f * v);
        const float den = 1.0f + ((ex * mg) / 3.75f);
        return (((1.0f / den) * g) * r) * (v - e);
    }
    return (g * r) * (v - e);
}

// NeuralRefractoriness::get_effect, spike_train/mod.rs:68-73, 84-86, 174-176
static __device__ __noinline__ float refract_effect(int kind, float k, uint32_t timestep, uint32_t last, float v_max,
                                                float v_resting, float dt) {
    const float a = v_max - v_resting;
    const float td = (float)(timestep - last);
    if (kind == SNN_REFRACT_DELTA_DIRAC) return a * expf((-1.f / (k / dt)) * (td * td)) + v_resting;
    return a * expf((-1.f / (k / dt)) * td) + v_resting;
}

__device__ __forceinline__ float ldf(const float *p, size_t i) { return __ldg(p + i); }

// m.powf(3.) and n.powf(4.) of the ion-channel currents (ion_channels/mod.rs:226-231, 275-278).  The reference calls libm's
// powf (within 1 ulp of the exact power); CUDA's powf is ~75 instructions with up to 4 ulp of error, the products below are 2-3
// instructions with at most 1.5 ulp — closer to what the reference computes AND a tenth of the Hodgkin-Huxley step's
// instruction stream.  (The HH path is tolerance-checked either way: its expf calls already differ from glibc's in the last bit.)
__device__ __forceinline__ float pow3f(float x) { return (x * x) * x; }
__device__ __forceinline__ float pow4f(float x) { const float x2 = x * x; return x2 * x2; }

// ------------------------------------------------------------------------------------------------
// halo synchronisation over NVLink peer memory (multi-GPU row strips)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(unsigned long long *p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

// Spin until the neighbour's arrival counter reaches `epoch`.  Bounded by `timeout_ns` (SNN_OPT_HALO_TIMEOUT_MS, default
// 30 s; run() has already met the neighbours on the host before the first step kernel, so only a neighbour that died or
// runs a different number of steps gets here): a dead neighbour must not hang this GPU.  On time-out the error flag is
// raised — every later kernel of the run returns at once (halo_failed), the host reports SNN_GPU_WAIT_ERROR.
__device__ __forceinline__ bool halo_wait(const unsigned long long *flag, unsigned long long epoch, unsigned int *err,
                                          unsigned long long timeout_ns) {
    if (ld_acquire_sys(flag) >= epoch) return true;
    const unsigned long long t0 = global_timer_ns();
    while (ld_acquire_sys(flag) < epoch) {
        __nanosleep(64);
        if (global_timer_ns() - t0 > timeout_ns || *(volatile unsigned int *)err) { atomicExch(err, 1u); return false; }
    }
    // counters of the waits that had to spin (err[2], err[3] = halo_done[4], [5]): time spent and number.  Nothing reads them; they
    // stay because the window kernel compiled without them took 0.6 us longer per step on the 10^7-neuron bench lattice
    // (295.9 vs 295.3 us, B200 at 1000 W)
    atomicAdd(err + 2, (unsigned int)((global_timer_ns() - t0) >> 4));
    atomicAdd(err + 3, 1u);
    return true;
}
// a halo wait of this run has timed out: the ghosts are stale, stop stepping (uniform over the grid once the flag is visible)
// (CTA-uniform: called by every thread of the CTA before anything else)
__device__ __forceinline__ bool halo_failed(const StepParams &p) {
    if (!(p.halo[0].active | p.halo[1].active | p.n_gpeers)) return false;
    return __syncthreads_or(*(volatile unsigned int *)(p.halo_done + 2) != 0u) != 0;
}


// ------------------------------------------------------------------------------------------------
// general-graph partition: ghosts of any rank, exported through per-neuron lists
// ------------------------------------------------------------------------------------------------
// Protocol: rank r publishes "step s complete" to every peer when ALL of its warps are done with step s (exports written AND
// ghost reads finished).  A warp of step s that reads ghosts, or writes a peer's ghosts, first waits until every peer has
// completed step s - 1: the ghosts it reads are then the peers' step s - 1 exports, and the ghost slots it overwrites (the parity
// the peer read in ITS step s - 1) are no longer being read.  Ranks are never more than one step apart.
__device__ __forceinline__ void gpart_wait(const StepParams &p, uint32_t slice, uint32_t lane) {
    if (!p.n_gpeers) return;
    if (p.gslice[slice] == 0u) return;   // warp-uniform: an interior slice neither reads ghosts nor exports
    if (lane == 0) {
        for (uint32_t q = 0; q < p.n_gpeers; ++q)
            if (!halo_wait(p.gpeers[q].my_flag, p.halo_epoch, p.halo_done + 2, p.halo_timeout_ns)) break;
    }
    __syncwarp();
}

// after neuron_step: copy this neuron's new state into the ghost slots of every peer that lists it, then count the warp as done;
// the last warp of the step raises every peer's completion counter.  BCM: BCM Izhikevich neurons, whose current_activity is
// exported too (the peers' BCM edge kernels read it)
template <bool BCM>
__device__ __forceinline__ void gpart_export_publish(const StepParams &p, uint32_t slice, uint32_t lane, uint32_t ln, bool valid) {
    if (!p.n_gpeers) return;
    const bool exports = (p.gslice[slice] & 2u) != 0u;
    if (exports && valid) {
        const uint32_t i = p.own0 + ln;
        for (uint32_t e = p.gexp_off[ln]; e < p.gexp_off[ln + 1]; ++e) {
            const uint32_t ent = __ldg(p.gexp_ent + e), dst = ent & kColIdxMask;
            const GPeer &G = p.gpeers[ent >> 28];
            G.v[p.out_par][dst] = p.v_out[i];
            G.lft[p.out_par][dst] = p.lft_out[i];
            for (int ty = 0; ty < kNT; ++ty)
                if (p.nt_used & (1u << ty)) G.t[p.out_par][(size_t)ty * G.t_stride + dst] = p.t_out[(size_t)ty * p.t_stride + i];
            if constexpr (BCM) bcm_gpeer_act(p, ent >> 28, p.out_par)[dst] = p.f[F_CUR_ACT][ln];
        }
    }
    __syncwarp();
    if (lane == 0) {
        if (exports) __threadfence_system();
        else __threadfence();
        const unsigned int done = atomicAdd(&p.halo_done[6], 1u) + 1u;
        if (done == p.n_gslices) {
            p.halo_done[6] = 0u;
            __threadfence_system();
            for (uint32_t q = 0; q < p.n_gpeers; ++q) st_release_sys(p.gpeers[q].peer_flag, p.halo_epoch + 1ull);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// source policies
// ------------------------------------------------------------------------------------------------
struct GlobalSrc {
    // per-thread HBM loads: issue every parameter load before the edge loop so that the latencies overlap
    static constexpr bool kEarlyLoads = true;
    static constexpr bool kCheapEdges = false;
    static constexpr bool kWide = false;
    static constexpr uint32_t kWidth = 0;   // slice width known at run time only
    static constexpr bool kStencil = false;  // col words come from the table (gather_edges8)
    const StepParams &p;
    uint32_t lnc;   // clamped local neuron number
    uint32_t i;     // node index
    uint32_t lane;
    uint32_t k0, k1;  // k-rows of this warp's slice
    const float *t0;  // CHEMG == 1: row of the single neurotransmitter type in t_in
    template <int SLOT> __device__ __forceinline__ float f() const { return __ldg(p.f[SLOT] + lnc); }
    template <int SLOT> __device__ __forceinline__ float state() const { return p.f[SLOT][lnc]; }
    __device__ __forceinline__ float v() const { return p.v_in[i]; }
    __device__ __forceinline__ int lft() const { return p.lft_in[i]; }
    __device__ __forceinline__ uint32_t flags() const { return p.node_flags[i]; }
    // plain load: the multi-step kernel (step_multi.cu) reads words that an earlier step of the same launch wrote
    __device__ __forceinline__ uint32_t spk_prev_word(uint32_t warp_global) const { return p.spk_in[(p.own0 >> 5) + warp_global]; }
    __device__ __forceinline__ float t_own(int ty) const { return p.t_in[(size_t)ty * p.t_stride + i]; }
    __device__ __forceinline__ float nt(int slot, int ty) const { return __ldg(p.nt[slot] + (size_t)ty * p.nt_stride + i); }
    __device__ __forceinline__ float rc(int slot, int ty) const { return __ldg(p.rc[slot] + (size_t)ty * p.rc_stride + lnc); }
    __device__ __forceinline__ float rc_state(int slot, int ty) const { return p.rc[slot][(size_t)ty * p.rc_stride + lnc]; }
    __device__ __forceinline__ uint32_t width() const { return k1 - k0; }
    __device__ __forceinline__ uint32_t col(uint32_t kk) const { return __ldg(p.col + (size_t)(k0 + kk) * 32u + lane); }
    __device__ __forceinline__ float wgt(uint32_t kk) const { return p.wgt[(size_t)(k0 + kk) * 32u + lane]; }
    __device__ __forceinline__ float *wgt_ptr(uint32_t kk) const { return p.wgt + (size_t)(k0 + kk) * 32u + lane; }
    // neighbour gathers: a handle is whatever addresses presynaptic node j (here: j itself, through L1/L2)
    typedef uint32_t Handle;
    __device__ __forceinline__ Handle gh(uint32_t j) const { return j; }
    __device__ __forceinline__ float gv(Handle h) const { return p.v_in[h]; }
    __device__ __forceinline__ int glft(Handle h) const { return p.lft_in[h]; }
    __device__ __forceinline__ float gt0(Handle h) const { return t0[h]; }
    __device__ __forceinline__ float gt(Handle h, int ty) const { return p.t_in[(size_t)ty * p.t_stride + h]; }
};

// ------------------------------------------------------------------------------------------------
// in-edge gather
// ------------------------------------------------------------------------------------------------
struct EdgeAcc {
    float acc_e;
    uint32_t n_in;
    float acc_t[kNT];
    uint32_t cnt[kNT];
    bool fast8;   // warp-uniform: every lane had exactly 8 in-edges (and, CHEMG == 1, all of them release the type):
                  // the averaging divisions are by 8 = exact multiplications by 0.125
    bool fast8t;  // CHEMG == 3, warp-uniform: fast8 and every presynaptic neuron releases all three types
    bool skip;    // two-pass wide kernels: this CTA summed one accumulator and another CTA of the slice finishes the step
};

// The lazily applied STDP of the previous step for one chunk of U edges (see gather_edges); shared by both gathers.
//
// Spikes are rare (~0.2 % of the neurons per step in the bench workload) but a warp that meets one used to walk its
// U edges serially through a divergent call of stdp_delta (ncu, profiles/r1_step_win_active_full.txt: +20 % kernel
// time at that spike rate because the slow warp holds its shared-memory stage).  The work is spread over the warp
// instead, with the same stdp_delta evaluations on the same operands (bit-identical weights):
//   * out-edge rule (the presynaptic neuron spiked): delta(prev, last_firing_time of this lane) does not depend on the
//     edge, so every lane evaluates it once, without divergence;
//   * in-edge rule (this lane's neuron spiked): its U deltas delta(lj[u], prev) are evaluated by lanes 0..U-1 in
//     parallel and shuffled back.
template <int U, bool NET, class SRC>
__device__ __forceinline__ void stdp_chunk(const StepParams &p, const SRC &src, uint32_t kk, const uint32_t (&c)[U], const uint32_t (&j)[U],
                                           const int (&lj)[U], float (&w)[U], bool post_trig, int lft_me, int li, int prev) {
    constexpr uint32_t kAll = 0xffffffffu;
    {   // one cheap test per chunk decides whether the warp has anything to do
        bool any = post_trig;
#pragma unroll
        for (int u = 0; u < U; ++u) any |= (lj[u] == prev);
        if (!__any_sync(kAll, any)) return;
    }
    uint32_t pre_mask = 0;
#pragma unroll
    for (int u = 0; u < U; ++u) {
        bool pre_trig = c[u] != kColPad && lj[u] == prev;
        if (NET) {
            if (pre_trig) pre_trig = !(c[u] & kColTrainBit) && p.lat[lat_index(p, j[u] - p.own0)].do_plasticity != 0;
        } else {
            pre_trig = pre_trig && p.lat[0].do_plasticity != 0;
        }
        pre_mask |= (pre_trig ? 1u : 0u) << u;
    }
    const uint32_t post_lanes = __ballot_sync(kAll, post_trig);
    const bool any_pre = __any_sync(kAll, pre_mask != 0u);
    if (post_lanes == 0u && !any_pre) return;   // warp-uniform
    const int lane = (int)(threadIdx.x & 31u);
    float d_pre = 0.f;
    if (any_pre) d_pre = stdp_delta(p.lat[li], prev, lft_me);
    for (uint32_t rem = post_lanes; rem != 0u; rem &= rem - 1u) {
        const int src_lane = __ffs((int)rem) - 1;
        int t_pre = -1;
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int x = __shfl_sync(kAll, lj[u], src_lane);
            if (lane == u) t_pre = x;
        }
        const int li_src = NET ? __shfl_sync(kAll, li, src_lane) : 0;
        const float d = (lane < U) ? stdp_delta(p.lat[li_src], t_pre, prev) : 0.f;
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const float x = __shfl_sync(kAll, d, u);
            if (lane == src_lane && c[u] != kColPad) w[u] = w[u] + x;
        }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
        const bool in_rule = post_trig && c[u] != kColPad, out_rule = (pre_mask >> u) & 1u;
        if (in_rule || out_rule) {
            float wu = w[u];                 // the in-edge delta was added above
            if (out_rule) wu = wu + d_pre;   // both rules on one edge: t_pre == t_post, both deltas are 0
            w[u] = wu;
            *src.wgt_ptr(kk + u) = wu;
        }
    }
}

// The same lazy STDP for sources whose weight rows sit in a shared-memory stage (step_win.cu).  It runs BEFORE the
// gather loads the weights and updates them in place (stage and HBM), so the common path carries no register state of
// the rare path: the weight registers are loaded afterwards, and a warp without a trigger leaves after one vote.
template <class SRC>
__device__ __forceinline__ void stdp_chunk8_staged(const StepParams &p, const SRC &src, const uint32_t (&c)[8], const int (&lj)[8],
                                                   bool post_trig, int lft_me, int li, int prev) {
    constexpr uint32_t kAll = 0xffffffffu;
    {
        bool any = post_trig;
#pragma unroll
        for (int u = 0; u < 8; ++u) any |= (lj[u] == prev);
        if (!__any_sync(kAll, any)) return;
    }
    const bool plastic = p.lat[0].do_plasticity != 0;
    uint32_t pre_mask = 0;
#pragma unroll
    for (int u = 0; u < 8; ++u) pre_mask |= ((plastic && c[u] != kColPad && lj[u] == prev) ? 1u : 0u) << u;
    const int lane = (int)(threadIdx.x & 31u);
    // in-edge rule: the 8 deltas of a neuron that spiked are evaluated by 8 lanes in parallel, four spiking neurons per round
    // (lane group g = lane / 8 serves the g-th spiking lane of the round), so that a synchronous burst costs a quarter of the
    // rounds
    for (uint32_t rem = __ballot_sync(kAll, post_trig); rem != 0u;) {
        int psrc[4];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
            psrc[g] = rem ? __ffs((int)rem) - 1 : -1;
            rem &= rem - 1u;   // 0 stays 0
        }
        const int g_me = lane >> 3, u_me = lane & 7;
        const int my_src = g_me == 0 ? psrc[0] : (g_me == 1 ? psrc[1] : (g_me == 2 ? psrc[2] : psrc[3]));
        int t_pre = -1;
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int x = __shfl_sync(kAll, lj[u], my_src < 0 ? 0 : my_src);
            if (u_me == u) t_pre = x;
        }
        const float d = (my_src >= 0) ? stdp_delta(p.lat[li], t_pre, prev) : 0.f;
        // which group serves this lane (if it is one of the round's spiking lanes)
        const int g_of_me = lane == psrc[0] ? 0 : (lane == psrc[1] ? 1 : (lane == psrc[2] ? 2 : (lane == psrc[3] ? 3 : -1)));
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const float x = __shfl_sync(kAll, d, (g_of_me < 0 ? 0 : g_of_me) * 8 + u);
            if (g_of_me >= 0 && c[u] != kColPad) src.wgt_update(u, src.wgt(u) + x);
        }
    }
    // out-edge rule: delta(prev, own last_firing_time) is the same for every edge of a lane
    if (__any_sync(kAll, pre_mask != 0u)) {
        const float d_pre = stdp_delta(p.lat[li], prev, lft_me);
#pragma unroll
        for (int u = 0; u < 8; ++u)
            if ((pre_mask >> u) & 1u) src.wgt_update(u, src.wgt(u) + d_pre);   // both rules on one edge: both deltas are 0
    }
    src.wgt_updates_done();
}

// Gather for sources whose slices are exactly 8 k-rows wide (radius-1 stencil tables, step_win.cu): one chunk, no loop.
// FULL (warp-uniform): no lane of the warp has a padding slot and, with a single neurotransmitter type, every
// presynaptic neuron releases it — the per-edge validity / type tests and the in-edge counters fold away.  The
// accumulation order and every rounding are those of gather_edges (a skipped `+ 0` term of a padding slot is exact).
// STEN (with FULL): a full warp of a stencil tile (WinSrc): slot u is node i + stencil_off(u), every presynaptic node releases
// stencil_nt(), and c[] only answers validity tests (every slot holds an edge).
template <int CHEMG, bool STDP, bool FULL, bool FULLT, bool STEN, class SRC>
__device__ __forceinline__ void gather_edges8_body(const StepParams &p, const SRC &src, uint32_t i, float v, float gap, int lft_me,
                                                   bool post_trig, int li, uint32_t ty0, const uint32_t (&c)[8], EdgeAcc &A) {
    constexpr int U = 8;
    const bool pending = STDP && p.apply_pending;
    const bool do_e = p.electrical != 0;
    const int prev = (int)p.clock - 1;
    uint32_t j[U];
    typename SRC::Handle h[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
        if constexpr (STEN) j[u] = i + src.stencil_off(u);
        else j[u] = (FULL || c[u] != kColPad) ? (c[u] & kColIdxMask) : i;
        // a full row of a generated radius-1 stencil lists its presynaptic neurons in ascending order: three in the row
        // above, the two side neighbours, three in the row below
        h[u] = FULL ? src.gh_row(u < 3 ? 0 : (u < 5 ? 1 : 2), j[u]) : src.gh(j[u]);   // u folds after unrolling
    }
    if (pending) {
        int lj[U];
#pragma unroll
        for (int u = 0; u < U; ++u) lj[u] = src.glft(h[u]);
        stdp_chunk8_staged(p, src, c, lj, post_trig, lft_me, li, prev);
    }
    float w[U];
#pragma unroll
    for (int u = 0; u < U; ++u) w[u] = src.wgt(u);
    float vj[U];
#pragma unroll
    for (int u = 0; u < U; ++u) vj[u] = do_e ? src.gv(h[u]) : v;
    float tj[U][CHEMG == 3 ? kNT : 1];
    if (CHEMG == 1) {
#pragma unroll
        for (int u = 0; u < U; ++u) tj[u][0] = src.gt0(h[u]);
    } else if (CHEMG == 3) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
            uint32_t m = (FULL || c[u] != kColPad) ? (c[u] >> kColNtShift) : 0u;
            if constexpr (STEN) m = src.stencil_nt();
#pragma unroll
            for (int ty = 0; ty < kNT; ++ty) tj[u][ty] = (FULLT || (m & (1u << ty))) ? src.gt(h[u], ty) : 0.f;
        }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
        const bool ok = FULL || c[u] != kColPad;
        const float wu = w[u];
        if (do_e) {
            const float final_input = gap * (vj[u] - v);  // gap_junction, neuron/mod.rs:54-60
            A.acc_e = A.acc_e + final_input * wu;
        }
        if (CHEMG == 1) {
            const float term = tj[u][0] * wu;
            if (FULL) {
                A.acc_t[0] = A.acc_t[0] + term;
            } else {
                const bool has = ok && ((c[u] >> (kColNtShift + ty0)) & 1u);
                A.acc_t[0] = A.acc_t[0] + (has ? term : 0.f);
                A.cnt[0] += has ? 1u : 0u;
            }
        } else if (CHEMG == 3) {
            if (FULLT) {
                // every presynaptic neuron releases every type: the same terms in the same order, without masks and counters
#pragma unroll
                for (int ty = 0; ty < kNT; ++ty) A.acc_t[ty] = A.acc_t[ty] + tj[u][ty] * wu;
            } else {
                uint32_t m = ok ? (c[u] >> kColNtShift) : 0u;
                if constexpr (STEN) m = src.stencil_nt();
#pragma unroll
                for (int ty = 0; ty < kNT; ++ty) {
                    const bool has = (m >> ty) & 1u;
                    const float term = tj[u][ty] * wu;
                    A.acc_t[ty] = A.acc_t[ty] + (has ? term : 0.f);
                    A.cnt[ty] += has ? 1u : 0u;
                }
            }
        }
        if (!FULL) A.n_in += ok ? 1u : 0u;
    }
    if (FULL) {
        A.n_in = 8u;
        if (CHEMG == 1) A.cnt[0] = 8u;
        if (FULLT) {
#pragma unroll
            for (int ty = 0; ty < kNT; ++ty) A.cnt[ty] = 8u;
        }
    }
}

template <int CHEMG, bool STDP, class SRC>
__device__ __forceinline__ void gather_edges8(const StepParams &p, const SRC &src, uint32_t i, float v, float gap, int lft_me,
                                              bool post_trig, int li, uint32_t ty0, EdgeAcc &A) {
    uint32_t c[8];
    if constexpr (SRC::kStencil) {
        // FULL needs, with one neurotransmitter type, that every presynaptic node releases it: uniform over the launch here
        const uint32_t nt = src.stencil_nt();
        if (src.stencil_full() && (CHEMG != 1 || ((nt >> ty0) & 1u))) {
#pragma unroll
            for (int u = 0; u < 8; ++u) c[u] = 0u;
            A.fast8 = true;
            A.fast8t = CHEMG == 3 && nt == 7u;
            if (CHEMG == 3 && A.fast8t) gather_edges8_body<CHEMG, STDP, true, true, true>(p, src, i, v, gap, lft_me, post_trig, li, ty0, c, A);
            else gather_edges8_body<CHEMG, STDP, true, false, true>(p, src, i, v, gap, lft_me, post_trig, li, ty0, c, A);
            return;
        }
        src.stencil_cols(c);   // border warps
    } else {
#pragma unroll
        for (int u = 0; u < 8; ++u) c[u] = src.col(u);
    }
    // sliced-ELL rows keep their valid entries first (sell_grid_kernel / sell_from_csr_kernel pad at the end), so a valid
    // last slot means a full row
    bool lane_full = c[7] != kColPad;
    const uint32_t all = c[0] & c[1] & c[2] & c[3] & c[4] & c[5] & c[6] & c[7];
    if (CHEMG == 1) lane_full = lane_full && ((all >> (kColNtShift + ty0)) & 1u);
    A.fast8 = __all_sync(0xffffffffu, lane_full);
    A.fast8t = false;
    if (CHEMG == 3) A.fast8t = A.fast8 && __all_sync(0xffffffffu, ((all >> kColNtShift) & 7u) == 7u);
    if (CHEMG == 3 && A.fast8t) gather_edges8_body<CHEMG, STDP, true, true, false>(p, src, i, v, gap, lft_me, post_trig, li, ty0, c, A);
    else if (A.fast8) gather_edges8_body<CHEMG, STDP, true, false, false>(p, src, i, v, gap, lft_me, post_trig, li, ty0, c, A);
    else gather_edges8_body<CHEMG, STDP, false, false, false>(p, src, i, v, gap, lft_me, post_trig, li, ty0, c, A);
}

// CHEMG: 0 = no chemical gather, 1 = exactly one neurotransmitter type in the whole node array (type index ty0),
//        3 = general per-edge type masks.  NET: the node array holds several lattices and/or spike trains.
//
// Edges are consumed in chunks of 8 (slice widths are padded to a multiple of 4): first all coalesced col/weight
// loads of the chunk, then all neighbour gathers, then the strictly ordered accumulation.  Eight independent
// requests per thread keep enough bytes in flight to cover HBM latency; the arithmetic order is the canonical one
// (ascending presynaptic index).  Padding slots carry weight 0 and gather the neuron itself, so they add an exact
// +0 and need no branch.
template <int CHEMG, bool STDP, bool NET, class SRC>
__device__ __forceinline__ void gather_edges(const StepParams &p, const SRC &src, uint32_t i, float v, float gap, int lft_me,
                                             bool post_trig, int li, uint32_t ty0, EdgeAcc &A) {
    constexpr int U = 8;
    const uint32_t width = SRC::kWidth ? SRC::kWidth : src.width();
    const bool pending = STDP && p.apply_pending;
    const bool do_e = p.electrical != 0;
    const int prev = (int)p.clock - 1;
    for (uint32_t kk = 0; kk < width; kk += U) {
        const bool full = kk + U <= width;
        uint32_t c[U];
        float w[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (u < 4 || full) { c[u] = src.col(kk + u); w[u] = SRC::kCheapEdges ? 0.f : src.wgt(kk + u); }
            else { c[u] = kColPad; w[u] = 0.f; }
        }
        uint32_t j[U];
        typename SRC::Handle h[U];
#pragma unroll
        for (int u = 0; u < U; ++u) { j[u] = (c[u] == kColPad) ? i : (c[u] & kColIdxMask); h[u] = src.gh(j[u]); }
        float vj[U];
        if (do_e) {
#pragma unroll
            for (int u = 0; u < U; ++u) vj[u] = src.gv(h[u]);
        } else {
#pragma unroll
            for (int u = 0; u < U; ++u) vj[u] = v;
        }
        int lj[U];
        if (pending) {
            // a spike train steps AFTER the neurons and their STDP (neuron/mod.rs:2573-2591): the rule of step s must
            // see the train's last_firing_time from before its step-s iterate, which still sits in the other
            // ping-pong buffer (the train kernel of this step has not run yet)
#pragma unroll
            for (int u = 0; u < U; ++u) lj[u] = (NET && (c[u] & kColTrainBit) && c[u] != kColPad) ? p.lft_out[j[u]] : src.glft(h[u]);
        } else {
#pragma unroll
            for (int u = 0; u < U; ++u) lj[u] = -1;
        }
        float tj[U][CHEMG == 3 ? kNT : 1];
        if (CHEMG == 1) {
#pragma unroll
            for (int u = 0; u < U; ++u) tj[u][0] = src.gt0(h[u]);
        } else if (CHEMG == 3) {
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const uint32_t m = (c[u] == kColPad) ? 0u : (c[u] >> kColNtShift);
#pragma unroll
                for (int ty = 0; ty < kNT; ++ty) tj[u][ty] = (m & (1u << ty)) ? src.gt(h[u], ty) : 0.f;
            }
        }
        // lazy application of the previous step's STDP while the edges stream by: in-edge rule if the post neuron spiked
        // last step, out-edge rule if the pre neuron did (update_weights_from_neurons, neuron/mod.rs:849-881, 2308-2417);
        // both use the post lattice's rule.  No edge can get two non-zero updates in one step.  Spikes are rare: one
        // test per chunk decides whether the slow path runs at all.
        if (SRC::kCheapEdges) {
            // operands in shared memory: re-read instead of holding 16 registers across the gather latency
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (u < 4 || full) { c[u] = src.col(kk + u); w[u] = src.wgt(kk + u); }
        }
        if (pending) stdp_chunk<U, NET>(p, src, kk, c, j, lj, w, post_trig, lft_me, li, prev);
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const bool ok = c[u] != kColPad;
            const float wu = w[u];
            if (do_e) {
                float final_input = gap * (vj[u] - v);  // gap_junction, neuron/mod.rs:54-60
                if (NET) {
                    if (ok && (c[u] & kColTrainBit)) {
                        // spike_train_gap_junction, neuron/mod.rs:119-137
                        const uint32_t tjx = j[u] - p.train0;
                        const int lt = p.lft_in[j[u]];
                        const float v_rest = ldf(p.tf[TF_VREST], tjx);
                        if (lt < 0) final_input = v_rest;
                        else
                            final_input = gap * refract_effect(p.refract, ldf(p.tf[TF_K], tjx), p.clock, (uint32_t)lt,
                                                               ldf(p.tf[TF_VTH], tjx), v_rest, ldf(p.tf[TF_DT], tjx));
                    }
                }
                A.acc_e = A.acc_e + final_input * wu;
            }
            if (CHEMG == 1) {
                // weight_neurotransmitter_concentration + aggregate, iterate_and_spike/mod.rs:2837-2866
                const bool has = ok && ((c[u] >> (kColNtShift + ty0)) & 1u);
                const float term = tj[u][0] * wu;
                A.acc_t[0] = A.acc_t[0] + (has ? term : 0.f);
                A.cnt[0] += has ? 1u : 0u;
            } else if (CHEMG == 3) {
                const uint32_t m = ok ? (c[u] >> kColNtShift) : 0u;
#pragma unroll
                for (int ty = 0; ty < kNT; ++ty) {
                    const bool has = (m >> ty) & 1u;
                    const float term = tj[u][ty] * wu;
                    A.acc_t[ty] = A.acc_t[ty] + (has ? term : 0.f);
                    A.cnt[ty] += has ? 1u : 0u;
                }
            }
            A.n_in += ok ? 1u : 0u;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// in-edge gather for wide rows (step_wide.cu): a whole CTA serves one 32-row slice
// ------------------------------------------------------------------------------------------------
// A LatticeNetwork like BASELINE.json configs[3] has few neurons with ~10^3 in-edges each (784 spike trains -> every
// excitatory neuron): with one thread per row the general kernel walks those edges serially in 25 warps on the whole GPU
// (1.6 ms per step).  Here the per-edge work (coalesced col/weight loads, neighbour gathers, spike-train refractoriness,
// lazy STDP, the products) is spread over all warps of the CTA — warp w takes k-rows w, w + W, ... of a chunk, lane = row —
// and parked in shared memory; the leader warp then adds the parked terms in ascending presynaptic order.  The terms and
// the order of the additions are those of gather_edges, so the sums are bit-identical.
constexpr int kWideUnroll = 4;         // k-rows per helper thread and chunk
constexpr int kWideWarps = 16;         // warps per CTA: one leader + 15 helpers
constexpr uint32_t kWideChunk = kWideUnroll * (kWideWarps - 1);   // 60 k-rows per chunk (slice widths are multiples of 4)
constexpr uint32_t kWideSumBufs = 8;   // chunk buffers of the sum pass of the two-pass wide kernels (7 copies in flight)
// shared memory of one chunk buffer (two of them: the helpers fill one while the leader drains the other)
__host__ __device__ constexpr uint32_t wide_buf_bytes(int chemg) { return kWideChunk * 32u * (4u + (chemg == 3 ? 4u * kNT : (chemg == 1 ? 4u : 0u)) + 1u); }

// Small networks (BASELINE.json configs[3]: 1 584 nodes): the whole node state a wide slice gathers from — V, both
// last_firing_time buffers, the neurotransmitter concentrations and, per spike train, the refractoriness term of
// spike_train_gap_junction (a function of the train alone: evaluated once per train and step instead of once per edge) — is
// copied into shared memory when the CTA starts its slice.  The helpers' per-edge gathers then are shared-memory reads: the two
// dependent L2 round trips per chunk (40 % long-scoreboard stalls, profiles/r1_step_wide_c4_pipelined_full.txt) are gone and only
// the coalesced col / weight stream still comes from L2.  Same values, same arithmetic: bit-identical.
struct WideStage {
    const float *v; const int *lft_in, *lft_out; const float *t;   // [n_nodes], [n_nodes], [n_nodes], [kNT][n_nodes]
    const float *eff; const uint8_t *never;                        // per train: refractoriness term (or v_resting), "has never fired"
    uint32_t n_nodes;                                              // 0 = not staged (gathers go to global memory)
};
__host__ __device__ constexpr uint32_t wide_stage_bytes(uint32_t n_nodes, uint32_t n_trains) {
    return ((n_nodes * 4u * (3u + (uint32_t)kNT) + n_trains * 4u + n_trains + 15u) / 16u) * 16u;
}
constexpr uint32_t kWideStageMaxNodes = 4096;

struct WideSrc : GlobalSrc {
    static constexpr bool kWide = true;
    uint32_t warp, n_warps;
    unsigned char *sm;    // 2 x wide_buf_bytes: [kWideChunk][32] f32 electrical terms, [types][kWideChunk][32] f32 chemical terms,
                          // [kWideChunk][32] u8 flags (bit 0: edge present, bits 1..3: presynaptic node releases type 0..2)
    WideStage st;
    // split mode for very wide slices (one SM cannot issue a 1 200-wide slice's per-edge instructions fast enough):
    //   0  one CTA does everything;
    //   1  "terms" pass: this CTA computes the per-edge terms of chunk `chunk` only and parks them in global scratch (all SMs share
    //      the slices' chunks);
    //   2  "sum" pass: the helpers copy the parked chunks into shared memory, the leader adds them in order and steps the neurons.
    uint32_t mode, chunk;     // sum pass: `chunk` is the accumulator this CTA sums (0: electrical, 1 + ty: neurotransmitter type)
    unsigned char *scratch;   // [slice][chunks_cap] chunk buffers of wide_buf_bytes(CHEMG), then the partial sums (wide_part_offset)
    uint32_t chunks_cap;
    uint32_t n_slices;
};
// after the chunk buffers: per slice (1 + kNT) x 32 partial sums (f32), (1 + kNT) x 32 counts (u32), one arrival counter (u32)
__host__ __device__ constexpr size_t wide_part_bytes_per_slice() { return (size_t)(1 + kNT) * 32u * 8u + 16u; }

// every thread of the CTA: fill the stage (called before neuron_step; ends with a CTA barrier)
template <bool NET>
__device__ __forceinline__ WideStage wide_stage_fill(const StepParams &p, unsigned char *base, bool enable) {
    WideStage S{};
    if (!enable) return S;
    const uint32_t n = p.n_nodes, nt = NET ? p.n_trains : 0u;
    float *sv = reinterpret_cast<float *>(base);
    int *sli = reinterpret_cast<int *>(sv + n), *slo = sli + n;
    float *stt = reinterpret_cast<float *>(slo + n);
    float *seff = stt + (size_t)kNT * n;
    uint8_t *snev = reinterpret_cast<uint8_t *>(seff + nt);
    for (uint32_t j = threadIdx.x; j < n; j += blockDim.x) {
        sv[j] = p.v_in[j];
        sli[j] = p.lft_in[j];
        slo[j] = p.lft_out[j];
#pragma unroll
        for (int ty = 0; ty < kNT; ++ty) stt[(size_t)ty * n + j] = (p.nt_used & (1u << ty)) ? p.t_in[(size_t)ty * p.t_stride + j] : 0.f;
    }
    if constexpr (NET) {
        for (uint32_t tj = threadIdx.x; p.electrical && tj < nt; tj += blockDim.x) {
            // spike_train_gap_junction, neuron/mod.rs:119-137: v_resting if the train has never fired, else the refractoriness term
            const int lt = p.lft_in[p.train0 + tj];
            const float v_rest = ldf(p.tf[TF_VREST], tj);
            float e = v_rest;
            if (lt >= 0) e = refract_effect(p.refract, ldf(p.tf[TF_K], tj), p.clock, (uint32_t)lt, ldf(p.tf[TF_VTH], tj), v_rest, ldf(p.tf[TF_DT], tj));
            seff[tj] = e;
            snev[tj] = lt < 0 ? 1u : 0u;
        }
    }
    __syncthreads();
    S.v = sv; S.lft_in = sli; S.lft_out = slo; S.t = stt; S.eff = seff; S.never = snev; S.n_nodes = n;
    return S;
}

template <int CHEMG, bool STDP, bool NET, class SRC>
__device__ __forceinline__ void gather_edges_wide(const StepParams &p, const SRC &src, uint32_t i, float v, float gap, int lft_me,
                                                  bool post_trig, int li, uint32_t ty0, EdgeAcc &A) {
    const uint32_t width = src.width();
    const bool pending = STDP && p.apply_pending;
    const bool do_e = p.electrical != 0;
    const int prev = (int)p.clock - 1;
    const uint32_t lane = src.lane;
    constexpr uint32_t HW = kWideWarps - 1;
    constexpr uint32_t kTerms = kWideChunk * 32u;
    constexpr uint32_t kTypes = CHEMG == 3 ? (uint32_t)kNT : (CHEMG == 1 ? 1u : 0u);
    const uint32_t n_chunks = (width + kWideChunk - 1u) / kWideChunk;
    const WideStage &SG = src.st;
    const bool staged = SG.n_nodes != 0u;   // CTA-uniform
    // ---- phase A (helper warps): the terms of chunk c into buffer c & 1 — kWideUnroll k-rows per thread: all col/weight loads,
    // then every gather they address (V, last_firing_time, t, the spike-train constants), then the arithmetic
    // split (two-pass mode): the chemical terms are parked already masked (`has ? term : 0`, the very operand the sum adds) and the
    // per-row edge counts of the chunk replace the per-term flag bytes, so the ordered sum is one load and one add per term
    auto phase_a_to = [&](uint32_t ci, unsigned char *buf, bool split) {
        float *sm_e = reinterpret_cast<float *>(buf);
        float *sm_t = sm_e + kTerms;
        uint8_t *sm_f = reinterpret_cast<uint8_t *>(sm_t + kTypes * kTerms);
        const uint32_t kk = ci * kWideChunk;
        const uint32_t kn = min(kWideChunk, width - kk);
        uint32_t lc[1 + kNT] = {0u, 0u, 0u, 0u};
        for (uint32_t kb = src.warp - 1u; kb < kn; kb += kWideUnroll * HW) {
            uint32_t c[kWideUnroll], j[kWideUnroll];
            float w[kWideUnroll];
            bool live[kWideUnroll], ok[kWideUnroll], train[kWideUnroll];
#pragma unroll
            for (int u = 0; u < kWideUnroll; ++u) {
                const uint32_t k = kb + (uint32_t)u * HW;
                live[u] = k < kn;
                c[u] = live[u] ? src.col(kk + k) : kColPad;
                w[u] = live[u] ? src.wgt(kk + k) : 0.f;
            }
            float vj[kWideUnroll], tj[kWideUnroll][CHEMG == 3 ? kNT : 1], tfv[kWideUnroll][4];
            int lj[kWideUnroll], lt[kWideUnroll];
#pragma unroll
            for (int u = 0; u < kWideUnroll; ++u) {
                ok[u] = c[u] != kColPad;
                j[u] = ok[u] ? (c[u] & kColIdxMask) : i;
                train[u] = NET && ok[u] && (c[u] & kColTrainBit);
                vj[u] = do_e ? (staged ? SG.v[j[u]] : p.v_in[j[u]]) : v;
                // see gather_edges: a spike train's last_firing_time of before its step-s iterate sits in the other buffer
                lj[u] = pending ? (staged ? (train[u] ? SG.lft_out[j[u]] : SG.lft_in[j[u]]) : (train[u] ? p.lft_out[j[u]] : p.lft_in[j[u]])) : -1;
                lt[u] = -1;
                if (NET) {
                    if (train[u] && do_e) {
                        const uint32_t tjx = j[u] - p.train0;
                        if (staged) {
                            // the train's term was evaluated once for the whole CTA (wide_stage_fill): tfv[0] carries it
                            lt[u] = SG.never[tjx] ? -1 : 0;
                            tfv[u][0] = SG.eff[tjx];
                        } else {
                            lt[u] = p.lft_in[j[u]];
                            tfv[u][0] = ldf(p.tf[TF_VREST], tjx); tfv[u][1] = ldf(p.tf[TF_K], tjx);
                            tfv[u][2] = ldf(p.tf[TF_VTH], tjx); tfv[u][3] = ldf(p.tf[TF_DT], tjx);
                        }
                    }
                }
                if (CHEMG == 1) {
                    tj[u][0] = staged ? SG.t[(size_t)ty0 * SG.n_nodes + j[u]] : src.gt0(j[u]);
                } else if (CHEMG == 3) {
                    const uint32_t m = ok[u] ? (c[u] >> kColNtShift) & 7u : 0u;
#pragma unroll
                    for (int ty = 0; ty < kNT; ++ty) tj[u][ty] = (m & (1u << ty)) ? (staged ? SG.t[(size_t)ty * SG.n_nodes + j[u]] : src.gt(j[u], ty)) : 0.f;
                }
            }
#pragma unroll
            for (int u = 0; u < kWideUnroll; ++u) {
                if (!live[u]) continue;
                const uint32_t k = kb + (uint32_t)u * HW;
                float wu = w[u];
                if (pending) {
                    bool pre_trig = ok[u] && lj[u] == prev;
                    if (NET) {
                        if (pre_trig) pre_trig = !train[u] && p.lat[lat_index(p, j[u] - p.own0)].do_plasticity != 0;
                    } else {
                        pre_trig = pre_trig && p.lat[0].do_plasticity != 0;
                    }
                    if ((post_trig && ok[u]) || pre_trig) {
                        const float d = stdp_delta(p.lat[li], lj[u], lft_me);
                        wu = wu + d;
                        if (post_trig && pre_trig) wu = wu + d;
                        *src.wgt_ptr(kk + k) = wu;
                    }
                }
                float final_input = gap * (vj[u] - v);  // gap_junction, neuron/mod.rs:54-60
                if (NET) {
                    if (train[u] && do_e) {
                        // spike_train_gap_junction, neuron/mod.rs:119-137
                        if (lt[u] < 0) final_input = tfv[u][0];
                        else if (staged) final_input = gap * tfv[u][0];
                        else final_input = gap * refract_effect(p.refract, tfv[u][1], p.clock, (uint32_t)lt[u], tfv[u][2], tfv[u][0], tfv[u][3]);
                    }
                }
                sm_e[k * 32u + lane] = final_input * wu;
                uint32_t f = ok[u] ? 1u : 0u;
                lc[0] += f;
                if (CHEMG == 1) {
                    const bool has = ok[u] && ((c[u] >> (kColNtShift + ty0)) & 1u);
                    const float term = tj[u][0] * wu;
                    sm_t[k * 32u + lane] = split ? (has ? term : 0.f) : term;
                    f |= has ? 2u : 0u;
                    lc[1] += has ? 1u : 0u;
                } else if (CHEMG == 3) {
                    const uint32_t m = ok[u] ? (c[u] >> kColNtShift) & 7u : 0u;
#pragma unroll
                    for (int ty = 0; ty < kNT; ++ty) {
                        const float term = tj[u][ty] * wu;
                        sm_t[((uint32_t)ty * kWideChunk + k) * 32u + lane] = split ? (((m >> ty) & 1u) ? term : 0.f) : term;
                        lc[1 + ty] += (m >> ty) & 1u;
                    }
                    f |= m << 1;
                }
                if (!split) sm_f[k * 32u + lane] = (uint8_t)f;
            }
        }
        if (split) {
            // per-row counts of the chunk: every helper thread adds its share into shared counters, the record takes the place of
            // the flag bytes (helpers only: named barrier 1 over the (kWideWarps - 1) * 32 helper threads)
            __shared__ uint32_t s_cnt[(1 + kNT) * 32];
            const uint32_t t = (src.warp - 1u) * 32u + lane;
            if (t < (1 + kNT) * 32u) s_cnt[t] = 0u;
            asm volatile("bar.sync 1, %0;" ::"n"((kWideWarps - 1) * 32) : "memory");
#pragma unroll
            for (int q = 0; q < 1 + kNT; ++q) if (lc[q]) atomicAdd(&s_cnt[q * 32 + lane], lc[q]);
            asm volatile("bar.sync 1, %0;" ::"n"((kWideWarps - 1) * 32) : "memory");
            if (t < (1 + kNT) * 32u) reinterpret_cast<uint32_t *>(sm_f)[t] = s_cnt[t];
        }
    };
    auto phase_a = [&](uint32_t ci, uint32_t bi) { phase_a_to(ci, src.sm + bi * wide_buf_bytes(CHEMG), false); };
    // ---- phase B (leader warp): add the parked terms of chunk c in ascending presynaptic order
    auto phase_b = [&](uint32_t ci, uint32_t bi) {
        const unsigned char *buf = src.sm + bi * wide_buf_bytes(CHEMG);
        const float *sm_e = reinterpret_cast<const float *>(buf);
        const float *sm_t = sm_e + kTerms;
        const uint8_t *sm_f = reinterpret_cast<const uint8_t *>(sm_t + kTypes * kTerms);
        const uint32_t kn = min(kWideChunk, width - ci * kWideChunk);
        // 4 k-rows per iteration (kn is a multiple of 4): their loads are issued together, the additions stay strictly ordered
        for (uint32_t k0b = 0; k0b < kn; k0b += 4u) {
            uint32_t f[4];
            float te[4], tt[4][CHEMG == 3 ? kNT : 1];
#pragma unroll
            for (uint32_t q = 0; q < 4u; ++q) {
                const uint32_t k = k0b + q;
                f[q] = sm_f[k * 32u + lane];
                te[q] = sm_e[k * 32u + lane];
                if (CHEMG == 1) tt[q][0] = sm_t[k * 32u + lane];
                if (CHEMG == 3) {
#pragma unroll
                    for (int ty = 0; ty < kNT; ++ty) tt[q][ty] = sm_t[((uint32_t)ty * kWideChunk + k) * 32u + lane];
                }
            }
#pragma unroll
            for (uint32_t q = 0; q < 4u; ++q) {
                if (do_e) A.acc_e = A.acc_e + te[q];
                if (CHEMG == 1) {
                    const bool has = (f[q] >> 1) & 1u;
                    A.acc_t[0] = A.acc_t[0] + (has ? tt[q][0] : 0.f);
                    A.cnt[0] += has ? 1u : 0u;
                } else if (CHEMG == 3) {
#pragma unroll
                    for (int ty = 0; ty < kNT; ++ty) {
                        const bool has = (f[q] >> (1 + ty)) & 1u;
                        A.acc_t[ty] = A.acc_t[ty] + (has ? tt[q][ty] : 0.f);
                        A.cnt[ty] += has ? 1u : 0u;
                    }
                }
                A.n_in += f[q] & 1u;
            }
        }
    };
    if (n_chunks == 0u) {   // uniform over the CTA: a slice without in-edges
        if (src.mode == 2u && src.chunk != 0u) A.skip = true;   // sum pass: one of the accumulator CTAs steps the neurons
        return;
    }
    const uint32_t warp_slice = (i - p.own0) >> 5;   // every lane of every warp of the CTA works on the same slice
    if (src.mode == 1u) {
        // terms pass: one chunk, parked in global memory (phase_a writes through generic pointers)
        if (src.chunk < n_chunks && src.warp != 0u) phase_a_to(src.chunk, src.scratch + ((size_t)warp_slice * src.chunks_cap + src.chunk) * wide_buf_bytes(CHEMG), true);
        return;
    }
    if (src.mode == 2u) {
        // sum pass: the helpers stream the parked chunks from L2 into the two shared-memory buffers (plain 16-byte copies, a few
        // instructions per k-row instead of ~180), the leader adds them in ascending presynaptic order
        // The sums of a slice are independent chains (electrical, one per neurotransmitter type): each gets its own CTA, which
        // streams only its array of every parked chunk (7.5 KB per chunk instead of 32 KB — one SM's latency-bound L2 stream was
        // the limit of a single summing CTA) and adds it in ascending presynaptic order.  The CTA that finishes last collects
        // the partial sums and steps the slice's neurons.
        constexpr uint32_t kAcc = 1u + kTypes;
        const uint32_t a = src.chunk;   // accumulator of this CTA (CTA-uniform)
        constexpr uint32_t kArr = kTerms * 4u;   // bytes of one array of a chunk
        static_assert(kArr % 16u == 0u && kArr / 16u <= (kWideWarps - 1) * 32u, "one 16-byte copy per helper thread and chunk");
        const uint32_t rec_off = (1u + kTypes) * kArr;   // count record of a chunk (phase_a_to, split)
        // shared memory: kWideSumBufs x (array + one 128-byte count row)
        constexpr uint32_t kSlot = kArr + 128u;
        auto fetch = [&](uint32_t ci) {
            const unsigned char *g = src.scratch + ((size_t)warp_slice * src.chunks_cap + ci) * wide_buf_bytes(CHEMG);
            const uint32_t d = (uint32_t)__cvta_generic_to_shared(src.sm + (ci % kWideSumBufs) * kSlot);
            const uint32_t t = (src.warp - 1u) * 32u + lane;
            if (t < kArr / 16u) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d + t * 16u), "l"(g + (size_t)a * kArr + (size_t)t * 16u) : "memory");
            if (t < 8u) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d + kArr + t * 16u), "l"(g + rec_off + (size_t)a * 128u + (size_t)t * 16u) : "memory");
        };
        auto commit = [&]() { asm volatile("cp.async.commit_group;" ::: "memory"); };
        float part = 0.f;
        uint32_t pcnt = 0u;
        auto sum_chunk = [&](uint32_t ci) {
            const float *arr = reinterpret_cast<const float *>(src.sm + (ci % kWideSumBufs) * kSlot);
            const uint32_t kn = min(kWideChunk, width - ci * kWideChunk);
            for (uint32_t k0b = 0; k0b < kn; k0b += 12u) {   // kn is a multiple of 4
                float te[12];
#pragma unroll
                for (uint32_t q = 0; q < 12u; ++q) te[q] = arr[min(k0b + q, kn - 1u) * 32u + lane];
#pragma unroll
                for (uint32_t q = 0; q < 12u; ++q) if (k0b + q < kn) part = part + te[q];
            }
            pcnt += reinterpret_cast<const uint32_t *>(arr + kTerms)[lane];
        };
        static_assert(kWideSumBufs * kSlot <= 2u * wide_buf_bytes(CHEMG) || true, "");
        if (src.warp != 0u) {
            for (uint32_t c = 0; c + 1u < kWideSumBufs; ++c) { if (c < n_chunks) fetch(c); commit(); }
            asm volatile("cp.async.wait_group %0;" ::"n"(kWideSumBufs - 2) : "memory");   // chunk 0 has landed
        }
        __syncthreads();
        for (uint32_t c = 0; c < n_chunks; ++c) {
            if (src.warp == 0u) {
                sum_chunk(c);
            } else {
                if (c + kWideSumBufs - 1u < n_chunks) fetch(c + kWideSumBufs - 1u);   // into the buffer the leader finished before the last barrier
                commit();
                asm volatile("cp.async.wait_group %0;" ::"n"(kWideSumBufs - 2) : "memory");   // chunk c + 1 has landed
            }
            __syncthreads();
        }
        if (src.warp != 0u) return;
        // publish the partial sum; the last CTA of the slice gathers all of them
        unsigned char *pb = src.scratch + (size_t)src.n_slices * src.chunks_cap * wide_buf_bytes(CHEMG) + (size_t)warp_slice * wide_part_bytes_per_slice();
        float *psum = reinterpret_cast<float *>(pb);
        uint32_t *pcn = reinterpret_cast<uint32_t *>(pb + (1 + kNT) * 32u * 4u);
        unsigned int *arrive = reinterpret_cast<unsigned int *>(pb + (1 + kNT) * 32u * 8u);
        __stcg(psum + a * 32u + lane, part);
        __stcg(pcn + a * 32u + lane, pcnt);
        __threadfence();
        __syncwarp();
        unsigned int old = 0u;
        if (lane == 0) old = atomicAdd(arrive, 1u);
        old = __shfl_sync(0xffffffffu, old, 0);
        if (old + 1u != kAcc) { A.skip = true; return; }
        if (lane == 0) *arrive = 0u;   // ready for the next timestep (the next launch is stream-ordered after this kernel)
        __threadfence();
        A.acc_e = __ldcg(psum + lane);
        A.n_in = __ldcg(pcn + lane);
        if (CHEMG == 1) { A.acc_t[0] = __ldcg(psum + 32u + lane); A.cnt[0] = __ldcg(pcn + 32u + lane); }
        if (CHEMG == 3) {
#pragma unroll
            for (int ty = 0; ty < kNT; ++ty) { A.acc_t[ty] = __ldcg(psum + (1u + (uint32_t)ty) * 32u + lane); A.cnt[ty] = __ldcg(pcn + (1u + (uint32_t)ty) * 32u + lane); }
        }
        return;
    }
    // software pipeline over the chunks: while the leader adds chunk c, the helpers already compute chunk c + 1
    if (src.warp != 0u) phase_a(0u, 0u);
    __syncthreads();
    for (uint32_t c = 0; c < n_chunks; ++c) {
        if (src.warp == 0u) phase_b(c, c & 1u);
        else if (c + 1u < n_chunks) phase_a(c + 1u, (c + 1u) & 1u);
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------
// one neuron, one timestep
// ------------------------------------------------------------------------------------------------
// warp_global: slice index (neuron-local word index of the spike bitmask); ln: local neuron number; lnc: clamped copy
// used for addressing by invalid lanes of the last warp.
template <int MODEL, int CHEMG, bool NTREL, bool STDP, bool NET, class SRC>
__device__ __forceinline__ void neuron_step(const StepParams &p, const SRC &src, uint32_t warp_global, uint32_t lane,
                                            uint32_t ln, uint32_t lnc, bool valid, bool export_lo, bool export_hi) {
    const uint32_t i = p.own0 + lnc;
    // row strips: does any lane of this warp export to a neighbour (warp-uniform)?  Interior warps — all but a few dozen of a
    // strip's tiles — skip every export test: the window kernel is co-limited by its instruction stream, and ~35 extra
    // instructions per warp and tile on the common path cost 5 % of the step (measured on 2 GPUs, tools/diag_halo.py)
    const bool part = __any_sync(0xffffffffu, export_lo | export_hi);
    // ---- own state and parameters ------------------------------------------------------------------
    float v = src.v();
    const float gap = src.template f<F_GAP>();
    const float dt = src.template f<F_DT>();
    constexpr bool BCM = MODEL == SNN_MODEL_BCM_IZHIKEVICH;
    constexpr bool NEEDS_CM = NTREL || BCM || MODEL == SNN_MODEL_HODGKIN_HUXLEY || MODEL == SNN_MODEL_IZHIKEVICH ||
                              MODEL == SNN_MODEL_LEAKY_IZHIKEVICH || MODEL == SNN_MODEL_ADAPTIVE_LEAKY_INTEGRATE_AND_FIRE ||
                              MODEL == SNN_MODEL_ADAPTIVE_EXP_LEAKY_INTEGRATE_AND_FIRE;
    float c_m = 1.f, v_th = 0.f;
    if (SRC::kEarlyLoads) { if constexpr (NEEDS_CM) c_m = src.template f<F_CM>(); v_th = src.template f<F_VTH>(); }
    const int lft_me = (STDP || p.lft_pp) ? src.lft() : 0;
    const uint32_t spk_word_in = (NTREL || BCM) ? src.spk_prev_word(warp_global) : 0u;
    // Hodgkin-Huxley: the "was increasing" word of this warp is the one global load on the consumers' path of the staged kernels.
    // Issued here, its latency overlaps the gather; next to its use (after stores it might alias) every warp sat out a full
    // memory round trip per tile (30 % of the stall samples, profiles/r1_step_win_hh_full.txt)
    uint32_t wi_word_early = 0u;
    if constexpr (MODEL == SNN_MODEL_HODGKIN_HUXLEY) wi_word_early = p.was_inc[warp_global];
    const bool spiking_prev = (spk_word_in >> lane) & 1u;
    const uint32_t flags = NTREL ? src.flags() : 0u;
    constexpr bool IZH = MODEL == SNN_MODEL_IZHIKEVICH || MODEL == SNN_MODEL_LEAKY_IZHIKEVICH || BCM;
    constexpr bool IF4 = MODEL == SNN_MODEL_LEAKY_INTEGRATE_AND_FIRE || MODEL == SNN_MODEL_QUADRATIC_INTEGRATE_AND_FIRE ||
                         MODEL == SNN_MODEL_ADAPTIVE_LEAKY_INTEGRATE_AND_FIRE || MODEL == SNN_MODEL_ADAPTIVE_EXP_LEAKY_INTEGRATE_AND_FIRE;
    constexpr bool ADAPT = MODEL == SNN_MODEL_ADAPTIVE_LEAKY_INTEGRATE_AND_FIRE || MODEL == SNN_MODEL_ADAPTIVE_EXP_LEAKY_INTEGRATE_AND_FIRE;
    constexpr bool LEAKY = MODEL == SNN_MODEL_LEAKY_INTEGRATE_AND_FIRE || ADAPT;
    // model parameters (only the ones this model reads are loaded; the rest fold away).  With HBM-sourced operands the
    // loads are issued before the edge loop (latency overlap); with shared-memory operands they are deferred until
    // after it (they are cheap, and not holding them across the loop saves ~15 registers = one more resident CTA).
    float w_adapt = 0.f, pa = 0.f, pb = 0.f, pc = 0.f, pd = 0.f, tau_m = 1.f, e_l = 0.f, v_reset = 0.f, integ = 0.f, refr = 0.f,
          tref = 0.f, g_l = 1.f, leak = 0.f, alpha = 0.f, beta = 0.f;
    auto load_model_params = [&]() {
        if constexpr (IZH || ADAPT) w_adapt = src.template state<F_W>();
        if constexpr (IZH) { pa = src.template f<F_A>(); pb = src.template f<F_B>(); pc = src.template f<F_C>(); pd = src.template f<F_D>(); }
        if constexpr (IZH || IF4) tau_m = src.template f<F_TAUM>();
        if constexpr (LEAKY || MODEL == SNN_MODEL_LEAKY_IZHIKEVICH) e_l = src.template f<F_EL>();
        if constexpr (IF4 || MODEL == SNN_MODEL_SIMPLE_LEAKY_INTEGRATE_AND_FIRE) v_reset = src.template f<F_VRESET>();
        if constexpr (IF4) { integ = src.template f<F_INTEG>(); refr = src.template state<F_REFR>(); tref = src.template f<F_TREF>(); }
        if constexpr (LEAKY) { g_l = src.template f<F_GL>(); leak = src.template f<F_LEAK>(); }
        if constexpr (ADAPT || MODEL == SNN_MODEL_QUADRATIC_INTEGRATE_AND_FIRE) alpha = src.template f<F_ALPHA>();
        if constexpr (ADAPT) beta = src.template f<F_BETA>();
    };
    if (SRC::kEarlyLoads) load_model_params();

    // the single neurotransmitter type of the CHEMG == 1 fast path
    const uint32_t ty0 = (CHEMG == 1) ? (uint32_t)(__ffs((int)p.nt_used) - 1) : 0u;

    int li = 0;
    bool post_trig = false;
    if (STDP) {
        li = NET ? lat_index(p, lnc) : 0;
        post_trig = p.apply_pending && p.lat[li].do_plasticity && lft_me == (int)p.clock - 1;
    }

    // ---- gather over in-edges (ascending presynaptic index = canonical summation order) ----------
    EdgeAcc A;
    A.acc_e = 0.f; A.n_in = 0;
#pragma unroll
    for (int ty = 0; ty < kNT; ++ty) { A.acc_t[ty] = 0.f; A.cnt[ty] = 0; }
    const bool do_e = p.electrical != 0;
    const bool do_c = NTREL && p.chemical != 0;
    A.fast8 = false; A.fast8t = false; A.skip = false;
    if constexpr (SRC::kWidth == 8 && !NET) gather_edges8<CHEMG, STDP>(p, src, i, v, gap, lft_me, post_trig, li, ty0, A);
    else if constexpr (SRC::kWide) gather_edges_wide<CHEMG, STDP, NET>(p, src, i, v, gap, lft_me, post_trig, li, ty0, A);
    else gather_edges<CHEMG, STDP, NET>(p, src, i, v, gap, lft_me, post_trig, li, ty0, A);
    if constexpr (SRC::kWide) {
        // the helpers of a wide slice, the CTAs of the terms pass and all but the last accumulator CTA of the sum pass are done;
        // the leader warp steps the 32 neurons
        if (src.warp != 0 || src.mode == 1u || A.skip) return;
    }
    if (!SRC::kEarlyLoads) { load_model_params(); if constexpr (NEEDS_CM) c_m = src.template f<F_CM>(); v_th = src.template f<F_VTH>(); }
    // neuron/mod.rs:722-729: divide by the number of incoming edges (1 if none)
    // (x / 8 == x * 0.125 exactly, subnormals included: both round the same real number)
    float input = 0.f;
    if (do_e) input = A.fast8 ? A.acc_e * 0.125f : A.acc_e / (A.n_in == 0 ? 1.f : (float)A.n_in);

    // ---- receptors (iterate_with_neurotransmitter_and_spike: kinetics then currents from pre-update V)
    float rc_total = 0.f;
    if (NTREL) {
        const uint32_t rcm = flags >> 4;
        if (do_c) {
#pragma unroll
            for (int ty = 0; ty < kNT; ++ty) {
                if (!(p.rc_used & (1u << ty))) continue;
                if (!(rcm & (1u << ty))) continue;
                float r = src.rc_state(RCF_R, ty);
                const uint32_t cnt = (CHEMG == 1) ? (ty == (int)ty0 ? A.cnt[0] : 0u) : A.cnt[ty];
                if (cnt > 0) {
                    const float acc = (CHEMG == 1) ? A.acc_t[0] : A.acc_t[ty];
                    const float tin = ((CHEMG == 1 && A.fast8) || (CHEMG == 3 && A.fast8t)) ? acc * 0.125f : acc / (float)cnt;
                    float k1 = 0.f, k2 = 0.f;
                    if (p.rck != SNN_RC_APPROXIMATE) { k1 = src.rc(RCF_K1, ty); k2 = src.rc(RCF_K2, ty); }
                    r = rc_apply(p.rck, r, k1, k2, tin, dt);
                    if (valid) p.rc[RCF_R][(size_t)ty * p.rc_stride + lnc] = r;
                }
                const float mg = (ty == SNN_NT_NMDA) ? src.rc(RCF_MG, ty) : 0.f;
                rc_total += receptor_current(ty, src.rc(RCF_G, ty), src.rc(RCF_E, ty), mg, r, v);
            }
        } else if (MODEL == SNN_MODEL_HODGKIN_HUXLEY) {
            // hodgkin_huxley/mod.rs:161-164: the electrical-only path still subtracts the stored ligand currents
#pragma unroll
            for (int ty = 0; ty < kNT; ++ty)
                if ((p.rc_used & (1u << ty)) && (rcm & (1u << ty))) rc_total += p.rc[RCF_CUR][(size_t)ty * p.rc_stride + lnc];
        }
    }
    const float rc_dv = rc_total * (dt / c_m);  // Ionotropic::get_receptor_currents, iterate_and_spike/mod.rs:1286-1304

    // ---- neuron update --------------------------------------------------------------------------
    bool spike = false;
    float v_release;  // membrane voltage seen by the neurotransmitter kinetics (post-update, pre-reset)
    if constexpr (BCM) {
        // BCMIzhikevichNeuron activity bookkeeping, integrate_and_fire/mod.rs:1458-1467 / :1485-1494: runs before the
        // Izhikevich update and sees the spike flag of the previous step.  The two iterate variants of the reference
        // normalise current_activity differently (window * dt vs window); both are restated literally.
        uint32_t num_spikes = __float_as_uint(src.template state<F_NSPK>());
        if (spiking_prev) num_spikes += 1u;
        float fr_clock = src.template state<F_FRCLK>() + dt;
        const float fr_window = src.template f<F_FRWIN>();
        if (fr_clock >= fr_window) {
            fr_clock = 0.f;
            const float current_activity = p.chemical ? (float)num_spikes / fr_window : (float)num_spikes / (fr_window * dt);
            const float period = (float)__float_as_uint(src.template f<F_PERIOD>());
            float average_activity = src.template state<F_AVG_ACT>();
            average_activity = average_activity - average_activity / period;
            average_activity = average_activity + current_activity / period;
            if (valid) { p.f[F_CUR_ACT][lnc] = current_activity; p.f[F_AVG_ACT][lnc] = average_activity; }
        }
        if (valid) { p.f[F_NSPK][lnc] = __uint_as_float(num_spikes); p.f[F_FRCLK][lnc] = fr_clock; }
    }
    if constexpr (IZH) {
        float dv;
        if constexpr (MODEL != SNN_MODEL_LEAKY_IZHIKEVICH)  // integrate_and_fire/mod.rs:1255-1260 (also :1446-1451, BCM)
            dv = (((((0.04f * (v * v)) + (5.f * v)) + 140.f) - w_adapt) + input) * (dt / c_m);
        else                                            // :1342-1348
            dv = (((((0.04f * (v * v)) + (5.f * v)) + 140.f) - (w_adapt * (v - e_l))) + input) * (dt / c_m);
        const float dw = (pa * (pb * v - w_adapt)) * (dt / tau_m);  // :1225-1231
        if (do_c) v += dv + (-rc_dv); else v += dv;               // :226, :246
        w_adapt += dw;
        v_release = v;
        if (v >= v_th) {                                            // izhikevich_handle_spiking :1235-1247
            spike = true;
            v = pc;
            w_adapt += pd;
        }
        if (valid) p.f[F_W][lnc] = w_adapt;
    } else if constexpr (IF4) {
        float dw = 0.f, dv;
        if constexpr (MODEL == SNN_MODEL_LEAKY_INTEGRATE_AND_FIRE) {  // :176-181
            dv = ((leak * (v - e_l)) + (integ * (input / g_l))) * (dt / tau_m);
        } else if constexpr (MODEL == SNN_MODEL_QUADRATIC_INTEGRATE_AND_FIRE) {  // :324-327
            dv = (((alpha * (v - v_reset)) * (v - src.template f<F_VC>())) + integ * input) * (dt / tau_m);
        } else {
            if constexpr (MODEL == SNN_MODEL_ADAPTIVE_LEAKY_INTEGRATE_AND_FIRE)  // :1035-1041
                dv = (((leak * (v - e_l)) + (integ * (input / g_l))) - (w_adapt / g_l)) * (dt / c_m);
            else {                                                                  // :1138-1145
                const float sf = src.template f<F_SLOPE>();
                dv = ((((leak * (v - e_l)) + (sf * expf((v - v_th) / sf))) + (integ * (input / g_l))) - (w_adapt / g_l)) * (dt / c_m);
            }
            dw = (alpha * (v - e_l) - w_adapt) * (dt / tau_m);  // :1002-1009
        }
        if (do_c) v += dv + (-rc_dv); else v += dv;
        if (ADAPT) w_adapt += dw;
        v_release = v;
        // impl_default_handle_spiking :87-102 / adaptive_handle_spiking :1013-1029
        if (refr > 0.f) {
            v = v_reset;
            refr -= 1.f;
        } else if (v >= v_th) {
            spike = true;
            v = v_reset;
            if (ADAPT) w_adapt += beta;
            refr = tref / dt;
        }
        if (valid) {
            p.f[F_REFR][lnc] = refr;
            if (ADAPT) p.f[F_W][lnc] = w_adapt;
        }
    } else if constexpr (MODEL == SNN_MODEL_SIMPLE_LEAKY_INTEGRATE_AND_FIRE) {
        const float dv = (src.template f<F_G>() * (v - src.template f<F_E>()) + input) * dt;  // :1592-1594
        if (do_c) v += dv + (-rc_dv); else v += dv;
        v_release = v;
        if (v >= v_th) { spike = true; v = v_reset; }  // :1579-1590
    } else {  // Hodgkin-Huxley, hodgkin_huxley/mod.rs:156-241; ion_channels/mod.rs:40-44, 219-235, 268-281, 310-312
        const float last_voltage = v;
        float m = src.template state<F_M>(), h = src.template state<F_H>(), n = src.template state<F_N>();
        const float m_alpha = 0.1f * ((v + 40.f) / (1.f - expf(-(v + 40.f) / 10.f)));
        const float m_beta = 4.f * expf(-(v + 65.f) / 18.f);
        const float h_alpha = 0.07f * expf(-(v + 65.f) / 20.f);
        const float h_beta = 1.f / (expf(-(v + 35.f) / 10.f) + 1.f);
        m += dt * (m_alpha * (1.f - m) - m_beta * m);
        h += dt * (h_alpha * (1.f - h) - h_beta * h);
        const float i_na = ((pow3f(m) * h) * src.template f<F_GNA>()) * (v - src.template f<F_ENA>());
        const float n_alpha = (0.01f * (v + 55.f)) / (1.f - expf(-(v + 55.f) / 10.f));
        const float n_beta = 0.125f * expf(-(v + 65.f) / 80.f);
        n += dt * (n_alpha * (1.f - n) - n_beta * n);
        const float i_k = (pow4f(n) * src.template f<F_GK>()) * (v - src.template f<F_EK>());
        const float i_kl = src.template f<F_GKL>() * (v - src.template f<F_EKL>());
        const float i_sum = input - ((i_na + i_k) + i_kl);
        v += (dt * i_sum) / c_m - rc_dv;
        v_release = v;
        const bool was_increasing = (wi_word_early >> lane) & 1u;
        const bool increasing_right_now = last_voltage < v;
        spike = (v > v_th) && was_increasing && !increasing_right_now;
        const uint32_t wi_new = __ballot_sync(0xffffffffu, increasing_right_now && valid);
        if (lane == 0) p.was_inc[warp_global] = wi_new;
        if (valid) { p.f[F_M][lnc] = m; p.f[F_H][lnc] = h; p.f[F_N][lnc] = n; }
    }

    // ---- neurotransmitter release: post-update voltage, previous step's spike flag
    //      (intermediate_delegate/mod.rs:18-24, integrate_and_fire/mod.rs:229)
    if (NTREL) {
        const uint32_t ntm = flags & 0xFu;
#pragma unroll
        for (int ty = 0; ty < kNT; ++ty) {
            if (!(p.nt_used & (1u << ty))) continue;
            if (!(ntm & (1u << ty))) continue;
            const float t_old = src.t_own(ty);
            float p1 = 0.f, p2 = 0.f;
            if (p.ntk != SNN_NT_DISCRETE_SPIKE) p1 = src.nt(NTF_P1, ty);
            if (p.ntk == SNN_NT_DESTEXHE) p2 = src.nt(NTF_P2, ty);
            const float t_new = nt_apply(p.ntk, t_old, src.nt(NTF_TMAX, ty), p1, p2, v_release, spiking_prev, dt);
            if (valid) {
                p.t_out[(size_t)ty * p.t_stride + i] = t_new;
                if (part) {   // uniform: one branch instead of two predicated address computations on single-GPU handles
                    if (export_lo) p.halo[0].peer_t[p.out_par][(size_t)ty * p.halo[0].peer_t_stride + p.halo[0].peer_node0 + (ln - p.halo[0].first)] = t_new;
                    if (export_hi) p.halo[1].peer_t[p.out_par][(size_t)ty * p.halo[1].peer_t_stride + p.halo[1].peer_node0 + (ln - p.halo[1].first)] = t_new;
                }
            }
        }
    }

    // ---- spike compaction: one bit per neuron, one word per warp --------------------------------
    const uint32_t spk_word = __ballot_sync(0xffffffffu, spike && valid);
    if (lane == 0) {
        p.spk_out[(p.own0 >> 5) + warp_global] = spk_word;
        if (p.spike_hist) p.spike_hist[warp_global] = spk_word;
    }
    if (valid) {
        p.v_out[i] = v;
        // set_last_firing_time(Some(internal_clock)), neuron/mod.rs:964-966
        int lft_new = lft_me;
        if (p.lft_pp) { lft_new = spike ? (int)p.clock : lft_me; p.lft_out[i] = lft_new; }
        else if (spike) { lft_new = (int)p.clock; p.lft_out[i] = lft_new; }
        if (p.grid_hist) p.grid_hist[ln] = v;  // GridVoltageHistory::update, neuron/mod.rs:293-296
        if (part && export_lo) {
            const HaloDir &H = p.halo[0];
            const uint32_t dst = H.peer_node0 + (ln - H.first);
            H.peer_v[p.out_par][dst] = v;
            if (p.lft_pp) H.peer_lft[p.out_par][dst] = lft_new;
            if constexpr (BCM) bcm_halo_act(p, 0, p.out_par)[dst] = p.f[F_CUR_ACT][lnc];   // read by the neighbour's BCM edge kernel
        }
        if (part && export_hi) {
            const HaloDir &H = p.halo[1];
            const uint32_t dst = H.peer_node0 + (ln - H.first);
            H.peer_v[p.out_par][dst] = v;
            if (p.lft_pp) H.peer_lft[p.out_par][dst] = lft_new;
            if constexpr (BCM) bcm_halo_act(p, 1, p.out_par)[dst] = p.f[F_CUR_ACT][lnc];
        }
    }
}

// ---- multi-GPU: does this warp's slice touch a halo?  If so wait for the neighbour's previous step first.
__device__ __forceinline__ void halo_import(const StepParams &p, uint32_t warp_global, uint32_t lane, uint32_t ln, bool valid,
                                            bool &export_lo, bool &export_hi) {
    export_lo = export_hi = false;
    if (!(p.halo[0].active | p.halo[1].active)) return;
    const uint32_t w0 = warp_global * 32u, w1 = min(w0 + 32u, p.n_neurons);
    const bool near_lo = p.halo[0].active && w0 < p.halo[0].first + p.halo[0].count;
    const bool near_hi = p.halo[1].active && w1 > p.halo[1].first;
    if (near_lo) {
        if (lane == 0) halo_wait(p.halo[0].my_flag, p.halo_epoch, p.halo_done + 2, p.halo_timeout_ns);
        __syncwarp();
    }
    if (near_hi) {
        if (lane == 0) halo_wait(p.halo[1].my_flag, p.halo_epoch, p.halo_done + 2, p.halo_timeout_ns);
        __syncwarp();
    }
    export_lo = near_lo && valid && ln >= p.halo[0].first && ln < p.halo[0].first + p.halo[0].count;
    export_hi = near_hi && valid && ln >= p.halo[1].first && ln < p.halo[1].first + p.halo[1].count;
}

// ---- multi-GPU, window kernel: ghosts arrive through the producer's TMA copies (it does the waiting), consumers only
// need to know which of their neurons are exported
__device__ __forceinline__ void halo_export_flags(const StepParams &p, uint32_t ln, bool valid, bool &export_lo, bool &export_hi) {
    export_lo = export_hi = false;
    if (!(p.halo[0].active | p.halo[1].active)) return;
    export_lo = p.halo[0].active && valid && ln >= p.halo[0].first && ln < p.halo[0].first + p.halo[0].count;
    export_hi = p.halo[1].active && valid && ln >= p.halo[1].first && ln < p.halo[1].first + p.halo[1].count;
}

// ---- multi-GPU: publish "my boundary values of this step have landed" to each neighbour.  Every exporting warp
// fences its remote stores, then bumps a local counter; the last one raises the neighbour's arrival flag.
__device__ __forceinline__ void halo_publish(const StepParams &p, uint32_t warp_global, uint32_t lane) {
    if (!(p.halo[0].active | p.halo[1].active)) return;
    const uint32_t w0 = warp_global * 32u, w1 = min(w0 + 32u, p.n_neurons);
#pragma unroll
    for (int d = 0; d < 2; ++d) {
        const HaloDir &H = p.halo[d];
        if (!H.active) continue;
        const bool mine = w0 < H.first + H.count && w1 > H.first;
        if (!mine) continue;
        __syncwarp();
        if (lane == 0) {
            __threadfence_system();
            const uint32_t first_w = H.first >> 5, last_w = (H.first + H.count - 1) >> 5;
            const uint32_t n_warps = last_w - first_w + 1;
            const unsigned int done = atomicAdd(&p.halo_done[d], 1u) + 1u;
            if (done == n_warps) {
                p.halo_done[d] = 0u;
                __threadfence_system();
                st_release_sys(H.peer_flag, p.halo_epoch + 1ull);
            }
        }
    }
}

}  // namespace snn
