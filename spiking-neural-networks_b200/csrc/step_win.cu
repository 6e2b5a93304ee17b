// step_win.cu — the step kernel for 8-neighbour (radius-1) stencil lattices: one persistent CTA per SM, every operand
// staged by TMA, including the neighbour rows.
//
// Why: the L1-gather kernels (kernels.cu, step_tma.cu) spend their time on ~24 dependent neighbour gathers per neuron
// and on ~870 issued instructions per 32 neurons (ncu, profiles/r1_step_tma_full.txt: 53 % issue slots, 32 % of stall
// samples on the long scoreboard, 40 % of DRAM peak).  For a row-major lattice the presynaptic neurons of a tile of
// 256 consecutive neurons lie in three contiguous index ranges of the node arrays (the tile's own range and the same
// range one row up / one row down, each widened by one neuron), so here the producer lane copies those three windows
// of V, last_firing_time and t with TMA bulk copies next to the tile's own parameters and col/weight rows.  Consumer
// warps then run the shared neuron_step (step_body.cuh — same arithmetic, bit-identical results) on shared memory
// only: no global load is left on their critical path, operand offsets are compile-time immediates (WinLayout,
// common.h), and HBM latency is hidden by the depth of the stage ring instead of by warp occupancy.
//
// CTA = G groups of 8 consumer warps + kWinProducers producer warps; tile n of the CTA goes to group n % G and stage n % S.
// The col words are read and used (the window is selected by comparing the presynaptic index against the tile's bounds),
// so any per-edge weight / type content of the sliced-ELL table keeps working; only the index pattern must be the
// radius-1 stencil that set_graph_grid generates.  When tile_params_kernel has found every col word of every tile equal
// to stencil_cols (STEN), the col words are not staged at all: full warps derive their neighbours from their own index,
// border warps compute the words with stencil_cols, and both run the same arithmetic on them as the kernel that reads them.
#include <type_traits>

#include "step_body.cuh"
#include "tma_util.cuh"

namespace snn {

// shared-memory loads with a compile-time immediate offset.  `volatile` keeps them between the mbarrier wait and the
// mbarrier arrive of their stage (both volatile asm); ptxas still schedules them freely inside that span.
template <uint32_t OFF> __device__ __forceinline__ float lds_f32(uint32_t addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1+%2];" : "=f"(v) : "r"(addr), "n"(OFF));
    return v;
}
template <uint32_t OFF> __device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1+%2];" : "=r"(v) : "r"(addr), "n"(OFF));
    return v;
}
template <uint32_t OFF> __device__ __forceinline__ uint32_t lds_u8(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1+%2];" : "=r"(v) : "r"(addr), "n"(OFF));
    return v;
}
__device__ __forceinline__ float lds_f32_rt(uint32_t addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}

// UNI: every neuron of the tile has the parameters of its first one (WinLayout::o_row): f<>(), nt() and rc() read that row
// ROWS: the stage has a row (win_layout(..., rows = true))
// STEN: every tile is a stencil tile (kTileStencil): no col words in the stage (gather_edges8 asks stencil_full() instead)
template <int MODEL, int CHEMG, bool NTREL, bool STDP, bool ROWS, bool UNI, bool STEN>
struct WinSrc {
    static constexpr bool kEarlyLoads = false;   // operands sit in shared memory: read them where they are used
    static constexpr bool kCheapEdges = false;
    static constexpr bool kWide = false;
    static constexpr bool kStencil = STEN;
    static_assert(!STEN || ROWS, "the full-warp mask of a stencil tile is in its tile row");
    static constexpr uint32_t kWidth = kWinWidth;
    static __host__ __device__ constexpr WinLayout lay() { return win_layout(MODEL, CHEMG, NTREL, STDP, ROWS, STEN); }

    const StepParams &p;
    const WinParams &wp;
    uint32_t me;                // shared address of this stage + 4 * (neuron within the tile): per-neuron operand rows
    uint32_t own;               // shared address of this neuron inside a (row-relative) window row
    uint32_t edge;              // shared address of this lane's first col word relative to o_col (weights: + o_wgt - o_col)
    uint32_t lo_thr, hi_thr;    // presynaptic node index < lo_thr: upper window, > hi_thr: lower window
    uint32_t d0, d1, d2;        // shared address of V[node 0] as seen through the upper / middle / lower window (mod 2^32)
    uint32_t k0g, lane;         // first k-row of this warp's slice in the global edge arrays
    uint32_t tid;               // neuron within the tile
    uint32_t row;               // shared address of this stage's tile row

    template <int SLOT> __device__ __forceinline__ float f() const {
        static_assert(win_field_param(MODEL, NTREL, SLOT), "not a parameter of this model (win_field_read, win_field_state)");
        if constexpr (UNI) return lds_f32<lay().r_f[SLOT] * 4u>(row);
        else return lds_f32<lay().o_f[SLOT]>(me);
    }
    template <int SLOT> __device__ __forceinline__ float state() const {
        static_assert(win_field_read(MODEL, NTREL, SLOT) && win_field_state(SLOT), "not a state field of this model (win_field_state)");
        return lds_f32<lay().o_f[SLOT]>(me);
    }
    __device__ __forceinline__ float v() const { return lds_f32<lay().o_vwin + kWinRowBytes>(own); }
    __device__ __forceinline__ int lft() const {
        return (int)lds_u32<lay().o_lwin + (lay().lrows == 3 ? kWinRowBytes : 0u)>(own);
    }
    // flags: one byte per neuron; `me` advances 4 bytes per neuron, the byte row needs 1
    __device__ __forceinline__ uint32_t flags() const { return lds_u8<lay().o_flags>(me - 3u * tid); }
    // one word per warp, used late (neurotransmitter release): a plain read-only load, issued early by the compiler
    __device__ __forceinline__ uint32_t spk_prev_word(uint32_t warp_global) const { return __ldg(p.spk_in + (p.own0 >> 5) + warp_global); }
    __device__ __forceinline__ float t_own(int ty) const {
        constexpr uint32_t o = lay().o_twin, tr = lay().trows;
        const uint32_t q = (CHEMG == 1) ? 0u : (uint32_t)ty;
        return lds_f32_rt(own + o + (q * tr + (tr == 3 ? 1u : 0u)) * kWinRowBytes);
    }
    // slot and ty are constants after neuron_step's loops unroll: the row offsets fold into the loads
    __device__ __forceinline__ float nt(int slot, int ty) const {
        if constexpr (UNI) return lds_f32_rt(row + (lay().r_nt + (uint32_t)(slot * kNT + ty)) * 4u);
        else return lds_f32_rt(me + wp.o_nt[slot][ty]);
    }
    __device__ __forceinline__ float rc(int slot, int ty) const {
        if constexpr (UNI) return lds_f32_rt(row + (lay().r_rc + (uint32_t)((slot - RCF_K1) * kNT + ty)) * 4u);
        else return lds_f32_rt(me + wp.o_rc[slot][ty]);
    }
    __device__ __forceinline__ float rc_state(int slot, int ty) const { return lds_f32_rt(me + wp.o_rc[slot][ty]); }
    __device__ __forceinline__ uint32_t width() const { return kWinWidth; }
    __device__ __forceinline__ uint32_t col(uint32_t kk) const {
        static_assert(!STEN, "a stencil stage has no col words");
        return lds_u32<lay().o_col>(edge + kk * 128u);
    }
    // STEN: this warp is full (warp-uniform; from the tile row), the lattice-wide release mask, the node index offset of slot u
    // of a full row, and the col words of this lane (border warps)
    __device__ __forceinline__ bool stencil_full() const { return (lds_u32<0>(row) >> (kTileFullShift + (tid >> 5))) & 1u; }
    __device__ __forceinline__ uint32_t stencil_nt() const { return wp.stencil_nt; }
    __device__ __forceinline__ uint32_t stencil_off(int u) const {
        return u < 3 ? (uint32_t)(u - 1) - wp.cols : (u < 5 ? (uint32_t)(2 * u - 7) : wp.cols + (uint32_t)(u - 6));
    }
    __device__ __forceinline__ void stencil_cols(uint32_t (&c)[8]) const {
        snn::stencil_cols(k0g * 4u + lane, p.n_neurons, wp.cols, wp.row0_global, wp.rows_global, p.own0, wp.stencil_nt, c);
    }
    __device__ __forceinline__ float wgt(uint32_t kk) const { return lds_f32<lay().o_wgt>(edge + kk * 128u); }
    __device__ __forceinline__ float *wgt_ptr(uint32_t kk) const { return p.wgt + (size_t)(k0g + kk) * 32u + lane; }
    // STDP: the new weight goes to the stage (this step's gather reads it from there) and to HBM
    __device__ __forceinline__ void wgt_update(uint32_t kk, float x) const {
        asm volatile("st.shared.f32 [%0+%1], %2;" ::"r"(edge + kk * 128u), "n"(lay().o_wgt), "f"(x) : "memory");
        *wgt_ptr(kk) = x;
    }
    // generic-proxy stores into a stage that TMA (async proxy) overwrites after the empty barrier
    __device__ __forceinline__ void wgt_updates_done() const { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

    // neighbour gathers: the handle is the shared address of V[j] inside whichever window holds node j
    typedef uint32_t Handle;
    __device__ __forceinline__ Handle gh(uint32_t j) const {
        uint32_t d = d1;
        if (j < lo_thr) d = d0;
        if (j > hi_thr) d = d2;
        return d + j * 4u;
    }
    __device__ __forceinline__ Handle gh_row(int row, uint32_t j) const { return (row == 0 ? d0 : (row == 1 ? d1 : d2)) + j * 4u; }
    __device__ __forceinline__ float gv(Handle h) const { return lds_f32<lay().o_vwin>(h); }
    __device__ __forceinline__ int glft(Handle h) const {
        static_assert(!STDP || lay().lrows == 3, "gathered last_firing_time needs all three window rows");
        return (int)lds_u32<lay().o_lwin>(h);
    }
    __device__ __forceinline__ float gt0(Handle h) const { return lds_f32<lay().o_twin>(h); }
    __device__ __forceinline__ float gt(Handle h, int ty) const { return lds_f32_rt(h + lay().o_twin + (uint32_t)ty * 3u * kWinRowBytes); }
};

// Order in which the CTAs take the tiles.  Whole lattices: ascending, or descending on odd timesteps (the tail of the arrays that
// the previous step left in L2 is what this step reads first).  Row strips: the tiles that import ghosts / export boundary rows
// go FIRST, so a strip's exports of step s leave at the start of step s and its neighbour — which needs them at the start of its
// step s + 1 — finds them long arrived: the NVLink store / fence / flag latency (~10 us) is off the critical path of every step.
template <bool ROWS>
__device__ __forceinline__ uint32_t win_tile_of(const StepParams &p, const WinParams &wp, uint32_t seq) {
    const uint32_t nb = ROWS ? wp.first_end : wp.first_lo + wp.first_hi;
    if (seq < wp.first_lo) return seq;
    if (seq < nb) return wp.n_tiles - 1u - (seq - wp.first_lo);
    const uint32_t k = seq - nb, n_int = wp.n_tiles - nb;
    return wp.first_lo + (p.reverse ? n_int - 1u - k : k);
}

constexpr int kWinProducers = 4;   // producer warps per CTA; together they issue the copies of every tile
template <int G> constexpr int win_threads() { return (G * 8 + kWinProducers) * 32; }

// Which tiles read their parameter row (WinParams::tile_par).  Each case is its own kernel: compiled with both step variants, the
// kernel's code doubles and its registers are allocated over both, which cost 2-8 % on lattices whose tiles all stream (measured on
// one B200 at 1000 W: 1000 x 1000 LIF + STDP 23.6 -> 25.5 us per step, Hodgkin-Huxley 2048 x 2048 317 -> 323 us).  kRowsNone has
// the stage layout, stream order and loop code of the kernel before tile rows (win_layout(..., rows = false)); kRowsSome runs with
// two consumer groups (win_groups).
enum WinRows : int { kRowsNone = 0, kRowsAll = 1, kRowsSome = 2 };

// STEN (kRowsAll only): every tile is a stencil tile, see WinSrc
template <int MODEL, int CHEMG, bool NTREL, bool STDP, int G, int ROWS, bool STEN>
__global__ void __launch_bounds__(win_threads<G>(), 1)
step_win_kernel(const __grid_constant__ StepParams p, const __grid_constant__ WinParams wp) {
    extern __shared__ __align__(128) unsigned char smem[];
    constexpr bool R = ROWS != kRowsNone;
    static_assert(!STEN || ROWS == kRowsAll, "stencil stages are built for lattices whose tiles all read their rows");
    constexpr WinLayout L = win_layout(MODEL, CHEMG, NTREL, STDP, R, STEN);
    const uint32_t S = wp.stages;
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + (size_t)S * wp.stage_bytes);
    uint64_t *empty = full + S;
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    if (threadIdx.x == 0) {
        for (uint32_t s = 0; s < S; ++s) {
            mbar_init(&full[s], kWinProducers);   // every producer warp announces its share of the bytes
            mbar_init(&empty[s], 8);   // the eight warps of the group that consumed the stage
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    pdl_wait();   // everything above ran while the previous timestep's kernel was still draining (launch_pdl)
    if (halo_failed(p)) return;
    if (p.dbg && blockIdx.x == 0 && threadIdx.x == 0) {
        unsigned long long gt;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt));
        p.dbg[0] = (unsigned long long)clock64(); p.dbg[1] = gt;
    }

    if (warp >= G * 8) {
        // ---- producers: kWinProducers warps fill every stage TOGETHER.  A cp.async.bulk costs its warp ~32 ns of issue
        // time whatever its size or the number of active lanes (tools/tma_bench.cu: 1 warp sustains 4.3 TB/s chip-wide with
        // 1 KB copies, 2 warps 7.0 TB/s), and a tile needs ~45 of them: one warp per tile put 1.4 us of serial issue in
        // front of every stage.  Copy k of a tile is issued by warp k % P, lane k / P; each warp announces its own bytes
        // on the stage's full barrier (initialised to P arrivals).
        const uint32_t q = warp - G * 8;
        bool waited_lo = !p.halo[0].active, waited_hi = !p.halo[1].active;
        const uint32_t ty0 = (CHEMG == 1) ? (uint32_t)(__ffs((int)p.nt_used) - 1) : 0u;
        const bool lft_on = wp.lft_copy != 0;
        uint32_t n_t = 0, t_types[kNT] = {0, 0, 0};
        if constexpr (NTREL) {
            for (uint32_t k = 0; k < L.tslots; ++k) {
                const uint32_t ty = (CHEMG == 1) ? ty0 : k;
                if (p.nt_used & (1u << ty)) t_types[n_t++] = k;
            }
        }
        // this lane's copy: a per-tile contiguous operand stream, or window row r of node array arr (0: V, 1:
        // last_firing_time, 2..: t slots)
        const uint32_t idx = q + kWinProducers * lane;
        const bool is_stream = idx < wp.n_streams;
        const bool is_par = is_stream && idx >= wp.n_state;   // a parameter stream: non-uniform tiles only
        const uint32_t wv = idx - wp.n_streams, arr = wv / 3u, r = wv - arr * 3u;
        bool is_win = !is_stream && arr < 2u + n_t;
        if (is_win && arr == 1u) is_win = lft_on && (L.lrows == 3 || r == 1u);
        if (is_win && arr >= 2u) is_win = (L.trows == 3 || r == 1u);
        TmaStream my{nullptr, 0u, 0u};
        if (is_stream) my = wp.st[idx];
        // uniform flag of the next tile, loaded one tile ahead (its L2 latency overlaps the empty-barrier wait and the copies of
        // the tile before); only needed when some tiles are uniform and others stream their parameters
        constexpr bool flags_needed = ROWS == kRowsSome;
        auto uniform_of = [&](uint32_t seq) -> uint32_t {
            return (flags_needed && seq < wp.n_tiles) ? __ldg(wp.tile_par + (size_t)win_tile_of<R>(p, wp, seq) * wp.row_words) & kTileUniform : 0u;
        };
        uint32_t uni_next = uniform_of(blockIdx.x);
        uint32_t s = 0, ph = 0;
        for (uint32_t tile_seq = blockIdx.x; tile_seq < wp.n_tiles; tile_seq += gridDim.x) {
            const uint32_t tile = win_tile_of<R>(p, wp, tile_seq);
            const bool uni = uni_next != 0u;
            uni_next = uniform_of(tile_seq + gridDim.x);
            mbar_wait_backoff(&empty[s], ph ^ 1u);   // the whole warp probes: no divergent lane-0 loop with 31 lanes parked at a reconvergence barrier
            const uint32_t ts = tile * kWinTile;   // first local neuron of the tile
            // multi-GPU: ghost rows are written by the neighbouring GPU over NVLink; they must have landed before TMA reads
            // them.  Tiles whose upper window reaches below own0 read lower ghosts, tiles whose lower window reaches past the
            // last owned neuron read upper ghosts.
            bool ghosts = false;
            if (!waited_lo && ts <= wp.cols) {
                if (lane == 0) halo_wait(p.halo[0].my_flag, p.halo_epoch, p.halo_done + 2, p.halo_timeout_ns);
                waited_lo = ghosts = true;
            }
            if (!waited_hi && ts + kWinTile + 1u + wp.cols > p.n_neurons) {
                if (lane == 0) halo_wait(p.halo[1].my_flag, p.halo_epoch, p.halo_done + 2, p.halo_timeout_ns);
                waited_hi = ghosts = true;
            }
            unsigned char *dst = smem + (size_t)s * wp.stage_bytes;
            const void *src = nullptr;
            uint32_t bytes = 0;
            if (is_stream && !(is_par && uni)) {
                src = my.src + (size_t)tile * my.bytes_per_tile;
                dst += my.smem_off;
                bytes = my.bytes_per_tile;
            } else if (is_win) {
                // window row r: node indices [a4, a4 + kWinRowElems) with a4 = floor4(own0 + ts + (r - 1) * cols - 1), clamped
                // to the allocation
                const int64_t a = (int64_t)p.own0 + ts + ((int64_t)r - 1) * wp.cols - 1;
                const int64_t a4 = a & ~(int64_t)3;
                const int64_t b = a4 < 0 ? 0 : a4;
                const int64_t e = (a4 + kWinRowElems) > (int64_t)wp.node_cap ? (int64_t)wp.node_cap : (a4 + kWinRowElems);
                if (e > b) {
                    bytes = (uint32_t)(e - b) * 4u;
                    const uint32_t so = (uint32_t)(b - a4) * 4u;   // bytes skipped at the front of the window row
                    if (arr == 0u) {
                        dst += L.o_vwin + r * kWinRowBytes + so;
                        src = p.v_in + b;
                    } else if (arr == 1u) {
                        dst += L.o_lwin + (L.lrows == 3 ? r : 0u) * kWinRowBytes + so;
                        src = p.lft_in + b;
                    } else {
                        const uint32_t k = t_types[arr - 2u];
                        const uint32_t ty = (CHEMG == 1) ? ty0 : k;
                        dst += L.o_twin + (k * L.trows + (L.trows == 3 ? r : 0u)) * kWinRowBytes + so;
                        src = p.t_in + (size_t)ty * p.t_stride + b;
                    }
                }
            }
            const uint32_t tx = __reduce_add_sync(0xffffffffu, bytes);
            if (lane == 0) mbar_arrive_expect_tx(&full[s], tx);
            __syncwarp();
            if (ghosts) fence_proxy_async();   // lane 0's acquire of the arrival flag, then every lane's TMA reads of the ghosts
            if (bytes) tma_bulk_g2s(dst, src, bytes, &full[s]);
            if (++s == S) { s = 0; ph ^= 1u; }
        }
        return;
    }

    // ---- consumers: group g takes the CTA's tiles g, g + G, ...; 8 warps x 32 neurons per tile --------------------
    const uint32_t g = warp >> 3, wg = warp & 7u, tid = threadIdx.x & 255u;
    const uint32_t smem_s = smem_u32(smem);
    uint32_t s = g % S, ph = (g / S) & 1u;
    for (uint32_t tile_seq = blockIdx.x + g * gridDim.x; tile_seq < wp.n_tiles; tile_seq += G * gridDim.x) {
        const uint32_t tile = win_tile_of<R>(p, wp, tile_seq);
        const uint32_t warp_global = tile * 8u + wg;
        const uint32_t ln = warp_global * 32u + lane;
        const bool active = warp_global * 32u < p.n_neurons;
        const bool valid = ln < p.n_neurons;
        const uint32_t lnc = valid ? ln : p.n_neurons - 1;
        bool export_lo = false, export_hi = false;
        // only the few tiles at the two ends of a strip touch a halo (CTA-uniform test): everything else runs the plain step
        const bool boundary = tile < wp.bnd_lo || tile + wp.bnd_hi >= wp.n_tiles;
        if (boundary) halo_export_flags(p, ln, valid, export_lo, export_hi);
        // A group returns to a stage only every lcm(S, G) / S rounds, and a parity wait cannot tell "round k landed" from
        // "round k - 1 is still landing" (two phases apart).  Bulk copies of different stages complete out of order, so
        // first make sure that round k - 1 of this stage has been consumed (the empty barrier; a producer that issued this
        // warp's previous tile has already seen round k - 2 consumed, so this wait is unambiguous), then wait for the data.
        if (R ? wp.ring_check != 0u : S % G != 0u) mbar_wait(&empty[s], ph ^ 1u);
        mbar_wait(&full[s], ph);
        if (active) {
            const uint32_t ts_node = p.own0 + tile * kWinTile;
            const uint32_t st = smem_s + s * wp.stage_bytes;
            // shared address of V[node 0] through window row r: st + r * row_bytes - 4 * floor4(ts_node + (r - 1) * cols - 1)
            const int32_t a0 = (int32_t)ts_node - (int32_t)wp.cols - 1, a1 = (int32_t)ts_node - 1, a2 = (int32_t)ts_node + (int32_t)wp.cols - 1;
            const uint32_t d0 = st + 0u * kWinRowBytes - (uint32_t)(a0 & ~3) * 4u;
            const uint32_t d1 = st + 1u * kWinRowBytes - (uint32_t)(a1 & ~3) * 4u;
            const uint32_t d2 = st + 2u * kWinRowBytes - (uint32_t)(a2 & ~3) * 4u;
            // this neuron inside a row-relative window: node (ts_node + tid) sits (ts_node + tid - floor4(a1)) elements in
            const uint32_t own = st + ((uint32_t)((int32_t)ts_node - (a1 & ~3)) + tid) * 4u;
            auto step = [&](auto uni) {
                const WinSrc<MODEL, CHEMG, NTREL, STDP, R, decltype(uni)::value, STEN> src{
                    p, wp, st + tid * 4u, own, st + (wg * kWinWidth * 32u + lane) * 4u, ts_node ? ts_node - 1u : 0u, ts_node + kWinTile,
                    d0, d1, d2, warp_global * kWinWidth, lane, tid, st + L.o_row};
                neuron_step<MODEL, CHEMG, NTREL, STDP, false>(p, src, warp_global, lane, ln, lnc, valid, export_lo, export_hi);
            };
            if constexpr (ROWS == kRowsNone) step(std::false_type{});
            else if constexpr (ROWS == kRowsAll) step(std::true_type{});
            else if (lds_u32<L.o_row>(st) & kTileUniform) step(std::true_type{});   // CTA-uniform
            else step(std::false_type{});
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[s]);
        if (boundary && active) halo_publish(p, warp_global, lane);
        s += G;
        if (s >= S) { s -= S; ph ^= 1u; }
    }
    if (p.dbg && blockIdx.x == 0 && threadIdx.x == 0) {
        unsigned long long gt;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt));
        p.dbg[2] = (unsigned long long)clock64(); p.dbg[3] = gt;
    }
}

// ------------------------------------------------------------------------------------------------
// launcher
// ------------------------------------------------------------------------------------------------
cudaError_t launch_step_win(const StepParams &p, const WinParams &wp, const StepSpec &spec, unsigned grid, cudaStream_t s) {
    if (p.n_neurons == 0) return cudaSuccess;
    const size_t smem = (size_t)wp.stages * wp.stage_bytes + 2 * wp.stages * sizeof(uint64_t);
    return dispatch_step(spec, cudaErrorInvalidValue, [&](auto k) {
        using K = decltype(k);
        if constexpr (K::NET) {
            return cudaErrorInvalidValue;   // single lattices only
        } else {
            constexpr int G = win_groups(K::MODEL, K::CHEMG, false), GM = win_groups(K::MODEL, K::CHEMG, true);
            auto launch = [&](auto kern, int threads) {
                cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                if (e != cudaSuccess) return e;
                return launch_pdl(pdl_ok(p), kern, dim3(grid), dim3(threads), smem, s, p, wp);
            };
            if (wp.tile_par == nullptr) return launch(step_win_kernel<K::MODEL, K::CHEMG, K::NTREL, K::STDP, G, kRowsNone, false>, win_threads<G>());
            if (wp.n_streams == wp.n_state) {
                if (wp.stencil) return launch(step_win_kernel<K::MODEL, K::CHEMG, K::NTREL, K::STDP, G, kRowsAll, true>, win_threads<G>());
                return launch(step_win_kernel<K::MODEL, K::CHEMG, K::NTREL, K::STDP, G, kRowsAll, false>, win_threads<G>());
            }
            return launch(step_win_kernel<K::MODEL, K::CHEMG, K::NTREL, K::STDP, GM, kRowsSome, false>, win_threads<GM>());
        }
    });
}

// one CTA per tile, one thread per neuron (see TileParSrc); thread t checks lane t % 32 of the tile's warp t / 32 in the table
__global__ void __launch_bounds__(kWinTile) tile_params_kernel(const __grid_constant__ TileParSrc a, uint32_t *rows, unsigned int *counts) {
    __shared__ uint32_t full_warps;
    const uint32_t tile = blockIdx.x, ts = tile * kWinTile, ln = ts + threadIdx.x;
    const bool valid = ln < a.n_neurons;
    uint32_t *row = rows + (size_t)tile * a.row_words;
    if (threadIdx.x == 0) full_warps = 0u;
    bool same = true;
    for (uint32_t k = 0; k < a.n_par; ++k) {
        const uint32_t first = __ldg(a.src[k] + ts);
        if (valid) same = same && __ldg(a.src[k] + ts + threadIdx.x) == first;
        if (threadIdx.x == 0) row[a.word[k]] = first;
    }
    uint32_t c[8];
    stencil_cols(ln, a.n_neurons, a.cols, a.row0_global, a.rows_global, a.own0, a.stencil_nt, c);
    // the slices of a uniform-width table: warp w's k-row u at ((tile * 8 + w) * 8 + u) * 32 (allocated for whole tiles)
    const uint32_t *cw = a.col + ((size_t)(ln >> 5) * kWinWidth) * 32u + (threadIdx.x & 31u);
    bool sten = true;
#pragma unroll
    for (int u = 0; u < 8; ++u) sten = sten && __ldg(cw + u * 32) == c[u];
    const bool full = __all_sync(0xffffffffu, c[7] != kColPad);
    __syncthreads();
    if (full && (threadIdx.x & 31u) == 0u) atomicOr(&full_warps, 1u << (threadIdx.x >> 5));
    const bool uni = __syncthreads_and(same) != 0;
    const bool all_sten = __syncthreads_and(sten) != 0;
    if (threadIdx.x == 0) {
        row[0] = (uni ? kTileUniform : 0u) | (all_sten ? kTileStencil : 0u) | full_warps << kTileFullShift;
        if (!uni) atomicAdd(counts, 1u);
        if (!all_sten) atomicAdd(counts + 1, 1u);
    }
}

cudaError_t launch_tile_params(const TileParSrc &a, uint32_t *rows, unsigned int *counts, cudaStream_t s) {
    if (a.n_tiles == 0) return cudaSuccess;
    tile_params_kernel<<<a.n_tiles, kWinTile, 0, s>>>(a, rows, counts);
    return cudaGetLastError();
}

}  // namespace snn
