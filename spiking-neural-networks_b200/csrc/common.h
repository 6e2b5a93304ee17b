// common.h — shared host/device declarations of the B200 lattice engine.
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/snn_b200.h"
#include "step_spec.h"

#include <cstdlib>
#include <utility>

namespace snn {

// Programmatic dependent launch: a kernel launched through launch_pdl may be scheduled while its predecessor in the stream is
// still draining (its CTAs take the SMs the predecessor's CTAs leave); it must execute pdl_wait() before it touches anything the
// predecessor wrote — that returns once the predecessor grid has completed and its writes are visible.  Hides the launch latency
// and the prologue (barrier initialisation, parameter loads) behind the predecessor's tail.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
#endif
// Measured (profiles/README.md, round 2): step kernels gain 2.5-3 us per launch (1000 x 1000 lattice 26.5 -> 23.4 us per step,
// wide-row network 30.6 -> 28.0 us); the persistent per-edge reward kernel LOSES 90 us per step as a dependent launch (its three
// CTAs per SM arrive one by one as the step kernel's CTAs drain).  `allow` = false launches plainly: the per-edge kernels, and
// every kernel of row strips and general-graph partitions (measured: the same 10^7-neuron lattice over 4 GPUs takes 83.8 us per
// step with dependent launches and 79.8 us without — the early CTAs of the next step only add to the neighbour handshake's
// critical path).
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(bool allow, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args &&...args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = allow ? 1u : 0u;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

constexpr int kNT = SNN_NUM_NT_TYPES;

// ---- sliced-ELL in-edge storage (slice height = one warp) -------------------------------------
// col word: bits 0..27 presynaptic node index (local), 28..30 neurotransmitter types the
// presynaptic node releases, 31 presynaptic node is a spike train.  0xFFFFFFFF = padding.
constexpr uint32_t kColPad = 0xFFFFFFFFu;
constexpr uint32_t kColIdxMask = 0x0FFFFFFFu;
constexpr uint32_t kColNtShift = 28;
constexpr uint32_t kColTrainBit = 0x80000000u;
constexpr uint64_t kMaxNodes = 0x0FFFFFFEull;

// device code unrolls the loop that follows (host compilers do not know the pragma)
#ifdef __CUDA_ARCH__
#define SNN_UNROLL _Pragma("unroll")
#else
#define SNN_UNROLL
#endif

// The col words of one row of a radius-1 Moore stencil table, as sell_grid_kernel writes them: slot k holds the k-th in-bounds
// neighbour of local neuron ln in ascending node index, OR'd with `nt` << kColNtShift (the generator passes 0 and stamps each
// neighbour's own release bits); the slots past the last neighbour, and every slot of a lane ln >= n, hold kColPad.  The lattice
// has rows_global rows of `cols` cells; local neuron 0 is the first cell of row row0_global and has node index own0.
__host__ __device__ __forceinline__ void stencil_cols(uint32_t ln, uint32_t n, uint32_t cols, uint32_t row0_global, uint32_t rows_global,
                                                      uint32_t own0, uint32_t nt, uint32_t (&c)[8]) {
    const bool valid = ln < n;
    const uint32_t r = valid ? ln / cols : 0u, x = valid ? ln - r * cols : 0u;
    const bool up = r + row0_global > 0u, dn = r + row0_global + 1u < rows_global, lf = x > 0u, rt = x + 1u < cols;
    const uint32_t me = own0 + ln, hi = nt << kColNtShift;
    uint32_t k = 0;
SNN_UNROLL
    for (int u = 0; u < 8; ++u) c[u] = kColPad;
    // candidate q: three in the row above, the two side neighbours, three in the row below; it can only fill slots u <= q
SNN_UNROLL
    for (int q = 0; q < 8; ++q) {
        const int dr = q < 3 ? -1 : (q < 5 ? 0 : 1);
        const int dc = q < 3 ? q - 1 : (q < 5 ? 2 * q - 7 : q - 6);
        const bool ok = valid && (dr < 0 ? up : (dr > 0 ? dn : true)) && (dc < 0 ? lf : (dc > 0 ? rt : true));
        const uint32_t w = (me + (uint32_t)dr * cols + (uint32_t)dc) | hi;
SNN_UNROLL
        for (int u = 0; u <= q; ++u)
            if (ok && k == (uint32_t)u) c[u] = w;
        k += ok ? 1u : 0u;
    }
}

// ---- per-neuron device field slots (index into StepParams::f) ---------------------------------
enum NeuronSlot : int {
    F_GAP = 0, F_DT, F_CM, F_VTH, F_VRESET, F_REFR, F_TREF, F_LEAK, F_INTEG, F_EL, F_GL, F_TAUM,
    F_ALPHA, F_BETA, F_SLOPE, F_W, F_VC, F_A, F_B, F_C, F_D, F_G, F_E,
    F_GNA, F_ENA, F_M, F_H, F_GK, F_EK, F_N, F_GKL, F_EKL,
    // BCMIzhikevichNeuron activity bookkeeping (period and num_spikes hold u32 bit patterns)
    F_AVG_ACT, F_CUR_ACT, F_PERIOD, F_NSPK, F_FRCLK, F_FRWIN,
    // derived (written by the finalize kernel only, never inside the step loop)
    F_NA_CUR, F_M_ALPHA, F_M_BETA, F_H_ALPHA, F_H_BETA, F_K_CUR, F_N_ALPHA, F_N_BETA, F_KL_CUR,
    F_COUNT
};

// per spike-train device field slots
enum TrainSlot : int { TF_VTH = 0, TF_VREST, TF_DT, TF_K, TF_CHANCE, TF_RATE, TF_STEP, TF_ICLOCK, TF_COUNTER, TF_COUNT };

// per-type (type-major, stride = node/neuron capacity) chemical arrays
enum NtSlot : int { NTF_TMAX = 0, NTF_P1 /* clearance | v_p | decay */, NTF_P2 /* k_p */, NTF_COUNT };
enum RcSlot : int { RCF_R = 0, RCF_K1 /* alpha | r_max */, RCF_K2 /* beta | decay */, RCF_G, RCF_E, RCF_MG, RCF_CUR, RCF_COUNT };

struct LatInfo {  // one per neuron lattice, device table
    uint32_t base;        // first neuron (local neuron number)
    uint32_t n;
    float a_plus, a_minus, tau_plus, tau_minus, dt;
    uint32_t do_plasticity;
    uint32_t grid_hist;   // record grid voltage history
    uint32_t spike_hist;
    uint64_t hist_off;    // float offset of this lattice inside one history step record
};

constexpr int kMaxLattices = 16;

// halo export of one direction (multi-GPU row strips): owned neurons [first, first+count) are also
// written into the peer's ghost slots starting at node index peer_node0
struct HaloDir {
    uint32_t first, count, peer_node0;
    uint32_t my_ghost0;          // node index of the ghost slots the peer fills for me
    float *peer_v[2];            // peer's V ping-pong buffers (device pointers mapped through CUDA IPC)
    int *peer_lft[2];
    float *peer_t[2];            // type-major, stride peer_t_stride
    uint64_t peer_t_stride;
    unsigned long long *peer_flag;   // peer-side arrival counter for data coming from me
    unsigned long long *my_flag;     // my arrival counter for data coming from this peer
    // second pair, reward-modulated strips: "the per-edge kernel of step s has finished reading its old ghosts" — the step
    // kernel of s + 1 waits for it instead of my_flag, because it overwrites those ghost slots in the neighbour's slab
    unsigned long long *peer_flag2;
    unsigned long long *my_flag2;
    uint32_t active;
};

// general-graph partition (contiguous node ranges, arbitrary in-edges): one entry per rank this rank exchanges with
constexpr int kMaxRanks = 16;
struct GPeer {
    float *v[2]; int *lft[2]; float *t[2];   // the peer's node arrays (both parities), mapped through CUDA IPC or addressed directly
    uint64_t t_stride;
    unsigned long long *peer_flag;           // the peer's "rank r has completed step s" counter for me
    unsigned long long *my_flag;             // my counter for that peer
};

struct StepParams {
    // index space
    uint32_t own0;        // node index of neuron 0 (multiple of 32)
    uint32_t n_neurons;   // neurons stepped by this kernel
    uint32_t n_nodes;     // neurons + ghosts + spike trains
    uint32_t clock;       // internal clock value stamped on spikes of this step
    uint32_t apply_pending;  // lazy STDP: apply last step's weight updates while streaming the edges
    uint32_t electrical, chemical;
    uint32_t nt_used, rc_used;   // union over nodes of present neurotransmitter / receptor types
    int ntk, rck, refract;
    // graph
    const uint32_t *slice_off;
    uint32_t uniform_width;   // != 0: every slice has this many k-rows (slice_off[s] == s * uniform_width)
    const uint32_t *col;
    float *wgt;
    // shared node arrays
    const float *v_in;  float *v_out;
    const int *lft_in;  int *lft_out;
    uint32_t lft_pp;     // lft is ping-ponged (else in == out, written on spike only)
    const uint32_t *spk_in; uint32_t *spk_out;
    const float *t_in; float *t_out; uint64_t t_stride;   // type-major [kNT][t_stride]
    const uint8_t *node_flags;  // per node: nt mask | rc mask << 4
    // neuron arrays
    float *f[F_COUNT];
    uint32_t *was_inc;          // HH bitmask
    float *nt[NTF_COUNT]; uint64_t nt_stride;   // per node
    float *rc[RCF_COUNT]; uint64_t rc_stride;   // per neuron
    // spike trains (nodes [train0, train0+n_trains))
    uint32_t train0, n_trains;
    const float *tf[TF_COUNT];   // on BCM Izhikevich partitions: the activity exchange (BcmSlot)
    // lattices
    const LatInfo *lat; int n_lat;
    // histories: this step's record
    float *grid_hist;           // nullptr = off
    uint32_t *spike_hist;       // bit words, one per warp of neurons
    // halos
    HaloDir halo[2];
    unsigned long long halo_epoch;   // value the arrival counters must reach before ghosts are read
    uint32_t out_par;                // parity of the *_out ping-pong buffers (same on every rank)
    unsigned int *halo_done;         // [2] per-direction CTA completion counters
    unsigned long long halo_timeout_ns;   // bound of one in-kernel wait for a neighbouring strip
    // general-graph partition: ghosts are gather lists, not contiguous rows
    const GPeer *gpeers; uint32_t n_gpeers;
    const uint32_t *gexp_off, *gexp_ent;    // per owned neuron: export entries (peer slot << 28 | node index in the peer's arrays)
    const uint8_t *gslice;                  // per slice: bit 0 reads ghosts, bit 1 has exporting neurons
    uint32_t n_gslices;
    uint32_t reverse;                // window kernel: sweep the tiles back to front (alternates per step: the tail of the
                                     // arrays that the previous step left in L2 is what this step reads first)
    // window kernel: {clock64, globaltimer} of CTA 0 at its start and end, when non-null.  The engine leaves it null; the stamps
    // stay because the window kernel compiled without them took 1.0 us longer per step on the 10^7-neuron bench lattice (296.3 vs
    // 295.3 us, B200 at 1000 W)
    unsigned long long *dbg;
};

// BCM Izhikevich partitions: current_activity travels to the neighbours next to V and last_firing_time, into node-indexed
// ping-pong buffers of their slabs.  A partitioned handle holds one neuron lattice and no spike trains, so the pointers ride in
// the spike-train slots StepParams::tf (null on every other handle).  New members of HaloDir, GPeer or StepParams would move the
// parameters, and with them change the code, of every other kernel.
enum BcmSlot : int {
    TFB_HALO_ACT = 0,    // tf[TFB_HALO_ACT + 2 * direction + parity]: the neighbour's activity buffer (addressed like HaloDir::peer_v)
    TFB_GPEER_ACT = 4,   // a float *const * table, [2 * peer slot + parity]: the same for general-graph peers (addressed like GPeer::v)
    TFB_ACT_GHOST = 5,   // my own buffer of parity out_par: the ghosts' activity after this step (BCM edge kernel)
};
static_assert((int)TFB_ACT_GHOST < (int)TF_COUNT, "the BCM activity pointers must fit into StepParams::tf");
#ifdef __CUDACC__
__device__ __forceinline__ float *bcm_halo_act(const StepParams &p, uint32_t d, uint32_t par) {
    return const_cast<float *>(p.tf[TFB_HALO_ACT + 2u * d + par]);
}
__device__ __forceinline__ float *bcm_gpeer_act(const StepParams &p, uint32_t q, uint32_t par) {
    return reinterpret_cast<float *const *>(p.tf[TFB_GPEER_ACT])[2u * q + par];
}
#endif

struct TrainParams {
    uint32_t train0, n_trains, clock; int kind; int ntk;
    uint64_t seed;
    uint64_t draw;   // per-handle count of spike-train steps: the Philox counter (survives reset_timing)
    const float *v_in; float *v_out;
    const int *lft_in; int *lft_out; uint32_t lft_pp;
    const uint32_t *spk_in; uint32_t *spk_out;
    const float *t_in; float *t_out; uint64_t t_stride;
    const uint8_t *node_flags;
    float *nt[NTF_COUNT]; uint64_t nt_stride;
    float *tf[TF_COUNT];
    const uint64_t *ft_off; const float *ft;   // preset firing times CSR
    // per train-lattice clocks: lattice l covers trains [tl_base[l], tl_base[l+1]) and stamps tl_clock[l]
    int n_tl; uint32_t tl_base[kMaxLattices + 1]; uint32_t tl_clock[kMaxLattices];
    float *grid_hist; uint32_t *spike_hist;   // this step's record over all trains (nullptr = off)
};

// ---- multi-step kernel (step_multi.cu): a whole chunk of timesteps in one cooperative launch ----------
struct MultiParams {
    uint32_t steps;           // timesteps of this launch
    uint32_t first_pending;   // the first of them applies the previous step's pending STDP (0 only at the first step of a run)
    uint32_t cur, lft_loc;    // parities of the current V / t / spike buffers and of the current last_firing_time at launch
    uint32_t lft_pp;
    uint32_t train_sync;      // the spike trains of a step wait for all of its neurons (lazy STDP reads the trains' lft_out)
    float *v[2]; int *lft[2]; uint32_t *spk[2]; float *t[2];
    float *grid_hist; uint32_t *spike_hist; float *tgrid_hist; uint32_t *tspike_hist;   // staged history of the chunk (record s at + s * row)
    uint64_t n_neurons, n_words, n_trains, t_words;
    unsigned int *barrier;    // grid-wide arrival counter, zero at launch
    uint32_t wide_stage;      // wide-row variant: stage the node state in shared memory (small networks)
    uint32_t cache_rows;      // the stencil rows and parameters may live in registers for the whole launch (nothing rewrites them)
};
// dry = only report whether the configuration is eligible (cudaSuccess) without launching
cudaError_t launch_step_multi(const StepParams &p, const TrainParams &t, const MultiParams &m, const StepSpec &spec, bool wide, int device,
                              bool dry, cudaStream_t s);

// ---- TMA-staged step kernel (step_tma.cu) -----------------------------------------------------
constexpr int kTmaTile = 256;            // neurons per tile
constexpr int kTmaConsumerWarps = 8;
constexpr int kTmaThreads = (kTmaConsumerWarps + 1) * 32;   // + one producer warp
constexpr int kMaxTmaStreams = 56;

struct TmaStream {           // one contiguous operand range per tile
    const unsigned char *src;
    uint32_t bytes_per_tile;  // multiple of 16
    uint32_t smem_off;        // multiple of 128, inside a stage
};

struct TmaParams {
    uint32_t n_tiles, n_streams, stage_bytes, stages, tx_bytes;
    TmaStream st[kMaxTmaStreams];
    // byte offsets inside a stage of each logical operand
    uint32_t o_v, o_lft, o_flags, o_col, o_wgt;
    uint32_t o_t[kNT];
    uint32_t o_f[F_COUNT];
    uint32_t o_nt[NTF_COUNT][kNT];
    uint32_t o_rc[RCF_COUNT][kNT];
};

cudaError_t launch_step_tma(const StepParams &p, const TmaParams &tp, const StepSpec &spec, unsigned grid, cudaStream_t s);

// ---- window-staged step kernel (step_win.cu): radius-1 stencil lattices ----------------------
// One persistent CTA per SM; every operand of a 256-neuron tile, INCLUDING the three neighbour row windows of the node
// arrays (V, last_firing_time, t), is moved into a shared-memory stage by TMA bulk copies.  The stage layout of
// everything but the per-type chemical parameters is a compile-time function of the kernel's template arguments, so
// operand addresses are immediates.
constexpr uint32_t kWinTile = 256;                      // neurons per tile (8 consumer warps)
constexpr uint32_t kWinRowElems = kWinTile + 8;         // a window row: tile + 1 neighbour each side + 16-byte alignment slack
constexpr uint32_t kWinRowBytes = kWinRowElems * 4;     // 1056
constexpr uint32_t kWinWidth = 8;                       // k-rows per slice of a radius-1 stencil
constexpr uint32_t kWinEdgeBytes = 8 * kWinWidth * 32 * 4;  // col (or weight) bytes per tile

struct WinLayout {
    uint32_t lrows, trows, tslots;   // window rows kept for last_firing_time / t, neurotransmitter type slots
    uint32_t o_vwin, o_lwin, o_twin, o_spk, o_flags, o_wgt;
    uint32_t o_col;                  // 0xFFFFFFFF = stencil: every tile's col words are those of stencil_cols, none staged
    uint32_t o_f[F_NA_CUR];          // 0xFFFFFFFF = not read by this model
    // rows (some tile reads its parameter row): the state fields first, then the row, then the parameters, so that a stage without
    // per-neuron parameters ends at uni_end; without rows every field in slot order and no row (o_row = 0xFFFFFFFF)
    uint32_t o_row;                  // the tile's parameter row (copied from the tile table, see win_field_param)
    uint32_t uni_end;                // first byte after the part every tile fills (state fields and the row; multiple of 16)
    uint32_t fixed_end;              // first byte after the compile-time part (multiple of 128)
    // the tile row, in 32-bit words: [0] flags (kTileUniform, kTileStencil, kTileFullShift), then the first neuron's parameters: r_f[slot] for the model's, [r_nt + NtSlot * kNT + type] for the neurotransmitters',
    // [r_rc + (RcSlot - RCF_K1) * kNT + type] for the receptors' (words of kinetics this run does not read stay 0)
    uint32_t r_f[F_NA_CUR];
    uint32_t r_nt, r_rc;
    uint32_t row_bytes;              // multiple of 16
};

// fields the step of `model` reads (must mirror neuron_step, step_body.cuh)
__host__ __device__ constexpr bool win_field_read(int model, bool ntrel, int slot) {
    const bool bcm = model == SNN_MODEL_BCM_IZHIKEVICH;
    const bool izh = model == SNN_MODEL_IZHIKEVICH || model == SNN_MODEL_LEAKY_IZHIKEVICH || bcm;
    const bool adapt = model == SNN_MODEL_ADAPTIVE_LEAKY_INTEGRATE_AND_FIRE || model == SNN_MODEL_ADAPTIVE_EXP_LEAKY_INTEGRATE_AND_FIRE;
    const bool if4 = model == SNN_MODEL_LEAKY_INTEGRATE_AND_FIRE || model == SNN_MODEL_QUADRATIC_INTEGRATE_AND_FIRE || adapt;
    const bool leaky = model == SNN_MODEL_LEAKY_INTEGRATE_AND_FIRE || adapt;
    const bool qif = model == SNN_MODEL_QUADRATIC_INTEGRATE_AND_FIRE;
    const bool simple = model == SNN_MODEL_SIMPLE_LEAKY_INTEGRATE_AND_FIRE;
    const bool hh = model == SNN_MODEL_HODGKIN_HUXLEY;
    switch (slot) {
    case F_GAP: case F_DT: case F_VTH: return true;
    case F_CM: return ntrel || hh || izh || adapt;
    case F_W: return izh || adapt;
    case F_A: case F_B: case F_C: case F_D: return izh;
    case F_TAUM: return izh || if4;
    case F_EL: return leaky || model == SNN_MODEL_LEAKY_IZHIKEVICH;
    case F_VRESET: return if4 || simple;
    case F_INTEG: case F_REFR: case F_TREF: return if4;
    case F_GL: case F_LEAK: return leaky;
    case F_ALPHA: return adapt || qif;
    case F_BETA: return adapt;
    case F_VC: return qif;
    case F_SLOPE: return model == SNN_MODEL_ADAPTIVE_EXP_LEAKY_INTEGRATE_AND_FIRE;
    case F_G: case F_E: return simple;
    case F_GNA: case F_ENA: case F_M: case F_H: case F_GK: case F_EK: case F_N: case F_GKL: case F_EKL: return hh;
    case F_AVG_ACT: case F_CUR_ACT: case F_PERIOD: case F_NSPK: case F_FRCLK: case F_FRWIN: return bcm;
    default: return false;
    }
}

// State among the fields win_field_read lists: neuron_step reads them through src.state<SLOT>() or writes them back.  The
// others are parameters, read through src.f<SLOT>() only; with the neurotransmitter parameters (src.nt()) and the receptor
// parameters (src.rc(): every receptor field but RCF_R, which is state and read through src.rc_state()) they are what a tile
// whose neurons all share them takes from its tile row instead of from per-neuron streams.  WinSrc asserts both lists.
__host__ __device__ constexpr bool win_field_state(int slot) {
    switch (slot) {
    case F_W: case F_REFR: case F_M: case F_H: case F_N: case F_AVG_ACT: case F_CUR_ACT: case F_NSPK: case F_FRCLK: return true;
    default: return false;
    }
}
__host__ __device__ constexpr bool win_field_param(int model, bool ntrel, int slot) {
    return win_field_read(model, ntrel, slot) && !win_field_state(slot);
}

// word 0 of a tile row (WinLayout): every neuron of the tile has the first one's parameters (bit patterns); every col word of the
// tile is that of stencil_cols for the lattice-wide release mask WinParams::stencil_nt; bit kTileFullShift + w: warp w of the
// tile is full (32 valid lanes with 8 in-edges each)
constexpr uint32_t kTileUniform = 1u, kTileStencil = 2u, kTileFullShift = 8;

__host__ __device__ constexpr WinLayout win_layout(int model, int chemg, bool ntrel, bool stdp, bool rows, bool stencil) {
    WinLayout L{};
    uint32_t off = 0;
    L.lrows = stdp ? 3u : 1u;
    L.trows = chemg ? 3u : 1u;
    L.tslots = !ntrel ? 0u : (chemg == 1 ? 1u : (uint32_t)kNT);
    L.o_vwin = off; off += 3u * kWinRowBytes;
    L.o_lwin = off; off += L.lrows * kWinRowBytes;
    L.o_twin = off; off += L.tslots * L.trows * kWinRowBytes;
    off = (off + 127u) & ~127u;
    L.o_spk = off; off += 128u;
    L.o_flags = off; off += kWinTile;
    L.o_col = 0xFFFFFFFFu;
    if (!stencil) { L.o_col = off; off += kWinEdgeBytes; }
    L.o_wgt = off; off += kWinEdgeBytes;
    uint32_t w = 1;
    for (int s = 0; s < F_NA_CUR; ++s) {
        L.o_f[s] = 0xFFFFFFFFu;
        L.r_f[s] = 0;
        if (win_field_read(model, ntrel, s) && (win_field_state(s) || !rows)) { L.o_f[s] = off; off += kWinTile * 4u; }
        if (win_field_param(model, ntrel, s)) L.r_f[s] = w++;
    }
    L.r_nt = w; if (ntrel) w += NTF_COUNT * kNT;
    L.r_rc = w; if (ntrel) w += (RCF_MG - RCF_K1 + 1) * kNT;
    L.row_bytes = (w * 4u + 15u) & ~15u;
    L.o_row = 0xFFFFFFFFu;
    if (rows) {
        L.o_row = off; off += L.row_bytes;
        L.uni_end = off;
        off = (off + 127u) & ~127u;
        for (int s = 0; s < F_NA_CUR; ++s)
            if (win_field_param(model, ntrel, s)) { L.o_f[s] = off; off += kWinTile * 4u; }
    }
    if (!rows) L.uni_end = off;
    L.fixed_end = off;
    return L;
}

struct WinParams {
    uint32_t n_tiles, n_streams, stage_bytes, stages;
    uint32_t n_state;             // streams [0, n_state) go to every tile, [n_state, n_streams) (parameters) to non-uniform tiles only
    uint32_t node_cap;            // elements allocated per node array (window copies are clamped to [0, node_cap))
    uint32_t cols;
    uint32_t lft_copy;            // copy last_firing_time windows at all (STDP or ping-ponged lft)
    uint32_t first_lo, first_hi;  // row strips: this many tiles at the front / back of the strip touch a halo and are stepped first
    uint32_t bnd_lo, bnd_hi;      // tiles at the front / back that import ghosts or export boundary rows (0, 0 on whole lattices)
    TmaStream st[kMaxTmaStreams]; // per-tile contiguous operands (src + tile * bytes_per_tile)
    uint32_t o_nt[NTF_COUNT][kNT];   // run-time part of the stage layout: per-type chemical parameters
    uint32_t o_rc[RCF_COUNT][kNT];
    // tile rows [n_tiles][row_words] (WinLayout::r_f ...), copied into every stage by the stream n_state - 1; nullptr: no tile is
    // uniform (no row is copied, the stage layout is win_layout(..., rows = false))
    const uint32_t *tile_par;
    uint32_t row_words;
    // first_lo + first_hi, and stages % consumer groups != 0, for the kernels that read tile rows: held in registers as values
    // (as the kernel without rows holds them) they made those kernels spill
    uint32_t first_end, ring_check;
    // every tile is a stencil tile (kTileStencil) and reads its parameter row: the kernel without col words (win_layout(...,
    // stencil = true)), with the release mask of every node and the rows of the lattice that stencil_cols needs for the border
    // warps
    uint32_t stencil, stencil_nt, row0_global, rows_global;
};

// groups of 8 consumer warps per CTA (register budget: 65536 / ((groups * 8 + 1) * 32))
// models with wide operand sets (Hodgkin-Huxley, three neurotransmitter types): fewer, fatter stages
// mixed: the kernel for lattices with both uniform and streaming tiles, which carries both step variants (with 3 groups and 72
// registers, the variants of AdEx and simple LIF with chemistry and STDP spilled)
__host__ __device__ constexpr int win_groups(int model, int chemg, bool mixed) {
    return (mixed || model == SNN_MODEL_HODGKIN_HUXLEY || chemg == 3) ? 2 : 3;
}

cudaError_t launch_step_win(const StepParams &p, const WinParams &wp, const StepSpec &spec, unsigned grid, cudaStream_t s);

// Tile rows of the window kernel: per kWinTile tile of [0, n_neurons), word 0 has kTileUniform when every valid neuron of the
// tile has the bit pattern of the tile's first neuron in every src[k] (compared as 32-bit words: -0.0 != +0.0, a NaN equals only
// its own payload), kTileStencil when the tile's 8 x 8 x 32 words of the uniform-width table `col` equal those of stencil_cols
// (cols, row0_global, rows_global, own0, stencil_nt) bit for bit, and the tile's full warps; word word[k] = the first neuron's
// src[k].  The other words are left as they are.  counts[0] += tiles without kTileUniform, counts[1] += tiles without kTileStencil.
constexpr int kWinMaxPar = 48;
struct TileParSrc {
    const uint32_t *src[kWinMaxPar];   // indexed by local neuron number
    uint32_t word[kWinMaxPar];
    uint32_t n_par, row_words, n_neurons, n_tiles;
    const uint32_t *col;
    uint32_t cols, row0_global, rows_global, own0, stencil_nt;
};
cudaError_t launch_tile_params(const TileParSrc &a, uint32_t *rows, unsigned int *counts, cudaStream_t s);

// ---- kernel launchers (kernels.cu) ------------------------------------------------------------
cudaError_t launch_step(const StepParams &p, const StepSpec &spec, cudaStream_t s);
// same contract as launch_step, one CTA per slice (step_wide.cu): graphs with wide rows, single-GPU handles only
constexpr uint32_t kWideMinWidth = 48;   // mean k-rows per slice from which the wide kernel is used
// scratch != nullptr: two passes (per-edge terms of every slice chunk on its own CTA, parked in `scratch`: chunks_cap buffers of
// wide_chunk_bytes(chemg) per slice; then the ordered sums) — very wide slices, where one SM per slice is issue-bound
// trains != nullptr (two-pass mode only): the spike trains of the timestep are stepped by extra CTAs of the sum pass
cudaError_t launch_step_wide(const StepParams &p, const StepSpec &spec, unsigned char *scratch, uint32_t chunks_cap, const TrainParams *trains,
                             cudaStream_t s);
uint32_t wide_chunk_bytes(int chemg);
uint32_t wide_chunk_krows();
size_t wide_part_bytes();   // per slice, after the chunk buffers: partial sums, counts and the arrival counter of the sum pass (zeroed once)
inline bool pdl_ok(const StepParams &p) { return !(p.halo[0].active | p.halo[1].active) && p.n_gpeers == 0u; }   // see launch_pdl
inline bool pdl_ok(const TrainParams &) { return true; }
cudaError_t launch_trains(const TrainParams &p, cudaStream_t s);
cudaError_t launch_flush_stdp(const StepParams &p, cudaStream_t s);
// RewardModulatedSTDP::update_weight on every edge, both calls of the timestep (p.lft_in = last_firing_time before the step,
// p.lft_out = after it)
// BCM::update_weight on the edges of the neurons that spiked in the step just computed (p.spk_out).  On partitioned handles
// (p.halo active or p.n_gpeers != 0) p.halo_epoch is the value the neighbours' step kernels of this timestep publish.
struct BcmParams { float decay, average_scalar, dt; };
cudaError_t launch_bcm_edges(const StepParams &p, const BcmParams &b, cudaStream_t s);
struct RstdpParams {
    float dopamine, tau_c, a_plus, a_minus, tau_plus, tau_minus, dt;
    uint8_t *counter; float *dw, *c;
    uint32_t canonical;   // every edge has counter == 0 and dw == 0 between timesteps (see rstdp_edge_kernel)
    // the STDP term depends on the two spike times only through their integer difference: tab[0][k] = term for t_post - t_pre = k,
    // tab[1][k] for t_pre - t_post = k (k = 1 .. tab_n - 1, the last entry stands for every larger difference: the term has
    // underflowed to +-0 there).  Filled by rstdp_table_kernel with the very function the kernel would call: bit-identical.
    const float *tab; uint32_t tab_n;
};
cudaError_t launch_rstdp_table(const RstdpParams &r, float *tab, uint32_t tab_n, cudaStream_t s);
cudaError_t launch_rstdp_edges(const StepParams &p, const RstdpParams &r, cudaStream_t s);
// RewardModulatedLatticeNetwork (neuron/mod.rs:3455-5455): the post-step weight pass over the rows of its reward-modulated
// lattices.  lat[] follows StepParams::lat (neuron lattices in node order).
struct RnetLat {
    float dopamine, tau_c, a_plus, a_minus, tau_plus, tau_minus, dt;
    uint32_t flags;   // bit 0: a RewardModulatedLattice; bit 1: its do_modulation
};
struct RnetParams {
    RnetLat lat[kMaxLattices];
    // per post lattice, 2 bits per presynaptic class q (q < kMaxLattices: neuron lattice q; q = kMaxLattices + t: spike-train lattice
    // t): 0 leave the edge alone, 1 own graph (two modulator calls), 2 RewardModulatedWeight block (one call), 3 Weight block fed by
    // a plain lattice (STDP with the input lattice's parameters)
    uint64_t kinds[kMaxLattices];
    uint32_t n_lat, nbase[kMaxLattices + 1];    // neuron lattice l covers local neuron numbers [nbase[l], nbase[l+1])
    uint32_t n_tl, tl_base[kMaxLattices + 1];   // spike-train lattice t covers node indices [train0 + tl_base[t], train0 + tl_base[t+1])
    uint32_t train0;
    uint8_t *counter; float *dw, *c;   // TraceRSTDP members next to StepParams::wgt (same element index)
    uint32_t canonical;                // own-graph edges have counter == 0 and dw == 0 between timesteps (see the kernel)
    const float *tab; uint32_t tab_n;  // per neuron lattice l, 2 * tab_n floats at tab + l * 2 * tab_n (layout of RstdpParams::tab); nullptr = formula
};
cudaError_t launch_rstdp_net_edges(const StepParams &p, const RnetParams &r, cudaStream_t s);
cudaError_t launch_finalize(const StepParams &p, int model, const float *v_prev, cudaStream_t s);
cudaError_t launch_sell_from_csr(const uint64_t *row_ptr, const uint32_t *pre, const float *w, const uint8_t *node_flags,
                                 uint32_t train0, uint32_t n_rows, const uint32_t *slice_off, uint32_t *col, float *wgt,
                                 cudaStream_t s);
cudaError_t launch_sell_grid(uint32_t rows_local, uint32_t cols, uint32_t row0_global, uint32_t rows_global,
                             uint32_t radius, float weight, uint32_t own0, const uint8_t *node_flags, uint32_t width,
                             uint32_t *slice_off, uint32_t *col, float *wgt, cudaStream_t s);
cudaError_t launch_halo_push(const StepParams &p, cudaStream_t s);
cudaError_t launch_gpart_push(const StepParams &p, cudaStream_t s);
// per (step, lattice): sum of V and sum of (V - ref) over the lattice's neurons, f64, fixed reduction order
cudaError_t launch_history_reduce(const float *grid, uint64_t n_neurons, uint32_t steps, const uint32_t *lat_base, const uint32_t *lat_n,
                                  const float *lat_ref, int n_lat, double *out, cudaStream_t s);
// node_flags[i] <- (node_flags[i] & ~(0xF << shift)) | (mask of the non-zero words of src[i*3 .. i*3+2]) << shift; *changed |= any
// counts[i] = number of the `steps` staged raster records in which node i spiked (SpikeHistory::aggregate)
cudaError_t launch_spike_count(const uint32_t *words, uint32_t steps, uint64_t n_words, uint64_t n, uint32_t *counts, cudaStream_t s);
cudaError_t launch_pack_flags(const uint32_t *src, uint8_t *node_flags, uint64_t n, int shift, unsigned int *changed, cudaStream_t s);
cudaError_t launch_fill_u32(uint32_t *p, uint32_t v, uint64_t n, cudaStream_t s);
cudaError_t launch_bits_from_u32(const uint32_t *src, uint32_t *words, uint64_t n, uint64_t bit0, cudaStream_t s);
cudaError_t launch_u32_from_bits(const uint32_t *words, uint32_t *dst, uint64_t n, uint64_t bit0, cudaStream_t s);
cudaError_t launch_transpose_in(const float *src_nm, float *dst_tm, uint64_t n, uint64_t stride, cudaStream_t s);
cudaError_t launch_transpose_out(const float *src_tm, float *dst_nm, uint64_t n, uint64_t stride, cudaStream_t s);
// graph history (graph_history.cu): row_off[0 .. 32 n_slices] = exclusive prefix sum of the valid entries per table row, and one
// record of every table weight in canonical CSR order written to out[0 .. row_off[32 n_slices]); max_width = widest slice in k-rows
cudaError_t launch_graph_row_offsets(const uint32_t *col, const uint32_t *slice_off, uint32_t n_slices, uint32_t *row_off, cudaStream_t s);
cudaError_t launch_graph_record(const float *wgt, const uint32_t *slice_off, const uint32_t *row_off, uint32_t n_slices,
                                uint32_t max_width, float *out, cudaStream_t s);
// inclusive prefix sum of v[0, n) in place (one CTA: for the short arrays of per-tile or per-row counts)
cudaError_t launch_scan_u32(uint32_t *v, uint64_t n, cudaStream_t s);

// spike events (spike_events.cu): one lattice's bits [bit0, bit1) of a staged raster whose record s starts at raster + s * stride;
// words [w0, w0 + nw) hold them.  Its items (one per word and record) start at item0; an event is bit - bit0 + add.
struct EvSeg {
    const uint32_t *raster;
    uint32_t stride, w0, nw, bit0, bit1, add, item0;
};
struct EvParams {
    EvSeg seg[2 * kMaxLattices];   // neuron lattices, then spike-train lattices, in item order
    uint32_t n_seg, steps, n_items;
};
uint32_t ev_tiles(uint32_t n_items);
// tile_off[0 .. ev_tiles(n_items)]: events before each tile, the chunk's total last
cudaError_t launch_spike_event_count(const EvParams &p, uint32_t *tile_off, cudaStream_t s);
// events[0 .. total) in canonical order, rec_off[seg * steps + s] = events before record s of segment seg
cudaError_t launch_spike_event_scatter(const EvParams &p, const uint32_t *tile_off, uint32_t *events, uint32_t *rec_off, cudaStream_t s);

}  // namespace snn
