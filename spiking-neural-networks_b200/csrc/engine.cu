// engine.cu — host runtime: device memory layout, named-field I/O, graph ingestion, the step loop.
#include "engine.h"
#include <chrono>
#include <cmath>

#include <algorithm>
#include <atomic>
#include <thread>
#include <cstdio>
#include <cstring>
#include <functional>
#include <numeric>

namespace snn {

#define CK(call, status)                                                          \
    do {                                                                          \
        cudaError_t _e = (call);                                                  \
        if (_e != cudaSuccess) return cuda_fail(_e, (status), #call);             \
    } while (0)

static inline uint64_t round_up(uint64_t x, uint64_t m) { return (x + m - 1) / m * m; }

// Host -> device copy that has LANDED when it returns.  A plain cudaMemcpy from pageable memory may return once the data sits in
// the driver's staging buffer; the engine's kernels run on a non-blocking stream that does not wait for the legacy stream's DMA,
// so a kernel launched right after could read an array whose tail has not arrived yet (seen as garbage in the last slices of a
// rebuilt graph).  Copy on the engine's stream and wait for it.
static cudaError_t h2d_sync(void *dst, const void *src, size_t bytes, cudaStream_t s) {
    if (bytes == 0) return cudaSuccess;
    cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, s);
    return e != cudaSuccess ? e : cudaStreamSynchronize(s);
}

template <class T>
static cudaError_t dev_alloc(T **p, size_t n) {
    *p = nullptr;
    return cudaMalloc((void **)p, std::max<size_t>(n, 1) * sizeof(T));
}

static uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

Engine::Engine(int model_, int ntk_, int rck_, int train_kind_, int refract_, int device_)
    : model(model_), ntk(ntk_), rck(rck_), train_kind(train_kind_), refract(refract_), device(device_) {
    // handles of one process get distinct (but reproducible) default keys: two networks built the same way must not replay the
    // same Poisson noise; SNN_OPT_RNG_SEED pins the key
    static std::atomic<uint64_t> serial{0};
    seed = splitmix64(0x5EED5EEDull + serial.fetch_add(1));
}

static void unmap_peer(PeerMap &m) {
    if (m.ipc) { cudaIpcCloseMemHandle(m.slab); cudaIpcCloseMemHandle(m.flags); }
    m = PeerMap{};
}

Engine::~Engine() {
    if (device >= 0) cudaSetDevice(device);
    for (auto &m : strip_map_) unmap_peer(m);
    for (auto &G : gpeers_) unmap_peer(G.map);
    if (d_gpeers_) cudaFree(d_gpeers_);
    if (d_gexp_off_) cudaFree(d_gexp_off_);
    if (d_gexp_ent_) cudaFree(d_gexp_ent_);
    if (d_gslice_) cudaFree(d_gslice_);
    if (d_gact_) cudaFree(d_gact_);
    free_device();
    if (flags_) cudaFree(flags_);
    if (halo_done_) cudaFree(halo_done_);
    if (multi_barrier_) cudaFree(multi_barrier_);
    if (stdp_tab_) cudaFree(stdp_tab_);
    if (wide_scratch_) cudaFree(wide_scratch_);
    if (scratch_) cudaFree(scratch_);
    if (ghist_row_off_) cudaFree(ghist_row_off_);
    if (ev_bounce_) cudaFreeHost(ev_bounce_);
    if (ev0_) cudaEventDestroy(ev0_);
    if (ev1_) cudaEventDestroy(ev1_);
    if (stream_) cudaStreamDestroy(stream_);
}

int Engine::cuda_fail(cudaError_t e, int status, const char *what) {
    char buf[512];
    snprintf(buf, sizeof buf, "%s: %s (%s)", what, cudaGetErrorString(e), cudaGetErrorName(e));
    last_error = buf;
    cudaGetLastError();
    return status;
}

int Engine::init() {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        cudaGetLastError();
        return fail(SNN_GPU_GET_DEVICE_FAILURE, "no CUDA device available (this library has no CPU fallback)");
    }
    if (device < 0) {
        if (cudaGetDevice(&device) != cudaSuccess) return fail(SNN_GPU_GET_DEVICE_FAILURE, "cudaGetDevice failed");
    }
    if (device >= count) return fail(SNN_GPU_GET_DEVICE_FAILURE, "device ordinal out of range");
    CK(cudaSetDevice(device), SNN_GPU_GET_DEVICE_FAILURE);
    CK(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking), SNN_GPU_QUEUE_FAILURE);
    CK(cudaEventCreate(&ev0_), SNN_GPU_QUEUE_FAILURE);
    CK(cudaEventCreate(&ev1_), SNN_GPU_QUEUE_FAILURE);
    // [0],[1] step arrivals from rank-1 / rank+1, [2],[3] edge-kernel arrivals, [8 + r] general-graph partition: rank r completed a step
    CK(dev_alloc(&flags_, 8 + kMaxRanks), SNN_GPU_BUFFER_CREATE_ERROR);
    CK(cudaMemsetAsync(flags_, 0, (8 + kMaxRanks) * sizeof(unsigned long long), stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    CK(dev_alloc(&multi_barrier_, 1), SNN_GPU_BUFFER_CREATE_ERROR);
    CK(dev_alloc(&halo_done_, 8), SNN_GPU_BUFFER_CREATE_ERROR);  // [0],[1] completion counters, [2] halo time-out flag, [3] per-edge kernel CTAs done, [4],[5] halo wait counters, [6] general-partition slices done
    CK(cudaMemsetAsync(halo_done_, 0, 8 * sizeof(unsigned int), stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    CK(cudaStreamSynchronize(stream_), SNN_GPU_WAIT_ERROR);
    return SNN_OK;
}

int Engine::ensure_scratch(size_t bytes) {
    if (bytes <= scratch_bytes_) return SNN_OK;
    if (scratch_) cudaFree(scratch_);
    scratch_ = nullptr; scratch_bytes_ = 0;
    CK(cudaMalloc(&scratch_, bytes), SNN_GPU_BUFFER_CREATE_ERROR);
    scratch_bytes_ = bytes;
    return SNN_OK;
}

Lat *Engine::find(uint64_t id) {
    for (auto &L : lats_) if (L.id == id) return &L;
    return nullptr;
}
const Lat *Engine::find(uint64_t id) const {
    for (auto &L : lats_) if (L.id == id) return &L;
    return nullptr;
}

// ------------------------------------------------------------------------------------------------
// layout
// ------------------------------------------------------------------------------------------------
void Engine::compute_layout() {
    // canonical order: neuron lattices by ascending id, then spike-train lattices by ascending id
    std::stable_sort(lats_.begin(), lats_.end(), [](const Lat &a, const Lat &b) {
        if (a.is_train != b.is_train) return !a.is_train;
        return a.id < b.id;
    });
    n_neurons = n_trains = 0;
    for (auto &L : lats_) {
        if (L.is_train) { L.off = n_trains; n_trains += L.n; }
        else { L.off = n_neurons; n_neurons += L.n; }
    }
    // row strips: `halo_` ghost rows on each side that has a neighbour; general-graph partition: the ghost lists themselves
    const uint32_t halo_lo = gpart_ ? (uint32_t)g_lo_.size() : ((part_world > 1 && part_rank > 0) ? halo_ : 0);
    const uint32_t halo_hi = gpart_ ? (uint32_t)g_hi_.size() : ((part_world > 1 && part_rank < part_world - 1) ? halo_ : 0);
    own0_ = (uint32_t)round_up(halo_lo, 32);
    train0_ = (uint32_t)round_up(own0_ + n_neurons, 32);
    // upper ghosts follow the owned neurons without a gap: the stencil generator addresses the row below the strip as
    // own0 + rows_local * cols + c
    ghost_hi0_ = (part_world > 1) ? own0_ + (uint32_t)n_neurons : train0_;
    n_nodes_ = (part_world > 1) ? ghost_hi0_ + halo_hi : train0_ + (uint32_t)n_trains;
    // capacities cover whole 256-neuron tiles so that the TMA-staged kernel may copy full tiles past the last neuron
    node_cap_ = round_up(std::max<uint64_t>(n_nodes_, 1), 32) + kTmaTile + 32;
    neuron_cap_ = round_up(std::max<uint64_t>(n_neurons, 1), kTmaTile);
    train_cap_ = round_up(std::max<uint64_t>(n_trains, 1), 32);
}

void Engine::free_device() {
    auto fr = [](auto *&p) { if (p) cudaFree(p); p = nullptr; };
    if (slab_) cudaFree(slab_);
    slab_ = nullptr;
    V_[0] = V_[1] = nullptr; LFT_[0] = LFT_[1] = nullptr; T_[0] = T_[1] = nullptr; ACT_[0] = ACT_[1] = nullptr;
    fr(SPK_[0]); fr(SPK_[1]); fr(was_inc_);
    node_flags_ = nullptr;   // lives in the slab
    for (auto &p : NT_) fr(p);
    for (auto &p : F_) fr(p);
    for (auto &p : RC_) fr(p);
    for (auto &p : TF_) fr(p);
    fr(ft_off_); fr(ft_); fr(d_lat_);
    fr(slice_off_); fr(col_); fr(wgt_);
    fr(tile_par_); tile_par_bytes_ = 0; tile_par_dirty_ = true;
    free_reward_arrays();
    chem_alloc_ = false;
    graph_dirty_ = true;
    grid_fast_ = false;
}

static cudaError_t fill_f32(float *p, float v, uint64_t n, cudaStream_t s) {
    uint32_t b; memcpy(&b, &v, 4);
    return launch_fill_u32((uint32_t *)p, b, n, s);
}

int Engine::alloc_device() {
    CK(cudaSetDevice(device), SNN_GPU_GET_DEVICE_FAILURE);
    // slab: V[2], LFT[2] (+ T[2] once chemistry is touched) in one allocation so that a neighbouring rank can
    // map all halo-visible arrays with one CUDA IPC handle
    const size_t vb = round_up(node_cap_ * 4, 256);
    slab_off_v_[0] = 0; slab_off_v_[1] = vb; slab_off_lft_[0] = 2 * vb; slab_off_lft_[1] = 3 * vb;
    // node flags ride in the slab too: a neighbouring strip reads the neurotransmitter type sets of my boundary rows at attach time
    const size_t fbytes = round_up(node_cap_, 256);
    slab_off_flags_ = 4 * vb;
    // BCM Izhikevich strips and partitions: ACT[2] after the flags (the model is fixed at create time, so BCM plasticity may be
    // switched on at any point before run; no other handle carries these bytes)
    const bool act = model == SNN_MODEL_BCM_IZHIKEVICH && part_world > 1;
    slab_off_act_[0] = act ? 4 * vb + fbytes : 0; slab_off_act_[1] = act ? 5 * vb + fbytes : 0;
    slab_off_t_[0] = (act ? 6 * vb : 4 * vb) + fbytes; slab_off_t_[1] = slab_off_t_[0] + round_up(node_cap_ * 4 * kNT, 256);
    slab_bytes_ = slab_off_t_[0];  // T appended by ensure_chem (which reallocates the slab)
    CK(cudaMalloc(&slab_, slab_bytes_), SNN_GPU_BUFFER_CREATE_ERROR);
    node_flags_ = (uint8_t *)slab_ + slab_off_flags_;
    for (int k = 0; k < 2; ++k) {
        V_[k] = (float *)((char *)slab_ + slab_off_v_[k]);
        LFT_[k] = (int *)((char *)slab_ + slab_off_lft_[k]);
        if (act) {
            ACT_[k] = (float *)((char *)slab_ + slab_off_act_[k]);
            CK(fill_f32(ACT_[k], 0.f, node_cap_, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
        }
        CK(fill_f32(V_[k], 0.f, node_cap_, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
        CK(launch_fill_u32((uint32_t *)LFT_[k], 0xFFFFFFFFu, node_cap_, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
        CK(dev_alloc(&SPK_[k], node_cap_ / 32 + 1), SNN_GPU_BUFFER_CREATE_ERROR);
        CK(launch_fill_u32(SPK_[k], 0u, node_cap_ / 32 + 1, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    }
    CK(cudaMemsetAsync(node_flags_, 0, node_cap_, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    h_node_flags_.assign(node_cap_, 0);
    flags_cache_valid_ = false;
    // neuron fields used by this model
    for (int i = 0; i < kNumNeuronFields; ++i) {
        const FieldDef &fd = kNeuronFields[i];
        if (fd.kind != FK_NEURON_DEV || !(fd.models & SNN_M(model))) continue;
        CK(dev_alloc(&F_[fd.slot], neuron_cap_), SNN_GPU_BUFFER_CREATE_ERROR);
        CK(fill_f32(F_[fd.slot], neuron_default(model, fd.kind, fd.slot), neuron_cap_, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    }
    if (model == SNN_MODEL_HODGKIN_HUXLEY) {
        CK(dev_alloc(&was_inc_, neuron_cap_ / 32 + 1), SNN_GPU_BUFFER_CREATE_ERROR);
        CK(launch_fill_u32(was_inc_, 0u, neuron_cap_ / 32 + 1, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    }
    // neuron voltage default
    if (n_neurons)
        CK(fill_f32(V_[0] + own0_, neuron_default(model, FK_V, 0), n_neurons, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    if (n_neurons) CK(fill_f32(V_[1] + own0_, neuron_default(model, FK_V, 0), n_neurons, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    // trains
    if (n_trains) {
        for (int s = 0; s < TF_COUNT; ++s) {
            CK(dev_alloc(&TF_[s], train_cap_), SNN_GPU_BUFFER_CREATE_ERROR);
            CK(fill_f32(TF_[s], train_default(s), train_cap_, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
        }
        std::vector<uint64_t> zero(n_trains + 1, 0);
        CK(dev_alloc(&ft_off_, n_trains + 1), SNN_GPU_BUFFER_CREATE_ERROR);
        CK(cudaMemcpyAsync(ft_off_, zero.data(), (n_trains + 1) * 8, cudaMemcpyHostToDevice, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
        CK(dev_alloc(&ft_, 1), SNN_GPU_BUFFER_CREATE_ERROR);
        CK(cudaStreamSynchronize(stream_), SNN_GPU_WAIT_ERROR);
    }
    CK(dev_alloc(&d_lat_, kMaxLattices), SNN_GPU_BUFFER_CREATE_ERROR);
    for (auto &L : lats_) {
        if (L.is_train) continue;
        if (L.cold[0].size() != L.n) L.cold[0].assign(L.n, neuron_default(model, FK_NEURON_COLD, 0));
        if (L.cold[1].size() != L.n) L.cold[1].assign(L.n, neuron_default(model, FK_NEURON_COLD, 1));
    }
    cur_ = 0; lft_loc_ = 0;
    CK(cudaStreamSynchronize(stream_), SNN_GPU_WAIT_ERROR);
    return SNN_OK;
}

int Engine::ensure_chem() {
    if (chem_alloc_) return SNN_OK;
    if (layout_frozen_) return fail(SNN_UNSUPPORTED, "chemical fields must be set before the halo slab is exported");
    CK(cudaSetDevice(device), SNN_GPU_GET_DEVICE_FAILURE);
    // grow the slab to hold T[2]
    const size_t tb = round_up(node_cap_ * 4 * kNT, 256);
    const size_t new_bytes = slab_off_t_[0] + 2 * tb;
    void *ns = nullptr;
    CK(cudaMalloc(&ns, new_bytes), SNN_GPU_BUFFER_CREATE_ERROR);
    CK(cudaMemcpyAsync(ns, slab_, slab_bytes_, cudaMemcpyDeviceToDevice, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    CK(cudaMemsetAsync((char *)ns + slab_off_t_[0], 0, 2 * tb, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    CK(cudaStreamSynchronize(stream_), SNN_GPU_WAIT_ERROR);
    cudaFree(slab_);
    slab_ = ns; slab_bytes_ = new_bytes;
    for (int k = 0; k < 2; ++k) {
        V_[k] = (float *)((char *)slab_ + slab_off_v_[k]);
        LFT_[k] = (int *)((char *)slab_ + slab_off_lft_[k]);
        T_[k] = (float *)((char *)slab_ + slab_off_t_[k]);
        if (ACT_[k]) ACT_[k] = (float *)((char *)slab_ + slab_off_act_[k]);
    }
    node_flags_ = (uint8_t *)slab_ + slab_off_flags_;
    for (int s = 0; s < NTF_COUNT; ++s) {
        CK(dev_alloc(&NT_[s], node_cap_ * kNT), SNN_GPU_BUFFER_CREATE_ERROR);
        CK(fill_f32(NT_[s], nt_default(ntk, s), node_cap_ * kNT, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    }
    for (int s = 0; s < RCF_COUNT; ++s) {
        CK(dev_alloc(&RC_[s], neuron_cap_ * kNT), SNN_GPU_BUFFER_CREATE_ERROR);
        for (int ty = 0; ty < kNT; ++ty)
            CK(fill_f32(RC_[s] + (size_t)ty * neuron_cap_, rc_default(rck, ty, s), neuron_cap_, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    }
    CK(cudaStreamSynchronize(stream_), SNN_GPU_WAIT_ERROR);
    chem_alloc_ = true;
    tile_par_dirty_ = true;
    return SNN_OK;
}

int Engine::set_partition(uint32_t rows_g, uint32_t cols, int rank, int world) {
    if (!lats_.empty()) return fail(SNN_INVALID_ARGUMENT, "set_partition must precede add_lattice");
    if (world < 1 || rank < 0 || rank >= world) return fail(SNN_INVALID_ARGUMENT, "bad partition rank/world");
    part_rank = rank; part_world = world; rows_global = rows_g;
    row0_global = snn_partition_begin(rows_g, world, rank);
    halo_ = world > 1 ? cols : 0;  // one grid row; grows with the stencil radius (connect_grid)
    return SNN_OK;
}

int Engine::add_lattice(uint64_t id, uint32_t rows, uint32_t cols, bool is_train, bool is_reward) {
    // LatticeNetwork::add_lattice / add_spike_train_lattice, neuron/mod.rs:1663-1698
    if (find(id)) return fail(SNN_NET_GRAPH_ID_ALREADY_PRESENT, "Graph id already present in network, id: " + std::to_string(id));
    if (!is_train && n_neuron_lattices() >= kMaxLattices) return fail(SNN_UNSUPPORTED, "too many lattices");
    if (part_world > 1 && (!lats_.empty() || is_train)) return fail(SNN_UNSUPPORTED, "a partitioned handle holds exactly one neuron lattice");
    if (is_reward && (is_train || part_world > 1 || reward_mode || bcm_mode))
        return fail(SNN_UNSUPPORTED, "reward-modulated lattices of a network: single-GPU network handles only");
    Lat nl;
    nl.is_reward = is_reward;   // RewardModulatedLatticeNetwork::add_reward_modulated_lattice, neuron/mod.rs:3615-3634
    nl.id = id; nl.rows = rows; nl.cols = cols; nl.n = (uint64_t)rows * cols; nl.is_train = is_train;
    if ((is_train ? n_trains : n_neurons) + nl.n + 64ull * (part_world > 1 ? cols : 0) > kMaxNodes)
        return fail(SNN_UNSUPPORTED, "lattice too large for one device (node index is 28 bits)");
    // lattices are added at set-up time; the single-lattice (large) case never has anything to snapshot
    if (dev_weights_newer_) { int r = sync_weights_to_host(); if (r) return r; }
    return relayout([&]() { lats_.push_back(nl); });
}

// Rebuild the device layout after `change` alters its parameters: snapshot every field through the public get path, free,
// change, allocate, restore.
int Engine::relayout(const std::function<void()> &change) {
    struct FieldSnap { uint64_t id; std::string name; int dtype; uint64_t count; std::vector<uint8_t> data; };
    std::vector<FieldSnap> snaps;
    const bool had_chem = chem_alloc_;
    int r = SNN_OK;
    for (auto &L : lats_) {
        for_each_field(L, [&](const FieldDef &fd, const char *name) {
            const bool is_chem = fd.kind == FK_NT_FLAGS || fd.kind == FK_NT_T || fd.kind == FK_NT || fd.kind == FK_RC_FLAGS || fd.kind == FK_RC;
            if (is_chem && !had_chem) return false;
            FieldSnap f{L.id, name, fd.dtype, L.n * fd.per, {}};
            f.data.resize(std::max<uint64_t>(f.count, 1) * 4);
            r = get_field(L.id, name, f.data.data(), f.count, fd.dtype);
            if (!r) snaps.push_back(std::move(f));
            return r != SNN_OK;
        });
        if (r) return r;
    }
    const uint64_t saved_clock = internal_clock;
    free_device();
    change();
    compute_layout();
    r = alloc_device();
    if (r) return r;
    if (had_chem) { r = ensure_chem(); if (r) return r; }
    for (auto &f : snaps) {
        r = set_field(f.id, f.name.c_str(), f.data.data(), f.count, f.dtype);
        if (r) return r;
    }
    // re-upload preset firing times
    for (auto &L : lats_)
        if (L.is_train && !L.ft_off.empty()) {
            std::vector<uint64_t> off = L.ft_off; std::vector<float> t = L.ft;
            r = set_preset_firing_times(L.id, off.data(), t.data(), L.n, t.size());
            if (r) return r;
        }
    internal_clock = saved_clock;
    graph_dirty_ = true;
    return SNN_OK;
}

// ------------------------------------------------------------------------------------------------
// field directory
// ------------------------------------------------------------------------------------------------
static bool field_visible(const FieldDef &fd, int kind_bit, int ntk_) {
    if (!(fd.models & SNN_M(kind_bit))) return false;
    if (fd.kind == FK_NT && fd.aux && !(fd.aux & SNN_M(ntk_))) return false;
    return true;
}

// The directory of lattice L in index order: f(fd, name) for every field of this handle's model (or train kind) and kinetics,
// until f returns true.  Receptor fields are generated per type (fd.name == nullptr); `name` then points into a buffer of this
// call that the next field overwrites.
template <class F>
void Engine::for_each_field(const Lat &L, F &&f) const {
    const FieldDef *tab = L.is_train ? kTrainFields : kNeuronFields;
    const int n = L.is_train ? kNumTrainFields : kNumNeuronFields;
    for (int i = 0; i < n; ++i)
        if (field_visible(tab[i], L.is_train ? train_kind : model, ntk) && f(tab[i], tab[i].name)) return;
    if (L.is_train) return;
    char buf[128];
    for (int ty = 0; ty < kNT; ++ty)
        for (const RcFieldDef &rf : kRcFields) {
            if (rf.nmda_only && ty != SNN_NT_NMDA) continue;
            if (rf.kinetics_mask && !(rf.kinetics_mask & SNN_M(rck))) continue;
            snprintf(buf, sizeof buf, "receptors$%s%s", kRcTypeNames[ty], rf.suffix);
            if (f(FieldDef{nullptr, SNN_F32, 1, FK_RC, rf.slot, ty, kAllModels}, (const char *)buf)) return;
        }
}

int Engine::field_count(uint64_t id, uint32_t *count) const {
    const Lat *L = find(id);
    if (!L) return SNN_NET_ID_NOT_FOUND_IN_LATTICES;
    uint32_t c = 0;
    for_each_field(*L, [&](const FieldDef &, const char *) { ++c; return false; });
    *count = c;
    return SNN_OK;
}

static thread_local char g_name_buf[128];

int Engine::field_info(uint64_t id, uint32_t index, const char **name, int32_t *dtype, uint32_t *per) const {
    const Lat *L = find(id);
    if (!L) return SNN_NET_ID_NOT_FOUND_IN_LATTICES;
    uint32_t c = 0;
    bool found = false;
    for_each_field(*L, [&](const FieldDef &fd, const char *nm) {
        if (c++ != index) return false;
        // a generated receptor name is handed out from this thread's buffer, valid until the next call that returns one
        *name = fd.name ? fd.name : strcpy(g_name_buf, nm);
        *dtype = fd.dtype; *per = fd.per;
        return found = true;
    });
    return found ? SNN_OK : SNN_INVALID_ARGUMENT;
}

int Engine::lookup_field(const Lat &L, const char *name, FieldDef *out) const {
    bool found = false;
    for_each_field(L, [&](const FieldDef &fd, const char *nm) {
        if (strcmp(nm, name)) return false;
        *out = fd;
        return found = true;
    });
    return found ? SNN_OK : SNN_UNKNOWN_FIELD;
}

// ------------------------------------------------------------------------------------------------
// field I/O
// ------------------------------------------------------------------------------------------------
int Engine::set_bits(uint32_t *words, const uint32_t *host_u32, uint64_t n, uint64_t bit0) {
    int r = ensure_scratch(n * 4);
    if (r) return r;
    CK(cudaMemcpyAsync(scratch_, host_u32, n * 4, cudaMemcpyHostToDevice, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    CK(launch_bits_from_u32((const uint32_t *)scratch_, words, n, bit0, stream_), SNN_GPU_QUEUE_FAILURE);
    CK(cudaStreamSynchronize(stream_), SNN_GPU_WAIT_ERROR);
    return SNN_OK;
}

int Engine::get_bits(const uint32_t *words, uint32_t *host_u32, uint64_t n, uint64_t bit0) {
    int r = ensure_scratch(n * 4);
    if (r) return r;
    CK(launch_u32_from_bits(words, (uint32_t *)scratch_, n, bit0, stream_), SNN_GPU_QUEUE_FAILURE);
    CK(cudaMemcpyAsync(host_u32, scratch_, n * 4, cudaMemcpyDeviceToHost, stream_), SNN_GPU_BUFFER_READ_ERROR);
    CK(cudaStreamSynchronize(stream_), SNN_GPU_WAIT_ERROR);
    return SNN_OK;
}

int Engine::field_io(Lat &L, const FieldDef &fd, void *data, uint64_t count, bool set) {
    CK(cudaSetDevice(device), SNN_GPU_GET_DEVICE_FAILURE);
    const uint64_t n = L.n;
    if (n == 0) return SNN_OK;
    const uint32_t no = node_off(L);
    const cudaMemcpyKind dir = set ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost;
    const int wr = set ? SNN_GPU_BUFFER_WRITE_ERROR : SNN_GPU_BUFFER_READ_ERROR;
    auto plain = [&](void *dev, uint64_t elems) -> int {
        if (set) CK(cudaMemcpyAsync(dev, data, elems * 4, dir, stream_), wr);
        else CK(cudaMemcpyAsync(data, dev, elems * 4, dir, stream_), wr);
        CK(cudaStreamSynchronize(stream_), SNN_GPU_WAIT_ERROR);
        return SNN_OK;
    };
    // neuron-major [n][3] host <-> type-major device [3][stride] at element offset `o`
    auto typed = [&](float *dev_tm, uint64_t stride, uint64_t o) -> int {
        int r = ensure_scratch(n * kNT * 4);
        if (r) return r;
        if (set) {
            CK(cudaMemcpyAsync(scratch_, data, n * kNT * 4, cudaMemcpyHostToDevice, stream_), wr);
            CK(launch_transpose_in((const float *)scratch_, dev_tm + o, n, stride, stream_), SNN_GPU_QUEUE_FAILURE);
        } else {
            CK(launch_transpose_out(dev_tm + o, (float *)scratch_, n, stride, stream_), SNN_GPU_QUEUE_FAILURE);
            CK(cudaMemcpyAsync(data, scratch_, n * kNT * 4, cudaMemcpyDeviceToHost, stream_), wr);
        }
        CK(cudaStreamSynchronize(stream_), SNN_GPU_WAIT_ERROR);
        return SNN_OK;
    };
    if (set && (fd.kind == FK_NEURON_DEV || fd.kind == FK_NT || fd.kind == FK_RC)) tile_par_dirty_ = true;
    switch (fd.kind) {
    case FK_NEURON_DEV:
        return plain(F_[fd.slot] + L.off, n);
    case FK_NEURON_COLD:
        if (set) memcpy(L.cold[fd.slot].data(), data, n * 4); else memcpy(data, L.cold[fd.slot].data(), n * 4);
        return SNN_OK;
    case FK_V:
        return plain(V_[cur_] + no, n);
    case FK_LFT: {
        int r = plain(LFT_[lft_loc_] + no, n);
        if (r) return r;
        if (set && part_world > 1)  // keep both parities coherent for the halo protocol
            CK(cudaMemcpyAsync(LFT_[lft_loc_ ^ 1] + no, LFT_[lft_loc_] + no, n * 4, cudaMemcpyDeviceToDevice, stream_), wr);
            CK(cudaStreamSynchronize(stream_), SNN_GPU_WAIT_ERROR);
        return SNN_OK;
    }
    case FK_SPIKING:
        return set ? set_bits(SPK_[cur_], (const uint32_t *)data, n, no) : get_bits(SPK_[cur_], (uint32_t *)data, n, no);
    case FK_WAS_INC:
        return set ? set_bits(was_inc_, (const uint32_t *)data, n, L.off) : get_bits(was_inc_, (uint32_t *)data, n, L.off);
    case FK_NT_FLAGS:
    case FK_RC_FLAGS: {
        const int shift = fd.kind == FK_NT_FLAGS ? 0 : 4;
        uint32_t *h = (uint32_t *)data;
        if (set) {
            int r = ensure_chem();
            if (r) return r;
            bool changed = false;
            if (n >= (1u << 16)) {
                // large lattices: pack on the device (a host loop over 3 n words costs more than the copy), then refresh
                // the host mirror only if something changed
                r = ensure_scratch(n * kNT * 4 + 16);
                if (r) return r;
                unsigned int *d_changed = (unsigned int *)((char *)scratch_ + n * kNT * 4);
                CK(cudaMemsetAsync(d_changed, 0, 4, stream_), wr);
                CK(cudaMemcpyAsync(scratch_, h, n * kNT * 4, cudaMemcpyHostToDevice, stream_), wr);
                CK(launch_pack_flags((const uint32_t *)scratch_, node_flags_ + no, n, shift, d_changed, stream_), SNN_GPU_QUEUE_FAILURE);
                unsigned int hc = 0;
                CK(cudaMemcpyAsync(&hc, d_changed, 4, cudaMemcpyDeviceToHost, stream_), wr);
                CK(cudaStreamSynchronize(stream_), SNN_GPU_WAIT_ERROR);
                changed = hc != 0;
                if (changed) CK(cudaMemcpy(h_node_flags_.data() + no, node_flags_ + no, n, cudaMemcpyDeviceToHost), SNN_GPU_BUFFER_READ_ERROR);
            } else {
                for (uint64_t i = 0; i < n; ++i) {
                    uint8_t m = 0;
                    for (int ty = 0; ty < kNT; ++ty) if (h[i * kNT + ty]) m |= (uint8_t)(1u << ty);
                    uint8_t &f = h_node_flags_[no + i];
                    const uint8_t nf = (uint8_t)((f & ~(0xFu << shift)) | (m << shift));
                    changed |= nf != f;
                    f = nf;
                }
                if (changed) {
                    CK(cudaMemcpyAsync(node_flags_ + no, h_node_flags_.data() + no, n, cudaMemcpyHostToDevice, stream_), wr);
                    CK(cudaStreamSynchronize(stream_), SNN_GPU_WAIT_ERROR);
                }
            }
            if (!changed) return SNN_OK;
            flags_cache_valid_ = false;
            if (shift == 0) {
                // the presynaptic type bits are baked into the edge words: re-encode at the next run
                if (dev_weights_newer_) { r = sync_weights_to_host(); if (r) return r; }
                graph_dirty_ = true;
            }
        } else {
            for (uint64_t i = 0; i < n; ++i)
                for (int ty = 0; ty < kNT; ++ty) h[i * kNT + ty] = (h_node_flags_[no + i] >> (shift + ty)) & 1u;
        }
        return SNN_OK;
    }
    case FK_NT_T: {
        if (set) { int r = ensure_chem(); if (r) return r; }
        if (!chem_alloc_) { memset(data, 0, n * kNT * 4); return SNN_OK; }
        return typed(T_[cur_], node_cap_, no);
    }
    case FK_NT: {
        if (set) { int r = ensure_chem(); if (r) return r; }
        if (!chem_alloc_) {
            float *o = (float *)data;
            for (uint64_t i = 0; i < n * kNT; ++i) o[i] = nt_default(ntk, fd.slot);
            return SNN_OK;
        }
        return typed(NT_[fd.slot], node_cap_, no);
    }
    case FK_RC: {
        if (set) { int r = ensure_chem(); if (r) return r; }
        if (!chem_alloc_) {
            float *o = (float *)data;
            for (uint64_t i = 0; i < n; ++i) o[i] = rc_default(rck, fd.aux, fd.slot);
            return SNN_OK;
        }
        return plain(RC_[fd.slot] + (size_t)fd.aux * neuron_cap_ + L.off, n);
    }
    case FK_TRAIN_DEV:
    case FK_TRAIN_COUNTER:
        return plain(TF_[fd.slot] + L.off, n);
    }
    (void)count;
    return SNN_UNKNOWN_FIELD;
}

int Engine::set_field(uint64_t id, const char *name, const void *data, uint64_t count, int dtype) {
    Lat *L = find(id);
    if (!L) return fail(SNN_NET_ID_NOT_FOUND_IN_LATTICES, "Id not present in lattices, id: " + std::to_string(id));
    if (!name || (!data && L->n)) return fail(SNN_INVALID_ARGUMENT, "null argument");
    FieldDef fd;
    if (lookup_field(*L, name, &fd)) return fail(SNN_UNKNOWN_FIELD, std::string("unknown field: ") + name);
    if (dtype != fd.dtype) return fail(SNN_DTYPE_MISMATCH, std::string("dtype mismatch for field: ") + name);
    if (count != L->n * (uint64_t)fd.per) return fail(SNN_SIZE_MISMATCH, std::string("size mismatch for field: ") + name);
    return field_io(*L, fd, const_cast<void *>(data), count, true);
}

int Engine::get_field(uint64_t id, const char *name, void *out, uint64_t count, int dtype) {
    Lat *L = find(id);
    if (!L) return fail(SNN_NET_ID_NOT_FOUND_IN_LATTICES, "Id not present in lattices, id: " + std::to_string(id));
    if (!name || (!out && L->n)) return fail(SNN_INVALID_ARGUMENT, "null argument");
    FieldDef fd;
    if (lookup_field(*L, name, &fd)) return fail(SNN_UNKNOWN_FIELD, std::string("unknown field: ") + name);
    if (dtype != fd.dtype) return fail(SNN_DTYPE_MISMATCH, std::string("dtype mismatch for field: ") + name);
    if (count != L->n * (uint64_t)fd.per) return fail(SNN_SIZE_MISMATCH, std::string("size mismatch for field: ") + name);
    return field_io(*L, fd, out, count, false);
}

int Engine::fill_field(uint64_t id, const char *name, uint32_t bits, int dtype) {
    Lat *L = find(id);
    if (!L) return fail(SNN_NET_ID_NOT_FOUND_IN_LATTICES, "Id not present in lattices, id: " + std::to_string(id));
    FieldDef fd;
    if (!name || lookup_field(*L, name, &fd)) return fail(SNN_UNKNOWN_FIELD, std::string("unknown field: ") + (name ? name : "(null)"));
    if (dtype != fd.dtype) return fail(SNN_DTYPE_MISMATCH, std::string("dtype mismatch for field: ") + name);
    if (L->n == 0) return SNN_OK;
    CK(cudaSetDevice(device), SNN_GPU_GET_DEVICE_FAILURE);
    tile_par_dirty_ = true;
    // fast device-side fills for the plain arrays; everything else goes through the host path
    uint32_t *dev = nullptr;
    switch (fd.kind) {
    case FK_NEURON_DEV: dev = (uint32_t *)(F_[fd.slot] + L->off); break;
    case FK_V: dev = (uint32_t *)(V_[cur_] + node_off(*L)); break;
    case FK_TRAIN_DEV: case FK_TRAIN_COUNTER: dev = (uint32_t *)(TF_[fd.slot] + L->off); break;
    case FK_RC: { int r = ensure_chem(); if (r) return r; dev = (uint32_t *)(RC_[fd.slot] + (size_t)fd.aux * neuron_cap_ + L->off); break; }
    default: break;
    }
    if (dev) {
        CK(launch_fill_u32(dev, bits, L->n, stream_), SNN_GPU_QUEUE_FAILURE);
        CK(cudaStreamSynchronize(stream_), SNN_GPU_WAIT_ERROR);
        return SNN_OK;
    }
    std::vector<uint32_t> tmp(L->n * fd.per, bits);
    return field_io(*L, fd, tmp.data(), tmp.size(), true);
}

int Engine::set_preset_firing_times(uint64_t id, const uint64_t *offsets, const float *times, uint64_t nt, uint64_t n_times) {
    Lat *L = find(id);
    if (!L || !L->is_train) return fail(SNN_NET_ID_NOT_FOUND_IN_LATTICES, "Id not present in spike train lattices");
    if (train_kind != SNN_TRAIN_PRESET) return fail(SNN_UNSUPPORTED, "spike train type has no firing_times");
    if (nt != L->n || !offsets || offsets[nt] != n_times) return fail(SNN_SIZE_MISMATCH, "firing_times size mismatch");
    L->ft_off.assign(offsets, offsets + nt + 1);
    L->ft.assign(times, times + n_times);
    // rebuild the concatenated CSR over all train lattices
    std::vector<uint64_t> off(n_trains + 1, 0);
    std::vector<float> all;
    for (auto &X : lats_) {
        if (!X.is_train) continue;
        for (uint64_t i = 0; i < X.n; ++i) {
            off[X.off + i] = all.size();
            if (!X.ft_off.empty()) all.insert(all.end(), X.ft.begin() + X.ft_off[i], X.ft.begin() + X.ft_off[i + 1]);
        }
    }
    off[n_trains] = all.size();
    CK(cudaSetDevice(device), SNN_GPU_GET_DEVICE_FAILURE);
    if (ft_) cudaFree(ft_);
    CK(dev_alloc(&ft_, all.size()), SNN_GPU_BUFFER_CREATE_ERROR);
    CK(h2d_sync(ft_off_, off.data(), off.size() * 8, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    if (!all.empty()) CK(h2d_sync(ft_, all.data(), all.size() * 4, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    return SNN_OK;
}

// ------------------------------------------------------------------------------------------------
// general-graph partition (SURVEY 8e, second half): contiguous node ranges per rank, in-edges from any node of any rank
// ------------------------------------------------------------------------------------------------
// Node order on a rank: [ghosts below my range, ascending global index | my neurons | ghosts above], so local order == global
// order and the canonical (ascending presynaptic index) summation order of every row is the one of the unpartitioned lattice.
int Engine::gpart_enable(const std::vector<uint32_t> &remote) {
    if (layout_frozen_) return fail(SNN_UNSUPPORTED, "the graph of a partitioned handle cannot change its reach after the slab was exported");
    const uint64_t cols = lats_[0].cols, g0 = (uint64_t)row0_global * cols, g1 = g0 + n_neurons;
    std::vector<uint32_t> lo, hi;
    for (uint32_t g : remote) (g < g0 ? lo : hi).push_back(g);
    (void)g1;
    if (gpart_ && lo == g_lo_ && hi == g_hi_) return SNN_OK;
    for (int d = 0; d < 2; ++d) if (halo_dir_[d].active) return fail(SNN_UNSUPPORTED, "handle already attached as a row strip");
    int r = relayout([&]() { gpart_ = true; g_lo_ = lo; g_hi_ = hi; });
    if (r) return r;
    gpeers_.clear();
    gpart_dirty_ = true;
    return SNN_OK;
}

int64_t Engine::global_to_node(uint64_t g) const {
    const uint64_t cols = lats_.empty() ? 0 : lats_[0].cols, g0 = (uint64_t)row0_global * cols;
    if (g >= g0 && g < g0 + n_neurons) return (int64_t)own0_ + (int64_t)(g - g0);
    if (!gpart_) {
        const int64_t node = (int64_t)g + (int64_t)own0_ - (int64_t)g0;
        return (node < 0 || node >= (int64_t)n_nodes_) ? -1 : node;
    }
    const std::vector<uint32_t> &v = g < g0 ? g_lo_ : g_hi_;
    auto it = std::lower_bound(v.begin(), v.end(), (uint32_t)g);
    if (it == v.end() || *it != g) return -1;
    const uint64_t k = (uint64_t)(it - v.begin());
    return g < g0 ? (int64_t)own0_ - (int64_t)g_lo_.size() + (int64_t)k : (int64_t)ghost_hi0_ + (int64_t)k;
}

uint64_t Engine::node_to_global(uint32_t node) const {
    const uint64_t cols = lats_.empty() ? 0 : lats_[0].cols, g0 = (uint64_t)row0_global * cols;
    if (node >= own0_ && node < own0_ + n_neurons) return g0 + (node - own0_);
    if (!gpart_) return (uint64_t)((int64_t)node + (int64_t)g0 - (int64_t)own0_);
    if (node < own0_) return g_lo_[node - (own0_ - (uint32_t)g_lo_.size())];
    return g_hi_[node - ghost_hi0_];
}

Engine::GPeerHost *Engine::gpeer(int rank, bool create) {
    for (auto &g : gpeers_) if (g.rank == rank) return &g;
    if (!create) return nullptr;
    GPeerHost g; g.rank = rank;
    auto it = gpeers_.begin();
    while (it != gpeers_.end() && it->rank < rank) ++it;
    return &*gpeers_.insert(it, std::move(g));
}

int Engine::check_peer_rank(int peer) {
    if (part_world <= 1 || peer < 0 || peer >= part_world || peer == part_rank) return fail(SNN_INVALID_ARGUMENT, "bad peer rank");
    return SNN_OK;
}

int Engine::gpart_wants(int peer, uint32_t *global_idx, uint64_t capacity, uint64_t *n, uint32_t *first_slot) {
    if (int r = check_peer_rank(peer)) return r;
    if (n) *n = 0;
    if (first_slot) *first_slot = 0;
    if (!gpart_) return SNN_OK;   // a row strip has no gather lists
    const uint64_t cols = lats_[0].cols;
    const uint64_t q0 = (uint64_t)snn_partition_begin(rows_global, part_world, peer) * cols, q1 = (uint64_t)snn_partition_begin(rows_global, part_world, peer + 1) * cols;
    const std::vector<uint32_t> &v = peer < part_rank ? g_lo_ : g_hi_;
    auto a = std::lower_bound(v.begin(), v.end(), (uint32_t)q0), b = std::lower_bound(v.begin(), v.end(), (uint32_t)std::min<uint64_t>(q1, 0xFFFFFFFFull));
    const uint64_t cnt = (uint64_t)(b - a);
    if (n) *n = cnt;
    const uint32_t base = peer < part_rank ? own0_ - (uint32_t)g_lo_.size() : ghost_hi0_;
    if (first_slot) *first_slot = base + (uint32_t)(a - v.begin());
    if (global_idx) {
        if (capacity < cnt) return fail(SNN_SIZE_MISMATCH, "index buffer too small");
        std::copy(a, b, global_idx);
    }
    return SNN_OK;
}

int Engine::gpart_set_exports(int peer, const uint32_t *global_idx, uint64_t n, uint32_t first_slot_at_peer) {
    if (int r = check_peer_rank(peer)) return r;
    if (n && !global_idx) return fail(SNN_INVALID_ARGUMENT, "null argument");
    if (!gpart_) return fail(SNN_INVALID_ARGUMENT, "not a general-graph partition (set SNN_OPT_GENERAL_PARTITION before the graph on every rank)");
    if (n == 0 && !gpeer(peer, false)) return SNN_OK;
    const uint64_t cols = lats_[0].cols, g0 = (uint64_t)row0_global * cols;
    GPeerHost *G = gpeer(peer, true);
    G->exp_local.clear();
    for (uint64_t k = 0; k < n; ++k) {
        if (global_idx[k] < g0 || global_idx[k] >= g0 + n_neurons) return fail(SNN_GRAPH_POSITION_NOT_FOUND, "Position not found, position: " + std::to_string(global_idx[k]));
        if (k && global_idx[k] <= global_idx[k - 1]) return fail(SNN_INVALID_ARGUMENT, "export list must be ascending");
        G->exp_local.push_back((uint32_t)(global_idx[k] - g0));
    }
    G->peer_slot0 = first_slot_at_peer;
    gpart_dirty_ = true;
    return SNN_OK;
}

int Engine::gpart_attach(int peer, const IpcBlob *blob, Engine *local) {
    if (int r = check_peer_rank(peer)) return r;
    if (!gpart_) return fail(SNN_INVALID_ARGUMENT, "not a general-graph partition (set SNN_OPT_GENERAL_PARTITION before the graph on every rank)");
    CK(cudaSetDevice(device), SNN_GPU_GET_DEVICE_FAILURE);
    const GPeerHost *old = gpeer(peer, false);
    if (old && old->attached) return fail(SNN_INVALID_ARGUMENT, "peer already attached");
    GPeerHost G = old ? *old : GPeerHost{};
    G.rank = peer;
    int r = map_peer(blob, local, peer, &G.map, &G.view);
    if (r) return r;
    // the ghosts that this peer owns: slots slot0 .. slot0 + cnt - 1, at the peer's neuron numbers node_to_global(slot) - q0
    uint64_t cnt = 0; uint32_t slot0 = 0;
    r = gpart_wants(peer, nullptr, 0, &cnt, &slot0);
    if (!r && cnt) {
        const uint64_t q0 = (uint64_t)snn_partition_begin(rows_global, part_world, peer) * lats_[0].cols;
        std::vector<uint32_t> pick(cnt);
        for (uint64_t k = 0; k < cnt; ++k) pick[k] = (uint32_t)(node_to_global(slot0 + (uint32_t)k) - q0);
        r = import_ghost_flags(slot0, (const uint8_t *)G.map.slab + G.view.off_flags + G.view.own0, G.view.n_neurons, pick, false);
    }
    if (r) { unmap_peer(G.map); return r; }
    G.attached = true;
    *gpeer(peer, true) = std::move(G);
    layout_frozen_ = true;
    if (local) { local->layout_frozen_ = true; local_peers_.push_back(local); }
    gpart_dirty_ = true;
    return SNN_OK;
}

int Engine::gpart_build_device() {
    if (!gpart_dirty_) return SNN_OK;
    auto fr = [](auto *&p) { if (p) cudaFree(p); p = nullptr; };
    fr(d_gpeers_); fr(d_gexp_off_); fr(d_gexp_ent_); fr(d_gslice_); fr(d_gact_);
    if (gpeers_.size() > 15) return fail(SNN_UNSUPPORTED, "too many peers");
    std::vector<GPeer> hp(std::max<size_t>(gpeers_.size(), 1));
    std::vector<float *> act(2 * hp.size(), nullptr);
    std::vector<std::vector<uint32_t>> per(n_neurons);
    for (size_t q = 0; q < gpeers_.size(); ++q) {
        GPeerHost &G = gpeers_[q];
        if (!G.attached) return fail(SNN_INVALID_ARGUMENT, "general-graph partition: rank " + std::to_string(G.rank) + " is not attached");
        GPeer &D = hp[q];
        for (int k = 0; k < 2; ++k) {
            D.v[k] = (float *)((char *)G.map.slab + G.view.off_v[k]);
            D.lft[k] = (int *)((char *)G.map.slab + G.view.off_lft[k]);
            D.t[k] = (float *)((char *)G.map.slab + G.view.off_t[k]);
            if (ACT_[0]) act[2 * q + k] = (float *)((char *)G.map.slab + G.view.off_act[k]);
        }
        D.t_stride = G.view.t_stride;
        D.peer_flag = (unsigned long long *)G.map.flags + 8 + part_rank;
        D.my_flag = flags_ + 8 + G.rank;
        for (size_t k = 0; k < G.exp_local.size(); ++k) per[G.exp_local[k]].push_back(((uint32_t)q << 28) | (G.peer_slot0 + (uint32_t)k));
    }
    std::vector<uint32_t> off(n_neurons + 1, 0), ent;
    std::vector<uint8_t> gs(std::max<size_t>(n_slices_, 1), 0);
    for (uint64_t i = 0; i < n_neurons; ++i) {
        off[i] = (uint32_t)ent.size();
        ent.insert(ent.end(), per[i].begin(), per[i].end());
        if (!per[i].empty()) gs[i / 32] |= 2u;
    }
    off[n_neurons] = (uint32_t)ent.size();
    for (size_t sl = 0; sl < h_gslice_.size() && sl < gs.size(); ++sl) gs[sl] |= h_gslice_[sl] & 1u;
    CK(dev_alloc(&d_gpeers_, hp.size()), SNN_GPU_BUFFER_CREATE_ERROR);
    CK(dev_alloc(&d_gexp_off_, off.size()), SNN_GPU_BUFFER_CREATE_ERROR);
    CK(dev_alloc(&d_gexp_ent_, ent.size()), SNN_GPU_BUFFER_CREATE_ERROR);
    CK(dev_alloc(&d_gslice_, gs.size()), SNN_GPU_BUFFER_CREATE_ERROR);
    CK(h2d_sync(d_gpeers_, hp.data(), hp.size() * sizeof(GPeer), stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    CK(h2d_sync(d_gexp_off_, off.data(), off.size() * 4, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    CK(h2d_sync(d_gexp_ent_, ent.data(), ent.size() * 4, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    CK(h2d_sync(d_gslice_, gs.data(), gs.size(), stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    if (ACT_[0]) {
        CK(dev_alloc(&d_gact_, act.size()), SNN_GPU_BUFFER_CREATE_ERROR);
        CK(h2d_sync(d_gact_, act.data(), act.size() * sizeof(float *), stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    }
    gpart_dirty_ = false;
    return SNN_OK;
}

// ------------------------------------------------------------------------------------------------
// graph ingestion
// ------------------------------------------------------------------------------------------------
static int check_connect(Engine &E, uint64_t pre_id, uint64_t post_id, Lat **A, Lat **B) {
    // LatticeNetwork::connect preconditions, neuron/mod.rs:1852-1862
    Lat *pre = E.find(pre_id), *post = E.find(post_id);
    if (post && post->is_train)
        return E.fail(SNN_NET_POSTSYNAPTIC_LATTICE_CANNOT_BE_SPIKE_TRAIN,
                      "Postsynaptic lattice cannot be a spike train lattice because spike trains cannot take inputs");
    if (!pre) return E.fail(SNN_NET_PRESYNAPTIC_ID_NOT_FOUND, "Presynaptic id not present in network, id: " + std::to_string(pre_id));
    if (!post) return E.fail(SNN_NET_POSTSYNAPTIC_ID_NOT_FOUND, "Postsynaptic id not present in network, id: " + std::to_string(post_id));
    *A = pre; *B = post;
    return SNN_OK;
}

static void sort_rows(Block &b) {
    const uint64_t n = b.row_ptr.size() - 1;
    std::vector<std::pair<uint32_t, float>> tmp;
    for (uint64_t q = 0; q < n; ++q) {
        const uint64_t s = b.row_ptr[q], e = b.row_ptr[q + 1];
        bool sorted = true;
        for (uint64_t k = s + 1; k < e; ++k) if (b.pre[k - 1] > b.pre[k]) { sorted = false; break; }
        if (sorted) continue;
        tmp.clear();
        for (uint64_t k = s; k < e; ++k) tmp.emplace_back(b.pre[k], b.w[k]);
        std::stable_sort(tmp.begin(), tmp.end(), [](auto &x, auto &y) { return x.first < y.first; });
        for (uint64_t k = s; k < e; ++k) { b.pre[k] = tmp[k - s].first; b.w[k] = tmp[k - s].second; }
    }
}

int Engine::connect_dense(uint64_t pre_id, uint64_t post_id, const uint32_t *connections, const float *weights,
                          const uint32_t *itp, uint64_t n_pre, uint64_t n_post) {
    Lat *A, *B;
    int r = check_connect(*this, pre_id, post_id, &A, &B);
    if (r) return r;
    if (n_pre != A->n || n_post != B->n) return fail(SNN_GRAPH_DIMENSIONS_DO_NOT_MATCH, "Dimensions do not match");
    if (n_pre != 0 && n_post != 0 && (!connections || !weights)) return fail(SNN_INVALID_ARGUMENT, "null graph pointers");
    if ((r = refuse_if_graph_history("connect"))) return r;
    if (part_world > 1) return fail(SNN_UNSUPPORTED, "dense graphs are not supported on partitioned handles");
    if (itp) {
        if (pre_id != post_id) return fail(SNN_INVALID_ARGUMENT, "index_to_position only applies to an internal graph");
        for (uint64_t i = 0; i < n_pre; ++i)
            if (itp[i] >= n_pre) return fail(SNN_GRAPH_POSITION_NOT_FOUND, "Position not found, position: " + std::to_string(itp[i]));
    }
    if (dev_weights_newer_) { r = sync_weights_to_host(); if (r) return r; }
    Block b;
    b.kind = Block::CSR;
    b.row_ptr.assign(n_post + 1, 0);
    // rows are indexed by cell position; graph index g maps to position itp[g]
    std::vector<uint64_t> cnt(n_post + 1, 0);
    for (uint64_t q = 0; q < n_post; ++q) {
        const uint64_t qp = itp ? itp[q] : q;
        uint64_t c = 0;
        for (uint64_t p = 0; p < n_pre; ++p) if (connections[p * n_post + q]) c++;
        cnt[qp] = c;
    }
    for (uint64_t q = 0; q < n_post; ++q) b.row_ptr[q + 1] = b.row_ptr[q] + cnt[q];
    b.pre.resize(b.row_ptr[n_post]); b.w.resize(b.row_ptr[n_post]);
    for (uint64_t q = 0; q < n_post; ++q) {
        const uint64_t qp = itp ? itp[q] : q;
        uint64_t o = b.row_ptr[qp];
        for (uint64_t p = 0; p < n_pre; ++p)
            if (connections[p * n_post + q]) { b.pre[o] = (uint32_t)(itp ? itp[p] : p); b.w[o] = weights[p * n_post + q]; ++o; }
    }
    if (itp) sort_rows(b);
    blocks_[{pre_id, post_id}] = std::move(b);
    graph_dirty_ = true;
    return SNN_OK;
}

int Engine::connect_csr(uint64_t pre_id, uint64_t post_id, const uint64_t *row_ptr, const uint32_t *pre, const float *weights,
                        uint64_t n_post, uint64_t nnz) {
    Lat *A, *B;
    int r = check_connect(*this, pre_id, post_id, &A, &B);
    if (r) return r;
    if (n_post != B->n) return fail(SNN_GRAPH_DIMENSIONS_DO_NOT_MATCH, "Dimensions do not match");
    if (!row_ptr || (nnz && (!pre || !weights))) return fail(SNN_INVALID_ARGUMENT, "null graph pointers");
    if (row_ptr[0] != 0 || row_ptr[n_post] != nnz) return fail(SNN_SIZE_MISMATCH, "row_ptr does not match nnz");
    const uint64_t pre_limit = part_world > 1 ? (uint64_t)rows_global * A->cols : A->n;
    for (uint64_t k = 0; k < nnz; ++k)
        if (pre[k] >= pre_limit) return fail(SNN_GRAPH_PRESYNAPTIC_NOT_FOUND, "Presynaptic position not found, position: " + std::to_string(pre[k]));
    for (uint64_t q = 0; q < n_post; ++q)
        if (row_ptr[q + 1] < row_ptr[q]) return fail(SNN_INVALID_ARGUMENT, "row_ptr must be non-decreasing");
    if ((r = refuse_if_graph_history("connect"))) return r;
    if (dev_weights_newer_) { r = sync_weights_to_host(); if (r) return r; }
    Block b;
    b.kind = Block::CSR;
    b.row_ptr.assign(row_ptr, row_ptr + n_post + 1);
    b.pre.assign(pre, pre + nnz);
    b.w.assign(weights, weights + nnz);
    sort_rows(b);
    if (part_world > 1) {
        // edges that reach beyond the strip's halo rows (or any edge, once the handle is a general-graph partition): the ghosts
        // become gather lists of exactly the remote nodes this rank's rows read
        const int64_t g0 = (int64_t)row0_global * A->cols, g1 = g0 + (int64_t)A->n;
        bool beyond = gpart_ || force_gpart;
        std::vector<uint32_t> remote;
        for (uint64_t k = 0; k < nnz; ++k) {
            const int64_t g = b.pre[k];
            if (g >= g0 && g < g1) continue;
            remote.push_back((uint32_t)g);
            if (g < g0 - (int64_t)halo_ || g >= g1 + (int64_t)halo_) beyond = true;
        }
        if (beyond) {
            std::sort(remote.begin(), remote.end());
            remote.erase(std::unique(remote.begin(), remote.end()), remote.end());
            blocks_.clear();
            r = gpart_enable(remote);
            if (r) return r;
            A = B = find(pre_id);
        }
    }
    blocks_[{pre_id, post_id}] = std::move(b);
    graph_dirty_ = true;
    return SNN_OK;
}

int Engine::connect_grid(uint64_t id, uint32_t radius, float weight) {
    Lat *A, *B;
    int r = check_connect(*this, id, id, &A, &B);
    if (r) return r;
    if (radius > 7) return fail(SNN_UNSUPPORTED, "stencil radius too large");
    if ((r = refuse_if_graph_history("connect"))) return r;
    if (part_world > 1) {
        const uint32_t need = radius * A->cols;
        if (need > A->n && A->n) return fail(SNN_UNSUPPORTED, "strip is thinner than the stencil radius");
        if (need != halo_) {
            // re-layout with a halo of `radius` rows
            if (layout_frozen_) return fail(SNN_UNSUPPORTED, "cannot change the stencil after the halo slab was exported");
            r = relayout([&]() { halo_ = need; });
            if (r) return r;
        }
    }
    // the learned weights of every OTHER block live on the device until synced: replacing this block must not discard them
    if (dev_weights_newer_) {
        bool others = false;
        for (auto &kv : blocks_) others |= kv.first != std::make_pair(id, id);
        if (others) { r = sync_weights_to_host(); if (r) return r; }
    }
    Block b;
    b.kind = Block::GRID;
    b.radius = radius; b.weight = weight;
    blocks_[{id, id}] = std::move(b);
    dev_weights_newer_ = false;
    graph_dirty_ = true;
    return SNN_OK;
}

void Engine::materialize_grid(Block &b, const Lat &L) const {
    // host CSR of the Moore stencil (same enumeration order as sell_grid_kernel: ascending flat index)
    const int64_t R = b.radius, rows_g = part_world > 1 ? rows_global : L.rows, cols = L.cols;
    const int64_t r0 = part_world > 1 ? row0_global : 0;
    b.row_ptr.assign(L.n + 1, 0);
    b.pre.clear(); b.w.clear();
    for (int64_t i = 0; i < (int64_t)L.rows; ++i)
        for (int64_t j = 0; j < cols; ++j) {
            for (int64_t di = -R; di <= R; ++di)
                for (int64_t dj = -R; dj <= R; ++dj) {
                    const int64_t a = r0 + i + di, c = j + dj;
                    if ((di == 0 && dj == 0) || a < 0 || c < 0 || a >= rows_g || c >= cols) continue;
                    // pre index: global flat index on partitioned handles, local otherwise
                    b.pre.push_back((uint32_t)(a * cols + c));
                    b.w.push_back(b.weight);
                }
            b.row_ptr[i * cols + j + 1] = b.pre.size();
        }
    b.kind = Block::CSR;
    b.from_grid_radius = b.radius;
}

// `b` itself, or the host CSR of a stencil block materialised on `tmp`: the block stays a stencil, and with it the device fast
// path of finalize_graph
Block &Engine::csr_view(Block &b, const Lat &L, Block &tmp) const {
    if (b.kind != Block::GRID) return b;
    tmp = b;
    materialize_grid(tmp, L);
    return tmp;
}

// The row order of the device edge table: for every neuron lattice B (only `into`, if given), every row q and every block into B,
// f(B, q, A, b, k) with A the presynaptic lattice and k the offset of the block's edges within the row.  Blocks into a lattice
// follow the node offset of their presynaptic lattice, so that rows stay sorted by node index; each block's edges of the row
// keep its CSR order.  finalize_graph lays the table out in this order and every map from a host edge to a table element reads
// it back from here.  A stencil block is visited as its materialised copy.
template <class F>
void Engine::for_each_row_segment(F &&f, const Lat *into) {
    for (const Lat &B : lats_) {
        if (B.is_train || (into && &B != into)) continue;
        Block tmp;   // only a lattice's own graph can be a stencil
        std::vector<std::pair<const Lat *, Block *>> blocks;
        for (auto &kv : blocks_)
            if (kv.first.second == B.id) {
                const Lat *A = find(kv.first.first);
                if (A) blocks.emplace_back(A, &csr_view(kv.second, B, tmp));
            }
        std::sort(blocks.begin(), blocks.end(), [&](auto &x, auto &y) { return node_off(*x.first) < node_off(*y.first); });
        for (uint64_t q = 0; q < B.n; ++q) {
            uint64_t k = 0;
            for (auto &ab : blocks) {
                Block &b = *ab.second;
                f(B, q, *ab.first, b, k);
                k += b.row_ptr[q + 1] - b.row_ptr[q];
            }
        }
    }
}

static uint32_t stencil_width(uint32_t radius) { return (2 * radius + 1) * (2 * radius + 1) - 1; }

// k-rows of a uniform-width table: whole tiles of the TMA-staged kernel
static uint64_t uniform_table_krows(uint32_t n_slices, uint32_t width) { return round_up(n_slices, kTmaConsumerWarps) * width; }

// col_ / wgt_ for the table of which the builder writes the first sell_krows_ k-rows.  A uniform-width table (`width` > 0) is
// allocated to uniform_table_krows; the k-rows past the last slice are padding (col kColPad, weight 0).
int Engine::alloc_table(uint32_t width) {
    const uint64_t krows = width ? uniform_table_krows(n_slices_, width) : sell_krows_;
    CK(dev_alloc(&col_, krows * 32), SNN_GPU_BUFFER_CREATE_ERROR);
    CK(dev_alloc(&wgt_, krows * 32), SNN_GPU_BUFFER_CREATE_ERROR);
    if (!width) return SNN_OK;
    sell_alloc_krows_ = krows;
    if (krows > sell_krows_) {
        CK(cudaMemsetAsync(col_ + sell_krows_ * 32, 0xFF, (krows - sell_krows_) * 32 * 4, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
        CK(cudaMemsetAsync(wgt_ + sell_krows_ * 32, 0, (krows - sell_krows_) * 32 * 4, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    }
    return SNN_OK;
}

void Engine::refresh_flag_cache() const {
    if (flags_cache_valid_) return;
    uint32_t a = 0;
    for (uint32_t i = 0; i < n_nodes_; ++i) a |= h_node_flags_[i];
    nt_used_ = a & 0x7u; rc_used_ = (a >> 4) & 0x7u;
    flags_cache_valid_ = true;
}
uint32_t Engine::nt_used() const { refresh_flag_cache(); return nt_used_; }
uint32_t Engine::rc_used() const { refresh_flag_cache(); return rc_used_; }

int Engine::finalize_graph() {
    if (!graph_dirty_) return SNN_OK;
    tile_par_dirty_ = true;     // the col table is written below: the window kernel checks its stencil tiles again
    ghist_off_valid_ = false;   // the canonical order of the new table is counted again by the next run that records it
    free_reward_arrays();   // a rebuilt graph starts from TraceRSTDP::default traces
    CK(cudaSetDevice(device), SNN_GPU_GET_DEVICE_FAILURE);
    // the stencil fast path re-generates the table in place when its size is unchanged (set_graph_grid called again,
    // e.g. once per run by a caller that mirrors LatticeGPU's upload-everything-per-run behaviour)
    const uint32_t new_slices = (uint32_t)((n_neurons + 31) / 32);
    bool reuse = false;
    if (blocks_.size() == 1 && blocks_.begin()->second.kind == Block::GRID && col_ && wgt_ && slice_off_ && n_slices_ == new_slices) {
        reuse = sell_alloc_krows_ == uniform_table_krows(new_slices, stencil_width(blocks_.begin()->second.radius));
    }
    if (!reuse) {
        if (slice_off_) cudaFree(slice_off_);
        if (col_) cudaFree(col_);
        if (wgt_) cudaFree(wgt_);
        slice_off_ = col_ = nullptr; wgt_ = nullptr;
        sell_alloc_krows_ = 0;
    }
    grid_fast_ = false;
    uniform_width_ = 0;
    n_slices_ = new_slices;
    if (!reuse) CK(dev_alloc(&slice_off_, (size_t)n_slices_ + 1), SNN_GPU_BUFFER_CREATE_ERROR);
    // partitioned handles: ghost rows inherit the neurotransmitter type sets of the adjacent owned rows
    if (part_world > 1 && n_neurons && !gpart_) {
        // (until the neighbour is attached: attach_strip replaces them with the neighbour's real boundary flags)
        for (uint32_t g = 0; g < halo_; ++g) {
            if (part_rank > 0 && !ghost_flags_from_peer_[0]) h_node_flags_[own0_ - halo_ + g] = h_node_flags_[own0_ + (g % std::max<uint64_t>(n_neurons, 1))];
            if (part_rank < part_world - 1 && !ghost_flags_from_peer_[1]) h_node_flags_[ghost_hi0_ + g] = h_node_flags_[own0_ + n_neurons - halo_ + g];
        }
        CK(h2d_sync(node_flags_, h_node_flags_.data(), node_cap_, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
        flags_cache_valid_ = false;
    }
    const int n_neuron_lat = n_neuron_lattices();
    const Lat *only = n_neuron_lat == 1 ? &lats_[0] : nullptr;   // neuron lattices come first in lats_
    // fast path: one lattice whose only block is a grid stencil -> built directly in sliced-ELL form on the device
    if (n_neuron_lat == 1 && blocks_.size() == 1 && blocks_.begin()->second.kind == Block::GRID &&
        blocks_.begin()->first == std::make_pair(only->id, only->id)) {
        const Block &b = blocks_.begin()->second;
        const uint32_t width = stencil_width(b.radius);
        sell_krows_ = (uint64_t)n_slices_ * width;
        if (!reuse) { int r = alloc_table(width); if (r) return r; }
        if (n_neurons == 0) CK(cudaMemsetAsync(slice_off_, 0, 4, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
        CK(launch_sell_grid(only->rows, only->cols, part_world > 1 ? row0_global : 0, part_world > 1 ? rows_global : only->rows,
                            b.radius, b.weight, own0_, node_flags_, width, slice_off_, col_, wgt_, stream_), SNN_GPU_QUEUE_FAILURE);
        CK(cudaStreamSynchronize(stream_), SNN_GPU_WAIT_ERROR);
        grid_fast_ = true;
        uniform_width_ = width;
        max_slice_width_ = n_slices_ ? width : 0;
        graph_dirty_ = false;
        dev_weights_newer_ = false;
        return SNN_OK;
    }
    // general path: merge every block into one CSR over canonical node indices
    for (auto &kv : blocks_)
        if (kv.second.kind == Block::GRID) materialize_grid(kv.second, *find(kv.first.first));
    std::vector<uint64_t> row_ptr(n_neurons + 1, 0);
    for_each_row_segment([&](const Lat &B, uint64_t q, const Lat &, Block &b, uint64_t) {
        row_ptr[B.off + q + 1] += b.row_ptr[q + 1] - b.row_ptr[q];
    });
    for (uint64_t i = 0; i < n_neurons; ++i) row_ptr[i + 1] += row_ptr[i];
    const uint64_t nnz = row_ptr[n_neurons];
    std::vector<uint32_t> pre(std::max<uint64_t>(nnz, 1));
    std::vector<float> w(std::max<uint64_t>(nnz, 1));
    const int64_t node_shift = part_world > 1 ? (int64_t)own0_ - (int64_t)row0_global * (only ? only->cols : 0) : 0;
    std::vector<uint64_t> ghost_rows;   // general-graph partition: rows with an in-edge from a ghost
    bool beyond_halo = false;
    for_each_row_segment([&](const Lat &B, uint64_t q, const Lat &A, Block &b, uint64_t k) {
        uint64_t o = row_ptr[B.off + q] + k;
        for (uint64_t e = b.row_ptr[q]; e < b.row_ptr[q + 1]; ++e, ++o) {
            int64_t node = gpart_ ? global_to_node(b.pre[e]) : (part_world > 1 ? (int64_t)b.pre[e] + node_shift : (int64_t)node_off(A) + b.pre[e]);
            if (node < 0 || node >= (int64_t)n_nodes_) { beyond_halo = true; return; }
            if (gpart_ && (node < (int64_t)own0_ || node >= (int64_t)own0_ + (int64_t)n_neurons)) ghost_rows.push_back(B.off + q);
            pre[o] = (uint32_t)node; w[o] = b.w[e];
        }
    });
    if (beyond_halo) return fail(SNN_UNSUPPORTED, "edge reaches beyond the halo of this strip");
    std::vector<uint32_t> slice_off(n_slices_ + 1, 0);
    for (uint32_t s = 0; s < n_slices_; ++s) {
        uint64_t mx = 0;
        for (uint64_t r = (uint64_t)s * 32; r < std::min<uint64_t>((uint64_t)s * 32 + 32, n_neurons); ++r)
            mx = std::max(mx, row_ptr[r + 1] - row_ptr[r]);
        mx = round_up(mx, 4);  // the step kernel consumes edges in chunks of 4/8 without tail checks
        const uint64_t next = (uint64_t)slice_off[s] + mx;
        if (next > 0xFFFFFFF0ull / 32) return fail(SNN_UNSUPPORTED, "graph too large");
        slice_off[s + 1] = (uint32_t)next;
    }
    sell_krows_ = slice_off[n_slices_];
    // a materialised stencil (weights came back from the device: STDP, edit_weight) keeps the uniform-width layout of the
    // generator, so the window / TMA step kernels stay eligible after a rebuild
    uint32_t width = 0;
    if (n_neuron_lat == 1 && blocks_.size() == 1 && blocks_.begin()->second.from_grid_radius &&
        blocks_.begin()->first == std::make_pair(only->id, only->id)) {
        width = stencil_width(blocks_.begin()->second.from_grid_radius);
        for (uint32_t s = 0; s < n_slices_; ++s) {
            if (slice_off[s + 1] - slice_off[s] > width) { width = 0; break; }
        }
        if (width) {
            for (uint32_t s = 0; s <= n_slices_; ++s) slice_off[s] = s * width;
            sell_krows_ = (uint64_t)n_slices_ * width;
        }
    }
    max_slice_width_ = 0;
    for (uint32_t s = 0; s < n_slices_; ++s) max_slice_width_ = std::max(max_slice_width_, slice_off[s + 1] - slice_off[s]);
    int r = alloc_table(width);
    if (r) return r;
    CK(h2d_sync(slice_off_, slice_off.data(), ((size_t)n_slices_ + 1) * 4, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    uint64_t *d_rp = nullptr; uint32_t *d_pre = nullptr; float *d_w = nullptr;
    CK(dev_alloc(&d_rp, n_neurons + 1), SNN_GPU_BUFFER_CREATE_ERROR);
    CK(dev_alloc(&d_pre, nnz), SNN_GPU_BUFFER_CREATE_ERROR);
    CK(dev_alloc(&d_w, nnz), SNN_GPU_BUFFER_CREATE_ERROR);
    h2d_sync(d_rp, row_ptr.data(), (n_neurons + 1) * 8, stream_);
    if (nnz) { h2d_sync(d_pre, pre.data(), nnz * 4, stream_); h2d_sync(d_w, w.data(), nnz * 4, stream_); }
    cudaError_t e = launch_sell_from_csr(d_rp, d_pre, d_w, node_flags_, part_world > 1 ? 0xFFFFFFFFu : train0_, (uint32_t)n_neurons,
                                         slice_off_, col_, wgt_, stream_);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream_);
    cudaFree(d_rp); cudaFree(d_pre); cudaFree(d_w);
    if (e != cudaSuccess) return cuda_fail(e, SNN_GPU_QUEUE_FAILURE, "sell_from_csr");
    if (width) { grid_fast_ = true; uniform_width_ = width; }
    if (gpart_) {
        h_gslice_.assign(n_slices_, 0);
        for (uint64_t row : ghost_rows) h_gslice_[row / 32] |= 1u;
        gpart_dirty_ = true;
    }
    graph_dirty_ = false;
    dev_weights_newer_ = false;
    return SNN_OK;
}

// ------------------------------------------------------------------------------------------------
// RewardModulatedLattice
// ------------------------------------------------------------------------------------------------
int Engine::set_bcm_plasticity(bool enable, const snn_bcm_t *b) {
    if (enable && model != SNN_MODEL_BCM_IZHIKEVICH) return fail(SNN_INVALID_ARGUMENT, "BCM plasticity needs neurons with BCMActivity (SNN_MODEL_BCM_IZHIKEVICH)");
    if (enable && (n_neuron_lattices() > 1 || n_trains > 0)) return fail(SNN_UNSUPPORTED, "BCM plasticity: Lattice handles only (whole, row-strip or general-graph partitioned)");
    bcm_mode = enable;
    if (b) bcm = *b;
    return SNN_OK;
}

int Engine::set_reward_modulator(bool enable, bool modulate, const snn_rstdp_t *m) {
    if (enable && (n_neuron_lattices() > 1 || n_trains > 0)) return fail(SNN_UNSUPPORTED, "snn_lattice_set_reward_modulator is for single-lattice handles; networks add reward-modulated lattices with snn_network_add_reward_modulated_lattice");
    reward_mode = enable; do_modulation = modulate;
    if (m) rstdp = *m;
    if (!enable) free_reward_arrays();
    return SNN_OK;
}

// RewardModulatedLatticeNetwork: per-lattice modulators and the kind of the connecting blocks
int Engine::set_lattice_reward_modulator(uint64_t id, bool modulate, const snn_rstdp_t *m) {
    Lat *L = find(id);
    if (!L || !L->is_reward) return fail(SNN_INVALID_ARGUMENT, "not a reward-modulated lattice of this network, id: " + std::to_string(id));
    L->do_modulation = modulate;
    if (m) L->rstdp = *m;
    return SNN_OK;
}

int Engine::get_lattice_reward_modulator(uint64_t id, int32_t *modulate, snn_rstdp_t *m) {
    Lat *L = find(id);
    if (!L || !L->is_reward) return fail(SNN_INVALID_ARGUMENT, "not a reward-modulated lattice of this network, id: " + std::to_string(id));
    if (modulate) *modulate = L->do_modulation ? 1 : 0;
    if (m) *m = L->rstdp;
    return SNN_OK;
}

int Engine::set_connection_reward(uint64_t pre_id, uint64_t post_id, bool reward_modulated) {
    // connect_with_reward_modulation neuron/mod.rs:4076-4209: the block's values are RewardModulatedConnection::RewardModulatedWeight
    // (TraceRSTDP) instead of ::Weight(f32)
    const Lat *A = find(pre_id), *B = find(post_id);
    if (B && B->is_train)
        return fail(SNN_NET_POSTSYNAPTIC_LATTICE_CANNOT_BE_SPIKE_TRAIN, "Postsynaptic lattice cannot be a spike train lattice because spike trains cannot take inputs");
    if (!A) return fail(SNN_NET_PRESYNAPTIC_ID_NOT_FOUND, "Presynaptic id not present in network, id: " + std::to_string(pre_id));
    if (!(B && B->is_reward) && !A->is_reward)
        return fail(SNN_NET_CANNOT_CONNECT_WITH_REWARD_MODULATED_CONNECTION, "When connecting reward modulated network, at least one lattice has to be reward modulated");
    if (!B) return fail(SNN_NET_POSTSYNAPTIC_ID_NOT_FOUND, "Postsynaptic id not present in network, id: " + std::to_string(post_id));
    if (pre_id == post_id)
        return fail(SNN_NET_REWARD_MODULATED_CONNECTION_NOT_COMPATIBLE_INTERNALLY,
                    "When connecting reward modulated lattice, RewardModulatedConnection cannot be used to connect a reward modulated lattice internally");
    auto it = blocks_.find({pre_id, post_id});
    if (it == blocks_.end()) return fail(SNN_INVALID_ARGUMENT, "no such connecting block: connect it first");
    it->second.reward_conn = reward_modulated;
    return SNN_OK;
}

void Engine::free_reward_arrays() {
    if (rs_counter_) cudaFree(rs_counter_);
    if (rs_dw_) cudaFree(rs_dw_);
    if (rs_c_) cudaFree(rs_c_);
    rs_counter_ = nullptr; rs_dw_ = rs_c_ = nullptr; rs_elems_ = 0;
}

int Engine::ensure_reward_arrays() {
    const uint64_t elems = std::max<uint64_t>(std::max(sell_alloc_krows_, sell_krows_) * 32, 1);
    if (rs_counter_ && rs_elems_ == elems) return SNN_OK;
    free_reward_arrays();
    CK(dev_alloc(&rs_counter_, elems), SNN_GPU_BUFFER_CREATE_ERROR);
    CK(dev_alloc(&rs_dw_, elems), SNN_GPU_BUFFER_CREATE_ERROR);
    CK(dev_alloc(&rs_c_, elems), SNN_GPU_BUFFER_CREATE_ERROR);
    CK(cudaMemsetAsync(rs_counter_, 0, elems, stream_), SNN_GPU_BUFFER_WRITE_ERROR);   // TraceRSTDP::default: counter 0, dw 0, c 0
    CK(cudaMemsetAsync(rs_dw_, 0, elems * 4, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    CK(cudaMemsetAsync(rs_c_, 0, elems * 4, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    rs_elems_ = elems;
    rs_canonical_ = true;
    return SNN_OK;
}

bool Engine::has_reward_lattices() const {
    for (auto &L : lats_) if (L.is_reward) return true;
    return false;
}

// element index (k * 32 + lane) of every edge of block pre_id -> post_id, in the block's CSR order
int Engine::block_elements(uint64_t pre_id, uint64_t post_id, std::vector<size_t> *elems, Block **blk) {
    Lat *B = find(post_id);
    if (!find(pre_id) || !B || B->is_train) return fail(SNN_INVALID_ARGUMENT, "no such connection block");
    *blk = nullptr;
    elems->clear();
    auto it = blocks_.find({pre_id, post_id});
    if (it == blocks_.end()) return SNN_OK;
    *blk = &it->second;
    std::vector<uint32_t> so((size_t)n_slices_ + 1);
    CK(cudaStreamSynchronize(stream_), SNN_GPU_WAIT_ERROR);
    CK(cudaMemcpy(so.data(), slice_off_, so.size() * 4, cudaMemcpyDeviceToHost), SNN_GPU_BUFFER_READ_ERROR);
    for_each_row_segment([&](const Lat &, uint64_t q, const Lat &A, Block &b, uint64_t k) {
        if (A.id != pre_id) return;
        const uint64_t row = B->off + q;
        for (uint64_t i = 0; i < b.row_ptr[q + 1] - b.row_ptr[q]; ++i) elems->push_back((size_t)(so[row / 32] + k + i) * 32 + row % 32);
    }, B);
    return SNN_OK;
}

int Engine::get_block_traces(uint64_t pre_id, uint64_t post_id, uint32_t *counter, float *dw, float *c, uint64_t nnz) {
    if (!reward_mode && !has_reward_lattices()) return fail(SNN_INVALID_ARGUMENT, "handle holds no reward-modulated lattice");
    CK(cudaSetDevice(device), SNN_GPU_GET_DEVICE_FAILURE);
    int r = finalize_graph();
    if (r) return r;
    r = ensure_reward_arrays();
    if (r) return r;
    std::vector<size_t> el;
    Block *b = nullptr;
    r = block_elements(pre_id, post_id, &el, &b);
    if (r) return r;
    if (el.size() != nnz) return fail(SNN_SIZE_MISMATCH, "nnz mismatch");
    if (nnz == 0) return SNN_OK;
    std::vector<uint8_t> hc(rs_elems_);
    std::vector<float> hd(rs_elems_), hcc(rs_elems_);
    CK(cudaMemcpy(hc.data(), rs_counter_, rs_elems_, cudaMemcpyDeviceToHost), SNN_GPU_BUFFER_READ_ERROR);
    CK(cudaMemcpy(hd.data(), rs_dw_, rs_elems_ * 4, cudaMemcpyDeviceToHost), SNN_GPU_BUFFER_READ_ERROR);
    CK(cudaMemcpy(hcc.data(), rs_c_, rs_elems_ * 4, cudaMemcpyDeviceToHost), SNN_GPU_BUFFER_READ_ERROR);
    for (uint64_t e = 0; e < nnz; ++e) {
        if (counter) counter[e] = hc[el[e]];
        if (dw) dw[e] = hd[el[e]];
        if (c) c[e] = hcc[el[e]];
    }
    return SNN_OK;
}

int Engine::set_block_traces(uint64_t pre_id, uint64_t post_id, const float *weight, const uint32_t *counter, const float *dw, const float *c,
                             uint64_t nnz) {
    if (!reward_mode && !has_reward_lattices()) return fail(SNN_INVALID_ARGUMENT, "handle holds no reward-modulated lattice");
    CK(cudaSetDevice(device), SNN_GPU_GET_DEVICE_FAILURE);
    int r = finalize_graph();
    if (r) return r;
    r = ensure_reward_arrays();
    if (r) return r;
    r = sync_weights_to_host();   // the host copy of the weights must be current before parts of it are overwritten
    if (r) return r;
    std::vector<size_t> el;
    Block *b = nullptr;
    r = block_elements(pre_id, post_id, &el, &b);
    if (r) return r;
    if (el.size() != nnz) return fail(SNN_SIZE_MISMATCH, "nnz mismatch");
    if (nnz == 0) return SNN_OK;
    const uint64_t wel = std::max(sell_alloc_krows_, sell_krows_) * 32;
    std::vector<uint8_t> hc(rs_elems_);
    std::vector<float> hd(rs_elems_), hcc(rs_elems_), hw(rs_elems_);
    CK(cudaMemcpy(hc.data(), rs_counter_, rs_elems_, cudaMemcpyDeviceToHost), SNN_GPU_BUFFER_READ_ERROR);
    CK(cudaMemcpy(hd.data(), rs_dw_, rs_elems_ * 4, cudaMemcpyDeviceToHost), SNN_GPU_BUFFER_READ_ERROR);
    CK(cudaMemcpy(hcc.data(), rs_c_, rs_elems_ * 4, cudaMemcpyDeviceToHost), SNN_GPU_BUFFER_READ_ERROR);
    CK(cudaMemcpy(hw.data(), wgt_, std::min<uint64_t>(rs_elems_, wel) * 4, cudaMemcpyDeviceToHost), SNN_GPU_BUFFER_READ_ERROR);
    for (uint64_t e = 0; e < nnz; ++e) {
        const size_t o = el[e];
        if (weight) { hw[o] = weight[e]; if (b->kind == Block::CSR) b->w[e] = weight[e]; }
        // the canonical state concerns edges that get two calls per timestep: those of a reward-modulated lattice's own graph
        if (counter) { hc[o] = (uint8_t)counter[e]; if (counter[e] != 0u && pre_id == post_id) rs_canonical_ = false; }
        if (dw) { hd[o] = dw[e]; if (dw[e] != 0.f && pre_id == post_id) rs_canonical_ = false; }
        if (c) hcc[o] = c[e];
    }
    if (weight) CK(h2d_sync(wgt_, hw.data(), wel * 4, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    if (counter) CK(h2d_sync(rs_counter_, hc.data(), rs_elems_, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    if (dw) CK(h2d_sync(rs_dw_, hd.data(), rs_elems_ * 4, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    if (c) CK(h2d_sync(rs_c_, hcc.data(), rs_elems_ * 4, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    if (weight && b->kind == Block::GRID) dev_weights_newer_ = true;   // a stencil block's weights live on the device
    return SNN_OK;
}

int Engine::get_connection_traces(uint32_t *counter, float *dw, float *c, uint64_t nnz) {
    const Lat *only = nullptr;
    for (auto &L : lats_) if (!L.is_train) only = &L;
    if (!only || !reward_mode) return fail(SNN_INVALID_ARGUMENT, "handle is not a reward-modulated lattice");
    return get_block_traces(only->id, only->id, counter, dw, c, nnz);
}

int Engine::set_connection_traces(const float *weight, const uint32_t *counter, const float *dw, const float *c, uint64_t nnz) {
    const Lat *only = nullptr;
    for (auto &L : lats_) if (!L.is_train) only = &L;
    if (!only || !reward_mode) return fail(SNN_INVALID_ARGUMENT, "handle is not a reward-modulated lattice");
    return set_block_traces(only->id, only->id, weight, counter, dw, c, nnz);
}

int Engine::sync_weights_to_host() {
    if (!dev_weights_newer_) return SNN_OK;
    if (graph_dirty_ || !col_) { dev_weights_newer_ = false; return SNN_OK; }
    CK(cudaSetDevice(device), SNN_GPU_GET_DEVICE_FAILURE);
    std::vector<uint32_t> so((size_t)n_slices_ + 1), col(std::max<uint64_t>(sell_krows_ * 32, 1));
    std::vector<float> wg(std::max<uint64_t>(sell_krows_ * 32, 1));
    CK(cudaMemcpy(so.data(), slice_off_, so.size() * 4, cudaMemcpyDeviceToHost), SNN_GPU_BUFFER_READ_ERROR);
    if (sell_krows_) {
        CK(cudaMemcpy(col.data(), col_, sell_krows_ * 32 * 4, cudaMemcpyDeviceToHost), SNN_GPU_BUFFER_READ_ERROR);
        CK(cudaMemcpy(wg.data(), wgt_, sell_krows_ * 32 * 4, cudaMemcpyDeviceToHost), SNN_GPU_BUFFER_READ_ERROR);
    }
    for (auto &kv : blocks_)
        if (kv.second.kind == Block::GRID) materialize_grid(kv.second, *find(kv.first.first));
    for_each_row_segment([&](const Lat &B, uint64_t q, const Lat &, Block &b, uint64_t k) {
        const uint64_t row = B.off + q;
        for (uint64_t i = 0, e = b.row_ptr[q]; e < b.row_ptr[q + 1]; ++i, ++e) b.w[e] = wg[(size_t)(so[row / 32] + k + i) * 32 + row % 32];
    });
    dev_weights_newer_ = false;
    return SNN_OK;
}

int Engine::connection_nnz(uint64_t pre_id, uint64_t post_id, uint64_t *nnz) {
    Lat *A = find(pre_id), *B = find(post_id);
    if (!A || !B) return fail(SNN_NET_ID_NOT_FOUND_IN_LATTICES, "Id not present in lattices");
    auto it = blocks_.find({pre_id, post_id});
    if (it == blocks_.end()) { *nnz = 0; return SNN_OK; }
    if (it->second.kind == Block::GRID) {
        int r = sync_weights_to_host();
        if (r) return r;
        if (it->second.kind == Block::GRID) materialize_grid(it->second, *A);
    }
    *nnz = it->second.pre.size();
    return SNN_OK;
}

int Engine::get_connection_csr(uint64_t pre_id, uint64_t post_id, uint64_t *row_ptr, uint32_t *pre, float *weights,
                               uint64_t n_post, uint64_t nnz) {
    Lat *A = find(pre_id), *B = find(post_id);
    if (!A || !B || B->is_train) return fail(SNN_NET_ID_NOT_FOUND_IN_LATTICES, "Id not present in lattices");
    if (n_post != B->n) return fail(SNN_GRAPH_DIMENSIONS_DO_NOT_MATCH, "Dimensions do not match");
    int r = sync_weights_to_host();
    if (r) return r;
    auto it = blocks_.find({pre_id, post_id});
    if (it == blocks_.end()) {
        if (nnz) return fail(SNN_SIZE_MISMATCH, "nnz mismatch");
        if (row_ptr) std::fill(row_ptr, row_ptr + n_post + 1, 0);
        return SNN_OK;
    }
    Block tmp;
    const Block &b = csr_view(it->second, *A, tmp);
    if (b.pre.size() != nnz) return fail(SNN_SIZE_MISMATCH, "nnz mismatch");
    if (row_ptr) memcpy(row_ptr, b.row_ptr.data(), (n_post + 1) * 8);
    if (pre && nnz) memcpy(pre, b.pre.data(), nnz * 4);
    if (weights && nnz) memcpy(weights, b.w.data(), nnz * 4);
    return SNN_OK;
}

int Engine::get_connection_dense(uint64_t pre_id, uint64_t post_id, uint32_t *connections, float *weights, uint64_t n_pre,
                                 uint64_t n_post) {
    Lat *A = find(pre_id), *B = find(post_id);
    if (!A || !B || B->is_train) return fail(SNN_NET_ID_NOT_FOUND_IN_LATTICES, "Id not present in lattices");
    if (n_pre != A->n || n_post != B->n) return fail(SNN_GRAPH_DIMENSIONS_DO_NOT_MATCH, "Dimensions do not match");
    if (part_world > 1) return fail(SNN_UNSUPPORTED, "dense graphs are not supported on partitioned handles");
    int r = sync_weights_to_host();
    if (r) return r;
    if (connections) std::fill(connections, connections + n_pre * n_post, 0u);
    if (weights) std::fill(weights, weights + n_pre * n_post, 0.f);
    auto it = blocks_.find({pre_id, post_id});
    if (it == blocks_.end()) return SNN_OK;
    Block tmp;
    const Block &b = csr_view(it->second, *A, tmp);
    for (uint64_t q = 0; q < n_post; ++q)
        for (uint64_t k = b.row_ptr[q]; k < b.row_ptr[q + 1]; ++k) {
            const uint64_t idx = (uint64_t)b.pre[k] * n_post + q;
            if (connections) connections[idx] = 1;
            if (weights) weights[idx] = b.w[k];
        }
    return SNN_OK;
}

// ------------------------------------------------------------------------------------------------
// per-row graph access on the device table (Graph::get_incoming_connections / lookup_weight / edit_weight)
// ------------------------------------------------------------------------------------------------
int Engine::get_connection_rows(uint64_t pre_id, uint64_t post_id, uint64_t row_begin, uint64_t row_end, uint64_t *row_ptr, uint32_t *pre,
                                float *weights, uint64_t capacity, uint64_t *nnz_out) {
    Lat *A = find(pre_id), *B = find(post_id);
    if (!A || !B || B->is_train) return fail(SNN_NET_ID_NOT_FOUND_IN_LATTICES, "Id not present in lattices");
    if (row_begin > row_end || row_end > B->n) return fail(SNN_GRAPH_POSITION_NOT_FOUND, "Position not found, position: " + std::to_string(row_end));
    if (nnz_out) *nnz_out = 0;
    if (row_ptr) row_ptr[0] = 0;
    if (row_begin == row_end) return SNN_OK;
    CK(cudaSetDevice(device), SNN_GPU_GET_DEVICE_FAILURE);
    int r = finalize_graph();
    if (r) return r;
    const uint64_t g0 = B->off + row_begin, g1 = B->off + row_end;   // local neuron numbers
    const uint32_t s0 = (uint32_t)(g0 / 32), s1 = (uint32_t)((g1 - 1) / 32);
    std::vector<uint32_t> so(s1 - s0 + 2);
    CK(cudaStreamSynchronize(stream_), SNN_GPU_WAIT_ERROR);
    CK(cudaMemcpy(so.data(), slice_off_ + s0, so.size() * 4, cudaMemcpyDeviceToHost), SNN_GPU_BUFFER_READ_ERROR);
    const uint64_t k0 = so.front(), k1 = so.back();
    std::vector<uint32_t> col(std::max<uint64_t>((k1 - k0) * 32, 1));
    std::vector<float> wg(col.size());
    if (k1 > k0) {
        CK(cudaMemcpy(col.data(), col_ + k0 * 32, (k1 - k0) * 32 * 4, cudaMemcpyDeviceToHost), SNN_GPU_BUFFER_READ_ERROR);
        CK(cudaMemcpy(wg.data(), wgt_ + k0 * 32, (k1 - k0) * 32 * 4, cudaMemcpyDeviceToHost), SNN_GPU_BUFFER_READ_ERROR);
    }
    // node range of the presynaptic lattice; partitioned handles report GLOBAL flat indices (ghost nodes included)
    const int64_t a0 = part_world > 1 ? 0 : (int64_t)node_off(*A), a1 = part_world > 1 ? (int64_t)n_nodes_ : a0 + (int64_t)A->n;
    const int64_t shift = part_world > 1 ? (int64_t)row0_global * A->cols - (int64_t)own0_ : -a0;
    uint64_t o = 0;
    for (uint64_t g = g0; g < g1; ++g) {
        const uint32_t s = (uint32_t)(g / 32), lane = (uint32_t)(g % 32);
        for (uint64_t k = so[s - s0]; k < so[s - s0 + 1]; ++k) {
            const size_t e = (size_t)(k - k0) * 32 + lane;
            if (col[e] == kColPad) break;   // valid entries first
            const int64_t j = (int64_t)(col[e] & kColIdxMask);
            if (j < a0 || j >= a1) continue;
            if (o < capacity) { if (pre) pre[o] = gpart_ ? (uint32_t)node_to_global((uint32_t)j) : (uint32_t)(j + shift); if (weights) weights[o] = wg[e]; }
            ++o;
        }
        if (row_ptr) row_ptr[g - g0 + 1] = o;
    }
    if (nnz_out) *nnz_out = o;
    if (o > capacity && (pre || weights)) return fail(SNN_SIZE_MISMATCH, "edge buffers too small: " + std::to_string(o) + " edges in the row range");
    return SNN_OK;
}

int Engine::check_edge_endpoints(uint64_t pre_id, uint64_t post_id, uint64_t pre, uint64_t post, Lat **A, Lat **B) {
    *A = find(pre_id); *B = find(post_id);
    if (!*A || !*B || (*B)->is_train) return fail(SNN_NET_ID_NOT_FOUND_IN_LATTICES, "Id not present in lattices");
    // lookup_weight / edit_weight check the postsynaptic key first (graph/mod.rs:197-202, 209-214)
    if (post >= (*B)->n) return fail(SNN_GRAPH_POSTSYNAPTIC_NOT_FOUND, "Postsynaptic position not found, position: " + std::to_string(post));
    const uint64_t pre_limit = part_world > 1 ? (uint64_t)rows_global * (*A)->cols : (*A)->n;
    if (pre >= pre_limit) return fail(SNN_GRAPH_PRESYNAPTIC_NOT_FOUND, "Presynaptic position not found, position: " + std::to_string(pre));
    return SNN_OK;
}

int Engine::find_edge(uint64_t row, uint32_t j, int64_t *elem) {
    *elem = -1;
    const uint32_t s = (uint32_t)(row / 32), lane = (uint32_t)(row % 32);
    uint32_t so[2];
    CK(cudaStreamSynchronize(stream_), SNN_GPU_WAIT_ERROR);
    CK(cudaMemcpy(so, slice_off_ + s, 8, cudaMemcpyDeviceToHost), SNN_GPU_BUFFER_READ_ERROR);
    if (so[1] == so[0]) return SNN_OK;
    std::vector<uint32_t> col((size_t)(so[1] - so[0]) * 32);
    CK(cudaMemcpy(col.data(), col_ + (size_t)so[0] * 32, col.size() * 4, cudaMemcpyDeviceToHost), SNN_GPU_BUFFER_READ_ERROR);
    for (uint32_t k = 0; k < so[1] - so[0]; ++k) {
        const uint32_t c = col[(size_t)k * 32 + lane];
        if (c == kColPad) break;
        if ((c & kColIdxMask) == j) { *elem = ((int64_t)so[0] + k) * 32 + lane; break; }
    }
    return SNN_OK;
}

int Engine::lookup_weight(uint64_t pre_id, uint64_t post_id, uint64_t pre, uint64_t post, float *weight, int32_t *connected) {
    Lat *A, *B;
    int r = check_edge_endpoints(pre_id, post_id, pre, post, &A, &B);
    if (r) return r;
    *connected = 0; *weight = 0.f;
    CK(cudaSetDevice(device), SNN_GPU_GET_DEVICE_FAILURE);
    r = finalize_graph();
    if (r) return r;
    const int64_t node = part_world > 1 ? global_to_node(pre) : (int64_t)node_off(*A) + (int64_t)pre;
    if (node < 0 || node >= (int64_t)n_nodes_) return SNN_OK;   // partitioned: not among this rank's ghosts, cannot be connected
    int64_t e = -1;
    r = find_edge(B->off + post, (uint32_t)node, &e);
    if (r || e < 0) return r;
    CK(cudaMemcpy(weight, wgt_ + e, 4, cudaMemcpyDeviceToHost), SNN_GPU_BUFFER_READ_ERROR);
    *connected = 1;
    return SNN_OK;
}

int Engine::edit_weight(uint64_t pre_id, uint64_t post_id, uint64_t pre, uint64_t post, bool has, float weight) {
    Lat *A, *B;
    int r = check_edge_endpoints(pre_id, post_id, pre, post, &A, &B);
    if (r) return r;
    CK(cudaSetDevice(device), SNN_GPU_GET_DEVICE_FAILURE);
    r = finalize_graph();
    if (r) return r;
    const int64_t node = part_world > 1 ? global_to_node(pre) : (int64_t)node_off(*A) + (int64_t)pre;
    int64_t e = -1;
    if (node >= 0 && node < (int64_t)n_nodes_) { r = find_edge(B->off + post, (uint32_t)node, &e); if (r) return r; }
    if (e >= 0 && has) {
        // Some(w) over Some(_): the adjacency is unchanged, one word on the device
        CK(h2d_sync(wgt_ + e, &weight, 4, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
        dev_weights_newer_ = true;
        return SNN_OK;
    }
    if (e < 0 && !has) return SNN_OK;   // None over None
    if ((r = refuse_if_graph_history("adding or removing an edge"))) return r;
    // the adjacency changes (None -> Some, Some -> None): edit the host CSR of the block and rebuild the device table lazily
    if (part_world > 1) return fail(SNN_UNSUPPORTED, "adding or removing edges is not supported on partitioned handles (weights of existing edges are)");
    dev_weights_newer_ = true;   // the device holds the live weights (STDP, earlier in-place edits)
    r = sync_weights_to_host();
    if (r) return r;
    Block &b = blocks_[{pre_id, post_id}];
    if (b.kind == Block::GRID) materialize_grid(b, *A);
    b.from_grid_radius = 0;   // no longer the generator's adjacency
    if (b.row_ptr.size() != B->n + 1) b.row_ptr.assign(B->n + 1, 0);
    const uint64_t rs = b.row_ptr[post], re = b.row_ptr[post + 1];
    uint64_t pos = rs;
    while (pos < re && b.pre[pos] < pre) ++pos;
    if (has) {
        b.pre.insert(b.pre.begin() + pos, (uint32_t)pre);
        b.w.insert(b.w.begin() + pos, weight);
        for (uint64_t q = post + 1; q <= B->n; ++q) b.row_ptr[q] += 1;
    } else {
        b.pre.erase(b.pre.begin() + pos);
        b.w.erase(b.w.begin() + pos);
        for (uint64_t q = post + 1; q <= B->n; ++q) b.row_ptr[q] -= 1;
    }
    graph_dirty_ = true;
    return SNN_OK;
}

// ------------------------------------------------------------------------------------------------
// options
// ------------------------------------------------------------------------------------------------
int Engine::set_dt(float dt) {
    // LatticeNetwork::set_dt neuron/mod.rs:1655-1660; Lattice::set_dt :649-652; PoissonNeuron::set_dt
    // rescales chance_of_firing (spike_train/mod.rs:345-349)
    CK(cudaSetDevice(device), SNN_GPU_GET_DEVICE_FAILURE);
    for (auto &L : lats_) {
        if (L.n == 0) { if (!L.is_train) { L.stdp.dt = dt; if (L.is_reward) L.rstdp.dt = dt; } continue; }
        if (L.is_train) {
            std::vector<float> old(L.n), ch(L.n);
            CK(cudaMemcpy(old.data(), TF_[TF_DT] + L.off, L.n * 4, cudaMemcpyDeviceToHost), SNN_GPU_BUFFER_READ_ERROR);
            if (train_kind == SNN_TRAIN_POISSON) {
                CK(cudaMemcpy(ch.data(), TF_[TF_CHANCE] + L.off, L.n * 4, cudaMemcpyDeviceToHost), SNN_GPU_BUFFER_READ_ERROR);
                for (uint64_t i = 0; i < L.n; ++i) { const float scalar = dt / old[i]; ch[i] *= scalar; }
                CK(h2d_sync(TF_[TF_CHANCE] + L.off, ch.data(), L.n * 4, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
            }
            CK(fill_f32(TF_[TF_DT] + L.off, dt, L.n, stream_), SNN_GPU_QUEUE_FAILURE);
        } else {
            CK(fill_f32(F_[F_DT] + L.off, dt, L.n, stream_), SNN_GPU_QUEUE_FAILURE);
            tile_par_dirty_ = true;
            L.stdp.dt = dt;
            if (L.is_reward) L.rstdp.dt = dt;   // RewardModulatedLattice::set_dt, neuron/mod.rs:2867-2870
        }
    }
    if (reward_mode) rstdp.dt = dt;
    CK(cudaStreamSynchronize(stream_), SNN_GPU_WAIT_ERROR);
    return SNN_OK;
}

int Engine::reset_timing() {
    // neuron/mod.rs:405-420, 1710-1717
    CK(cudaSetDevice(device), SNN_GPU_GET_DEVICE_FAILURE);
    internal_clock = 0;
    for (auto &L : lats_) L.clock = 0;
    for (int k = 0; k < 2; ++k)
        if (LFT_[k]) CK(launch_fill_u32((uint32_t *)LFT_[k], 0xFFFFFFFFu, node_cap_, stream_), SNN_GPU_QUEUE_FAILURE);
    CK(cudaStreamSynchronize(stream_), SNN_GPU_WAIT_ERROR);
    return SNN_OK;
}

int Engine::reset_history() {
    for (auto &L : lats_) {
        L.grid_history.clear(); L.spike_history.clear(); L.spike_agg.clear(); L.average_history.clear(); L.eeg_history.clear(); L.hist_len = 0;
        L.ev_ptr.clear(); L.ev_neuron.clear();
    }
    graph_hist_.clear();
    return SNN_OK;
}

// ------------------------------------------------------------------------------------------------
// graph history (Graph::update_history, graph/mod.rs:278-284)
// ------------------------------------------------------------------------------------------------
bool Engine::graph_history_nonempty() const {
    for (auto &kv : graph_hist_) if (kv.second.steps) return true;
    return false;
}

// a record is the block's weights in a fixed edge order: the adjacency stays put until reset_history clears the records
int Engine::refuse_if_graph_history(const char *what) {
    if (!graph_history_nonempty()) return SNN_OK;
    return fail(SNN_UNSUPPORTED, std::string(what) + ": the adjacency cannot change while a graph history holds records (reset_history first)");
}

int Engine::graph_history_len(uint64_t pre_id, uint64_t post_id, uint64_t *steps, uint64_t *nnz) {
    const Lat *A = find(pre_id), *B = find(post_id);
    if (!A || !B || B->is_train) return fail(SNN_NET_ID_NOT_FOUND_IN_LATTICES, "Id not present in lattices");
    auto it = graph_hist_.find({pre_id, post_id});
    if (steps) *steps = it == graph_hist_.end() ? 0 : it->second.steps;
    if (nnz) *nnz = it == graph_hist_.end() ? 0 : it->second.nnz;
    return SNN_OK;
}

int Engine::get_graph_history(uint64_t pre_id, uint64_t post_id, float *out, uint64_t capacity) {
    const Lat *A = find(pre_id), *B = find(post_id);
    if (!A || !B || B->is_train) return fail(SNN_NET_ID_NOT_FOUND_IN_LATTICES, "Id not present in lattices");
    auto it = graph_hist_.find({pre_id, post_id});
    if (it == graph_hist_.end() || it->second.w.empty()) return SNN_OK;
    if (capacity < it->second.w.size()) return fail(SNN_SIZE_MISMATCH, "graph history buffer too small");
    if (!out) return fail(SNN_INVALID_ARGUMENT, "null argument");
    memcpy(out, it->second.w.data(), it->second.w.size() * 4);
    return SNN_OK;
}

int Engine::history_len(uint64_t id, uint64_t *steps) const {
    const Lat *L = find(id);
    if (!L) return SNN_NET_ID_NOT_FOUND_IN_LATTICES;
    *steps = L->hist_len;
    return SNN_OK;
}

int Engine::get_grid_history(uint64_t id, float *out, uint64_t capacity) {
    Lat *L = find(id);
    if (!L) return fail(SNN_NET_ID_NOT_FOUND_IN_LATTICES, "Id not present in lattices");
    if (capacity < L->grid_history.size()) return fail(SNN_SIZE_MISMATCH, "history buffer too small");
    if (!L->grid_history.empty()) memcpy(out, L->grid_history.data(), L->grid_history.size() * 4);
    return SNN_OK;
}

int Engine::get_reduced_history(uint64_t id, bool eeg, float *out, uint64_t capacity) {
    Lat *L = find(id);
    if (!L) return fail(SNN_NET_ID_NOT_FOUND_IN_LATTICES, "Id not present in lattices");
    const std::vector<float> &h = eeg ? L->eeg_history : L->average_history;
    if (capacity < h.size()) return fail(SNN_SIZE_MISMATCH, "history buffer too small");
    if (!h.empty()) memcpy(out, h.data(), h.size() * 4);
    return SNN_OK;
}

int Engine::set_eeg_parameters(uint64_t id, float reference_voltage, float distance, float conductivity) {
    Lat *L = find(id);
    if (!L || L->is_train) return fail(SNN_NET_ID_NOT_FOUND_IN_LATTICES, "Id not present in lattices");
    L->eeg_ref = reference_voltage; L->eeg_dist = distance; L->eeg_cond = conductivity;
    return SNN_OK;
}

int Engine::get_spike_aggregate(uint64_t id, int64_t *out, uint64_t capacity) {
    Lat *L = find(id);
    if (!L) return fail(SNN_NET_ID_NOT_FOUND_IN_LATTICES, "Id not present in lattices");
    // an empty history aggregates to an empty vector in the reference; here: zeros (the shape is known)
    if (capacity < L->n) return fail(SNN_SIZE_MISMATCH, "aggregate buffer too small");
    if (!out) return L->n ? fail(SNN_INVALID_ARGUMENT, "null argument") : SNN_OK;
    if (L->spike_agg.size() == L->n) memcpy(out, L->spike_agg.data(), L->n * 8);
    else std::fill(out, out + L->n, (int64_t)0);
    return SNN_OK;
}

int Engine::get_spike_history(uint64_t id, uint8_t *out, uint64_t capacity) {
    Lat *L = find(id);
    if (!L) return fail(SNN_NET_ID_NOT_FOUND_IN_LATTICES, "Id not present in lattices");
    if (capacity < L->spike_history.size()) return fail(SNN_SIZE_MISMATCH, "history buffer too small");
    if (!L->spike_history.empty()) memcpy(out, L->spike_history.data(), L->spike_history.size());
    return SNN_OK;
}

int Engine::spike_event_count(uint64_t id, uint64_t *steps, uint64_t *n_events) const {
    const Lat *L = find(id);
    if (!L) return SNN_NET_ID_NOT_FOUND_IN_LATTICES;
    if (steps) *steps = L->ev_ptr.empty() ? 0 : L->ev_ptr.size() - 1;
    if (n_events) *n_events = L->ev_neuron.size();
    return SNN_OK;
}

// `capacity` bounds the neuron array; step_ptr must hold steps + 1 entries (either pointer may be NULL)
int Engine::get_spike_events(uint64_t id, uint64_t *step_ptr, uint32_t *neuron, uint64_t capacity) {
    Lat *L = find(id);
    if (!L) return fail(SNN_NET_ID_NOT_FOUND_IN_LATTICES, "Id not present in lattices");
    if (neuron && capacity < L->ev_neuron.size()) return fail(SNN_SIZE_MISMATCH, "spike event buffer too small");
    if (step_ptr) {
        if (L->ev_ptr.empty()) step_ptr[0] = 0;
        else memcpy(step_ptr, L->ev_ptr.data(), L->ev_ptr.size() * 8);
    }
    if (neuron && !L->ev_neuron.empty()) memcpy(neuron, L->ev_neuron.data(), L->ev_neuron.size() * 4);
    return SNN_OK;
}

// ------------------------------------------------------------------------------------------------
// the step loop
// ------------------------------------------------------------------------------------------------
int Engine::upload_lat_table() {
    LatInfo tab[kMaxLattices];
    memset(tab, 0, sizeof tab);
    int k = 0;
    for (auto &L : lats_) {
        if (L.is_train) continue;
        tab[k].base = (uint32_t)L.off; tab[k].n = (uint32_t)L.n;
        tab[k].a_plus = L.stdp.a_plus; tab[k].a_minus = L.stdp.a_minus; tab[k].tau_plus = L.stdp.tau_plus;
        tab[k].tau_minus = L.stdp.tau_minus; tab[k].dt = L.stdp.dt;
        tab[k].do_plasticity = L.do_plasticity && !L.is_reward; tab[k].grid_hist = L.grid_hist; tab[k].spike_hist = L.spike_hist;
        ++k;
    }
    if (k == 0) k = 1;
    CK(cudaMemcpyAsync(d_lat_, tab, sizeof(LatInfo) * kMaxLattices, cudaMemcpyHostToDevice, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    CK(cudaStreamSynchronize(stream_), SNN_GPU_WAIT_ERROR);
    return SNN_OK;
}

void Engine::fill_step_params(StepParams &p) {
    memset(&p, 0, sizeof p);
    p.own0 = own0_; p.n_neurons = (uint32_t)n_neurons; p.n_nodes = n_nodes_;
    p.electrical = electrical; p.chemical = chemical;
    p.nt_used = nt_used(); p.rc_used = rc_used();
    p.ntk = ntk; p.rck = rck; p.refract = refract;
    p.slice_off = slice_off_; p.col = col_; p.wgt = wgt_;
    p.uniform_width = uniform_width_;
    p.t_stride = node_cap_; p.node_flags = node_flags_;
    for (int s = 0; s < F_COUNT; ++s) p.f[s] = F_[s];
    p.was_inc = was_inc_;
    for (int s = 0; s < NTF_COUNT; ++s) p.nt[s] = NT_[s];
    p.nt_stride = node_cap_;
    for (int s = 0; s < RCF_COUNT; ++s) p.rc[s] = RC_[s];
    p.rc_stride = neuron_cap_;
    p.train0 = train0_; p.n_trains = (uint32_t)n_trains;
    for (int s = 0; s < TF_COUNT; ++s) p.tf[s] = TF_[s];
    p.lat = d_lat_;
    p.n_lat = std::max(n_neuron_lattices(), 1);
    p.halo[0] = halo_dir_[0]; p.halo[1] = halo_dir_[1];
    p.halo_done = halo_done_;
    p.halo_timeout_ns = halo_timeout_ms * 1000000ull;
    if (gpart_ && !gpeers_.empty()) {
        p.gpeers = d_gpeers_; p.n_gpeers = (uint32_t)gpeers_.size();
        p.gexp_off = d_gexp_off_; p.gexp_ent = d_gexp_ent_; p.gslice = d_gslice_; p.n_gslices = n_slices_;
    }
    if (ACT_[0]) {   // a BCM Izhikevich partition (no spike trains): the train slots carry the activity exchange (BcmSlot)
        for (int d = 0; d < 2; ++d)
            for (int k = 0; k < 2; ++k) p.tf[TFB_HALO_ACT + 2 * d + k] = halo_act_[d][k];
        p.tf[TFB_GPEER_ACT] = reinterpret_cast<const float *>(d_gact_);
    }
}

// Operand streams of the TMA-staged kernel for the current configuration; false = not eligible (use the general kernel).
bool Engine::build_tma_params(TmaParams &tp, bool ntrel, bool stdp, bool lft_pp, int mode, unsigned *grid) {
    memset(&tp, 0xFF, sizeof tp);
    if (!grid_fast_ || !uniform_width_ || n_neurons == 0) return false;
    if (mode == 0) return false;
    // tiny lattices are launch-latency bound: the persistent kernel only pays off with at least a few tiles per SM
    if (mode < 2 && n_neurons < 64 * 1024) return false;
    uint32_t off = 0, n = 0;
    auto add = [&](const void *src, uint32_t bytes_per_tile) -> uint32_t {
        if (n >= (uint32_t)kMaxTmaStreams) return 0xFFFFFFFFu;
        tp.st[n].src = (const unsigned char *)src;
        tp.st[n].bytes_per_tile = bytes_per_tile;
        tp.st[n].smem_off = off;
        const uint32_t o = off;
        off += (uint32_t)round_up(bytes_per_tile, 128);
        ++n;
        return o;
    };
    const uint32_t fb = kTmaTile * 4;
    tp.o_v = add(V_[0] + own0_, fb);            // src patched per step (ping-pong)
    tp.o_lft = (stdp || lft_pp) ? add(LFT_[0] + own0_, fb) : 0u;
    tp.o_flags = ntrel ? add(node_flags_ + own0_, kTmaTile) : 0u;
    const uint32_t eb = kTmaConsumerWarps * uniform_width_ * 32u * 4u;
    tp.o_col = add(col_, eb);
    tp.o_wgt = add(wgt_, eb);
    for (int i = 0; i < kNumNeuronFields; ++i) {
        const FieldDef &fd = kNeuronFields[i];
        if (fd.kind != FK_NEURON_DEV || !(fd.models & SNN_M(model)) || fd.slot >= F_NA_CUR) continue;
        tp.o_f[fd.slot] = add(F_[fd.slot], fb);
    }
    if (ntrel) {
        const uint32_t ntu = nt_used(), rcu = rc_used();
        for (int ty = 0; ty < kNT; ++ty) {
            if (ntu & (1u << ty)) {
                tp.o_t[ty] = add(T_[0] + (size_t)ty * node_cap_ + own0_, fb);   // src patched per step
                tp.o_nt[NTF_TMAX][ty] = add(NT_[NTF_TMAX] + (size_t)ty * node_cap_ + own0_, fb);
                if (ntk != SNN_NT_DISCRETE_SPIKE) tp.o_nt[NTF_P1][ty] = add(NT_[NTF_P1] + (size_t)ty * node_cap_ + own0_, fb);
                if (ntk == SNN_NT_DESTEXHE) tp.o_nt[NTF_P2][ty] = add(NT_[NTF_P2] + (size_t)ty * node_cap_ + own0_, fb);
            }
            if (rcu & (1u << ty)) {
                tp.o_rc[RCF_R][ty] = add(RC_[RCF_R] + (size_t)ty * neuron_cap_, fb);
                tp.o_rc[RCF_G][ty] = add(RC_[RCF_G] + (size_t)ty * neuron_cap_, fb);
                tp.o_rc[RCF_E][ty] = add(RC_[RCF_E] + (size_t)ty * neuron_cap_, fb);
                if (rck != SNN_RC_APPROXIMATE) {
                    tp.o_rc[RCF_K1][ty] = add(RC_[RCF_K1] + (size_t)ty * neuron_cap_, fb);
                    tp.o_rc[RCF_K2][ty] = add(RC_[RCF_K2] + (size_t)ty * neuron_cap_, fb);
                }
                if (ty == SNN_NT_NMDA) tp.o_rc[RCF_MG][ty] = add(RC_[RCF_MG] + (size_t)ty * neuron_cap_, fb);
            }
        }
    }
    if (n >= (uint32_t)kMaxTmaStreams) return false;
    tp.n_streams = n;
    tp.stage_bytes = off;
    tp.tx_bytes = 0;
    for (uint32_t k = 0; k < n; ++k) tp.tx_bytes += tp.st[k].bytes_per_tile;
    tp.n_tiles = (uint32_t)((n_neurons + kTmaTile - 1) / kTmaTile);
    // shared-memory budget: as many resident CTAs per SM as the kernel's register budget allows (3, or 2 for
    // Hodgkin-Huxley / general neurotransmitter masks: tma_min_ctas in step_tma.cu) with at least two stages each
    const uint32_t budget = 220 * 1024;
    uint32_t ctas = 3, stages = (budget / ctas) / off;
    if (stages < 2) { ctas = 2; stages = (budget / ctas) / off; }
    if (stages < 2) { ctas = 1; stages = budget / off; }
    if (stages < 2) return false;
    stages = std::min<uint32_t>(stages, 4);
    if ((uint64_t)stages * off + 64 > 227 * 1024) return false;
    tp.stages = stages;
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    *grid = (unsigned)std::min<uint64_t>(tp.n_tiles, (uint64_t)sms * ctas);
    return true;
}

// Operand streams of the window-staged kernel (step_win.cu): radius-1 stencil lattices.
//
// Parameters (win_field_param, and the chemical ones the run reads) are the same in whole blocks of neurons in the common
// case (Lattice::populate copies one neuron into every cell): a tile whose neurons all share the first one's bit patterns
// takes them from its tile row (one copy of at most a few hundred bytes) instead of from one 1 KB stream per parameter.
// When no tile streams its parameters the stage has no room for them, and the ring gets deeper.
int Engine::build_win_params(WinParams &wp, int chemg, bool ntrel, bool stdp, bool lft_pp, int mode, unsigned *grid, bool *eligible) {
    *eligible = false;
    memset(&wp, 0xFF, sizeof wp);
    if (!grid_fast_ || uniform_width_ != kWinWidth || n_neurons == 0) return SNN_OK;
    if (mode == 0) return SNN_OK;
    // tiny lattices are launch-latency bound: the persistent kernel only pays off with at least a few tiles per SM
    if (mode < 2 && n_neurons < 64 * 1024) return SNN_OK;
    uint32_t cols = 0, lat_rows = 0;
    for (auto &L : lats_) if (!L.is_train) { cols = L.cols; lat_rows = L.rows; }
    if (cols == 0) return SNN_OK;
    // the layout with rows; the one without (every parameter streamed) is chosen below when no tile is uniform
    const WinLayout L = win_layout(model, chemg, ntrel, stdp, true, false);
    wp.n_tiles = (uint32_t)((n_neurons + kWinTile - 1) / kWinTile);
    // the parameters: array (per local neuron), word of the tile row, and where a non-uniform tile's stream of it goes
    // (the model's at compile-time offsets, the chemical ones at offsets assigned after the state part of the stage)
    TileParSrc tp{};
    uint32_t par_off[kWinMaxPar] = {}, *par_rt[kWinMaxPar] = {};
    auto par = [&](const float *src, uint32_t word, uint32_t smem_off, uint32_t *rt) {
        if (tp.n_par < (uint32_t)kWinMaxPar) {
            tp.src[tp.n_par] = (const uint32_t *)src; tp.word[tp.n_par] = word;
            par_off[tp.n_par] = smem_off; par_rt[tp.n_par] = rt;
        }
        ++tp.n_par;
    };
    for (int sl = 0; sl < F_NA_CUR; ++sl) {
        if (L.o_f[sl] == 0xFFFFFFFFu) continue;
        if (!F_[sl]) return SNN_OK;
        if (win_field_param(model, ntrel, sl)) par(F_[sl], L.r_f[sl], L.o_f[sl], nullptr);
    }
    const uint32_t ntu = ntrel ? nt_used() : 0u, rcu = ntrel ? rc_used() : 0u;
    for (int ty = 0; ty < kNT; ++ty) {
        auto nt = [&](int sl) { par(NT_[sl] + (size_t)ty * node_cap_ + own0_, L.r_nt + sl * kNT + ty, 0u, &wp.o_nt[sl][ty]); };
        auto rc = [&](int sl) { par(RC_[sl] + (size_t)ty * neuron_cap_, L.r_rc + (sl - RCF_K1) * kNT + ty, 0u, &wp.o_rc[sl][ty]); };
        if (ntu & (1u << ty)) {
            nt(NTF_TMAX);
            if (ntk != SNN_NT_DISCRETE_SPIKE) nt(NTF_P1);
            if (ntk == SNN_NT_DESTEXHE) nt(NTF_P2);
        }
        if (rcu & (1u << ty)) {
            rc(RCF_G);
            rc(RCF_E);
            if (rck != SNN_RC_APPROXIMATE) { rc(RCF_K1); rc(RCF_K2); }
            if (ty == SNN_NT_NMDA) rc(RCF_MG);
        }
    }
    if (tp.n_par > (uint32_t)kWinMaxPar) return SNN_OK;
    tp.row_words = L.row_bytes / 4u;
    tp.n_neurons = (uint32_t)n_neurons;
    tp.n_tiles = wp.n_tiles;
    // the stencil the tiles are checked against: the one sell_grid_kernel writes for this lattice (or strip), every node
    // releasing the union of the release types (a node that releases fewer makes its neighbours' tiles differ)
    tp.col = col_;
    tp.cols = cols;
    tp.row0_global = part_world > 1 ? row0_global : 0u;
    tp.rows_global = part_world > 1 ? rows_global : lat_rows;
    tp.own0 = (uint32_t)own0_;
    tp.stencil_nt = nt_used();
    const int r = refresh_tile_params(tp);
    if (r) return r;
    const uint32_t mixed = tile_par_counts_[0];
    const bool rows = mixed < wp.n_tiles;
    // a stage without col words when every tile is a stencil tile and reads its row.  Not for lattices whose tiles stream their
    // parameters: a variant for them (the row staged for its full-warp mask) measured 5 % slower on Hodgkin-Huxley (DESIGN.md §3)
    wp.stencil = rows && !mixed && tile_par_counts_[1] == 0u ? 1u : 0u;
    wp.stencil_nt = tp.stencil_nt;
    wp.row0_global = tp.row0_global;
    wp.rows_global = tp.rows_global;
    const WinLayout L0 = win_layout(model, chemg, ntrel, stdp, false, false);
    const WinLayout L1 = win_layout(model, chemg, ntrel, stdp, true, wp.stencil != 0u);

    uint32_t off = !rows ? L0.fixed_end : (mixed ? L.fixed_end : L1.uni_end), n = 0;
    auto add_at = [&](const void *src, uint32_t bytes_per_tile, uint32_t smem_off) {
        if (n >= (uint32_t)kMaxTmaStreams) { n = kMaxTmaStreams + 1; return; }
        wp.st[n].src = (const unsigned char *)src;
        wp.st[n].bytes_per_tile = bytes_per_tile;
        wp.st[n].smem_off = smem_off;
        ++n;
    };
    auto add = [&](const void *src, uint32_t bytes_per_tile) -> uint32_t {
        const uint32_t o = off;
        add_at(src, bytes_per_tile, o);
        off += (uint32_t)round_up(bytes_per_tile, 128);
        return o;
    };
    const uint32_t fb = kWinTile * 4;
    if (!rows) {
        // no tile is uniform: every operand streamed, in slot order (no row, no parameter region of its own)
        if (ntrel) add_at(node_flags_ + own0_, kWinTile, L0.o_flags);
        add_at(col_, kWinEdgeBytes, L0.o_col);
        add_at(wgt_, kWinEdgeBytes, L0.o_wgt);
        for (int sl = 0; sl < F_NA_CUR; ++sl)
            if (L0.o_f[sl] != 0xFFFFFFFFu) add_at(F_[sl], fb, L0.o_f[sl]);
        for (int ty = 0; ty < kNT; ++ty) {
            if (ntu & (1u << ty)) {
                wp.o_nt[NTF_TMAX][ty] = add(NT_[NTF_TMAX] + (size_t)ty * node_cap_ + own0_, fb);
                if (ntk != SNN_NT_DISCRETE_SPIKE) wp.o_nt[NTF_P1][ty] = add(NT_[NTF_P1] + (size_t)ty * node_cap_ + own0_, fb);
                if (ntk == SNN_NT_DESTEXHE) wp.o_nt[NTF_P2][ty] = add(NT_[NTF_P2] + (size_t)ty * node_cap_ + own0_, fb);
            }
            if (rcu & (1u << ty)) {
                wp.o_rc[RCF_R][ty] = add(RC_[RCF_R] + (size_t)ty * neuron_cap_, fb);
                wp.o_rc[RCF_G][ty] = add(RC_[RCF_G] + (size_t)ty * neuron_cap_, fb);
                wp.o_rc[RCF_E][ty] = add(RC_[RCF_E] + (size_t)ty * neuron_cap_, fb);
                if (rck != SNN_RC_APPROXIMATE) {
                    wp.o_rc[RCF_K1][ty] = add(RC_[RCF_K1] + (size_t)ty * neuron_cap_, fb);
                    wp.o_rc[RCF_K2][ty] = add(RC_[RCF_K2] + (size_t)ty * neuron_cap_, fb);
                }
                if (ty == SNN_NT_NMDA) wp.o_rc[RCF_MG][ty] = add(RC_[RCF_MG] + (size_t)ty * neuron_cap_, fb);
            }
        }
        wp.tile_par = nullptr;
        wp.n_state = n;
    } else {
        // every tile: flags, edges (the weights only, on stencil stages), state
        if (ntrel) add_at(node_flags_ + own0_, kWinTile, L1.o_flags);
        if (!wp.stencil) add_at(col_, kWinEdgeBytes, L1.o_col);
        add_at(wgt_, kWinEdgeBytes, L1.o_wgt);
        for (int sl = 0; sl < F_NA_CUR; ++sl)
            if (L1.o_f[sl] != 0xFFFFFFFFu && win_field_state(sl)) add_at(F_[sl], fb, L1.o_f[sl]);
        for (int ty = 0; ty < kNT; ++ty)
            if (rcu & (1u << ty)) wp.o_rc[RCF_R][ty] = add(RC_[RCF_R] + (size_t)ty * neuron_cap_, fb);
        wp.tile_par = tile_par_;
        add_at(tile_par_, L1.row_bytes, L1.o_row);
        wp.n_state = n;
        // non-uniform tiles: the parameters
        if (mixed)
            for (uint32_t k = 0; k < tp.n_par; ++k) {
                if (par_rt[k]) *par_rt[k] = add(tp.src[k], fb);
                else add_at(tp.src[k], fb, par_off[k]);
            }
    }
    wp.row_words = tp.row_words;
    if (n > (uint32_t)kMaxTmaStreams) return SNN_OK;
    wp.n_streams = n;
    wp.stage_bytes = (uint32_t)round_up(off, 16);
    wp.node_cap = (uint32_t)node_cap_;
    wp.cols = cols;
    wp.lft_copy = (stdp || lft_pp) ? 1u : 0u;
    // tiles whose windows reach ghost rows (they are also the ones that export): same predicates as the producer's waits
    wp.first_lo = wp.first_hi = wp.bnd_lo = wp.bnd_hi = 0;
    if (part_world > 1) {
        for (uint32_t t = 0; t < wp.n_tiles; ++t) {
            const uint64_t ts = (uint64_t)t * kWinTile;
            if (halo_dir_[0].active && ts <= cols) wp.first_lo++;
            if (halo_dir_[1].active && ts + kWinTile + 1u + cols > n_neurons) wp.first_hi++;
        }
        wp.bnd_lo = wp.first_lo; wp.bnd_hi = wp.first_hi;
        if (wp.first_lo + wp.first_hi > wp.n_tiles) wp.first_lo = wp.first_hi = 0;   // a strip of a few rows: every tile is a boundary tile
    }
    wp.first_end = wp.first_lo + wp.first_hi;
    const uint32_t G = (uint32_t)win_groups(model, chemg, rows && mixed);
    uint32_t stages = (224u * 1024u) / (wp.stage_bytes + 16u);
    stages = std::min<uint32_t>(stages, 8);
    if (stages < G) return SNN_OK;   // the consumer groups need a stage each
    wp.stages = stages;
    wp.ring_check = stages % G != 0u ? 1u : 0u;
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    *grid = (unsigned)std::min<uint64_t>((wp.n_tiles + G - 1) / G, (uint64_t)sms);
    if (*grid == 0) *grid = 1;
    *eligible = true;
    return SNN_OK;
}

int Engine::refresh_tile_params(const TileParSrc &a) {
    if (!tile_par_dirty_ && memcmp(&a, &tile_par_key_, sizeof a) == 0) return SNN_OK;
    const size_t bytes = (size_t)a.n_tiles * a.row_words * 4u;
    if (bytes + 16u > tile_par_bytes_) {
        if (tile_par_) cudaFree(tile_par_);
        tile_par_ = nullptr; tile_par_bytes_ = 0;
        CK(cudaMalloc((void **)&tile_par_, bytes + 16u), SNN_GPU_BUFFER_CREATE_ERROR);
        tile_par_bytes_ = bytes + 16u;
    }
    // the counts of non-uniform and of non-stencil tiles sit after the rows
    unsigned int *d_mixed = (unsigned int *)((char *)tile_par_ + bytes);
    CK(cudaMemsetAsync(tile_par_, 0, bytes + 16u, stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    CK(launch_tile_params(a, tile_par_, d_mixed, stream_), SNN_GPU_QUEUE_FAILURE);
    CK(cudaMemcpyAsync(tile_par_counts_, d_mixed, sizeof tile_par_counts_, cudaMemcpyDeviceToHost, stream_), SNN_GPU_BUFFER_READ_ERROR);
    CK(cudaStreamSynchronize(stream_), SNN_GPU_WAIT_ERROR);
    memcpy(&tile_par_key_, &a, sizeof a);   // compared bytewise above, padding included (build_win_params zeroes it)
    tile_par_dirty_ = false;
    return SNN_OK;
}

// Partition handles of ONE process (attach_local / gpart_attach_local) are stepped from one host thread each, and their kernels
// wait for each other on the device.  CUDA only guarantees progress if every kernel a kernel waits for was launched EARLIER:
// streams that happen to share a hardware work queue execute in launch order, so a waiting kernel queued ahead of the kernel it
// waits for would never see it start (observed as time-outs with 4 handles on one device).  Hence: before launching a kernel
// that waits for the counter value `need`, wait on the host until every local peer has launched the kernel that raises it.
void Engine::wait_local_peers_launched(unsigned long long need, bool second) {
    for (Engine *q : local_peers_) {
        const std::atomic<unsigned long long> &c = second ? q->launched_pub2_ : q->launched_pub_;
        const auto t0 = std::chrono::steady_clock::now();
        while (c.load(std::memory_order_acquire) < need) {
            std::this_thread::sleep_for(std::chrono::microseconds(5));
            // a peer that never runs: fall through after the halo time-out, the device-side wait then reports the error
            if (std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count() > (double)halo_timeout_ms) return;
        }
    }
}

// A per-edge pass of a partitioned handle that reads the neighbours' exports of this timestep's step kernel: it waits for the
// counter value of the step after mine, and my step kernel of this timestep is in the queue already.
void Engine::await_step_exports(StepParams &ep) {
    ep.halo_epoch = halo_epoch_ + 1;
    if (local_peers_.empty()) return;
    launched_pub_.store(halo_epoch_ + 1, std::memory_order_release);
    wait_local_peers_launched(halo_epoch_ + 1, false);
}

// The step path of a run: which kernel steps the neurons of one timestep.  The values are those SNN_OPT_STEP_PATH reports.
enum class StepPath : uint32_t {
    General = 1,     // one thread per neuron (kernels.cu)
    Wide = 2,        // one CTA per slice (step_wide.cu): wide rows
    WideSplit = 3,   // two passes, per-edge terms then ordered sums (step_wide.cu): very wide rows
    Tma = 4,         // TMA-staged persistent kernel (step_tma.cu): other uniform-width stencil lattices
    Win = 5          // window-staged persistent kernel (step_win.cu): radius-1 stencil lattices
};

// Decisions fixed for a whole run(), taken once by plan_run.
struct Engine::RunPlan {
    StepSpec spec;                                 // kernel specialisation (step_spec.h)
    bool rmod = false, rmod_part = false;          // reward-modulated lattice (rmod_part: a row strip of one)
    bool bcm_on = false;                           // BCM rule instead of STDP
    bool net_reward = false, net_rmod = false;     // reward-modulated lattices in a network (net_rmod: one of them modulates)
    bool lft_pp = false;                           // last_firing_time is ping-ponged
    // histories: grid (including the grid record the reductions read), its host copy, spikes, train grid / spikes, reductions
    bool want_grid = false, copy_grid = false, want_spk = false, want_tgrid = false, want_tspk = false, want_red = false;
    // the staged rasters also serve the spike events; copy_*: some lattice of the domain keeps the dense SpikeHistory
    bool copy_spk = false, copy_tspk = false, want_ev = false;
    bool ghist_on = false;
    std::vector<std::pair<uint64_t, uint64_t>> gh_keys;   // blocks whose graph records this run appends to
    StepPath path = StepPath::General;
    bool multi = false;          // a chunk of timesteps per cooperative launch (step_multi.cu)
    bool trains_fused = false;   // WideSplit: the spike trains ride in extra CTAs of the sum pass
    unsigned grid = 0;           // Win / Tma: persistent grid size
    uint32_t wide_chunks_cap = 0;   // WideSplit: chunk buffers per slice
    int tma_iv = -1, tma_il = -1, tma_it[kNT] = {-1, -1, -1};   // Tma: streams whose source ping-pongs (patched every step)
};

// The kernel parameter blocks of a run and its counters.  The step functions patch the per-step fields.
struct Engine::LaunchArgs {
    StepParams sp{};
    TrainParams tp{};
    WinParams win{};
    TmaParams tma{};
    RstdpParams rsp{};   // reward-modulated lattice: dopamine is patched every step
    RnetParams rnp{};    // reward-modulated network: the lattices' dopamine is patched every step
    uint64_t launches = 0;
    float total_ms = 0.f;
};

static constexpr size_t kEvBounceBytes = 4u << 20;

// History staging: chunks of timesteps are recorded on the device and drained to the host between chunks.  Owns the staging
// buffers of one run().
struct Engine::HistStage {
    Engine &e;
    const RunPlan &pl;
    const uint64_t n_words, t_words;
    uint64_t per_step_bytes = 0;   // staged bytes per timestep (0: nothing is recorded)
    uint64_t chunk = 0;            // timesteps per chunk
    float *grid = nullptr, *tgrid = nullptr;
    uint32_t *spk = nullptr, *tspk = nullptr;
    double *red = nullptr;
    uint32_t *red_lat = nullptr;
    std::vector<Lat *> red_lats;   // AverageVoltageHistory / EEGHistory lattices (lats_ is not resized inside run())
    // graph records of a chunk: one per step, plus the final one of a Lattice with STDP (taken after the end-of-run flush)
    float *ghist = nullptr;
    uint64_t gh_recs = 0;
    // how each requested block is cut out of a record: the whole record (the table holds that block only) or one contiguous range
    // per postsynaptic row
    struct GhPlan { GraphHist *h; bool whole; const Block *b; std::vector<uint64_t> src; };
    std::vector<GhPlan> gh_plans;

    HistStage(Engine &eng, const RunPlan &plan)
        : e(eng), pl(plan), n_words((eng.n_neurons + 31) / 32), t_words((eng.n_trains + 31) / 32) {}
    // spike events of a chunk: the lattices recorded (segment order of EvParams), per-tile offsets, per-record offsets, the events
    std::vector<Lat *> ev_lats;
    uint32_t *ev_tile = nullptr, *ev_rec = nullptr, *ev_buf = nullptr;
    uint64_t ev_cap = 0;

    ~HistStage() {
        cudaFree(grid); cudaFree(spk); cudaFree(tgrid); cudaFree(tspk); cudaFree(red); cudaFree(red_lat); cudaFree(ghist);
        cudaFree(ev_tile); cudaFree(ev_rec); cudaFree(ev_buf);
    }
    int cuda_fail(cudaError_t x, int status, const char *what) { return e.cuda_fail(x, status, what); }

    int init(uint64_t iterations);
    int plan_graph_history();
    // the records of step s of the chunk
    void point(StepParams &sp, uint64_t s) const {
        sp.grid_hist = pl.want_grid ? grid + s * e.n_neurons : nullptr;
        sp.spike_hist = pl.want_spk ? spk + s * n_words : nullptr;
    }
    void point(TrainParams &tp, uint64_t s) const {
        tp.grid_hist = pl.want_tgrid ? tgrid + s * e.n_trains : nullptr;
        tp.spike_hist = pl.want_tspk ? tspk + s * t_words : nullptr;
    }
    void point(MultiParams &mp, uint64_t s) const {
        mp.grid_hist = pl.want_grid ? grid + s * e.n_neurons : nullptr;
        mp.spike_hist = pl.want_spk ? spk + s * n_words : nullptr;
        mp.tgrid_hist = pl.want_tgrid ? tgrid + s * e.n_trains : nullptr;
        mp.tspike_hist = pl.want_tspk ? tspk + s * t_words : nullptr;
    }
    // Lattice::iterate records after the step's plasticity (neuron/mod.rs:973-979); lazily applied STDP lands in the table with
    // the next step kernel (or the end-of-run flush), so a Lattice with STDP records step k after step kernel k + 1.
    // LatticeNetwork records before the step's STDP (neuron/mod.rs:2565-2576): the table after step kernel k.  BCM is applied
    // right after the step.
    cudaError_t record_graph(uint64_t &launches) {
        if (!e.ghist_nnz_) { ++gh_recs; return cudaSuccess; }
        cudaError_t x = launch_graph_record(e.wgt_, e.slice_off_, e.ghist_row_off_, e.n_slices_, e.max_slice_width_,
                                            ghist + gh_recs * e.ghist_nnz_, e.stream_);
        if (x == cudaSuccess) { ++gh_recs; ++launches; }
        return x;
    }
    int drain(uint64_t steps);
    int drain_graph();
    int drain_events(uint64_t steps);
    int d2h(void *dst, const void *src, size_t bytes);
};

int Engine::HistStage::init(uint64_t iterations) {
    if (pl.ghist_on) { int r = plan_graph_history(); if (r) return r; }
    if (pl.want_grid) per_step_bytes += e.n_neurons * 4;
    if (pl.want_spk) per_step_bytes += n_words * 4;
    if (pl.want_tgrid) per_step_bytes += e.n_trains * 4;
    if (pl.want_tspk) per_step_bytes += t_words * 4;
    if (pl.ghist_on) per_step_bytes += std::max<uint64_t>(e.ghist_nnz_, 1) * 4;
    chunk = iterations;
    if (per_step_bytes) chunk = std::max<uint64_t>(1, std::min<uint64_t>(iterations, (256ull << 20) / per_step_bytes));
    if (pl.want_grid) CK(dev_alloc(&grid, chunk * e.n_neurons), SNN_GPU_BUFFER_CREATE_ERROR);
    if (pl.want_spk) CK(dev_alloc(&spk, chunk * n_words), SNN_GPU_BUFFER_CREATE_ERROR);
    if (pl.want_tgrid) CK(dev_alloc(&tgrid, chunk * e.n_trains), SNN_GPU_BUFFER_CREATE_ERROR);
    if (pl.want_tspk) CK(dev_alloc(&tspk, chunk * t_words), SNN_GPU_BUFFER_CREATE_ERROR);
    if (pl.want_red) {
        for (auto &L : e.lats_) if (!L.is_train && (L.avg_hist || L.eeg_hist)) red_lats.push_back(&L);
        const size_t nl = red_lats.size();
        std::vector<uint32_t> meta(3 * nl);
        for (size_t k = 0; k < nl; ++k) {
            meta[k] = (uint32_t)red_lats[k]->off; meta[nl + k] = (uint32_t)red_lats[k]->n;
            memcpy(&meta[2 * nl + k], &red_lats[k]->eeg_ref, 4);
        }
        CK(dev_alloc(&red, chunk * nl * 2), SNN_GPU_BUFFER_CREATE_ERROR);
        CK(dev_alloc(&red_lat, 3 * nl), SNN_GPU_BUFFER_CREATE_ERROR);
        CK(h2d_sync(red_lat, meta.data(), meta.size() * 4, e.stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    }
    if (pl.ghist_on && e.ghist_nnz_) CK(dev_alloc(&ghist, (chunk + 1) * e.ghist_nnz_), SNN_GPU_BUFFER_CREATE_ERROR);
    if (pl.want_ev) {
        uint64_t words = 0;
        for (int dom = 0; dom < 2; ++dom)
            for (auto &L : e.lats_)
                if (L.spike_events && L.is_train == (dom == 1)) {
                    ev_lats.push_back(&L);
                    if (L.n) words += (L.off + L.n + 31) / 32 - L.off / 32;
                }
        CK(dev_alloc(&ev_tile, (uint64_t)ev_tiles((uint32_t)(chunk * words)) + 1), SNN_GPU_BUFFER_CREATE_ERROR);
        CK(dev_alloc(&ev_rec, chunk * ev_lats.size()), SNN_GPU_BUFFER_CREATE_ERROR);
        if (!e.ev_bounce_) CK(cudaMallocHost(&e.ev_bounce_, kEvBounceBytes), SNN_GPU_BUFFER_CREATE_ERROR);
    }
    return SNN_OK;
}

// Device -> host through the pinned bounce buffer, on the engine's stream.
int Engine::HistStage::d2h(void *dst, const void *src, size_t bytes) {
    for (size_t o = 0; o < bytes; o += kEvBounceBytes) {
        const size_t b = std::min<size_t>(kEvBounceBytes, bytes - o);
        CK(cudaMemcpyAsync(e.ev_bounce_, (const char *)src + o, b, cudaMemcpyDeviceToHost, e.stream_), SNN_GPU_BUFFER_READ_ERROR);
        CK(cudaStreamSynchronize(e.stream_), SNN_GPU_WAIT_ERROR);
        memcpy((char *)dst + o, e.ev_bounce_, b);
    }
    return SNN_OK;
}

// The chunk's spike events (spike_events.cu): count, scan, size the event buffer from the total, scatter; then only the per-record
// offsets and the events cross to the host, appended to each lattice's lists.
int Engine::HistStage::drain_events(uint64_t steps) {
    EvParams p{};
    p.steps = (uint32_t)steps;
    std::vector<Lat *> segs;   // lattice of each segment (lattices without cells have none)
    uint64_t items = 0;
    for (Lat *L : ev_lats) {
        if (!L->n) continue;
        EvSeg &g = p.seg[p.n_seg++];
        g.raster = L->is_train ? tspk : spk;
        g.stride = (uint32_t)(L->is_train ? t_words : n_words);
        g.bit0 = (uint32_t)L->off; g.bit1 = (uint32_t)(L->off + L->n);
        g.w0 = g.bit0 / 32; g.nw = (g.bit1 + 31) / 32 - g.w0;
        // partitions own one lattice: its events are global flat indices of the whole lattice
        g.add = L->is_train ? 0u : e.row0_global * L->cols;
        g.item0 = (uint32_t)items;
        items += steps * g.nw;
        segs.push_back(L);
    }
    p.n_items = (uint32_t)items;
    const uint32_t tiles = ev_tiles(p.n_items);
    CK(launch_spike_event_count(p, ev_tile, e.stream_), SNN_GPU_QUEUE_FAILURE);
    uint32_t total = 0;
    int r = d2h(&total, ev_tile + tiles, 4);
    if (r) return r;
    if (total > ev_cap) {   // grown from the chunk's own total, never sized for the worst case up front
        const uint64_t cap = std::max<uint64_t>(total, 2 * ev_cap);
        cudaFree(ev_buf);
        ev_buf = nullptr; ev_cap = 0;
        CK(dev_alloc(&ev_buf, cap), SNN_GPU_BUFFER_CREATE_ERROR);
        ev_cap = cap;
    }
    CK(launch_spike_event_scatter(p, ev_tile, ev_buf, ev_rec, e.stream_), SNN_GPU_QUEUE_FAILURE);
    std::vector<uint32_t> rec((size_t)p.n_seg * steps + 1);
    if ((r = d2h(rec.data(), ev_rec, (rec.size() - 1) * 4))) return r;
    rec.back() = total;
    for (uint32_t k = 0; k < p.n_seg; ++k) {
        Lat &L = *segs[k];
        const uint32_t a = rec[(size_t)k * steps], b = rec[(size_t)(k + 1) * steps];
        const size_t o = L.ev_neuron.size();
        L.ev_neuron.resize(o + (b - a));
        if ((r = d2h(L.ev_neuron.data() + o, ev_buf + a, (size_t)(b - a) * 4))) return r;
        if (L.ev_ptr.empty()) L.ev_ptr.push_back(0);
        for (uint64_t s = 0; s < steps; ++s) L.ev_ptr.push_back(o + (rec[(size_t)k * steps + s + 1] - a));
    }
    for (Lat *L : ev_lats)
        if (!L->n) { if (L->ev_ptr.empty()) L->ev_ptr.push_back(0); L->ev_ptr.insert(L->ev_ptr.end(), steps, L->ev_neuron.size()); }
    return SNN_OK;
}

// Per-row offsets of the table's canonical order (once per graph build), then how each requested block is cut out of a record.
int Engine::HistStage::plan_graph_history() {
    if (!e.ghist_off_valid_) {
        if (e.ghist_row_off_) cudaFree(e.ghist_row_off_);
        e.ghist_row_off_ = nullptr;
        CK(dev_alloc(&e.ghist_row_off_, (size_t)e.n_slices_ * 32 + 1), SNN_GPU_BUFFER_CREATE_ERROR);
        CK(launch_graph_row_offsets(e.col_, e.slice_off_, e.n_slices_, e.ghist_row_off_, e.stream_), SNN_GPU_QUEUE_FAILURE);
        uint32_t tot = 0;
        CK(cudaMemcpyAsync(&tot, e.ghist_row_off_ + (size_t)e.n_slices_ * 32, 4, cudaMemcpyDeviceToHost, e.stream_), SNN_GPU_BUFFER_READ_ERROR);
        CK(cudaStreamSynchronize(e.stream_), SNN_GPU_WAIT_ERROR);
        e.ghist_nnz_ = tot;
        e.ghist_off_valid_ = true;
    }
    std::vector<uint64_t> roff;   // canonical row offsets of the table from the host blocks (several blocks only)
    for (auto &key : pl.gh_keys) {
        GhPlan gp{&e.graph_hist_[key], false, nullptr, {}};
        auto it = e.blocks_.find(key);
        if (it != e.blocks_.end() && e.blocks_.size() == 1) {
            gp.whole = true;
            gp.h->nnz = e.ghist_nnz_;
        } else if (it != e.blocks_.end()) {
            // finalize_graph's general path: every block is host CSR
            if (roff.empty()) {
                roff.assign(e.n_neurons + 1, 0);
                e.for_each_row_segment([&](const Lat &B, uint64_t q, const Lat &, Block &b, uint64_t) {
                    roff[B.off + q + 1] += b.row_ptr[q + 1] - b.row_ptr[q];
                });
                for (uint64_t i = 0; i < e.n_neurons; ++i) roff[i + 1] += roff[i];
                if (roff[e.n_neurons] != e.ghist_nnz_) return e.fail(SNN_GPU_BUFFER_READ_ERROR, "graph history: host and device tables disagree");
            }
            const Lat *B = e.find(key.second);
            gp.b = &it->second;
            gp.src.resize(B->n);
            e.for_each_row_segment([&](const Lat &, uint64_t q, const Lat &A, Block &, uint64_t k) {
                if (A.id == key.first) gp.src[q] = roff[B->off + q] + k;
            }, B);
            gp.h->nnz = it->second.pre.size();
        } else {
            gp.h->nnz = 0;   // a lattice without an internal graph: empty records
        }
        gh_plans.push_back(std::move(gp));
    }
    return SNN_OK;
}

// The graph records of the chunk: each requested block's weights cut out of the canonical order.
int Engine::HistStage::drain_graph() {
    const uint64_t nz = e.ghist_nnz_;
    cudaError_t x = cudaSuccess;
    if (nz && gh_plans.size() == 1 && gh_plans[0].whole) {
        std::vector<float> &w = gh_plans[0].h->w;   // straight into the block's record vector
        const size_t o = w.size();
        w.resize(o + gh_recs * nz);
        x = cudaMemcpy(w.data() + o, ghist, gh_recs * nz * 4, cudaMemcpyDeviceToHost);
    } else if (nz) {
        std::vector<float> hr(gh_recs * nz);
        x = cudaMemcpy(hr.data(), ghist, hr.size() * 4, cudaMemcpyDeviceToHost);
        for (auto &gp : gh_plans) {
            if (x != cudaSuccess || gp.h->nnz == 0) continue;
            std::vector<float> &w = gp.h->w;
            for (uint64_t k = 0; k < gh_recs; ++k) {
                const float *rec = hr.data() + k * nz;
                if (gp.whole) { w.insert(w.end(), rec, rec + nz); continue; }
                const size_t o = w.size();
                w.resize(o + gp.h->nnz);
                const uint64_t n_post = gp.src.size();
                for (uint64_t q = 0; q < n_post; ++q) {
                    const uint64_t a = gp.b->row_ptr[q], c = gp.b->row_ptr[q + 1] - a;
                    if (c) memcpy(w.data() + o + a, rec + gp.src[q], c * 4);
                }
            }
        }
    }
    if (x != cudaSuccess) return cuda_fail(x, SNN_GPU_BUFFER_READ_ERROR, "graph history drain");
    for (auto &gp : gh_plans) gp.h->steps += gh_recs;
    gh_recs = 0;
    return SNN_OK;
}

// The records of the chunk's `steps` timesteps, appended to the lattices' host histories.
int Engine::HistStage::drain(uint64_t steps) {
    if (pl.ghist_on && gh_recs) { int r = drain_graph(); if (r) return r; }
    if (pl.want_ev) { int r = drain_events(steps); if (r) return r; }
    if (!per_step_bytes) return SNN_OK;
    const uint64_t n_neurons = e.n_neurons, n_trains = e.n_trains;
    std::vector<float> hg, htg; std::vector<uint32_t> hs, hts;
    cudaError_t he = cudaSuccess;
    if (pl.copy_grid) { hg.resize(steps * n_neurons); he = cudaMemcpy(hg.data(), grid, hg.size() * 4, cudaMemcpyDeviceToHost); }
    if (he != cudaSuccess) return cuda_fail(he, SNN_GPU_BUFFER_READ_ERROR, "grid history drain");
    if (pl.want_red) {
        const size_t nl = red_lats.size();
        cudaError_t re = launch_history_reduce(grid, n_neurons, (uint32_t)steps, red_lat, red_lat + nl, (const float *)(red_lat + 2 * nl),
                                               (int)nl, red, e.stream_);
        std::vector<double> hr(steps * nl * 2);
        // stream_ is non-blocking: a copy on the legacy stream would not wait for the reduction
        if (re == cudaSuccess) re = cudaMemcpyAsync(hr.data(), red, hr.size() * 8, cudaMemcpyDeviceToHost, e.stream_);
        if (re == cudaSuccess) re = cudaStreamSynchronize(e.stream_);
        if (re != cudaSuccess) return cuda_fail(re, SNN_GPU_BUFFER_READ_ERROR, "history reduce");
        for (size_t k = 0; k < nl; ++k) {
            Lat &L = *red_lats[k];
            for (uint64_t s = 0; s < steps; ++s) {
                const double sum_v = hr[(s * nl + k) * 2], sum_dv = hr[(s * nl + k) * 2 + 1];
                // AverageVoltageHistory::update, neuron/mod.rs:310-316: sum / len as f32
                if (L.avg_hist) L.average_history.push_back((float)sum_v / (float)L.n);
                // EEGHistory::update, neuron/mod.rs:266-279: (1 / (4 pi sigma d)) * total_current
                if (L.eeg_hist) L.eeg_history.push_back((1.f / (4.f * 3.14159274101257324f * L.eeg_cond * L.eeg_dist)) * (float)sum_dv);
            }
            if (!L.grid_hist && !L.spike_hist) L.hist_len += steps;
        }
    }
    if (pl.copy_spk) { hs.resize(steps * n_words); he = cudaMemcpy(hs.data(), spk, hs.size() * 4, cudaMemcpyDeviceToHost); }
    if (he == cudaSuccess && pl.want_tgrid) { htg.resize(steps * n_trains); he = cudaMemcpy(htg.data(), tgrid, htg.size() * 4, cudaMemcpyDeviceToHost); }
    if (he == cudaSuccess && pl.copy_tspk) { hts.resize(steps * t_words); he = cudaMemcpy(hts.data(), tspk, hts.size() * 4, cudaMemcpyDeviceToHost); }
    if (he != cudaSuccess) return cuda_fail(he, SNN_GPU_BUFFER_READ_ERROR, "history drain");
    // SpikeHistory::aggregate (neuron/mod.rs:335-359): the sum over the chunk's steps is taken on the device from the staged
    // raster; the host only adds one count per neuron and chunk
    std::vector<uint32_t> cnt_n, cnt_t;
    for (int dom = 0; dom < 2 && he == cudaSuccess; ++dom) {
        const bool on = dom ? pl.copy_tspk : pl.copy_spk;
        const uint64_t dn = dom ? n_trains : n_neurons, dw = dom ? t_words : n_words;
        if (!on || dn == 0) continue;
        std::vector<uint32_t> &cnt = dom ? cnt_t : cnt_n;
        cnt.resize(dn);
        if (e.ensure_scratch(dn * 4)) { he = cudaErrorMemoryAllocation; break; }
        he = launch_spike_count(dom ? tspk : spk, (uint32_t)steps, dw, dn, (uint32_t *)e.scratch_, e.stream_);
        if (he == cudaSuccess) he = cudaMemcpyAsync(cnt.data(), e.scratch_, dn * 4, cudaMemcpyDeviceToHost, e.stream_);
        if (he == cudaSuccess) he = cudaStreamSynchronize(e.stream_);
    }
    if (he != cudaSuccess) return cuda_fail(he, SNN_GPU_BUFFER_READ_ERROR, "spike aggregate");
    for (auto &L : e.lats_) {
        if (!L.grid_hist && !L.spike_hist) continue;
        const uint64_t dom_n = L.is_train ? n_trains : n_neurons, dom_w = L.is_train ? t_words : n_words;
        const std::vector<float> &G = L.is_train ? htg : hg;
        const std::vector<uint32_t> &S = L.is_train ? hts : hs;
        if (L.spike_hist) {
            const std::vector<uint32_t> &cnt = L.is_train ? cnt_t : cnt_n;
            if (L.spike_agg.size() != L.n) L.spike_agg.assign(L.n, 0);
            for (uint64_t j = 0; j < L.n; ++j) L.spike_agg[j] += cnt[L.off + j];
        }
        for (uint64_t s = 0; s < steps; ++s) {
            if (L.grid_hist) L.grid_history.insert(L.grid_history.end(), G.begin() + s * dom_n + L.off, G.begin() + s * dom_n + L.off + L.n);
            if (L.spike_hist) {
                const size_t o = L.spike_history.size();
                L.spike_history.resize(o + L.n);
                for (uint64_t j = 0; j < L.n; ++j) {
                    const uint64_t b = L.off + j;
                    L.spike_history[o + j] = (uint8_t)((S[s * dom_w + (b >> 5)] >> (b & 31)) & 1u);
                }
            }
        }
        L.hist_len += steps;
    }
    return SNN_OK;
}

// Difference tables of the STDP term, one per lattice (lattice l at tab + l * 2 * tab_n, the layout of RstdpParams::tab), long
// enough for every exponential to have underflowed to zero at its end.  Only a, tau and dt of each entry are read.  *tab stays
// null when a time constant is out of range: the kernels evaluate the formula then.
int Engine::build_stdp_tables(const std::vector<RstdpParams> &lat, const float **tab, uint32_t *tab_n) {
    double reach = 0.0;
    bool ok = true;
    for (const RstdpParams &q : lat) {
        ok = ok && q.tau_plus > 0.f && q.tau_minus > 0.f && q.dt > 0.f;
        reach = std::max(reach, 110.0 * std::max((double)q.tau_plus, (double)q.tau_minus) / std::max((double)q.dt, 1e-30));
    }
    if (!ok || !(reach > 0 && reach < 60000.0)) return SNN_OK;
    const uint32_t n = (uint32_t)reach + 8u;
    const size_t need = lat.size() * 2u * n;
    if (stdp_tab_elems_ != need) {
        if (stdp_tab_) cudaFree(stdp_tab_);
        stdp_tab_ = nullptr; stdp_tab_elems_ = 0;
        CK(dev_alloc(&stdp_tab_, need), SNN_GPU_BUFFER_CREATE_ERROR);
        stdp_tab_elems_ = need;
    }
    for (size_t l = 0; l < lat.size(); ++l)   // the parameters may have changed since the last run
        CK(launch_rstdp_table(lat[l], stdp_tab_ + l * 2u * n, n, stream_), SNN_GPU_QUEUE_FAILURE);
    *tab = stdp_tab_; *tab_n = n;
    return SNN_OK;
}

// RewardModulatedLatticeNetwork: reward-modulated lattices next to plain lattices and spike trains.  Refuses the configurations
// the reference cannot run itself.
int Engine::build_rnet_params(RnetParams &rnp, bool *net_rmod) {
    if (part_world > 1 || reward_mode || bcm_mode) return fail(SNN_UNSUPPORTED, "reward-modulated lattice networks run on single-GPU network handles");
    // update_weights_from_neurons_across_(reward_)lattices looks the OUTGOING connecting edges up with the end points swapped and
    // unwraps the result (neuron/mod.rs:4760-4763, 4931-4934), and its incoming arms unwrap lattice kinds that need not be there
    // (:4727-4731, 4741-4747)
    for (auto &kv : blocks_) {
        if (kv.first.first == kv.first.second) continue;
        if (kv.second.kind != Block::GRID && kv.second.pre.empty()) continue;
        const Lat *A = find(kv.first.first), *B = find(kv.first.second);
        if (!A || !B) continue;
        if (A->is_reward && A->do_modulation)
            return fail(SNN_UNSUPPORTED, "connecting edges out of a reward-modulated lattice with do_modulation: the reference panics on them (neuron/mod.rs:4931-4934)");
        if (!A->is_train && !A->is_reward && A->do_plasticity)
            return fail(SNN_UNSUPPORTED, "connecting edges out of a plastic lattice of a reward-modulated network: the reference panics on them (neuron/mod.rs:4760-4763)");
        if (!B->is_reward && kv.second.reward_conn)
            return fail(SNN_UNSUPPORTED, "RewardModulatedWeight connections must end in a reward-modulated lattice");
        if (!B->is_reward && B->do_plasticity && A->is_reward)
            return fail(SNN_UNSUPPORTED, "a plastic lattice fed by a reward-modulated lattice: the reference panics on it (neuron/mod.rs:4727-4731)");
    }
    *net_rmod = false;
    std::map<uint64_t, int> cls;   // lattice id -> presynaptic class of RnetParams::kinds
    std::vector<const Lat *> nl;
    int kn = 0, kt = 0;
    for (auto &L : lats_) {
        if (L.is_train) { rnp.tl_base[kt] = (uint32_t)L.off; cls[L.id] = kMaxLattices + kt; ++kt; continue; }
        RnetLat &R = rnp.lat[kn];
        R.dopamine = L.rstdp.dopamine; R.tau_c = L.rstdp.tau_c; R.a_plus = L.rstdp.a_plus; R.a_minus = L.rstdp.a_minus;
        R.tau_plus = L.rstdp.tau_plus; R.tau_minus = L.rstdp.tau_minus; R.dt = L.rstdp.dt;
        R.flags = (L.is_reward ? 1u : 0u) | (L.is_reward && L.do_modulation ? 2u : 0u);
        *net_rmod |= L.is_reward && L.do_modulation && L.n > 0;
        rnp.nbase[kn] = (uint32_t)L.off;
        nl.push_back(&L);
        cls[L.id] = kn++;
    }
    rnp.n_lat = (uint32_t)kn; rnp.nbase[kn] = (uint32_t)n_neurons;
    rnp.n_tl = (uint32_t)kt; rnp.tl_base[kt] = (uint32_t)n_trains; rnp.train0 = train0_;
    for (int post = 0; post < kn; ++post) {
        if (!nl[post]->is_reward) continue;
        uint64_t k = 1ull << (2 * post);                                 // own graph
        for (int pre = 0; pre < kn; ++pre)
            if (pre != post && !nl[pre]->is_reward) k |= 3ull << (2 * pre);   // Weight block fed by a plain lattice (the default kind)
        rnp.kinds[post] = k;
    }
    for (auto &kv : blocks_)
        if (kv.second.reward_conn && kv.first.first != kv.first.second && cls.count(kv.first.first) && cls.count(kv.first.second)) {
            uint64_t &k = rnp.kinds[cls[kv.first.second]];
            const int q = cls[kv.first.first];
            k = (k & ~(3ull << (2 * q))) | (2ull << (2 * q));
        }
    if (!*net_rmod) return SNN_OK;
    int r = ensure_reward_arrays();
    if (r) return r;
    rnp.counter = rs_counter_; rnp.dw = rs_dw_; rnp.c = rs_c_;
    rnp.canonical = rs_canonical_ ? 1u : 0u;
    // one table per neuron lattice: the modulator's STDP term for a reward-modulated lattice, the lattice's own STDP for a plain
    // one (what Weight edges out of it use)
    std::vector<RstdpParams> tl(nl.size(), RstdpParams{});
    for (size_t l = 0; l < nl.size(); ++l) {
        const Lat &L = *nl[l];
        RstdpParams &q = tl[l];
        if (L.is_reward) { q.a_plus = L.rstdp.a_plus; q.a_minus = L.rstdp.a_minus; q.tau_plus = L.rstdp.tau_plus; q.tau_minus = L.rstdp.tau_minus; q.dt = L.rstdp.dt; }
        else { q.a_plus = L.stdp.a_plus; q.a_minus = L.stdp.a_minus; q.tau_plus = L.stdp.tau_plus; q.tau_minus = L.stdp.tau_minus; q.dt = L.stdp.dt; }
    }
    return build_stdp_tables(tl, &rnp.tab, &rnp.tab_n);
}

// Refusals, the device graph, and every decision fixed for the whole run, with the kernel parameter blocks it selects.
int Engine::plan_run(RunPlan &pl, LaunchArgs &a) {
    for (auto &L : lats_) if (!L.is_train && L.graph_hist) pl.gh_keys.emplace_back(L.id, L.id);
    if (conn_graph_hist)
        for (auto &kv : blocks_)
            if (kv.first.first != kv.first.second && (kv.second.kind == Block::GRID || !kv.second.pre.empty())) pl.gh_keys.push_back(kv.first);
    pl.ghist_on = !pl.gh_keys.empty();
    if (pl.ghist_on && part_world > 1) return fail(SNN_UNSUPPORTED, "graph history: whole-GPU handles only (not row strips or general-graph partitions)");
    if (pl.ghist_on && (reward_mode || has_reward_lattices()))
        return fail(SNN_UNSUPPORTED, "graph history: not recorded for reward-modulated lattices and networks (TraceRSTDP weights)");
    if (part_world > 1 && !gpart_) {
        if ((part_rank > 0 && !halo_dir_[0].active) || (part_rank < part_world - 1 && !halo_dir_[1].active))
            return fail(SNN_INVALID_ARGUMENT, "partitioned handle: neighbouring strips are not attached");
    }
    if (gpart_ && reward_mode) return fail(SNN_UNSUPPORTED, "general-graph partitions step plain, STDP and BCM lattices");
    CK(cudaSetDevice(device), SNN_GPU_GET_DEVICE_FAILURE);
    if (chemical) { int r = ensure_chem(); if (r) return r; }
    int r = finalize_graph();
    if (r) return r;
    r = upload_lat_table();
    if (r) return r;
    if (gpart_) { r = gpart_build_device(); if (r) return r; }

    for (auto &L : lats_) {
        if (!L.is_train) { pl.spec.stdp |= L.do_plasticity && !L.is_reward; pl.want_grid |= L.grid_hist; pl.copy_spk |= L.spike_hist; pl.want_red |= L.avg_hist || L.eeg_hist; }
        else { pl.want_tgrid |= L.grid_hist; pl.copy_tspk |= L.spike_hist; }
        pl.want_ev |= L.spike_events;
    }
    for (auto &L : lats_) {
        const bool stage = L.spike_hist || L.spike_events;
        (L.is_train ? pl.want_tspk : pl.want_spk) |= stage;
    }
    // AverageVoltageHistory / EEGHistory are reductions of the staged grid record (it stays on the device for them)
    pl.copy_grid = pl.want_grid;
    pl.want_grid = pl.want_grid || pl.want_red;
    pl.spec.model = model;
    pl.spec.ntrel = chem_alloc_ &&(chemical || nt_used() != 0 || (model == SNN_MODEL_HODGKIN_HUXLEY && rc_used() != 0));
    pl.spec.net = n_neuron_lattices() > 1 || n_trains > 0;
    if (chemical && pl.spec.ntrel && nt_used() != 0) pl.spec.chemg = (!pl.spec.net && __builtin_popcount(nt_used()) == 1) ? 1 : 3;
    // reward-modulated lattice: the modulator replaces the plasticity rule and needs last_firing_time before and after a step
    pl.rmod = reward_mode && do_modulation && n_neurons > 0;
    // BCM rule instead of STDP: applied by its own per-edge kernel right after each step (it reads the activities the step wrote)
    pl.bcm_on = bcm_mode && pl.spec.stdp && !reward_mode && n_neurons > 0;
    if (reward_mode || bcm_mode) pl.spec.stdp = false;
    if (pl.rmod) { r = ensure_reward_arrays(); if (r) return r; }
    a.rsp = RstdpParams{rstdp.dopamine, rstdp.tau_c, rstdp.a_plus, rstdp.a_minus, rstdp.tau_plus, rstdp.tau_minus, rstdp.dt,
                        rs_counter_, rs_dw_, rs_c_, rs_canonical_ ? 1u : 0u, nullptr, 0u};
    if (pl.rmod) { r = build_stdp_tables({a.rsp}, &a.rsp.tab, &a.rsp.tab_n); if (r) return r; }
    pl.net_reward = has_reward_lattices();
    if (pl.net_reward) { r = build_rnet_params(a.rnp, &pl.net_rmod); if (r) return r; }
    pl.lft_pp = pl.spec.stdp || pl.rmod || pl.net_rmod || (n_trains && electrical) || part_world > 1;
    pl.rmod_part = pl.rmod && part_world > 1;

    fill_step_params(a.sp);
    a.sp.lft_pp = pl.lft_pp;
    if (pl.rmod_part)   // step s + 1 overwrites ghost slots that the neighbour's per-edge kernel of step s still reads: wait for that one
        for (int d = 0; d < 2; ++d) a.sp.halo[d].my_flag = halo_dir_[d].my_flag2;
    if (n_trains) {
        TrainParams &tp = a.tp;
        tp.train0 = train0_; tp.n_trains = (uint32_t)n_trains; tp.kind = train_kind; tp.ntk = ntk; tp.seed = seed;
        tp.t_stride = node_cap_; tp.node_flags = node_flags_; tp.nt_stride = node_cap_;
        for (int s = 0; s < NTF_COUNT; ++s) tp.nt[s] = NT_[s];
        for (int s = 0; s < TF_COUNT; ++s) tp.tf[s] = TF_[s];
        tp.ft_off = ft_off_; tp.ft = ft_; tp.lft_pp = pl.lft_pp;
    }
    return plan_step_path(pl, a);
}

// The step path, and whether a whole chunk of timesteps goes into one launch.
int Engine::plan_step_path(RunPlan &pl, LaunchArgs &a) {
    // SNN_B200_TMA: 0 never takes the staged kernels, 2 takes them at any lattice size (the tests cover them at small sizes);
    // SNN_B200_WIN=0 leaves the window kernel out
    const char *tma_env = getenv("SNN_B200_TMA"), *win_env = getenv("SNN_B200_WIN");
    const int tma_mode = tma_env ? atoi(tma_env) : 1;
    const int win_mode = (win_env && atoi(win_env) == 0) ? 0 : tma_mode;
    bool win = false;
    if (!pl.spec.net) {
        const int r = build_win_params(a.win, pl.spec.chemg, pl.spec.ntrel, pl.spec.stdp, pl.lft_pp, win_mode, &pl.grid, &win);
        if (r) return r;
    }
    last_uniform_tiles = win ? a.win.n_tiles - tile_par_counts_[0] : 0u;
    last_stencil_tiles = win && a.win.stencil ? a.win.n_tiles : 0u;
    if (win) {
        pl.path = StepPath::Win;
    } else if (!pl.spec.net && build_tma_params(a.tma, pl.spec.ntrel, pl.spec.stdp, pl.lft_pp, tma_mode, &pl.grid)) {
        pl.path = StepPath::Tma;
        for (uint32_t k = 0; k < a.tma.n_streams; ++k) {
            if (a.tma.st[k].smem_off == a.tma.o_v) pl.tma_iv = (int)k;
            if ((pl.spec.stdp || pl.lft_pp) && a.tma.st[k].smem_off == a.tma.o_lft) pl.tma_il = (int)k;
            for (int ty = 0; ty < kNT; ++ty) if (a.tma.o_t[ty] != 0xFFFFFFFFu && a.tma.st[k].smem_off == a.tma.o_t[ty]) pl.tma_it[ty] = (int)k;
        }
    } else if (part_world == 1 && n_slices_ > 0 && sell_krows_ / n_slices_ >= kWideMinWidth) {
        // wide rows (hundreds of in-edges per neuron, e.g. all-to-all spike-train input): one CTA per slice.  Very wide slices
        // (hundreds of k-rows): one SM per slice cannot issue the per-edge instructions fast enough — two passes, the per-edge
        // terms of every (slice, chunk) on its own CTA, then the ordered sums (step_wide.cu)
        pl.path = sell_krows_ / n_slices_ >= 2 * wide_chunk_krows() ? StepPath::WideSplit : StepPath::Wide;
    }
    if (pl.path == StepPath::WideSplit) {
        pl.wide_chunks_cap = (max_slice_width_ + wide_chunk_krows() - 1) / wide_chunk_krows();
        const size_t chunks_bytes = (size_t)n_slices_ * pl.wide_chunks_cap * wide_chunk_bytes(pl.spec.chemg);
        const size_t need = chunks_bytes + (size_t)n_slices_ * wide_part_bytes();
        if (need != wide_scratch_bytes_) {
            if (wide_scratch_) cudaFree(wide_scratch_);
            wide_scratch_ = nullptr; wide_scratch_bytes_ = 0;
            CK(cudaMalloc((void **)&wide_scratch_, need), SNN_GPU_BUFFER_CREATE_ERROR);
            wide_scratch_bytes_ = need;
        }
        // the arrival counters of the sum pass start at zero (they reset themselves after every timestep)
        CK(cudaMemsetAsync(wide_scratch_ + chunks_bytes, 0, (size_t)n_slices_ * wide_part_bytes(), stream_), SNN_GPU_BUFFER_WRITE_ERROR);
        // the spike trains ride in extra CTAs of the sum pass (nothing in that pass reads train state; the terms pass, which
        // does, has completed) — one launch and one launch gap less per timestep
        pl.trains_fused = n_neurons && n_trains > 0;
    }
    // small lattices / networks (everything the staged kernels do not take): a whole chunk of timesteps per cooperative launch
    // (step_multi.cu).  SNN_OPT_STEPS_PER_GRAPH: 0 = as many as the history chunk holds, 1 = one launch per timestep, k = at most
    // k.  Graph records are taken between launches, and the two-pass wide kernels are one-launch-per-step kernels.
    pl.multi = part_world == 1 && n_neurons > 0 && (pl.path == StepPath::Wide || pl.path == StepPath::General) && !pl.bcm_on &&
               !reward_mode && !pl.net_reward && steps_per_graph != 1 && !pl.ghist_on;
    if (pl.multi) {
        MultiParams probe{};
        probe.wide_stage = (pl.path == StepPath::Wide && n_nodes_ <= 4096) ? 1u : 0u;
        pl.multi = launch_step_multi(a.sp, a.tp, probe, pl.spec, pl.path == StepPath::Wide, device, true, stream_) == cudaSuccess;
        cudaGetLastError();
    }
    last_step_path = (uint32_t)pl.path + (pl.multi ? 16u : 0u);
    return SNN_OK;
}

// Multi-GPU: push the current boundary state into the neighbours' ghost slots, then meet the neighbours on the host before any
// step kernel is enqueued: the in-kernel waits are bounded, so ordinary host-side skew between the ranks (Python work, history
// drains, allocation) must be absorbed here, where nothing has been computed yet.
int Engine::halo_rendezvous(const StepParams &sp, uint64_t &launches) {
    StepParams hp = sp;
    hp.v_in = V_[cur_]; hp.lft_in = LFT_[lft_loc_]; hp.t_in = T_[cur_]; hp.out_par = (uint32_t)cur_;
    hp.halo_epoch = halo_epoch_;
    if (lft_loc_ != cur_) {  // keep lft parity aligned with the V parity on partitioned handles
        cudaMemcpyAsync(LFT_[cur_], LFT_[lft_loc_], node_cap_ * 4, cudaMemcpyDeviceToDevice, stream_);
        lft_loc_ = cur_; hp.lft_in = LFT_[lft_loc_];
    }
    cudaError_t e = gpart_ ? launch_gpart_push(hp, stream_) : launch_halo_push(hp, stream_);
    if (e != cudaSuccess) return cuda_fail(e, SNN_GPU_QUEUE_FAILURE, "halo_push");
    halo_epoch_ += 1;
    launched_pub_.store(halo_epoch_, std::memory_order_release);
    launched_pub2_.store(halo_epoch_, std::memory_order_release);
    launches++;
    e = cudaStreamSynchronize(stream_);
    if (e != cudaSuccess) return cuda_fail(e, SNN_GPU_WAIT_ERROR, "halo_push");
    const auto t_wait0 = std::chrono::steady_clock::now();
    for (;;) {
        unsigned long long f[8 + kMaxRanks];
        e = cudaMemcpy(f, flags_, sizeof f, cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) return cuda_fail(e, SNN_GPU_BUFFER_READ_ERROR, "halo rendez-vous");
        bool ready = true;
        for (int d = 0; d < 2; ++d) if (halo_dir_[d].active && f[d] < halo_epoch_) ready = false;
        for (auto &G : gpeers_) if (f[8 + G.rank] < halo_epoch_) ready = false;
        if (ready) return SNN_OK;
        if (std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_wait0).count() > 4.0 * (double)halo_timeout_ms)
            return fail(SNN_GPU_WAIT_ERROR, "timed out waiting for the neighbouring strips to enter run() (is every rank calling run with the same number of steps?)");
        std::this_thread::sleep_for(std::chrono::microseconds(20));
    }
}

// The clock of every spike-train lattice: lattice l covers trains [tl_base[l], tl_base[l + 1]) and stamps tl_clock[l].
void Engine::fill_train_clocks(TrainParams &tp) const {
    tp.n_tl = 0;
    for (auto &L : lats_)
        if (L.is_train) { tp.tl_base[tp.n_tl] = (uint32_t)L.off; tp.tl_clock[tp.n_tl] = (uint32_t)L.clock; tp.n_tl++; }
    tp.tl_base[tp.n_tl] = (uint32_t)n_trains;
}

// `steps` timesteps in cooperative launches of up to steps_per_graph timesteps each (step_multi.cu).
int Engine::run_multi_chunk(const RunPlan &pl, LaunchArgs &a, const HistStage &hist, uint64_t steps, bool first_chunk) {
    StepParams &sp = a.sp;
    TrainParams &tp = a.tp;
    const bool wide = pl.path == StepPath::Wide;
    for (uint64_t s0 = 0; s0 < steps;) {
        const uint64_t k = steps_per_graph ? std::min<uint64_t>(steps_per_graph, steps - s0) : steps - s0;
        sp.clock = (uint32_t)internal_clock;
        sp.reverse = 0u;
        if (n_trains) {
            fill_train_clocks(tp);
            tp.draw = train_draws;
        }
        MultiParams mp{};
        mp.steps = (uint32_t)k; mp.first_pending = (first_chunk && s0 == 0) ? 0u : 1u;
        mp.cur = (uint32_t)cur_; mp.lft_loc = (uint32_t)lft_loc_; mp.lft_pp = pl.lft_pp ? 1u : 0u;
        mp.train_sync = (pl.spec.stdp && n_trains) ? 1u : 0u;
        for (int q = 0; q < 2; ++q) { mp.v[q] = V_[q]; mp.lft[q] = LFT_[q]; mp.spk[q] = SPK_[q]; mp.t[q] = T_[q]; }
        hist.point(mp, s0);
        mp.n_neurons = n_neurons; mp.n_words = hist.n_words; mp.n_trains = n_trains; mp.t_words = hist.t_words;
        mp.barrier = multi_barrier_;
        mp.cache_rows = !pl.spec.stdp ? 1u : 0u;
        mp.wide_stage = (wide && n_nodes_ <= 4096) ? 1u : 0u;
        cudaError_t e = cudaMemsetAsync(multi_barrier_, 0, sizeof(unsigned int), stream_);
        if (e == cudaSuccess) e = launch_step_multi(sp, tp, mp, pl.spec, wide, device, false, stream_);
        if (e != cudaSuccess) return cuda_fail(e, SNN_GPU_QUEUE_FAILURE, "launch_step_multi");
        a.launches++;
        // the host mirrors what the launch did to the ping-pong state and the clocks
        internal_clock += k;
        if (k & 1ull) { cur_ ^= 1; if (pl.lft_pp) lft_loc_ ^= 1; }
        if (n_trains) { train_draws += k; for (auto &L : lats_) if (L.is_train) L.clock += k; }
        s0 += k;
    }
    return SNN_OK;
}

// Timestep s of the chunk: the step kernel, the per-edge plasticity pass, the spike trains and the graph record, in the order
// the reference applies them.  The host-side launch publications of in-process strips keep this order (wait_local_peers_launched).
int Engine::run_step(const RunPlan &pl, LaunchArgs &a, HistStage &hist, uint64_t s, bool first, const float *reward) {
    StepParams &sp = a.sp;
    TrainParams &tp = a.tp;
    const int in = cur_, out = cur_ ^ 1;
    sp.clock = (uint32_t)internal_clock;
    // window kernel: sweep the tiles back to front every other step (the tail the previous step left in L2 is read first)
    sp.reverse = (internal_clock & 1ull) ? 1u : 0u;
    sp.apply_pending = (pl.spec.stdp && !first) ? 1u : 0u;
    sp.v_in = V_[in]; sp.v_out = V_[out];
    sp.spk_in = SPK_[in]; sp.spk_out = SPK_[out];
    sp.t_in = T_[in]; sp.t_out = T_[out];
    sp.lft_in = LFT_[lft_loc_]; sp.lft_out = LFT_[pl.lft_pp ? lft_loc_ ^ 1 : lft_loc_];
    hist.point(sp, s);
    sp.out_par = (uint32_t)out;
    sp.halo_epoch = halo_epoch_;
    if (!local_peers_.empty()) wait_local_peers_launched(halo_epoch_, pl.rmod_part);
    // spike-train parameters of this timestep (the trains step after the neurons, with their own clocks)
    auto fill_train_step = [&]() {
        tp.v_in = V_[in]; tp.v_out = V_[out]; tp.spk_in = SPK_[in]; tp.spk_out = SPK_[out];
        tp.t_in = T_[in]; tp.t_out = T_[out];
        tp.lft_in = sp.lft_in; tp.lft_out = sp.lft_out;
        fill_train_clocks(tp);
        tp.draw = train_draws++;
        hist.point(tp, s);
    };
    if (pl.trains_fused) fill_train_step();
    if (n_neurons) {
        cudaError_t e = cudaSuccess;
        const char *what = "launch_step";
        switch (pl.path) {
        case StepPath::Win:
            e = launch_step_win(sp, a.win, pl.spec, pl.grid, stream_);
            what = "launch_step_win";
            break;
        case StepPath::Tma:
            a.tma.st[pl.tma_iv].src = (const unsigned char *)(sp.v_in + own0_);
            if (pl.tma_il >= 0) a.tma.st[pl.tma_il].src = (const unsigned char *)(sp.lft_in + own0_);
            for (int ty = 0; ty < kNT; ++ty)
                if (pl.tma_it[ty] >= 0) a.tma.st[pl.tma_it[ty]].src = (const unsigned char *)(sp.t_in + (size_t)ty * node_cap_ + own0_);
            e = launch_step_tma(sp, a.tma, pl.spec, pl.grid, stream_);
            what = "launch_step_tma";
            break;
        case StepPath::Wide:
            e = launch_step_wide(sp, pl.spec, nullptr, 0u, nullptr, stream_);
            break;
        case StepPath::WideSplit:
            e = launch_step_wide(sp, pl.spec, wide_scratch_, pl.wide_chunks_cap, pl.trains_fused ? &tp : nullptr, stream_);
            break;
        case StepPath::General:
            e = launch_step(sp, pl.spec, stream_);
            break;
        }
        if (e != cudaSuccess) return cuda_fail(e, SNN_GPU_QUEUE_FAILURE, what);
        a.launches += pl.path == StepPath::WideSplit ? 2 : 1;   // terms pass + sum pass
    }
    if (reward_mode && reward) {
        // RewardModulatedSTDP::update, plasticity/mod.rs:193-195 (run_lattice_with_reward, neuron/mod.rs:3160-3172)
        rstdp.dopamine = rstdp.dopamine * expf(-rstdp.dt / rstdp.tau_d) + rstdp.tau_d * *reward;
    }
    if (pl.net_reward) {
        // RewardModulatedLatticeNetwork::run_lattices_with_reward (neuron/mod.rs:5280-5297): every reward-modulated lattice's
        // modulator takes the reward before iterate; then post_neuron_update_step's pass over their rows
        int kn = 0;
        for (auto &L : lats_) {
            if (L.is_train) continue;
            if (L.is_reward && reward) L.rstdp.dopamine = L.rstdp.dopamine * expf(-L.rstdp.dt / L.rstdp.tau_d) + L.rstdp.tau_d * *reward;
            a.rnp.lat[kn++].dopamine = L.rstdp.dopamine;
        }
        if (pl.net_rmod) {
            cudaError_t e = launch_rstdp_net_edges(sp, a.rnp, stream_);
            if (e != cudaSuccess) return cuda_fail(e, SNN_GPU_QUEUE_FAILURE, "launch_rstdp_net_edges");
            a.launches++;
        }
    }
    if (pl.bcm_on) {
        StepParams ep = sp;
        if (part_world > 1) {
            // the kernel reads the neighbours' step-s exports: their last_firing_time and current_activity of this step in my
            // ghost slots (see bcm_edge_body for why no second handshake is needed)
            ep.tf[TFB_ACT_GHOST] = ACT_[out];
            await_step_exports(ep);
        }
        cudaError_t e = launch_bcm_edges(ep, BcmParams{bcm.decay, bcm.average_scalar, bcm.dt}, stream_);
        if (e != cudaSuccess) return cuda_fail(e, SNN_GPU_QUEUE_FAILURE, "launch_bcm_edges");
        a.launches++;
    }
    if (pl.rmod) {
        a.rsp.dopamine = rstdp.dopamine;
        StepParams ep = sp;
        if (pl.rmod_part) {
            // the kernel needs the neighbours' step-s exports (their last_firing_time of this step in my ghost slots)
            for (int d = 0; d < 2; ++d) ep.halo[d].my_flag = halo_dir_[d].my_flag;
            await_step_exports(ep);
        }
        cudaError_t e = launch_rstdp_edges(ep, a.rsp, stream_);
        if (pl.rmod_part) launched_pub2_.store(halo_epoch_ + 1, std::memory_order_release);
        if (e != cudaSuccess) return cuda_fail(e, SNN_GPU_QUEUE_FAILURE, "launch_rstdp_edges");
        a.launches++;
    }
    if (part_world > 1) { halo_epoch_ += 1; launched_pub_.store(halo_epoch_, std::memory_order_release); }
    // LatticeNetwork::iterate: clock += 1, then the spike trains step with their own clocks (neuron/mod.rs:2582-2591)
    if (n_trains) {
        if (!pl.trains_fused) {
            fill_train_step();
            cudaError_t e = launch_trains(tp, stream_);
            if (e != cudaSuccess) return cuda_fail(e, SNN_GPU_QUEUE_FAILURE, "launch_trains");
            a.launches++;
        }
        for (auto &L : lats_) if (L.is_train) L.clock += 1;
    }
    if (pl.ghist_on && (is_network || !pl.spec.stdp || sp.apply_pending)) {
        cudaError_t e = hist.record_graph(a.launches);
        if (e != cudaSuccess) return cuda_fail(e, SNN_GPU_QUEUE_FAILURE, "launch_graph_record");
    }
    internal_clock += 1;
    cur_ = out;
    if (pl.lft_pp) lft_loc_ ^= 1;
    return SNN_OK;
}

// The last step's STDP is still pending after the last step kernel: apply it so that weights are final at the API boundary.
int Engine::flush_stdp(const RunPlan &pl, LaunchArgs &a, HistStage &hist) {
    StepParams fp = a.sp;
    fp.clock = (uint32_t)internal_clock;
    fp.lft_in = LFT_[lft_loc_];
    fp.lft_out = LFT_[lft_loc_ ^ 1];  // spike trains: last_firing_time from before their last iterate
    fp.halo_epoch = halo_epoch_;
    if (!local_peers_.empty()) wait_local_peers_launched(halo_epoch_, false);
    cudaError_t e = launch_flush_stdp(fp, stream_);
    if (e != cudaSuccess) return cuda_fail(e, SNN_GPU_QUEUE_FAILURE, "flush_stdp");
    a.launches++;
    if (pl.ghist_on && !is_network) {
        e = hist.record_graph(a.launches);
        if (e != cudaSuccess) return cuda_fail(e, SNN_GPU_QUEUE_FAILURE, "launch_graph_record");
    }
    return SNN_OK;
}

// After the last step: a neighbour's halo time-out, and the derived fields (receptor currents, HH gate rates / channel currents)
// from the retained pre-update V.
int Engine::finish_run(const RunPlan &pl, const StepParams &sp) {
    if (part_world > 1) {
        unsigned int err = 0;
        CK(cudaMemcpy(&err, halo_done_ + 2, 4, cudaMemcpyDeviceToHost), SNN_GPU_BUFFER_READ_ERROR);
        if (err) {
            cudaMemsetAsync(halo_done_, 0, 4 * sizeof(unsigned int), stream_);
            cudaStreamSynchronize(stream_);
            return fail(SNN_GPU_WAIT_ERROR, "timed out waiting for a neighbouring strip's halo (is every rank running the same number of steps?)");
        }
    }
    if (pl.spec.stdp || pl.rmod || pl.net_rmod || pl.bcm_on) dev_weights_newer_ = true;
    if ((chemical && chem_alloc_) || model == SNN_MODEL_HODGKIN_HUXLEY) {
        StepParams fp = sp;
        fp.chemical = chemical && chem_alloc_;
        CK(launch_finalize(fp, model, V_[cur_ ^ 1], stream_), SNN_GPU_QUEUE_FAILURE);
        CK(cudaStreamSynchronize(stream_), SNN_GPU_WAIT_ERROR);
    }
    return SNN_OK;
}

int Engine::run(uint64_t iterations, float *elapsed_ms, uint64_t *launches, const float *rewards) {
    if (elapsed_ms) *elapsed_ms = 0.f;
    if (launches) *launches = 0;
    // gpu_lattices/mod.rs:1089-1091: empty lattice or zero iterations -> Ok(()); neuron/mod.rs:1217: both flags off -> Ok(())
    if (iterations == 0 || (n_neurons == 0 && n_trains == 0)) return SNN_OK;
    if (!electrical && !chemical) return SNN_OK;
    if (internal_clock + iterations > 0x7FFFFFF0ull) return fail(SNN_UNSUPPORTED, "internal clock would overflow the i32 last_firing_time");
    RunPlan pl;
    LaunchArgs a;
    int r = plan_run(pl, a);
    if (r) return r;
    {
        HistStage hist(*this, pl);
        r = hist.init(iterations);
        if (!r && part_world > 1) r = halo_rendezvous(a.sp, a.launches);
        for (uint64_t done = 0; !r && done < iterations;) {
            const uint64_t steps = std::min(hist.chunk, iterations - done);
            cudaEventRecord(ev0_, stream_);
            if (pl.multi) r = run_multi_chunk(pl, a, hist, steps, done == 0);
            for (uint64_t s = 0; !pl.multi && !r && s < steps; ++s)
                r = run_step(pl, a, hist, s, done == 0 && s == 0, rewards ? rewards + done + s : nullptr);
            done += steps;
            if (!r && done == iterations && pl.spec.stdp) r = flush_stdp(pl, a, hist);
            if (r) break;
            cudaEventRecord(ev1_, stream_);
            cudaError_t e = cudaStreamSynchronize(stream_);
            if (e != cudaSuccess) { r = cuda_fail(e, SNN_GPU_WAIT_ERROR, "cudaStreamSynchronize(step loop)"); break; }
            float ms = 0.f;
            cudaEventElapsedTime(&ms, ev0_, ev1_);
            a.total_ms += ms;
            r = hist.drain(steps);
        }
    }   // the history staging buffers are freed here
    if (!r) r = finish_run(pl, a.sp);
    if (r) return r;
    if (elapsed_ms) *elapsed_ms = a.total_ms;
    if (launches) *launches = a.launches;
    return SNN_OK;
}

// ------------------------------------------------------------------------------------------------
// multi-GPU halo plumbing (CUDA IPC; the caller moves the blobs between ranks)
// ------------------------------------------------------------------------------------------------
static constexpr uint32_t kIpcMagic = 0x534E4E42u;   // "SNNB", first word of every IpcBlob

int Engine::ipc_export(IpcBlob *blob) {
    int r = ipc_export_layout(blob);
    if (r) return r;
    CK(cudaSetDevice(device), SNN_GPU_GET_DEVICE_FAILURE);
    CK(cudaIpcGetMemHandle(&blob->slab, slab_), SNN_GPU_BUFFER_CREATE_ERROR);
    CK(cudaIpcGetMemHandle(&blob->flags, flags_), SNN_GPU_BUFFER_CREATE_ERROR);
    layout_frozen_ = true;   // a neighbour will hold pointers into the slab
    return SNN_OK;
}

int Engine::ipc_export_layout(IpcBlob *blob) {
    if (part_world <= 1) return fail(SNN_INVALID_ARGUMENT, "handle is not partitioned");
    memset(blob, 0, sizeof *blob);
    blob->magic = kIpcMagic; blob->version = SNN_B200_ABI_VERSION;
    for (int k = 0; k < 2; ++k) {
        blob->off_v[k] = slab_off_v_[k]; blob->off_lft[k] = slab_off_lft_[k]; blob->off_t[k] = slab_off_t_[k];
        blob->off_act[k] = slab_off_act_[k];
    }
    blob->off_flags = slab_off_flags_;
    blob->t_stride = node_cap_;
    blob->own0 = own0_; blob->n_neurons = (uint32_t)n_neurons; blob->ghost_hi0 = ghost_hi0_; blob->halo = halo_;
    blob->cols = lats_.empty() ? 0 : lats_[0].cols; blob->chem = chem_alloc_;
    blob->rank = part_rank; blob->world = part_world;
    return SNN_OK;
}

// Checks a partition peer's layout against mine, then maps its slab and arrival counters: `local` is a handle of this process
// (addressed directly), else `blob` comes from another process's ipc_export (CUDA IPC).  Nothing is mapped and no peer access
// is enabled unless every check passes.
int Engine::map_peer(const IpcBlob *blob, Engine *local, int expect_rank, PeerMap *out, IpcBlob *view) {
    if (local) {
        if (local == this) return fail(SNN_INVALID_ARGUMENT, "bad peer handle");
        int r = local->ipc_export_layout(view);
        if (r) return fail(r, local->last_error);
    } else {
        *view = *blob;
    }
    if (view->magic != kIpcMagic || view->version != SNN_B200_ABI_VERSION) return fail(SNN_INVALID_ARGUMENT, "bad ipc blob");
    if (view->rank != expect_rank || view->world != part_world) return fail(SNN_INVALID_ARGUMENT, "ipc blob is not from that rank");
    if ((view->chem != 0) != chem_alloc_) return fail(SNN_INVALID_ARGUMENT, "the ranks disagree on chemistry");
    if (!gpart_) {
        if (view->halo != halo_) return fail(SNN_INVALID_ARGUMENT, "neighbouring strips disagree on halo width");
        if (halo_ > n_neurons || halo_ > view->n_neurons) return fail(SNN_UNSUPPORTED, "strip thinner than the halo");
    }
    if ((view->off_act[0] != 0) != (ACT_[0] != nullptr)) return fail(SNN_INVALID_ARGUMENT, "the ranks disagree on the neuron model");
    if (local) {
        if (local->device != device) {
            int can = 0;
            CK(cudaDeviceCanAccessPeer(&can, device, local->device), SNN_GPU_GET_DEVICE_FAILURE);
            if (!can) return fail(SNN_UNSUPPORTED, "no peer access between the two devices");
            cudaError_t e = cudaDeviceEnablePeerAccess(local->device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return cuda_fail(e, SNN_GPU_GET_DEVICE_FAILURE, "cudaDeviceEnablePeerAccess");
            cudaGetLastError();
        }
        *out = PeerMap{local->slab_, local->flags_, false};
        return SNN_OK;
    }
    void *slab = nullptr, *flags = nullptr;
    CK(cudaIpcOpenMemHandle(&slab, view->slab, cudaIpcMemLazyEnablePeerAccess), SNN_GPU_BUFFER_CREATE_ERROR);
    cudaError_t e = cudaIpcOpenMemHandle(&flags, view->flags, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
        cudaIpcCloseMemHandle(slab);
        return cuda_fail(e, SNN_GPU_BUFFER_CREATE_ERROR, "cudaIpcOpenMemHandle(flags)");
    }
    *out = PeerMap{slab, flags, true};
    return SNN_OK;
}

// Ghost nodes node0, node0 + 1, ... take the neurotransmitter / receptor type flags of the peer's neurons they mirror (the flags
// are baked into the col words of edges from ghosts): ghost node0 + k takes byte pick[k] of the `bytes` peer flag bytes at
// `peer_flags`.  `force` re-encodes the graph even when no flag changes.
int Engine::import_ghost_flags(uint32_t node0, const uint8_t *peer_flags, uint64_t bytes, const std::vector<uint32_t> &pick, bool force) {
    std::vector<uint8_t> pf(bytes);
    CK(cudaMemcpy(pf.data(), peer_flags, bytes, cudaMemcpyDefault), SNN_GPU_BUFFER_READ_ERROR);
    bool changed = force;
    for (size_t k = 0; k < pick.size(); ++k) {
        changed |= h_node_flags_[node0 + k] != pf[pick[k]];
        h_node_flags_[node0 + k] = pf[pick[k]];
    }
    if (!changed) return SNN_OK;
    CK(h2d_sync(node_flags_ + node0, h_node_flags_.data() + node0, pick.size(), stream_), SNN_GPU_BUFFER_WRITE_ERROR);
    flags_cache_valid_ = false;
    if (dev_weights_newer_) { int r = sync_weights_to_host(); if (r) return r; }
    graph_dirty_ = true;
    return SNN_OK;
}

// The neighbouring strip lives in another process (`blob`) or in this one (`local`: another handle on the same device, or on a
// device with peer access).  Both handles must attach each other.  On one device the caller steps in-process strips from separate
// host threads and keeps the strips small enough for their step kernels to be resident together (a strip's boundary warps spin on
// the neighbour's progress).
int Engine::attach_strip(int direction, const IpcBlob *blob, Engine *local) {
    if (part_world <= 1) return fail(SNN_INVALID_ARGUMENT, "handle is not partitioned");
    if (direction != -1 && direction != 1) return fail(SNN_INVALID_ARGUMENT, "direction must be -1 or +1");
    if (gpart_) return fail(SNN_INVALID_ARGUMENT, "a general-graph partition attaches its peers with gpart_attach");
    CK(cudaSetDevice(device), SNN_GPU_GET_DEVICE_FAILURE);
    const int d = direction < 0 ? 0 : 1;
    if (halo_dir_[d].active) return fail(SNN_INVALID_ARGUMENT, "direction already attached");
    PeerMap m;
    IpcBlob v;
    int r = map_peer(blob, local, part_rank + direction, &m, &v);
    if (r) return r;
    HaloDir H;
    memset(&H, 0, sizeof H);
    H.count = halo_;
    // d == 0: my first `halo` neurons go to the upper ghost slots of rank-1; d == 1: my last `halo` neurons go to
    // the lower ghost slots of rank+1
    H.first = d == 0 ? 0 : (uint32_t)n_neurons - halo_;
    H.peer_node0 = d == 0 ? v.ghost_hi0 : v.own0 - v.halo;
    H.my_ghost0 = d == 0 ? own0_ - halo_ : ghost_hi0_;
    for (int k = 0; k < 2; ++k) {
        H.peer_v[k] = (float *)((char *)m.slab + v.off_v[k]);
        H.peer_lft[k] = (int *)((char *)m.slab + v.off_lft[k]);
        H.peer_t[k] = (float *)((char *)m.slab + v.off_t[k]);
    }
    H.peer_t_stride = v.t_stride;
    // the neighbour's arrival counter for data coming from me: I am its rank+1 when d == 0 (slot 1), its rank-1 when d == 1 (slot 0)
    H.peer_flag = (unsigned long long *)m.flags + (d == 0 ? 1 : 0);
    H.my_flag = flags_ + d;
    H.peer_flag2 = H.peer_flag + 2;
    H.my_flag2 = H.my_flag + 2;
    H.active = 1;
    // my ghost rows mirror the neighbour's boundary rows: d == 0 the LAST halo_ neurons of rank - 1, d == 1 the FIRST halo_ of rank + 1
    std::vector<uint32_t> pick(halo_);
    std::iota(pick.begin(), pick.end(), 0u);
    r = import_ghost_flags(H.my_ghost0, (const uint8_t *)m.slab + v.off_flags + (d == 0 ? v.own0 + v.n_neurons - halo_ : v.own0), halo_,
                           pick, !ghost_flags_from_peer_[d]);
    if (r) { unmap_peer(m); return r; }
    ghost_flags_from_peer_[d] = true;
    halo_dir_[d] = H;
    for (int k = 0; k < 2; ++k) halo_act_[d][k] = ACT_[0] ? (float *)((char *)m.slab + v.off_act[k]) : nullptr;
    strip_map_[d] = m;
    layout_frozen_ = true;
    if (local) { local->layout_frozen_ = true; local_peers_.push_back(local); }
    return SNN_OK;
}

}  // namespace snn
