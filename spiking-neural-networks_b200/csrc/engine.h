// engine.h — host-side runtime of the lattice stepping engine (one CUDA device, one stream).
//
// An Engine is the device-resident twin of a reference `LatticeNetwork` (neuron/mod.rs:1538-1564):
// neuron lattices in ascending id order, then spike-train lattices, one canonical node index space,
// one in-edge table.  A reference `Lattice` is an Engine with a single lattice.
#pragma once
#include <atomic>
#include <cstdint>
#include <functional>
#include <map>
#include <string>
#include <utility>
#include <vector>

#include "common.h"
#include "fields.h"

namespace snn {

struct Lat {
    uint64_t id = 0;
    uint32_t rows = 0, cols = 0;
    uint64_t n = 0;
    bool is_train = false;
    uint64_t off = 0;  // offset inside its domain (local neuron number / local train number)
    bool do_plasticity = false, grid_hist = false, spike_hist = false;
    bool avg_hist = false, eeg_hist = false;        // AverageVoltageHistory / EEGHistory (neuron/mod.rs:231-322)
    bool graph_hist = false;                        // update_graph_history: records of this lattice's own graph (graph/mod.rs:278-284)
    bool spike_events = false;                      // SNN_OPT_UPDATE_SPIKE_EVENTS: compacted (step, cell) spike lists
    float eeg_ref = 0.007f, eeg_dist = 0.8f, eeg_cond = 251.f;   // EEGHistory::default, neuron/mod.rs:243-252
    std::vector<float> average_history, eeg_history;
    snn_stdp_t stdp{2.f, 2.f, 4.5f, 4.5f, 0.1f};  // STDP::default, plasticity/mod.rs:29-39
    // a member of RewardModulatedLatticeNetwork::reward_modulated_lattices (neuron/mod.rs:3470-3471): TraceRSTDP weights in its own
    // graph, a RewardModulatedSTDP modulator (RewardModulatedLattice::default, neuron/mod.rs:2760-2777)
    bool is_reward = false, do_modulation = true;
    snn_rstdp_t rstdp{0.f, 20.f, 0.0001f, 2.f, 2.f, 4.5f, 4.5f, 0.1f};
    uint64_t clock = 0;                           // SpikeTrainLattice::internal_clock
    std::vector<float> cold[2];                   // v_init, w_init
    std::vector<float> grid_history;
    std::vector<uint8_t> spike_history;
    std::vector<int64_t> spike_agg;                // SpikeHistory::aggregate, accumulated from device-side counts
    uint64_t hist_len = 0;
    // spike events: record k's cells are ev_neuron[ev_ptr[k] .. ev_ptr[k + 1]) (ev_ptr is empty before the first record)
    std::vector<uint64_t> ev_ptr;
    std::vector<uint32_t> ev_neuron;
    std::vector<uint64_t> ft_off;                 // preset firing times (CSR) of a train lattice
    std::vector<float> ft;
};

struct Block {  // connections pre lattice -> post lattice, CSR by post (pre ascending), or a grid stencil
    enum Kind { CSR, GRID } kind = CSR;
    std::vector<uint64_t> row_ptr;
    std::vector<uint32_t> pre;
    std::vector<float> w;
    uint32_t radius = 0;
    float weight = 1.f;
    // a materialised stencil (kind == CSR, adjacency still that of set_graph_grid(radius)): finalize_graph keeps the uniform-width
    // layout and with it the window / TMA step kernels; cleared when an edge is added or removed
    uint32_t from_grid_radius = 0;
    // connecting block of a RewardModulatedLatticeNetwork whose values are RewardModulatedWeight(TraceRSTDP) rather than Weight(f32)
    bool reward_conn = false;
};

struct IpcBlob {  // exchanged between neighbouring ranks by the caller (e.g. torch.distributed all_gather)
    uint32_t magic, version;
    cudaIpcMemHandle_t slab, flags;
    uint64_t off_v[2], off_lft[2], off_t[2], off_flags;
    uint64_t off_act[2];   // current_activity ping-pong of a BCM Izhikevich strip; 0 = the slab has none
    uint64_t t_stride;
    uint32_t own0, n_neurons, ghost_hi0, halo, cols, chem;
    int32_t rank, world;
};

struct PeerMap {  // a partition peer's slab and arrival counters as this process addresses them
    void *slab = nullptr, *flags = nullptr;
    bool ipc = false;   // opened from CUDA IPC handles (closed by the engine), else the pointers of a handle of this process
};

class Engine {
public:
    Engine(int model, int ntk, int rck, int train_kind, int refract, int device);
    ~Engine();
    int init();  // device selection + stream; returns snn_status

    // topology
    int add_lattice(uint64_t id, uint32_t rows, uint32_t cols, bool is_train, bool is_reward = false);
    int set_partition(uint32_t rows_global, uint32_t cols, int rank, int world);  // before add_lattice
    Lat *find(uint64_t id);
    const Lat *find(uint64_t id) const;

    // fields
    int field_count(uint64_t id, uint32_t *count) const;
    int field_info(uint64_t id, uint32_t index, const char **name, int32_t *dtype, uint32_t *per) const;
    int set_field(uint64_t id, const char *name, const void *data, uint64_t count, int dtype);
    int get_field(uint64_t id, const char *name, void *out, uint64_t count, int dtype);
    int fill_field(uint64_t id, const char *name, uint32_t bits, int dtype);
    int set_preset_firing_times(uint64_t id, const uint64_t *offsets, const float *times, uint64_t n_trains, uint64_t n_times);

    // graph
    int connect_dense(uint64_t pre_id, uint64_t post_id, const uint32_t *connections, const float *weights,
                      const uint32_t *index_to_position, uint64_t n_pre, uint64_t n_post);
    int connect_csr(uint64_t pre_id, uint64_t post_id, const uint64_t *row_ptr, const uint32_t *pre, const float *weights,
                    uint64_t n_post, uint64_t nnz);
    int connect_grid(uint64_t id, uint32_t radius, float weight);
    int connection_nnz(uint64_t pre_id, uint64_t post_id, uint64_t *nnz);
    int get_connection_csr(uint64_t pre_id, uint64_t post_id, uint64_t *row_ptr, uint32_t *pre, float *weights,
                           uint64_t n_post, uint64_t nnz);
    int get_connection_dense(uint64_t pre_id, uint64_t post_id, uint32_t *connections, float *weights, uint64_t n_pre,
                             uint64_t n_post);
    // CSR of the postsynaptic rows [row_begin, row_end) of the pre -> post block, decoded from the device table (no whole-graph
    // download): Graph::get_incoming_connections over a range of positions (graph/mod.rs:228-256)
    int get_connection_rows(uint64_t pre_id, uint64_t post_id, uint64_t row_begin, uint64_t row_end, uint64_t *row_ptr, uint32_t *pre,
                            float *weights, uint64_t capacity, uint64_t *nnz);
    // Graph::lookup_weight / edit_weight on flat indices (graph/mod.rs:196-226)
    int lookup_weight(uint64_t pre_id, uint64_t post_id, uint64_t pre, uint64_t post, float *weight, int32_t *connected);
    int edit_weight(uint64_t pre_id, uint64_t post_id, uint64_t pre, uint64_t post, bool has, float weight);

    // options
    int set_dt(float dt);
    int reset_timing();
    int reset_history();

    // run
    int run(uint64_t iterations, float *elapsed_ms, uint64_t *launches, const float *rewards = nullptr);

    // RewardModulatedLattice (neuron/mod.rs:2717-3416)
    int set_reward_modulator(bool enable, bool modulate, const snn_rstdp_t *m);
    int set_bcm_plasticity(bool enable, const snn_bcm_t *b);
    bool bcm_mode = false;
    snn_bcm_t bcm{0.1f, 0.1f, 0.1f};   // BCM::default, plasticity/mod.rs:91-97
    int set_lattice_reward_modulator(uint64_t id, bool modulate, const snn_rstdp_t *m);
    int get_lattice_reward_modulator(uint64_t id, int32_t *modulate, snn_rstdp_t *m);
    int set_connection_reward(uint64_t pre_id, uint64_t post_id, bool reward_modulated);
    bool has_reward_lattices() const;
    int block_elements(uint64_t pre_id, uint64_t post_id, std::vector<size_t> *elems, Block **blk);
    int get_block_traces(uint64_t pre_id, uint64_t post_id, uint32_t *counter, float *dw, float *c, uint64_t nnz);
    int set_block_traces(uint64_t pre_id, uint64_t post_id, const float *weight, const uint32_t *counter, const float *dw, const float *c, uint64_t nnz);
    int get_connection_traces(uint32_t *counter, float *dw, float *c, uint64_t nnz);
    int set_connection_traces(const float *weight, const uint32_t *counter, const float *dw, const float *c, uint64_t nnz);
    bool reward_mode = false, do_modulation = true;
    snn_rstdp_t rstdp{0.f, 20.f, 0.0001f, 2.f, 2.f, 4.5f, 4.5f, 0.1f};   // RewardModulatedSTDP::default, plasticity/mod.rs:176-189

    // histories
    int history_len(uint64_t id, uint64_t *steps) const;
    int get_grid_history(uint64_t id, float *out, uint64_t capacity);
    int get_spike_history(uint64_t id, uint8_t *out, uint64_t capacity);
    int get_spike_aggregate(uint64_t id, int64_t *out, uint64_t capacity);   // SpikeHistory::aggregate, neuron/mod.rs:335-359
    int get_reduced_history(uint64_t id, bool eeg, float *out, uint64_t capacity);
    int set_eeg_parameters(uint64_t id, float reference_voltage, float distance, float conductivity);
    // graph history: one record per timestep of the block pre_id -> post_id (pre_id == post_id: a lattice's own graph), nnz f32
    // weights in the order of get_connection_csr
    int graph_history_len(uint64_t pre_id, uint64_t post_id, uint64_t *steps, uint64_t *nnz);
    int get_graph_history(uint64_t pre_id, uint64_t post_id, float *out, uint64_t capacity);
    bool graph_history_nonempty() const;
    // spike events of one lattice: `steps` records (CSR by step, step_ptr has steps + 1 entries) of `n_events` cell indices
    int spike_event_count(uint64_t id, uint64_t *steps, uint64_t *n_events) const;
    int get_spike_events(uint64_t id, uint64_t *step_ptr, uint32_t *neuron, uint64_t capacity);

    // multi-GPU
    int ipc_export(IpcBlob *blob);
    // the attach calls take either the `blob` of another process's ipc_export (CUDA IPC) or a `local` handle of this process
    int attach_strip(int direction, const IpcBlob *blob, Engine *local);   // row strips: direction -1 = rank-1, +1 = rank+1
    // general-graph partition (contiguous node ranges, in-edges from anywhere): which of `peer`'s nodes this rank reads, which of
    // its own nodes `peer` reads, and the mapping of the peer's arrays
    int gpart_wants(int peer, uint32_t *global_idx, uint64_t capacity, uint64_t *n, uint32_t *first_slot);
    int gpart_set_exports(int peer, const uint32_t *global_idx, uint64_t n, uint32_t first_slot_at_peer);
    int gpart_attach(int peer, const IpcBlob *blob, Engine *local);
    bool is_gpart() const { return gpart_; }

    // public knobs (Lattice / LatticeNetwork pub fields, neuron/mod.rs:556-587, 1554-1563)
    bool electrical = true, chemical = false, parallel = false;
    // a LatticeNetwork handle (snn_network_create) rather than a Lattice: the two take their graph history records at different
    // points of the step (Lattice::iterate after the step's plasticity, LatticeNetwork::iterate before it)
    bool is_network = false;
    bool conn_graph_hist = false;   // LatticeNetwork::update_connecting_graph_history: records of every connecting block
    uint64_t internal_clock = 0;
    uint64_t seed;                  // Philox key of the Poisson trains: distinct per handle unless SNN_OPT_RNG_SEED sets it
    uint64_t train_draws = 0;       // Philox counter word: one per spike-train step of this handle, never reset (reset_timing
                                    // restarts the clocks, not the random stream: the reference draws from thread_rng)
    uint32_t steps_per_graph = 0;
    uint32_t last_step_path = 0;        // SNN_OPT_STEP_PATH: step path of the last run, path + 16 * multi (0: nothing run yet)
    uint32_t last_uniform_tiles = 0;    // SNN_OPT_UNIFORM_TILES: window-kernel tiles of the last run that read their parameter row
    uint32_t last_stencil_tiles = 0;    // SNN_OPT_STENCIL_TILES: window-kernel tiles of the last run that took their in-edge
                                        // indices from the stencil instead of the col table
    bool force_gpart = false;           // SNN_OPT_GENERAL_PARTITION: CSR graphs of a partitioned handle always use gather-list ghosts
    uint64_t halo_timeout_ms = 30000;   // multi-GPU: how long a step may wait for a neighbouring strip before SNN_GPU_WAIT_ERROR
    std::string last_error;

    int model, ntk, rck, train_kind, refract, device;
    uint64_t n_neurons = 0, n_trains = 0;
    // partition
    int part_rank = 0, part_world = 1;
    uint32_t rows_global = 0, row0_global = 0;

    int fail(int status, const std::string &msg) { last_error = msg; return status; }

private:
    // layout
    std::vector<Lat> lats_;
    uint32_t own0_ = 0, train0_ = 0, ghost_hi0_ = 0, n_nodes_ = 0, halo_ = 0;
    uint64_t node_cap_ = 0, neuron_cap_ = 0, train_cap_ = 0;
    // device arrays
    cudaStream_t stream_ = nullptr;
    cudaEvent_t ev0_ = nullptr, ev1_ = nullptr;
    void *slab_ = nullptr; size_t slab_bytes_ = 0;
    float *V_[2] = {nullptr, nullptr};
    int *LFT_[2] = {nullptr, nullptr};
    float *T_[2] = {nullptr, nullptr};
    uint64_t slab_off_v_[2] = {0, 0}, slab_off_lft_[2] = {0, 0}, slab_off_t_[2] = {0, 0}, slab_off_flags_ = 0;
    // BCM Izhikevich partitions only: node-indexed current_activity ping-pong, of which the ghost slots are filled by the
    // neighbours (the partitioned BCM edge kernel reads a ghost's activity there)
    float *ACT_[2] = {nullptr, nullptr};
    uint64_t slab_off_act_[2] = {0, 0};
    float *halo_act_[2][2] = {};   // the neighbours' buffers, [direction][parity] (BcmSlot TFB_HALO_ACT)
    bool ghost_flags_from_peer_[2] = {false, false};
    uint32_t *SPK_[2] = {nullptr, nullptr};
    uint8_t *node_flags_ = nullptr;
    std::vector<uint8_t> h_node_flags_;
    float *NT_[NTF_COUNT] = {};
    float *F_[F_COUNT] = {};
    uint32_t *was_inc_ = nullptr;
    float *RC_[RCF_COUNT] = {};
    float *TF_[TF_COUNT] = {};
    uint64_t *ft_off_ = nullptr; float *ft_ = nullptr;
    LatInfo *d_lat_ = nullptr;
    bool chem_alloc_ = false;
    int cur_ = 0;       // parity holding the current V / T / SPK state
    int lft_loc_ = 0;   // buffer holding the current last_firing_time
    bool derived_stale_ = false;
    // graph
    std::map<std::pair<uint64_t, uint64_t>, Block> blocks_;
    bool graph_dirty_ = true;
    bool dev_weights_newer_ = false;
    bool grid_fast_ = false;
    uint32_t *slice_off_ = nullptr, *col_ = nullptr; float *wgt_ = nullptr;
    // TraceRSTDP members next to wgt_ (same sliced-ELL positions), allocated on the first reward-modulated run
    uint8_t *rs_counter_ = nullptr; float *rs_dw_ = nullptr, *rs_c_ = nullptr; uint64_t rs_elems_ = 0;
    // difference tables of the STDP term (RstdpParams::tab of a reward-modulated lattice, RnetParams::tab of a network)
    float *stdp_tab_ = nullptr; size_t stdp_tab_elems_ = 0;
    int build_stdp_tables(const std::vector<RstdpParams> &lat, const float **tab, uint32_t *tab_n);
    int build_rnet_params(RnetParams &rnp, bool *net_rmod);
    bool rs_canonical_ = true;   // counter == 0 and dw == 0 on every edge (TraceRSTDP::default, kept by two calls per timestep)
    int ensure_reward_arrays();
    void free_reward_arrays();
    uint64_t sell_krows_ = 0, sell_alloc_krows_ = 0; uint32_t n_slices_ = 0, uniform_width_ = 0;
    uint32_t max_slice_width_ = 0;   // widest slice of the table, in k-rows
    // halo
    unsigned long long *flags_ = nullptr;  // [0] arrivals from rank-1, [1] arrivals from rank+1
    unsigned int *halo_done_ = nullptr;
    unsigned char *wide_scratch_ = nullptr; size_t wide_scratch_bytes_ = 0;   // parked per-edge terms of the two-pass wide kernels
    unsigned int *multi_barrier_ = nullptr;   // grid-wide arrival counter of the multi-step kernel
    HaloDir halo_dir_[2] = {};
    PeerMap strip_map_[2] = {};
    unsigned long long halo_epoch_ = 0;
    // general-graph partition
    struct GPeerHost {
        int rank = -1;
        std::vector<uint32_t> exp_local;   // my local neuron numbers this peer reads (ascending)
        uint32_t peer_slot0 = 0;           // node index in the peer's arrays where they go
        PeerMap map;
        bool attached = false;
        IpcBlob view{};
    };
    bool gpart_ = false, gpart_dirty_ = true;
    std::vector<uint32_t> g_lo_, g_hi_;    // global indices of the ghost nodes below / above my node range (ascending)
    std::vector<GPeerHost> gpeers_;        // ascending rank
    std::vector<uint8_t> h_gslice_;        // per slice: bit 0 = a row of the slice reads a ghost
    GPeer *d_gpeers_ = nullptr; uint32_t *d_gexp_off_ = nullptr, *d_gexp_ent_ = nullptr; uint8_t *d_gslice_ = nullptr;
    float **d_gact_ = nullptr;             // BCM Izhikevich: the peers' activity buffers (BcmSlot TFB_GPEER_ACT), else null
    GPeerHost *gpeer(int rank, bool create);
    int check_peer_rank(int peer);
    int gpart_build_device();
    int gpart_enable(const std::vector<uint32_t> &remote_sorted_unique);
    int64_t global_to_node(uint64_t g) const;
    uint64_t node_to_global(uint32_t node) const;
    // scratch
    void *scratch_ = nullptr; size_t scratch_bytes_ = 0;
    // graph history: host records per requested block, and the per-row offsets of the canonical CSR order of the device table
    // (32 * n_slices_ + 1 entries, rebuilt after each finalize_graph while some graph history is on)
    struct GraphHist { uint64_t steps = 0, nnz = 0; std::vector<float> w; };
    std::map<std::pair<uint64_t, uint64_t>, GraphHist> graph_hist_;
    uint32_t *ghist_row_off_ = nullptr;
    uint64_t ghist_nnz_ = 0;
    bool ghist_off_valid_ = false;
    int refuse_if_graph_history(const char *what);
    // spike events: pinned bounce buffer of the device-to-host copies (allocated by the first run that records events)
    void *ev_bounce_ = nullptr;

    int ipc_export_layout(IpcBlob *blob);
    int map_peer(const IpcBlob *blob, Engine *local, int expect_rank, PeerMap *out, IpcBlob *view);
    int import_ghost_flags(uint32_t node0, const uint8_t *peer_flags, uint64_t bytes, const std::vector<uint32_t> &pick, bool force);
    bool layout_frozen_ = false;   // pointers into or out of my slab exist: its layout must not change
    // in-process neighbours: host-side launch ordering (see wait_local_peers_launched)
    std::vector<Engine *> local_peers_;
    std::atomic<unsigned long long> launched_pub_{0}, launched_pub2_{0};
    void wait_local_peers_launched(unsigned long long need, bool second);
    void await_step_exports(StepParams &ep);
    int cuda_fail(cudaError_t e, int status, const char *what);
    int ensure_scratch(size_t bytes);
    void free_device();
    int alloc_device();
    int ensure_chem();
    int relayout(const std::function<void()> &change);
    void compute_layout();
    uint32_t node_off(const Lat &L) const { return (L.is_train ? train0_ : own0_) + (uint32_t)L.off; }
    int n_neuron_lattices() const { int n = 0; for (auto &L : lats_) n += !L.is_train; return n; }
    template <class F> void for_each_field(const Lat &L, F &&f) const;
    int lookup_field(const Lat &L, const char *name, FieldDef *out) const;
    int field_io(Lat &L, const FieldDef &fd, void *data, uint64_t count, bool set);
    int set_bits(uint32_t *words, const uint32_t *host_u32, uint64_t n, uint64_t bit0);
    int get_bits(const uint32_t *words, uint32_t *host_u32, uint64_t n, uint64_t bit0);
    template <class F> void for_each_row_segment(F &&f, const Lat *into = nullptr);
    int alloc_table(uint32_t width);
    int finalize_graph();
    int sync_weights_to_host();
    // element index of edge (pre node j -> neuron row) in the sliced-ELL arrays, or -1; the graph must be finalized
    int find_edge(uint64_t row, uint32_t j, int64_t *elem);
    int check_edge_endpoints(uint64_t pre_id, uint64_t post_id, uint64_t pre, uint64_t post, Lat **A, Lat **B);
    void materialize_grid(Block &b, const Lat &L) const;
    Block &csr_view(Block &b, const Lat &L, Block &tmp) const;
    uint32_t nt_used() const; uint32_t rc_used() const;
    void refresh_flag_cache() const;
    mutable bool flags_cache_valid_ = false;
    mutable uint32_t nt_used_ = 0, rc_used_ = 0;
    void fill_step_params(StepParams &p);
    void fill_train_clocks(TrainParams &tp) const;
    int upload_lat_table();
    // mode (SNN_B200_TMA): 0 not eligible, 1 lattices of at least 64 Ki neurons, 2 any size
    bool build_tma_params(TmaParams &tp, bool ntrel, bool stdp, bool lft_pp, int mode, unsigned *grid);
    // *eligible = false: the window kernel does not take this configuration (the status is that of the tile-row build)
    int build_win_params(WinParams &wp, int chemg, bool ntrel, bool stdp, bool lft_pp, int mode, unsigned *grid, bool *eligible);
    // window kernel: the tile rows (TileParSrc) and the numbers of tiles among them that are not uniform / not stencil tiles.
    // Rebuilt when a parameter array was written or moved, or the col table rewritten, since (tile_par_dirty_), or when a run
    // reads another set of arrays.
    uint32_t *tile_par_ = nullptr; size_t tile_par_bytes_ = 0;
    bool tile_par_dirty_ = true;
    TileParSrc tile_par_key_{};
    uint32_t tile_par_counts_[2] = {0, 0};
    int refresh_tile_params(const TileParSrc &a);

    // run(), phase by phase (engine.cu)
    struct RunPlan;      // decisions fixed for the whole run
    struct LaunchArgs;   // kernel parameter blocks and launch count
    struct HistStage;    // device staging of the recorded histories
    int plan_run(RunPlan &pl, LaunchArgs &a);
    int plan_step_path(RunPlan &pl, LaunchArgs &a);
    int halo_rendezvous(const StepParams &sp, uint64_t &launches);
    int run_multi_chunk(const RunPlan &pl, LaunchArgs &a, const HistStage &hist, uint64_t steps, bool first_chunk);
    int run_step(const RunPlan &pl, LaunchArgs &a, HistStage &hist, uint64_t s, bool first, const float *reward);
    int flush_stdp(const RunPlan &pl, LaunchArgs &a, HistStage &hist);
    int finish_run(const RunPlan &pl, const StepParams &sp);
};

}  // namespace snn
