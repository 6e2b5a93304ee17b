// snn_b200.hpp — C++17 host-side mirror of the reference's lattice API, header-only, ABOVE the C ABI (snn_b200.h).
//
// The reference's host language is Rust; this image has no Rust toolchain, so the host side that a Rust caller would see
// (`Lattice`, `SpikeTrainLattice`, `LatticeNetwork`, `RewardModulatedLattice`, `STDP`, `BCM`, `RewardModulatedSTDP`,
// `RunLattice::run_lattice`, `RunNetwork::run_lattices`; backend/src/neuron/mod.rs:556-1220, 1290-1428, 1538-2675, 2717-3416;
// plasticity/mod.rs) is mirrored here in C++ with the same names, argument meaning and error behaviour
// (`SpikingNeuralNetworksError` carries the reference's error variant as a status code, error/mod.rs).  Everything below is
// plumbing around `extern "C"` calls: no compute, no CPU fallback.  INTEGRATION.md shows the Rust binding of the same calls.
#pragma once
#include <cstdint>
#include <functional>
#include <map>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "snn_b200.h"

namespace snn_b200 {

using Position = std::pair<std::size_t, std::size_t>;   // (row, column), the reference's graph key (usize, usize)

// error/mod.rs:221-238 (GPUError), graph/mod.rs GraphError, LatticeNetworkError: one exception type, the variant in `status`
struct SpikingNeuralNetworksError : std::runtime_error {
    int status;
    SpikingNeuralNetworksError(int s, const std::string &what) : std::runtime_error(what), status(s) {}
};

struct STDP { float a_plus = 2.f, a_minus = 2.f, tau_plus = 4.5f, tau_minus = 4.5f, dt = 0.1f; };               // plasticity/mod.rs:14-39
struct BCM { float decay = 0.1f, average_scalar = 0.1f, dt = 0.1f; };                                          // :80-97
struct RewardModulatedSTDP {                                                                                     // :155-189
    float dopamine = 0.f, tau_d = 20.f, tau_c = 0.0001f, a_plus = 2.f, a_minus = 2.f, tau_plus = 4.5f, tau_minus = 4.5f, dt = 0.1f;
};

// `IzhikevichNeuron { gap_conductance: 10., ..Default::default() }`: a model plus the fields that differ from its Default
struct BaseNeuron {
    snn_model_t model = SNN_MODEL_IZHIKEVICH;
    snn_nt_kinetics_t neurotransmitter_kinetics = SNN_NT_APPROXIMATE;
    snn_receptor_kinetics_t receptor_kinetics = SNN_RC_APPROXIMATE;
    std::map<std::string, float> fields;   // e.g. {"gap_conductance", 10.f}
    BaseNeuron() = default;
    explicit BaseNeuron(snn_model_t m) : model(m) {}
    BaseNeuron &with(const std::string &name, float value) { fields[name] = value; return *this; }
};

namespace detail {
inline void check(int status, const char *last_error) {
    if (status == SNN_OK) return;
    std::string text = (last_error && *last_error) ? last_error : snn_status_string(status);
    throw SpikingNeuralNetworksError(status, text);
}
// connect(&|x, y| cond, Some(&|x, y| weight)) evaluated into CSR by postsynaptic cell (neuron/mod.rs:1134-1157): O(n_pre * n_post)
// predicate calls like the reference, without its dense 8 B * N^2 matrix
struct Csr { std::vector<uint64_t> row_ptr; std::vector<uint32_t> pre; std::vector<float> w; };
inline Csr evaluate(std::size_t pre_rows, std::size_t pre_cols, std::size_t post_rows, std::size_t post_cols,
                    const std::function<bool(Position, Position)> &cond, const std::function<float(Position, Position)> &weight) {
    Csr g;
    g.row_ptr.assign(post_rows * post_cols + 1, 0);
    for (std::size_t q = 0; q < post_rows * post_cols; ++q) {
        const Position y{q / post_cols, q % post_cols};
        for (std::size_t p = 0; p < pre_rows * pre_cols; ++p) {
            const Position x{p / pre_cols, p % pre_cols};
            if (cond(x, y)) { g.pre.push_back((uint32_t)p); g.w.push_back(weight ? weight(x, y) : 1.f); }
        }
        g.row_ptr[q + 1] = g.pre.size();
    }
    if (g.pre.empty()) { g.pre.push_back(0); g.w.push_back(0.f); }   // keep data() non-null for nnz == 0
    return g;
}
}  // namespace detail

// Graph::update_history records (graph/mod.rs:278-284): `steps` records of `nnz` weights, each in the edge order of the graph's CSR
// (snn_lattice_get_graph_csr / snn_network_get_connection_csr), record k at weights[k * nnz]
struct GraphHistory {
    std::size_t steps = 0, nnz = 0;
    std::vector<float> weights;
};

// Spike events (SNN_OPT_UPDATE_SPIKE_EVENTS): record k holds the flat cell indices that spiked in the k-th recorded step, ascending,
// in neurons[step_ptr[k] .. step_ptr[k + 1])
struct SpikeEvents {
    std::vector<uint64_t> step_ptr{0};
    std::vector<uint32_t> neurons;
    std::size_t steps() const { return step_ptr.size() - 1; }
};

// ----------------------------------------------------------------------------------------------------------------------------
// Lattice<T, AdjacencyMatrix, GridVoltageHistory, STDP, N>  (neuron/mod.rs:556-1220) on one B200
// ----------------------------------------------------------------------------------------------------------------------------
class Lattice {
public:
    // public fields of the reference struct (neuron/mod.rs:556-587)
    bool electrical_synapse = true, chemical_synapse = false, do_plasticity = false;
    bool update_grid_history = false, update_spike_history = false, parallel = false;
    bool update_graph_history = false;   // records after each step's plasticity (Lattice::iterate, neuron/mod.rs:973-979)
    bool update_spike_events = false;    // compacted spike lists next to (or instead of) the dense raster
    STDP plasticity;

    Lattice() = default;
    Lattice(const Lattice &) = delete;
    Lattice &operator=(const Lattice &) = delete;
    virtual ~Lattice() { if (h_) snn_lattice_destroy(h_); }

    // populate(&base_neuron, num_rows, num_cols), neuron/mod.rs:1105-1126: drops previous neurons and connections
    void populate(const BaseNeuron &base, std::size_t num_rows, std::size_t num_cols) {
        if (h_) { snn_lattice_destroy(h_); h_ = nullptr; }
        snn_lattice_desc_t d{};
        d.struct_size = sizeof d; d.model = base.model; d.nt_kinetics = base.neurotransmitter_kinetics;
        d.receptor_kinetics = base.receptor_kinetics; d.rows = (uint32_t)num_rows; d.cols = (uint32_t)num_cols;
        d.device = -1; d.part_rank = 0; d.part_world = 1;
        detail::check(snn_lattice_create(&d, &h_), snn_lattice_last_error(nullptr));
        rows_ = num_rows; cols_ = num_cols;
        for (auto &kv : base.fields) ck(snn_lattice_fill_field_f32(h_, kv.first.c_str(), kv.second));
    }
    std::size_t rows() const { return rows_; }
    std::size_t cols() const { return cols_; }
    std::size_t size() const { return rows_ * cols_; }

    // connect(&connecting_conditional, weight_logic), neuron/mod.rs:1134-1157
    void connect(const std::function<bool(Position, Position)> &cond, const std::function<float(Position, Position)> &weight = nullptr) {
        const detail::Csr g = detail::evaluate(rows_, cols_, rows_, cols_, cond, weight);
        ck(snn_lattice_set_graph_csr(need(), g.row_ptr.data(), g.pre.data(), g.w.data(), size(), g.row_ptr.back()));
    }
    // the predicate max(|dr|, |dc|) <= radius && x != y, generated on the device (10^7 neurons)
    void connect_grid(uint32_t radius = 1, float weight = 1.f) { ck(snn_lattice_set_graph_grid(need(), radius, weight)); }
    // graph.lookup_weight(&x, &y) -> Option<f32>, graph/mod.rs:196-206 (false = None)
    bool lookup_weight(Position x, Position y, float *weight) {
        int32_t connected = 0;
        ck(snn_lattice_lookup_weight(need(), x.first * cols_ + x.second, y.first * cols_ + y.second, weight, &connected));
        return connected != 0;
    }

    // one named field of every neuron, row-major (IterateAndSpikeGPU::convert_to_gpu naming, integrate_and_fire/mod.rs:729-773);
    // the vector form of Lattice::apply / cell_grid()
    void set_field(const std::string &name, const std::vector<float> &v) { ck(snn_lattice_set_field(need(), name.c_str(), v.data(), v.size(), SNN_F32)); }
    void set_field(const std::string &name, const std::vector<uint32_t> &v) { ck(snn_lattice_set_field(need(), name.c_str(), v.data(), v.size(), SNN_U32)); }
    void set_field(const std::string &name, const std::vector<int32_t> &v) { ck(snn_lattice_set_field(need(), name.c_str(), v.data(), v.size(), SNN_I32)); }
    void fill_field(const std::string &name, float value) { ck(snn_lattice_fill_field_f32(need(), name.c_str(), value)); }
    std::vector<float> get_field(const std::string &name, std::size_t per_neuron = 1) {
        std::vector<float> v(size() * per_neuron);
        ck(snn_lattice_get_field(need(), name.c_str(), v.data(), v.size(), SNN_F32));
        return v;
    }
    std::vector<int32_t> get_last_firing_times() {   // Option<usize> as i32, -1 = None
        std::vector<int32_t> v(size());
        ck(snn_lattice_get_field(need(), "last_firing_time", v.data(), v.size(), SNN_I32));
        return v;
    }
    // apply_given_position(&|pos, neuron| ...), neuron/mod.rs:440-449, for one field at a time
    void apply_given_position(const std::string &field, const std::function<float(Position, float)> &f) {
        std::vector<float> v = get_field(field);
        for (std::size_t i = 0; i < v.size(); ++i) v[i] = f(Position{i / cols_, i % cols_}, v[i]);
        set_field(field, v);
    }

    void set_dt(float dt) { ck(snn_lattice_set_dt(need(), dt)); plasticity.dt = dt; }   // neuron/mod.rs:649-652
    void reset_timing() { ck(snn_lattice_reset_timing(need())); }                        // :405-420
    std::size_t internal_clock() const {
        int64_t v = 0;
        if (h_) detail::check(snn_lattice_get_option(h_, SNN_OPT_INTERNAL_CLOCK, &v), snn_lattice_last_error(h_));
        return (std::size_t)v;
    }

    // RunLattice::run_lattice, neuron/mod.rs:1209-1219; a lattice that was never populated is empty: Ok(())
    virtual void run_lattice(std::size_t iterations) {
        if (!h_) return;
        push_options();
        ck(snn_lattice_run(h_, iterations));
    }

    // grid_history.history: [step][row][col] flattened; spike raster likewise (neuron/mod.rs:286-378)
    std::size_t history_len() { uint64_t n = 0; ck(snn_lattice_history_len(need(), &n)); return n; }
    std::vector<float> grid_history() {
        std::vector<float> v(history_len() * size());
        ck(snn_lattice_get_grid_history(need(), v.data(), v.size()));
        return v;
    }
    std::vector<uint8_t> spike_history() {
        std::vector<uint8_t> v(history_len() * size());
        ck(snn_lattice_get_spike_history(need(), v.data(), v.size()));
        return v;
    }
    void reset_history() { ck(snn_lattice_reset_history(need())); }
    GraphHistory graph_history() {
        GraphHistory g;
        uint64_t steps = 0, nnz = 0;
        ck(snn_lattice_graph_history_len(need(), &steps, &nnz));
        g.steps = steps; g.nnz = nnz;
        g.weights.resize(steps * nnz);
        ck(snn_lattice_get_graph_history(h_, g.weights.data(), g.weights.size()));
        return g;
    }
    SpikeEvents spike_events() {
        uint64_t steps = 0, n = 0;
        ck(snn_lattice_spike_event_count(need(), &steps, &n));
        SpikeEvents ev;
        ev.step_ptr.resize(steps + 1); ev.neurons.resize(n);
        ck(snn_lattice_get_spike_events(h_, ev.step_ptr.data(), ev.neurons.data(), n));
        return ev;
    }

    snn_lattice_t *handle() { return h_; }

protected:
    snn_lattice_t *h_ = nullptr;
    std::size_t rows_ = 0, cols_ = 0;
    snn_lattice_t *need() {
        if (!h_) throw SpikingNeuralNetworksError(SNN_INVALID_ARGUMENT, "lattice is not populated");
        return h_;
    }
    void ck(int status) const { detail::check(status, h_ ? snn_lattice_last_error(h_) : nullptr); }
    virtual void push_options() {
        ck(snn_lattice_set_option(h_, SNN_OPT_ELECTRICAL_SYNAPSE, electrical_synapse));
        ck(snn_lattice_set_option(h_, SNN_OPT_CHEMICAL_SYNAPSE, chemical_synapse));
        ck(snn_lattice_set_option(h_, SNN_OPT_DO_PLASTICITY, do_plasticity));
        ck(snn_lattice_set_option(h_, SNN_OPT_UPDATE_GRID_HISTORY, update_grid_history));
        ck(snn_lattice_set_option(h_, SNN_OPT_UPDATE_SPIKE_HISTORY, update_spike_history));
        ck(snn_lattice_set_option(h_, SNN_OPT_UPDATE_GRAPH_HISTORY, update_graph_history));
        ck(snn_lattice_set_option(h_, SNN_OPT_UPDATE_SPIKE_EVENTS, update_spike_events));
        ck(snn_lattice_set_option(h_, SNN_OPT_PARALLEL, parallel));
        const snn_stdp_t s{plasticity.a_plus, plasticity.a_minus, plasticity.tau_plus, plasticity.tau_minus, plasticity.dt};
        ck(snn_lattice_set_plasticity(h_, &s));
    }
};

// Lattice<BCMIzhikevichNeuron, ..., BCM, ...>: the plasticity rule is BCM (plasticity/mod.rs:80-112)
class BCMLattice : public Lattice {
public:
    BCM bcm_plasticity;
protected:
    void push_options() override {
        Lattice::push_options();
        const snn_bcm_t b{bcm_plasticity.decay, bcm_plasticity.average_scalar, bcm_plasticity.dt};
        ck(snn_lattice_set_bcm_plasticity(h_, 1, &b));
    }
};

// RewardModulatedLattice<TraceRSTDP, T, ..., RewardModulatedSTDP, N>, neuron/mod.rs:2717-3416
class RewardModulatedLattice : public Lattice {
public:
    bool do_modulation = true;                 // RewardModulatedLattice::default, :2762-2777
    RewardModulatedSTDP reward_modulator;
    // run_lattice_with_reward(reward), :3250-3257: one timestep, reward_modulator.update(reward) first
    void run_lattice_with_reward(float reward) {
        if (!h_) return;
        push_options();
        ck(snn_lattice_run_with_rewards(h_, &reward, 1));
        snn_rstdp_t m{};
        ck(snn_lattice_get_reward_modulator(h_, &m));
        reward_modulator.dopamine = m.dopamine;
    }
protected:
    void push_options() override {
        do_plasticity = false;
        Lattice::push_options();
        const RewardModulatedSTDP &r = reward_modulator;
        const snn_rstdp_t m{r.dopamine, r.tau_d, r.tau_c, r.a_plus, r.a_minus, r.tau_plus, r.tau_minus, r.dt};
        ck(snn_lattice_set_reward_modulator(h_, 1, do_modulation, &m));
    }
};

// ----------------------------------------------------------------------------------------------------------------------------
// LatticeNetwork (neuron/mod.rs:1538-2675): lattices and spike-train lattices by unique id, one connecting graph
// ----------------------------------------------------------------------------------------------------------------------------
class LatticeNetwork {
public:
    bool electrical_synapse = true, chemical_synapse = false;
    // records of every connecting block before each step's STDP (neuron/mod.rs:2565-2576); a lattice's own graph is recorded with
    // set_lattice_option(id, SNN_OPT_UPDATE_GRAPH_HISTORY, 1)
    bool update_connecting_graph_history = false;

    explicit LatticeNetwork(snn_model_t model = SNN_MODEL_IZHIKEVICH, snn_spike_train_t spike_train = SNN_TRAIN_POISSON,
                            snn_nt_kinetics_t ntk = SNN_NT_APPROXIMATE, snn_receptor_kinetics_t rck = SNN_RC_APPROXIMATE,
                            snn_refractoriness_t refractoriness = SNN_REFRACT_DELTA_DIRAC) {
        snn_network_desc_t d{};
        d.struct_size = sizeof d; d.model = model; d.nt_kinetics = ntk; d.receptor_kinetics = rck; d.spike_train = spike_train;
        d.refractoriness = refractoriness; d.device = -1;
        detail::check(snn_network_create(&d, &h_), snn_network_last_error(nullptr));
    }
    LatticeNetwork(const LatticeNetwork &) = delete;
    LatticeNetwork &operator=(const LatticeNetwork &) = delete;
    ~LatticeNetwork() { if (h_) snn_network_destroy(h_); }

    // add_lattice / add_spike_train_lattice, neuron/mod.rs:1663-1698 (GraphIDAlreadyPresent on a duplicate id)
    void add_lattice(std::size_t id, const BaseNeuron &base, std::size_t rows, std::size_t cols) {
        ck(snn_network_add_lattice(h_, id, (uint32_t)rows, (uint32_t)cols));
        dims_[id] = {rows, cols};
        for (auto &kv : base.fields) ck(snn_network_fill_field_f32(h_, id, kv.first.c_str(), kv.second));
    }
    void add_spike_train_lattice(std::size_t id, const std::map<std::string, float> &base_fields, std::size_t rows, std::size_t cols) {
        ck(snn_network_add_spike_train_lattice(h_, id, (uint32_t)rows, (uint32_t)cols));
        dims_[id] = {rows, cols};
        for (auto &kv : base_fields) ck(snn_network_fill_field_f32(h_, id, kv.first.c_str(), kv.second));
    }
    // connect(presynaptic_id, postsynaptic_id, &cond, weight_logic), neuron/mod.rs:1845-1930
    void connect(std::size_t pre_id, std::size_t post_id, const std::function<bool(Position, Position)> &cond,
                 const std::function<float(Position, Position)> &weight = nullptr) {
        // the library checks the ids in the reference's order: postsynaptic spike train, presynaptic id, postsynaptic id (:1852-1862)
        const Position a = dims_.count(pre_id) ? dims_[pre_id] : Position{0, 0}, b = dims_.count(post_id) ? dims_[post_id] : Position{0, 0};
        const detail::Csr g = detail::evaluate(a.first, a.second, b.first, b.second, cond, weight);
        ck(snn_network_connect_csr(h_, pre_id, post_id, g.row_ptr.data(), g.pre.data(), g.w.data(), b.first * b.second, g.row_ptr.back()));
    }
    void set_field(std::size_t id, const std::string &name, const std::vector<float> &v) { ck(snn_network_set_field(h_, id, name.c_str(), v.data(), v.size(), SNN_F32)); }
    std::vector<float> get_field(std::size_t id, const std::string &name) {
        uint64_t n = 0;
        ck(snn_network_lattice_size(h_, id, &n));
        std::vector<float> v(n);
        ck(snn_network_get_field(h_, id, name.c_str(), v.data(), v.size(), SNN_F32));
        return v;
    }
    void set_lattice_option(std::size_t id, snn_option_t option, int64_t value) { ck(snn_network_set_lattice_option(h_, id, option, value)); }
    void set_plasticity(std::size_t id, const STDP &p) {
        const snn_stdp_t s{p.a_plus, p.a_minus, p.tau_plus, p.tau_minus, p.dt};
        ck(snn_network_set_plasticity(h_, id, &s));
    }
    void set_dt(float dt) { ck(snn_network_set_dt(h_, dt)); }
    // RunNetwork::run_lattices, neuron/mod.rs:2667-2674
    void run_lattices(std::size_t iterations) {
        ck(snn_network_set_option(h_, SNN_OPT_ELECTRICAL_SYNAPSE, electrical_synapse));
        ck(snn_network_set_option(h_, SNN_OPT_CHEMICAL_SYNAPSE, chemical_synapse));
        ck(snn_network_set_option(h_, SNN_OPT_UPDATE_CONNECTING_GRAPH_HISTORY, update_connecting_graph_history));
        ck(snn_network_run(h_, iterations));
    }
    // the records of the block pre_id -> post_id (pre_id == post_id: the lattice's own graph)
    GraphHistory graph_history(std::size_t pre_id, std::size_t post_id) {
        GraphHistory g;
        uint64_t steps = 0, nnz = 0;
        ck(snn_network_graph_history_len(h_, pre_id, post_id, &steps, &nnz));
        g.steps = steps; g.nnz = nnz;
        g.weights.resize(steps * nnz);
        ck(snn_network_get_graph_history(h_, pre_id, post_id, g.weights.data(), g.weights.size()));
        return g;
    }
    std::vector<uint8_t> spike_history(std::size_t id) {
        uint64_t steps = 0, n = 0;
        ck(snn_network_history_len(h_, id, &steps));
        ck(snn_network_lattice_size(h_, id, &n));
        std::vector<uint8_t> v(steps * n);
        ck(snn_network_get_spike_history(h_, id, v.data(), v.size()));
        return v;
    }
    // spike events of lattice `id` (SNN_OPT_UPDATE_SPIKE_EVENTS through set_lattice_option), indices inside the lattice
    SpikeEvents spike_events(std::size_t id) {
        uint64_t steps = 0, n = 0;
        ck(snn_network_spike_event_count(h_, id, &steps, &n));
        SpikeEvents ev;
        ev.step_ptr.resize(steps + 1); ev.neurons.resize(n);
        ck(snn_network_get_spike_events(h_, id, ev.step_ptr.data(), ev.neurons.data(), n));
        return ev;
    }
    snn_network_t *handle() { return h_; }

protected:
    snn_network_t *h_ = nullptr;
    std::map<std::size_t, Position> dims_;
    void ck(int status) const { detail::check(status, h_ ? snn_network_last_error(h_) : nullptr); }
};

// RewardModulatedConnection<TraceRSTDP>, neuron/mod.rs:3418-3443: Weight(f32) or RewardModulatedWeight(TraceRSTDP{weight, ..default})
struct RewardModulatedConnection {
    float weight = 1.f;
    bool reward_modulated = false;
    static RewardModulatedConnection Weight(float w) { return {w, false}; }
    static RewardModulatedConnection RewardModulatedWeight(float w) { return {w, true}; }
};

// RewardModulatedLatticeNetwork (neuron/mod.rs:3455-5455): plain, reward-modulated and spike-train lattices over one connecting
// graph of RewardModulatedConnection values.  One connection kind per connecting block; the configurations on which the reference
// panics make run_lattices* throw SNN_UNSUPPORTED (include/snn_b200.h).
class RewardModulatedLatticeNetwork : public LatticeNetwork {
public:
    using LatticeNetwork::LatticeNetwork;

    // add_reward_modulated_lattice, :3615-3634
    void add_reward_modulated_lattice(std::size_t id, const BaseNeuron &base, std::size_t rows, std::size_t cols,
                                      const RewardModulatedSTDP &modulator = RewardModulatedSTDP(), bool do_modulation = true) {
        ck(snn_network_add_reward_modulated_lattice(h_, id, (uint32_t)rows, (uint32_t)cols));
        dims_[id] = {rows, cols};
        reward_ids_[id] = true;
        for (auto &kv : base.fields) ck(snn_network_fill_field_f32(h_, id, kv.first.c_str(), kv.second));
        set_reward_modulator(id, modulator, do_modulation);
    }
    void set_reward_modulator(std::size_t id, const RewardModulatedSTDP &r, bool do_modulation = true) {
        const snn_rstdp_t m{r.dopamine, r.tau_d, r.tau_c, r.a_plus, r.a_minus, r.tau_plus, r.tau_minus, r.dt};
        ck(snn_network_set_reward_modulator(h_, id, do_modulation, &m));
    }
    RewardModulatedSTDP reward_modulator(std::size_t id) {
        snn_rstdp_t m{};
        ck(snn_network_get_reward_modulator(h_, id, nullptr, &m));
        RewardModulatedSTDP r;
        r.dopamine = m.dopamine; r.tau_d = m.tau_d; r.tau_c = m.tau_c; r.a_plus = m.a_plus; r.a_minus = m.a_minus;
        r.tau_plus = m.tau_plus; r.tau_minus = m.tau_minus; r.dt = m.dt;
        return r;
    }
    // connect, :3836-3947: plain / spike-train lattices only (ConnectFunctionMustHaveNonRewardModulatedLattice otherwise); the
    // checks that need the two lattice maps live here, the others in the library, in the reference's order
    void connect(std::size_t pre_id, std::size_t post_id, const std::function<bool(Position, Position)> &cond,
                 const std::function<float(Position, Position)> &weight = nullptr) {
        const bool known_pre = dims_.count(pre_id) != 0;
        if (known_pre && (reward_ids_.count(post_id) || (dims_.count(post_id) && reward_ids_.count(pre_id))))
            detail::check(SNN_NET_CONNECT_FUNCTION_MUST_HAVE_NON_REWARD_MODULATED_LATTICE,
                          "Connect function must have non reward modulated lattices, connect with reward modulation instead");
        LatticeNetwork::connect(pre_id, post_id, cond, weight);
    }
    // connect_reward_modulated_lattice_interally, :4393-4413 (IDNotFoundInLattices for anything but a reward-modulated lattice)
    void connect_reward_modulated_lattice_interally(std::size_t id, const std::function<bool(Position, Position)> &cond,
                                                    const std::function<float(Position, Position)> &weight = nullptr) {
        if (!reward_ids_.count(id)) detail::check(SNN_NET_ID_NOT_FOUND_IN_LATTICES, ("Id not present in lattices, id: " + std::to_string(id)).c_str());
        LatticeNetwork::connect(id, id, cond, weight);
    }
    // connect_with_reward_modulation, :4076-4209
    void connect_with_reward_modulation(std::size_t pre_id, std::size_t post_id, const std::function<bool(Position, Position)> &cond,
                                        const std::function<RewardModulatedConnection(Position, Position)> &weight_logic) {
        const Position a = dims_.count(pre_id) ? dims_[pre_id] : Position{0, 0}, b = dims_.count(post_id) ? dims_[post_id] : Position{0, 0};
        int kinds = 0;
        const detail::Csr g = detail::evaluate(a.first, a.second, b.first, b.second, cond, [&](Position x, Position y) {
            const RewardModulatedConnection c = weight_logic(x, y);
            kinds |= c.reward_modulated ? 2 : 1;
            return c.weight;
        });
        if (kinds == 3) detail::check(SNN_UNSUPPORTED, "one connecting block holds one kind of RewardModulatedConnection");
        // the id checks in the reference's order (:4083-4107) before anything is changed; the block itself may not exist yet
        const int pre_check = snn_network_set_connection_reward_modulated(h_, pre_id, post_id, kinds == 2);
        if (pre_check != SNN_OK && pre_check != SNN_INVALID_ARGUMENT) ck(pre_check);
        ck(snn_network_connect_csr(h_, pre_id, post_id, g.row_ptr.data(), g.pre.data(), g.w.data(), b.first * b.second, g.row_ptr.back()));
        ck(snn_network_set_connection_reward_modulated(h_, pre_id, post_id, kinds == 2));
    }
    // run_lattices_with_reward, :5385-5392
    void run_lattices_with_reward(float reward) {
        ck(snn_network_set_option(h_, SNN_OPT_ELECTRICAL_SYNAPSE, electrical_synapse));
        ck(snn_network_set_option(h_, SNN_OPT_CHEMICAL_SYNAPSE, chemical_synapse));
        ck(snn_network_set_option(h_, SNN_OPT_UPDATE_CONNECTING_GRAPH_HISTORY, update_connecting_graph_history));
        ck(snn_network_run_with_rewards(h_, &reward, 1));
    }
    std::vector<float> connection_weights(std::size_t pre_id, std::size_t post_id) {
        uint64_t nnz = 0, n = 0;
        ck(snn_network_connection_nnz(h_, pre_id, post_id, &nnz));
        ck(snn_network_lattice_size(h_, post_id, &n));
        std::vector<uint64_t> rp(n + 1);
        std::vector<uint32_t> pre(nnz ? nnz : 1);
        std::vector<float> w(nnz ? nnz : 1);
        ck(snn_network_get_connection_csr(h_, pre_id, post_id, rp.data(), pre.data(), w.data(), n, nnz));
        w.resize(nnz);
        return w;
    }

private:
    std::map<std::size_t, bool> reward_ids_;
};

// SpikeTrainLattice<N, T, U> on its own (neuron/mod.rs:1290-1428; RunSpikeTrainLattice :1419-1428): a network that holds just this lattice
class SpikeTrainLattice {
public:
    bool update_grid_history = false, update_spike_history = false, update_spike_events = false;
    explicit SpikeTrainLattice(snn_spike_train_t kind = SNN_TRAIN_POISSON, std::size_t id = 0) : net_(SNN_MODEL_IZHIKEVICH, kind), id_(id) {}
    // populate(&base_spike_train, num_rows, num_cols), :1321-1341; base = the spike train's fields that differ from Default
    void populate(const std::map<std::string, float> &base_fields, std::size_t rows, std::size_t cols) {
        net_.add_spike_train_lattice(id_, base_fields, rows, cols);
    }
    void set_field(const std::string &name, const std::vector<float> &v) { net_.set_field(id_, name, v); }
    std::vector<float> get_field(const std::string &name) { return net_.get_field(id_, name); }
    void run_lattice(std::size_t iterations) {
        net_.set_lattice_option(id_, SNN_OPT_UPDATE_GRID_HISTORY, update_grid_history);
        net_.set_lattice_option(id_, SNN_OPT_UPDATE_SPIKE_HISTORY, update_spike_history);
        net_.set_lattice_option(id_, SNN_OPT_UPDATE_SPIKE_EVENTS, update_spike_events);
        net_.run_lattices(iterations);
    }
    std::vector<uint8_t> spike_history() { return net_.spike_history(id_); }
    SpikeEvents spike_events() { return net_.spike_events(id_); }

private:
    LatticeNetwork net_;
    std::size_t id_;
};

}  // namespace snn_b200
