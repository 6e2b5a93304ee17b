// capi.cu — the extern "C" boundary declared in include/snn_b200.h.
// No exception may cross it: every entry point catches and maps to a status code.
#include <cstring>
#include <new>
#include <string>

#include "engine.h"

using snn::Engine;

struct snn_network { Engine *e; };
struct snn_lattice { Engine *e; };

static thread_local std::string g_create_error;

#define SNN_TRY try {
#define SNN_CATCH(h)                                                                                \
    } catch (const std::bad_alloc &) {                                                              \
        if (h) (h)->e->last_error = "host allocation failed";                                       \
        return SNN_GPU_BUFFER_CREATE_ERROR;                                                         \
    } catch (const std::exception &ex) {                                                            \
        if (h) (h)->e->last_error = ex.what();                                                      \
        return SNN_INVALID_ARGUMENT;                                                                \
    } catch (...) {                                                                                 \
        return SNN_INVALID_ARGUMENT;                                                                \
    }

static const uint64_t kLatticeId = 0;  // the single lattice behind an snn_lattice_t

extern "C" {

int32_t snn_abi_version(void) { return SNN_B200_ABI_VERSION; }

const char *snn_status_string(int32_t s) {
    switch (s) {
    case SNN_OK: return "ok";
    // messages of GPUError's Display impl, backend/src/error/mod.rs:241-256
    case SNN_GPU_PROGRAM_COMPILE_FAILURE: return "Could not compile program";
    case SNN_GPU_KERNEL_COMPILE_FAILURE: return "Could not compile kernel";
    case SNN_GPU_BUFFER_CREATE_ERROR: return "Could not create buffer";
    case SNN_GPU_BUFFER_WRITE_ERROR: return "Could not write to buffer";
    case SNN_GPU_BUFFER_READ_ERROR: return "Could not read buffer";
    case SNN_GPU_WAIT_ERROR: return "Could not wait for event";
    case SNN_GPU_GET_DEVICE_FAILURE: return "Could not get device";
    case SNN_GPU_QUEUE_FAILURE: return "Could not queue";
    // GraphError, error/mod.rs:22-33
    case SNN_GRAPH_PRESYNAPTIC_NOT_FOUND: return "Presynaptic position not found";
    case SNN_GRAPH_POSTSYNAPTIC_NOT_FOUND: return "Postsynaptic position not found";
    case SNN_GRAPH_POSITION_NOT_FOUND: return "Position not found";
    case SNN_GRAPH_DIMENSIONS_DO_NOT_MATCH: return "Dimensions do not match";
    // LatticeNetworkError, error/mod.rs:50-83
    case SNN_NET_GRAPH_ID_ALREADY_PRESENT: return "Graph id already present in network";
    case SNN_NET_POSTSYNAPTIC_ID_NOT_FOUND: return "Postsynaptic id not present in network";
    case SNN_NET_PRESYNAPTIC_ID_NOT_FOUND: return "Presynaptic id not present in network";
    case SNN_NET_ID_NOT_FOUND_IN_LATTICES: return "Id not present in lattices";
    case SNN_NET_POSTSYNAPTIC_LATTICE_CANNOT_BE_SPIKE_TRAIN:
        return "Postsynaptic lattice cannot be a spike train lattice because spike trains cannot take inputs";
    case SNN_NET_CANNOT_CONNECT_WITH_REWARD_MODULATED_CONNECTION:
        return "When connecting reward modulated network, at least one lattice has to be reward modulated";
    case SNN_NET_REWARD_MODULATED_CONNECTION_NOT_COMPATIBLE_INTERNALLY:
        return "When connecting reward modulated lattice, RewardModulatedConnection cannot be used to connect a reward modulated lattice internally";
    case SNN_NET_CONNECT_FUNCTION_MUST_HAVE_NON_REWARD_MODULATED_LATTICE:
        return "Connect function must have non reward modulated lattices, connect with reward modulation instead";
    case SNN_INVALID_ARGUMENT: return "invalid argument";
    case SNN_UNKNOWN_FIELD: return "unknown field";
    case SNN_DTYPE_MISMATCH: return "dtype mismatch";
    case SNN_SIZE_MISMATCH: return "size mismatch";
    case SNN_UNSUPPORTED: return "unsupported";
    }
    return "unknown status";
}

const char *snn_lattice_last_error(const snn_lattice_t *h) { return h ? h->e->last_error.c_str() : g_create_error.c_str(); }
const char *snn_network_last_error(const snn_network_t *h) { return h ? h->e->last_error.c_str() : g_create_error.c_str(); }

int32_t snn_device_count(int32_t *count) {
    int c = 0;
    cudaError_t e = cudaGetDeviceCount(&c);
    if (count) *count = (e == cudaSuccess) ? c : 0;
    if (e != cudaSuccess || c == 0) { cudaGetLastError(); return SNN_GPU_GET_DEVICE_FAILURE; }
    return SNN_OK;
}

uint32_t snn_partition_begin(uint32_t rows, int32_t world, int32_t rank) {
    if (world <= 0) return 0;
    if (rank <= 0) return 0;
    if (rank >= world) return rows;
    // balanced contiguous row strips: the first (rows % world) ranks own one extra row
    const uint32_t base = rows / (uint32_t)world, extra = rows % (uint32_t)world;
    return (uint32_t)rank * base + ((uint32_t)rank < extra ? (uint32_t)rank : extra);
}

static bool valid_enums(int model, int ntk, int rck) {
    return model >= 0 && model < SNN_MODEL_COUNT && ntk >= 0 && ntk <= SNN_NT_EXPONENTIAL_DECAY && rck >= 0 &&
           rck <= SNN_RC_EXPONENTIAL_DECAY;
}

// ---------------------------------------------------------------------------------------------- lattice
int32_t snn_lattice_create(const snn_lattice_desc_t *desc, snn_lattice_t **out) {
    if (out) *out = nullptr;
    if (!desc || !out || desc->struct_size != sizeof(snn_lattice_desc_t)) { g_create_error = "bad descriptor"; return SNN_INVALID_ARGUMENT; }
    if (!valid_enums(desc->model, desc->nt_kinetics, desc->receptor_kinetics)) { g_create_error = "bad enum in descriptor"; return SNN_INVALID_ARGUMENT; }
    try {
        Engine *e = new Engine(desc->model, desc->nt_kinetics, desc->receptor_kinetics, SNN_TRAIN_POISSON, SNN_REFRACT_DELTA_DIRAC, desc->device);
        int r = e->init();
        const int world = desc->part_world <= 0 ? 1 : desc->part_world;
        uint32_t rows_local = desc->rows;
        if (!r && world > 1) {
            r = e->set_partition(desc->rows, desc->cols, desc->part_rank, world);
            rows_local = snn_partition_begin(desc->rows, world, desc->part_rank + 1) - snn_partition_begin(desc->rows, world, desc->part_rank);
        }
        if (!r) r = e->add_lattice(kLatticeId, rows_local, desc->cols, false);
        if (r) { g_create_error = e->last_error; delete e; return r; }
        *out = new snn_lattice{e};
        return SNN_OK;
    } catch (...) { g_create_error = "allocation failed"; return SNN_GPU_BUFFER_CREATE_ERROR; }
}

int32_t snn_lattice_destroy(snn_lattice_t *h) {
    if (!h) return SNN_OK;
    delete h->e; delete h;
    return SNN_OK;
}

int32_t snn_lattice_rows(const snn_lattice_t *h, uint32_t *rows_local, uint32_t *cols) {
    if (!h) return SNN_INVALID_ARGUMENT;
    const snn::Lat *L = h->e->find(kLatticeId);
    if (rows_local) *rows_local = L->rows;
    if (cols) *cols = L->cols;
    return SNN_OK;
}
int32_t snn_lattice_size(const snn_lattice_t *h, uint64_t *n) {
    if (!h || !n) return SNN_INVALID_ARGUMENT;
    *n = h->e->find(kLatticeId)->n;
    return SNN_OK;
}
int32_t snn_lattice_field_count(const snn_lattice_t *h, uint32_t *count) {
    if (!h || !count) return SNN_INVALID_ARGUMENT;
    return h->e->field_count(kLatticeId, count);
}
int32_t snn_lattice_field_info(const snn_lattice_t *h, uint32_t index, const char **name, int32_t *dtype, uint32_t *per) {
    if (!h || !name || !dtype || !per) return SNN_INVALID_ARGUMENT;
    return h->e->field_info(kLatticeId, index, name, dtype, per);
}
int32_t snn_lattice_set_field(snn_lattice_t *h, const char *name, const void *data, uint64_t count, int32_t dtype) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->set_field(kLatticeId, name, data, count, dtype); SNN_CATCH(h)
}
int32_t snn_lattice_fill_field_f32(snn_lattice_t *h, const char *name, float v) {
    if (!h) return SNN_INVALID_ARGUMENT;
    uint32_t b; memcpy(&b, &v, 4);
    SNN_TRY return h->e->fill_field(kLatticeId, name, b, SNN_F32); SNN_CATCH(h)
}
int32_t snn_lattice_fill_field_u32(snn_lattice_t *h, const char *name, uint32_t v) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->fill_field(kLatticeId, name, v, SNN_U32); SNN_CATCH(h)
}
int32_t snn_lattice_fill_field_i32(snn_lattice_t *h, const char *name, int32_t v) {
    if (!h) return SNN_INVALID_ARGUMENT;
    uint32_t b; memcpy(&b, &v, 4);
    SNN_TRY return h->e->fill_field(kLatticeId, name, b, SNN_I32); SNN_CATCH(h)
}
int32_t snn_lattice_get_field(snn_lattice_t *h, const char *name, void *out, uint64_t count, int32_t dtype) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->get_field(kLatticeId, name, out, count, dtype); SNN_CATCH(h)
}

int32_t snn_lattice_set_graph_dense(snn_lattice_t *h, const uint32_t *connections, const float *weights,
                                    const uint32_t *index_to_position, uint32_t n) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->connect_dense(kLatticeId, kLatticeId, connections, weights, index_to_position, n, n); SNN_CATCH(h)
}
int32_t snn_lattice_set_graph_csr(snn_lattice_t *h, const uint64_t *row_ptr, const uint32_t *pre, const float *weights, uint64_t n,
                                  uint64_t nnz) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->connect_csr(kLatticeId, kLatticeId, row_ptr, pre, weights, n, nnz); SNN_CATCH(h)
}
int32_t snn_lattice_set_graph_grid(snn_lattice_t *h, uint32_t radius, float weight) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->connect_grid(kLatticeId, radius, weight); SNN_CATCH(h)
}
int32_t snn_lattice_graph_nnz(snn_lattice_t *h, uint64_t *nnz) {
    if (!h || !nnz) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->connection_nnz(kLatticeId, kLatticeId, nnz); SNN_CATCH(h)
}
int32_t snn_lattice_get_graph_csr(snn_lattice_t *h, uint64_t *row_ptr, uint32_t *pre, float *weights, uint64_t n, uint64_t nnz) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->get_connection_csr(kLatticeId, kLatticeId, row_ptr, pre, weights, n, nnz); SNN_CATCH(h)
}
int32_t snn_lattice_get_graph_dense(snn_lattice_t *h, uint32_t *connections, float *weights, uint32_t n) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->get_connection_dense(kLatticeId, kLatticeId, connections, weights, n, n); SNN_CATCH(h)
}
int32_t snn_lattice_lookup_weight(snn_lattice_t *h, uint64_t pre, uint64_t post, float *weight, int32_t *connected) {
    if (!h || !weight || !connected) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->lookup_weight(kLatticeId, kLatticeId, pre, post, weight, connected); SNN_CATCH(h)
}
int32_t snn_lattice_edit_weight(snn_lattice_t *h, uint64_t pre, uint64_t post, int32_t connected, float weight) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->edit_weight(kLatticeId, kLatticeId, pre, post, connected != 0, weight); SNN_CATCH(h)
}
int32_t snn_lattice_get_graph_rows(snn_lattice_t *h, uint64_t row_begin, uint64_t row_end, uint64_t *row_ptr, uint32_t *pre, float *weights,
                                   uint64_t capacity, uint64_t *nnz) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->get_connection_rows(kLatticeId, kLatticeId, row_begin, row_end, row_ptr, pre, weights, capacity, nnz); SNN_CATCH(h)
}
int32_t snn_lattice_get_spike_aggregate(snn_lattice_t *h, int64_t *out, uint64_t capacity) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->get_spike_aggregate(kLatticeId, out, capacity); SNN_CATCH(h)
}

static int32_t engine_set_option(Engine *e, bool have_id, uint64_t id, int32_t option, int64_t value) {
    snn::Lat *L = have_id ? e->find(id) : nullptr;
    if (have_id && !L) return e->fail(SNN_NET_ID_NOT_FOUND_IN_LATTICES, "Id not present in lattices, id: " + std::to_string(id));
    switch (option) {
    case SNN_OPT_ELECTRICAL_SYNAPSE: e->electrical = value != 0; return SNN_OK;
    case SNN_OPT_CHEMICAL_SYNAPSE: e->chemical = value != 0; return SNN_OK;
    case SNN_OPT_PARALLEL: e->parallel = value != 0; return SNN_OK;
    case SNN_OPT_RNG_SEED: e->seed = (uint64_t)value; return SNN_OK;
    case SNN_OPT_STEPS_PER_GRAPH: e->steps_per_graph = (uint32_t)value; return SNN_OK;
    case SNN_OPT_GENERAL_PARTITION: e->force_gpart = value != 0; return SNN_OK;
    case SNN_OPT_HALO_TIMEOUT_MS:
        if (value <= 0) return e->fail(SNN_INVALID_ARGUMENT, "halo time-out must be positive");
        e->halo_timeout_ms = (uint64_t)value; return SNN_OK;
    case SNN_OPT_INTERNAL_CLOCK:
        if (value < 0) return e->fail(SNN_INVALID_ARGUMENT, "clock must be non-negative");
        if (L && L->is_train) L->clock = (uint64_t)value; else e->internal_clock = (uint64_t)value;
        return SNN_OK;
    case SNN_OPT_DO_PLASTICITY: if (!L) break; L->do_plasticity = value != 0; return SNN_OK;
    case SNN_OPT_UPDATE_GRID_HISTORY: if (!L) break; L->grid_hist = value != 0; return SNN_OK;
    case SNN_OPT_UPDATE_SPIKE_HISTORY: if (!L) break; L->spike_hist = value != 0; return SNN_OK;
    case SNN_OPT_UPDATE_AVERAGE_HISTORY: if (!L || L->is_train) break; L->avg_hist = value != 0; return SNN_OK;
    case SNN_OPT_UPDATE_EEG_HISTORY: if (!L || L->is_train) break; L->eeg_hist = value != 0; return SNN_OK;
    case SNN_OPT_UPDATE_GRAPH_HISTORY: if (!L || L->is_train) break; L->graph_hist = value != 0; return SNN_OK;
    case SNN_OPT_UPDATE_CONNECTING_GRAPH_HISTORY: if (L || !e->is_network) break; e->conn_graph_hist = value != 0; return SNN_OK;
    case SNN_OPT_UPDATE_SPIKE_EVENTS: if (!L) break; L->spike_events = value != 0; return SNN_OK;
    }
    return e->fail(SNN_INVALID_ARGUMENT, "unknown option or missing lattice id");
}

static int32_t engine_get_option(const Engine *e, bool have_id, uint64_t id, int32_t option, int64_t *value) {
    const snn::Lat *L = have_id ? e->find(id) : nullptr;
    if (have_id && !L) return SNN_NET_ID_NOT_FOUND_IN_LATTICES;
    switch (option) {
    case SNN_OPT_ELECTRICAL_SYNAPSE: *value = e->electrical; return SNN_OK;
    case SNN_OPT_CHEMICAL_SYNAPSE: *value = e->chemical; return SNN_OK;
    case SNN_OPT_PARALLEL: *value = e->parallel; return SNN_OK;
    case SNN_OPT_RNG_SEED: *value = (int64_t)e->seed; return SNN_OK;
    case SNN_OPT_STEPS_PER_GRAPH: *value = e->steps_per_graph; return SNN_OK;
    case SNN_OPT_STEP_PATH: *value = e->last_step_path; return SNN_OK;
    case SNN_OPT_UNIFORM_TILES: *value = e->last_uniform_tiles; return SNN_OK;
    case SNN_OPT_STENCIL_TILES: *value = e->last_stencil_tiles; return SNN_OK;
    case SNN_OPT_HALO_TIMEOUT_MS: *value = (int64_t)e->halo_timeout_ms; return SNN_OK;
    case SNN_OPT_GENERAL_PARTITION: *value = e->force_gpart || e->is_gpart(); return SNN_OK;
    case SNN_OPT_INTERNAL_CLOCK: *value = (int64_t)((L && L->is_train) ? L->clock : e->internal_clock); return SNN_OK;
    case SNN_OPT_DO_PLASTICITY: if (!L) break; *value = L->do_plasticity; return SNN_OK;
    case SNN_OPT_UPDATE_GRID_HISTORY: if (!L) break; *value = L->grid_hist; return SNN_OK;
    case SNN_OPT_UPDATE_SPIKE_HISTORY: if (!L) break; *value = L->spike_hist; return SNN_OK;
    case SNN_OPT_UPDATE_AVERAGE_HISTORY: if (!L) break; *value = L->avg_hist; return SNN_OK;
    case SNN_OPT_UPDATE_EEG_HISTORY: if (!L) break; *value = L->eeg_hist; return SNN_OK;
    case SNN_OPT_UPDATE_GRAPH_HISTORY: if (!L) break; *value = L->graph_hist; return SNN_OK;
    case SNN_OPT_UPDATE_CONNECTING_GRAPH_HISTORY: if (L || !e->is_network) break; *value = e->conn_graph_hist; return SNN_OK;
    case SNN_OPT_UPDATE_SPIKE_EVENTS: if (!L) break; *value = L->spike_events; return SNN_OK;
    }
    return SNN_INVALID_ARGUMENT;
}

int32_t snn_lattice_set_option(snn_lattice_t *h, int32_t option, int64_t value) {
    if (!h) return SNN_INVALID_ARGUMENT;
    return engine_set_option(h->e, true, kLatticeId, option, value);
}
int32_t snn_lattice_get_option(const snn_lattice_t *h, int32_t option, int64_t *value) {
    if (!h || !value) return SNN_INVALID_ARGUMENT;
    return engine_get_option(h->e, true, kLatticeId, option, value);
}
int32_t snn_lattice_set_plasticity(snn_lattice_t *h, const snn_stdp_t *stdp) {
    if (!h || !stdp) return SNN_INVALID_ARGUMENT;
    h->e->find(kLatticeId)->stdp = *stdp;
    return SNN_OK;
}
int32_t snn_lattice_get_plasticity(const snn_lattice_t *h, snn_stdp_t *stdp) {
    if (!h || !stdp) return SNN_INVALID_ARGUMENT;
    *stdp = h->e->find(kLatticeId)->stdp;
    return SNN_OK;
}
int32_t snn_lattice_set_dt(snn_lattice_t *h, float dt) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->set_dt(dt); SNN_CATCH(h)
}
int32_t snn_lattice_reset_timing(snn_lattice_t *h) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->reset_timing(); SNN_CATCH(h)
}
int32_t snn_lattice_set_bcm_plasticity(snn_lattice_t *h, int32_t enable, const snn_bcm_t *bcm) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->set_bcm_plasticity(enable != 0, bcm); SNN_CATCH(h)
}
int32_t snn_lattice_set_reward_modulator(snn_lattice_t *h, int32_t enable, int32_t do_modulation, const snn_rstdp_t *modulator) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->set_reward_modulator(enable != 0, do_modulation != 0, modulator); SNN_CATCH(h)
}
int32_t snn_lattice_get_reward_modulator(const snn_lattice_t *h, snn_rstdp_t *modulator) {
    if (!h || !modulator) return SNN_INVALID_ARGUMENT;
    *modulator = h->e->rstdp;
    return SNN_OK;
}
int32_t snn_lattice_run_with_rewards(snn_lattice_t *h, const float *rewards, uint64_t n_rewards) {
    if (!h || (n_rewards && !rewards)) return SNN_INVALID_ARGUMENT;
    if (!h->e->reward_mode) return h->e->fail(SNN_INVALID_ARGUMENT, "handle is not a reward-modulated lattice (snn_lattice_set_reward_modulator)");
    SNN_TRY return h->e->run(n_rewards, nullptr, nullptr, rewards); SNN_CATCH(h)
}
int32_t snn_lattice_get_connection_traces(snn_lattice_t *h, uint32_t *counter, float *dw, float *c, uint64_t nnz) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->get_connection_traces(counter, dw, c, nnz); SNN_CATCH(h)
}
int32_t snn_lattice_set_connection_traces(snn_lattice_t *h, const float *weight, const uint32_t *counter, const float *dw, const float *c,
                                          uint64_t nnz) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->set_connection_traces(weight, counter, dw, c, nnz); SNN_CATCH(h)
}
int32_t snn_lattice_run(snn_lattice_t *h, uint64_t iterations) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->run(iterations, nullptr, nullptr); SNN_CATCH(h)
}
int32_t snn_lattice_run_timed(snn_lattice_t *h, uint64_t iterations, float *elapsed_ms, uint64_t *kernel_launches) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->run(iterations, elapsed_ms, kernel_launches); SNN_CATCH(h)
}
int32_t snn_lattice_history_len(const snn_lattice_t *h, uint64_t *steps) {
    if (!h || !steps) return SNN_INVALID_ARGUMENT;
    return h->e->history_len(kLatticeId, steps);
}
int32_t snn_lattice_get_grid_history(snn_lattice_t *h, float *out, uint64_t capacity_floats) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->get_grid_history(kLatticeId, out, capacity_floats); SNN_CATCH(h)
}
int32_t snn_lattice_get_spike_history(snn_lattice_t *h, uint8_t *out, uint64_t capacity_bytes) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->get_spike_history(kLatticeId, out, capacity_bytes); SNN_CATCH(h)
}
int32_t snn_lattice_get_average_history(snn_lattice_t *h, float *out, uint64_t capacity_floats) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->get_reduced_history(kLatticeId, false, out, capacity_floats); SNN_CATCH(h)
}
int32_t snn_lattice_set_eeg_parameters(snn_lattice_t *h, float reference_voltage, float distance, float conductivity) {
    if (!h) return SNN_INVALID_ARGUMENT;
    return h->e->set_eeg_parameters(kLatticeId, reference_voltage, distance, conductivity);
}
int32_t snn_lattice_get_eeg_history(snn_lattice_t *h, float *out, uint64_t capacity_floats) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->get_reduced_history(kLatticeId, true, out, capacity_floats); SNN_CATCH(h)
}
int32_t snn_lattice_reset_history(snn_lattice_t *h) {
    if (!h) return SNN_INVALID_ARGUMENT;
    return h->e->reset_history();
}
int32_t snn_lattice_graph_history_len(snn_lattice_t *h, uint64_t *steps, uint64_t *nnz) {
    if (!h || !steps || !nnz) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->graph_history_len(kLatticeId, kLatticeId, steps, nnz); SNN_CATCH(h)
}
int32_t snn_lattice_get_graph_history(snn_lattice_t *h, float *out, uint64_t capacity_floats) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->get_graph_history(kLatticeId, kLatticeId, out, capacity_floats); SNN_CATCH(h)
}
int32_t snn_lattice_spike_event_count(const snn_lattice_t *h, uint64_t *steps, uint64_t *n_events) {
    if (!h || !steps || !n_events) return SNN_INVALID_ARGUMENT;
    return h->e->spike_event_count(kLatticeId, steps, n_events);
}
int32_t snn_lattice_get_spike_events(snn_lattice_t *h, uint64_t *step_ptr, uint32_t *neuron, uint64_t capacity) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->get_spike_events(kLatticeId, step_ptr, neuron, capacity); SNN_CATCH(h)
}

uint32_t snn_lattice_ipc_blob_size(void) { return (uint32_t)sizeof(snn::IpcBlob); }
int32_t snn_lattice_ipc_export(snn_lattice_t *h, void *blob) {
    if (!h || !blob) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->ipc_export((snn::IpcBlob *)blob); SNN_CATCH(h)
}
int32_t snn_lattice_ipc_attach(snn_lattice_t *h, int32_t direction, const void *blob) {
    if (!h || !blob) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->attach_strip(direction, (const snn::IpcBlob *)blob, nullptr); SNN_CATCH(h)
}
int32_t snn_lattice_attach_local(snn_lattice_t *h, int32_t direction, snn_lattice_t *neighbour) {
    if (!h || !neighbour) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->attach_strip(direction, nullptr, neighbour->e); SNN_CATCH(h)
}
int32_t snn_lattice_gpart_wants(snn_lattice_t *h, int32_t peer, uint32_t *global_idx, uint64_t capacity, uint64_t *n, uint32_t *first_slot) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->gpart_wants(peer, global_idx, capacity, n, first_slot); SNN_CATCH(h)
}
int32_t snn_lattice_gpart_set_exports(snn_lattice_t *h, int32_t peer, const uint32_t *global_idx, uint64_t n, uint32_t first_slot_at_peer) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->gpart_set_exports(peer, global_idx, n, first_slot_at_peer); SNN_CATCH(h)
}
int32_t snn_lattice_gpart_attach(snn_lattice_t *h, int32_t peer, const void *blob) {
    if (!h || !blob) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->gpart_attach(peer, (const snn::IpcBlob *)blob, nullptr); SNN_CATCH(h)
}
int32_t snn_lattice_gpart_attach_local(snn_lattice_t *h, int32_t peer, snn_lattice_t *peer_handle) {
    if (!h || !peer_handle) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->gpart_attach(peer, nullptr, peer_handle->e); SNN_CATCH(h)
}

// ---------------------------------------------------------------------------------------------- network
int32_t snn_network_create(const snn_network_desc_t *desc, snn_network_t **out) {
    if (out) *out = nullptr;
    if (!desc || !out || desc->struct_size != sizeof(snn_network_desc_t)) { g_create_error = "bad descriptor"; return SNN_INVALID_ARGUMENT; }
    if (!valid_enums(desc->model, desc->nt_kinetics, desc->receptor_kinetics) || desc->spike_train < 0 ||
        desc->spike_train > SNN_TRAIN_PRESET || desc->refractoriness < 0 || desc->refractoriness > SNN_REFRACT_EXPONENTIAL_DECAY) {
        g_create_error = "bad enum in descriptor";
        return SNN_INVALID_ARGUMENT;
    }
    try {
        Engine *e = new Engine(desc->model, desc->nt_kinetics, desc->receptor_kinetics, desc->spike_train, desc->refractoriness, desc->device);
        int r = e->init();
        if (r) { g_create_error = e->last_error; delete e; return r; }
        e->is_network = true;
        *out = new snn_network{e};
        return SNN_OK;
    } catch (...) { g_create_error = "allocation failed"; return SNN_GPU_BUFFER_CREATE_ERROR; }
}
int32_t snn_network_destroy(snn_network_t *h) {
    if (!h) return SNN_OK;
    delete h->e; delete h;
    return SNN_OK;
}
int32_t snn_network_add_lattice(snn_network_t *h, uint64_t id, uint32_t rows, uint32_t cols) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->add_lattice(id, rows, cols, false); SNN_CATCH(h)
}
int32_t snn_network_add_spike_train_lattice(snn_network_t *h, uint64_t id, uint32_t rows, uint32_t cols) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->add_lattice(id, rows, cols, true); SNN_CATCH(h)
}
int32_t snn_network_lattice_size(const snn_network_t *h, uint64_t id, uint64_t *n) {
    if (!h || !n) return SNN_INVALID_ARGUMENT;
    const snn::Lat *L = h->e->find(id);
    if (!L) return SNN_NET_ID_NOT_FOUND_IN_LATTICES;
    *n = L->n;
    return SNN_OK;
}
int32_t snn_network_field_count(const snn_network_t *h, uint64_t id, uint32_t *count) {
    if (!h || !count) return SNN_INVALID_ARGUMENT;
    return h->e->field_count(id, count);
}
int32_t snn_network_field_info(const snn_network_t *h, uint64_t id, uint32_t index, const char **name, int32_t *dtype, uint32_t *per) {
    if (!h || !name || !dtype || !per) return SNN_INVALID_ARGUMENT;
    return h->e->field_info(id, index, name, dtype, per);
}
int32_t snn_network_set_field(snn_network_t *h, uint64_t id, const char *name, const void *data, uint64_t count, int32_t dtype) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->set_field(id, name, data, count, dtype); SNN_CATCH(h)
}
int32_t snn_network_fill_field_f32(snn_network_t *h, uint64_t id, const char *name, float v) {
    if (!h) return SNN_INVALID_ARGUMENT;
    uint32_t b; memcpy(&b, &v, 4);
    SNN_TRY return h->e->fill_field(id, name, b, SNN_F32); SNN_CATCH(h)
}
int32_t snn_network_fill_field_u32(snn_network_t *h, uint64_t id, const char *name, uint32_t v) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->fill_field(id, name, v, SNN_U32); SNN_CATCH(h)
}
int32_t snn_network_fill_field_i32(snn_network_t *h, uint64_t id, const char *name, int32_t v) {
    if (!h) return SNN_INVALID_ARGUMENT;
    uint32_t b; memcpy(&b, &v, 4);
    SNN_TRY return h->e->fill_field(id, name, b, SNN_I32); SNN_CATCH(h)
}
int32_t snn_network_get_field(snn_network_t *h, uint64_t id, const char *name, void *out, uint64_t count, int32_t dtype) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->get_field(id, name, out, count, dtype); SNN_CATCH(h)
}
int32_t snn_network_set_preset_firing_times(snn_network_t *h, uint64_t id, const uint64_t *offsets, const float *times,
                                            uint64_t n_trains, uint64_t n_times) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->set_preset_firing_times(id, offsets, times, n_trains, n_times); SNN_CATCH(h)
}
int32_t snn_network_connect_dense(snn_network_t *h, uint64_t pre_id, uint64_t post_id, const uint32_t *connections,
                                  const float *weights, uint64_t n_pre, uint64_t n_post) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->connect_dense(pre_id, post_id, connections, weights, nullptr, n_pre, n_post); SNN_CATCH(h)
}
int32_t snn_network_connect_csr(snn_network_t *h, uint64_t pre_id, uint64_t post_id, const uint64_t *row_ptr, const uint32_t *pre,
                                const float *weights, uint64_t n_post, uint64_t nnz) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->connect_csr(pre_id, post_id, row_ptr, pre, weights, n_post, nnz); SNN_CATCH(h)
}
int32_t snn_network_connection_nnz(snn_network_t *h, uint64_t pre_id, uint64_t post_id, uint64_t *nnz) {
    if (!h || !nnz) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->connection_nnz(pre_id, post_id, nnz); SNN_CATCH(h)
}
int32_t snn_network_get_connection_dense(snn_network_t *h, uint64_t pre_id, uint64_t post_id, uint32_t *connections, float *weights,
                                         uint64_t n_pre, uint64_t n_post) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->get_connection_dense(pre_id, post_id, connections, weights, n_pre, n_post); SNN_CATCH(h)
}
int32_t snn_network_lookup_weight(snn_network_t *h, uint64_t pre_id, uint64_t post_id, uint64_t pre, uint64_t post, float *weight,
                                  int32_t *connected) {
    if (!h || !weight || !connected) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->lookup_weight(pre_id, post_id, pre, post, weight, connected); SNN_CATCH(h)
}
int32_t snn_network_edit_weight(snn_network_t *h, uint64_t pre_id, uint64_t post_id, uint64_t pre, uint64_t post, int32_t connected,
                                float weight) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY
    snn::Lat *B;   // LatticeNetwork::connect's id checks (neuron/mod.rs:1852-1862) before the graph's position checks
    if (!(B = h->e->find(post_id))) return h->e->fail(SNN_NET_POSTSYNAPTIC_ID_NOT_FOUND, "Postsynaptic id not present in network, id: " + std::to_string(post_id));
    if (B->is_train) return h->e->fail(SNN_NET_POSTSYNAPTIC_LATTICE_CANNOT_BE_SPIKE_TRAIN, "Postsynaptic lattice cannot be a spike train lattice because spike trains cannot take inputs");
    if (!h->e->find(pre_id)) return h->e->fail(SNN_NET_PRESYNAPTIC_ID_NOT_FOUND, "Presynaptic id not present in network, id: " + std::to_string(pre_id));
    return h->e->edit_weight(pre_id, post_id, pre, post, connected != 0, weight);
    SNN_CATCH(h)
}
int32_t snn_network_get_spike_aggregate(snn_network_t *h, uint64_t id, int64_t *out, uint64_t capacity) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->get_spike_aggregate(id, out, capacity); SNN_CATCH(h)
}
int32_t snn_network_set_option(snn_network_t *h, int32_t option, int64_t value) {
    if (!h) return SNN_INVALID_ARGUMENT;
    return engine_set_option(h->e, false, 0, option, value);
}
int32_t snn_network_get_option(const snn_network_t *h, int32_t option, int64_t *value) {
    if (!h || !value) return SNN_INVALID_ARGUMENT;
    return engine_get_option(h->e, false, 0, option, value);
}
int32_t snn_network_set_lattice_option(snn_network_t *h, uint64_t id, int32_t option, int64_t value) {
    if (!h) return SNN_INVALID_ARGUMENT;
    return engine_set_option(h->e, true, id, option, value);
}
int32_t snn_network_get_lattice_option(const snn_network_t *h, uint64_t id, int32_t option, int64_t *value) {
    if (!h || !value) return SNN_INVALID_ARGUMENT;
    return engine_get_option(h->e, true, id, option, value);
}
int32_t snn_network_set_plasticity(snn_network_t *h, uint64_t id, const snn_stdp_t *stdp) {
    if (!h || !stdp) return SNN_INVALID_ARGUMENT;
    snn::Lat *L = h->e->find(id);
    if (!L || L->is_train) return h->e->fail(SNN_NET_ID_NOT_FOUND_IN_LATTICES, "Id not present in lattices, id: " + std::to_string(id));
    L->stdp = *stdp;
    return SNN_OK;
}
int32_t snn_network_set_dt(snn_network_t *h, float dt) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->set_dt(dt); SNN_CATCH(h)
}
int32_t snn_network_reset_timing(snn_network_t *h) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->reset_timing(); SNN_CATCH(h)
}
int32_t snn_network_run(snn_network_t *h, uint64_t iterations) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->run(iterations, nullptr, nullptr); SNN_CATCH(h)
}
int32_t snn_network_get_connection_csr(snn_network_t *h, uint64_t pre_id, uint64_t post_id, uint64_t *row_ptr, uint32_t *pre, float *weights,
                                       uint64_t n_post, uint64_t nnz) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->get_connection_csr(pre_id, post_id, row_ptr, pre, weights, n_post, nnz); SNN_CATCH(h)
}
int32_t snn_network_add_reward_modulated_lattice(snn_network_t *h, uint64_t id, uint32_t rows, uint32_t cols) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->add_lattice(id, rows, cols, false, true); SNN_CATCH(h)
}
int32_t snn_network_set_reward_modulator(snn_network_t *h, uint64_t id, int32_t do_modulation, const snn_rstdp_t *modulator) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->set_lattice_reward_modulator(id, do_modulation != 0, modulator); SNN_CATCH(h)
}
int32_t snn_network_get_reward_modulator(snn_network_t *h, uint64_t id, int32_t *do_modulation, snn_rstdp_t *modulator) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->get_lattice_reward_modulator(id, do_modulation, modulator); SNN_CATCH(h)
}
int32_t snn_network_set_connection_reward_modulated(snn_network_t *h, uint64_t pre_id, uint64_t post_id, int32_t reward_modulated) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->set_connection_reward(pre_id, post_id, reward_modulated != 0); SNN_CATCH(h)
}
int32_t snn_network_run_with_rewards(snn_network_t *h, const float *rewards, uint64_t n_rewards) {
    if (!h || (n_rewards && !rewards)) return SNN_INVALID_ARGUMENT;
    if (!h->e->has_reward_lattices()) return h->e->fail(SNN_INVALID_ARGUMENT, "network holds no reward-modulated lattice");
    SNN_TRY return h->e->run(n_rewards, nullptr, nullptr, rewards); SNN_CATCH(h)
}
int32_t snn_network_get_connection_traces(snn_network_t *h, uint64_t pre_id, uint64_t post_id, uint32_t *counter, float *dw, float *c,
                                          uint64_t nnz) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->get_block_traces(pre_id, post_id, counter, dw, c, nnz); SNN_CATCH(h)
}
int32_t snn_network_set_connection_traces(snn_network_t *h, uint64_t pre_id, uint64_t post_id, const float *weight, const uint32_t *counter,
                                          const float *dw, const float *c, uint64_t nnz) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->set_block_traces(pre_id, post_id, weight, counter, dw, c, nnz); SNN_CATCH(h)
}
int32_t snn_network_run_timed(snn_network_t *h, uint64_t iterations, float *elapsed_ms, uint64_t *kernel_launches) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->run(iterations, elapsed_ms, kernel_launches); SNN_CATCH(h)
}
int32_t snn_network_history_len(const snn_network_t *h, uint64_t id, uint64_t *steps) {
    if (!h || !steps) return SNN_INVALID_ARGUMENT;
    return h->e->history_len(id, steps);
}
int32_t snn_network_get_grid_history(snn_network_t *h, uint64_t id, float *out, uint64_t capacity_floats) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->get_grid_history(id, out, capacity_floats); SNN_CATCH(h)
}
int32_t snn_network_get_average_history(snn_network_t *h, uint64_t id, float *out, uint64_t capacity_floats) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->get_reduced_history(id, false, out, capacity_floats); SNN_CATCH(h)
}
int32_t snn_network_set_eeg_parameters(snn_network_t *h, uint64_t id, float reference_voltage, float distance, float conductivity) {
    if (!h) return SNN_INVALID_ARGUMENT;
    return h->e->set_eeg_parameters(id, reference_voltage, distance, conductivity);
}
int32_t snn_network_get_eeg_history(snn_network_t *h, uint64_t id, float *out, uint64_t capacity_floats) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->get_reduced_history(id, true, out, capacity_floats); SNN_CATCH(h)
}
int32_t snn_network_get_spike_history(snn_network_t *h, uint64_t id, uint8_t *out, uint64_t capacity_bytes) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->get_spike_history(id, out, capacity_bytes); SNN_CATCH(h)
}
int32_t snn_network_reset_history(snn_network_t *h) {
    if (!h) return SNN_INVALID_ARGUMENT;
    return h->e->reset_history();
}
int32_t snn_network_graph_history_len(snn_network_t *h, uint64_t pre_id, uint64_t post_id, uint64_t *steps, uint64_t *nnz) {
    if (!h || !steps || !nnz) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->graph_history_len(pre_id, post_id, steps, nnz); SNN_CATCH(h)
}
int32_t snn_network_get_graph_history(snn_network_t *h, uint64_t pre_id, uint64_t post_id, float *out, uint64_t capacity_floats) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->get_graph_history(pre_id, post_id, out, capacity_floats); SNN_CATCH(h)
}
int32_t snn_network_spike_event_count(const snn_network_t *h, uint64_t id, uint64_t *steps, uint64_t *n_events) {
    if (!h || !steps || !n_events) return SNN_INVALID_ARGUMENT;
    return h->e->spike_event_count(id, steps, n_events);
}
int32_t snn_network_get_spike_events(snn_network_t *h, uint64_t id, uint64_t *step_ptr, uint32_t *neuron, uint64_t capacity) {
    if (!h) return SNN_INVALID_ARGUMENT;
    SNN_TRY return h->e->get_spike_events(id, step_ptr, neuron, capacity); SNN_CATCH(h)
}

}  // extern "C"
