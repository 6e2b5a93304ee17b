/*
 * snn_b200.h — C ABI of the B200-native lattice stepping engine.
 *
 * This is the drop-in boundary for the hot path behind the reference's
 * `Lattice::run_lattice` / `LatticeNetwork::run_lattices`
 * (backend/src/neuron/mod.rs:1199-1220, 2654-2675).  The shape mirrors the
 * reference's own accelerator boundary, `LatticeGPU` / `LatticeNetworkGPU`
 * (backend/src/neuron/gpu_lattices/mod.rs:327-511, 1081-1100, 1560-1656,
 * 3183-3212): host code owns neuron structs, flattens them row-major into one
 * named structure-of-arrays buffer per struct field
 * (`IterateAndSpikeGPU::convert_to_gpu`, iterate_and_spike/mod.rs:3156-3189;
 * `flatten_and_retrieve_field!`, :2438-2459), hands over the graph, calls run,
 * and reads the fields back.
 *
 * Rules of the boundary
 *  - plain pointers and sizes only; every host pointer is borrowed for the
 *    duration of the call;
 *  - no exceptions/aborts cross it: every function returns an int32 status;
 *  - status 1..8 are the reference's `GPUError` variants in declaration order
 *    (backend/src/error/mod.rs:221-238); 16.. are `GraphError`
 *    (error/mod.rs:15-20); 32.. are `LatticeNetworkError` (error/mod.rs:38-48);
 *  - a handle is NOT thread-safe (the reference's types are not Send/Sync
 *    either); one caller at a time;
 *  - there is NO CPU fallback: if no CUDA device is usable, create() returns
 *    SNN_GPU_GET_DEVICE_FAILURE;
 *  - empty lattices and 0 iterations are no-ops that return SNN_OK
 *    (gpu_lattices/mod.rs:1089-1091, 3196-3203).
 *
 * Field names and dtypes follow the reference's buffer map: f32 for floats,
 * u32 for bools, i32 for `Option<usize>` with -1 = None
 * (iterate_and_spike/mod.rs:3112-3134, 2453-2457).  Per-type chemical fields
 * are sized n*3 neuron-major, type order AMPA=0, NMDA=1, GABA=2
 * (iterate_and_spike/mod.rs:1322-1334, 2566-2656).
 */
#ifndef SNN_B200_H
#define SNN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define SNN_API __attribute__((visibility("default")))
#else
#define SNN_API
#endif

#define SNN_B200_ABI_VERSION 1

/* ---------------------------------------------------------------- status */
typedef enum snn_status {
    SNN_OK = 0,
    /* GPUError, backend/src/error/mod.rs:221-238 */
    SNN_GPU_PROGRAM_COMPILE_FAILURE = 1,
    SNN_GPU_KERNEL_COMPILE_FAILURE = 2,
    SNN_GPU_BUFFER_CREATE_ERROR = 3,
    SNN_GPU_BUFFER_WRITE_ERROR = 4,
    SNN_GPU_BUFFER_READ_ERROR = 5,
    SNN_GPU_WAIT_ERROR = 6,
    SNN_GPU_GET_DEVICE_FAILURE = 7,
    SNN_GPU_QUEUE_FAILURE = 8,
    /* GraphError, backend/src/error/mod.rs:15-20 */
    SNN_GRAPH_PRESYNAPTIC_NOT_FOUND = 16,
    SNN_GRAPH_POSTSYNAPTIC_NOT_FOUND = 17,
    SNN_GRAPH_POSITION_NOT_FOUND = 18,
    SNN_GRAPH_DIMENSIONS_DO_NOT_MATCH = 19,
    /* LatticeNetworkError, backend/src/error/mod.rs:38-48 */
    SNN_NET_GRAPH_ID_ALREADY_PRESENT = 32,
    SNN_NET_POSTSYNAPTIC_ID_NOT_FOUND = 33,
    SNN_NET_PRESYNAPTIC_ID_NOT_FOUND = 34,
    SNN_NET_ID_NOT_FOUND_IN_LATTICES = 35,
    SNN_NET_POSTSYNAPTIC_LATTICE_CANNOT_BE_SPIKE_TRAIN = 36,
    /* the RewardModulatedLatticeNetwork members of LatticeNetworkError, backend/src/error/mod.rs:55-62 */
    SNN_NET_CANNOT_CONNECT_WITH_REWARD_MODULATED_CONNECTION = 37,
    SNN_NET_REWARD_MODULATED_CONNECTION_NOT_COMPATIBLE_INTERNALLY = 38,
    SNN_NET_CONNECT_FUNCTION_MUST_HAVE_NON_REWARD_MODULATED_LATTICE = 39,
    /* argument errors of the C boundary itself (Rust's type system rules these out) */
    SNN_INVALID_ARGUMENT = 64,
    SNN_UNKNOWN_FIELD = 65,
    SNN_DTYPE_MISMATCH = 66,
    SNN_SIZE_MISMATCH = 67,
    SNN_UNSUPPORTED = 68
} snn_status_t;

/* ---------------------------------------------------------------- enums */
/* neuron models: backend/src/neuron/integrate_and_fire/mod.rs, hodgkin_huxley/mod.rs */
typedef enum snn_model {
    SNN_MODEL_LEAKY_INTEGRATE_AND_FIRE = 0,       /* :106-215   */
    SNN_MODEL_QUADRATIC_INTEGRATE_AND_FIRE = 1,   /* :257-365   */
    SNN_MODEL_ADAPTIVE_LEAKY_INTEGRATE_AND_FIRE = 2,     /* :919-1051  */
    SNN_MODEL_ADAPTIVE_EXP_LEAKY_INTEGRATE_AND_FIRE = 3, /* :1053-1155 */
    SNN_MODEL_IZHIKEVICH = 4,                     /* :1157-1268 */
    SNN_MODEL_LEAKY_IZHIKEVICH = 5,               /* :1270-1356 */
    SNN_MODEL_SIMPLE_LEAKY_INTEGRATE_AND_FIRE = 6,/* :1522-1630 */
    SNN_MODEL_HODGKIN_HUXLEY = 7,                 /* hodgkin_huxley/mod.rs:48-242 */
    SNN_MODEL_BCM_IZHIKEVICH = 8,                 /* :1358-1520 (Izhikevich + BCMActivity bookkeeping) */
    SNN_MODEL_COUNT = 9
} snn_model_t;

/* NeurotransmitterKinetics impls, iterate_and_spike/mod.rs:122-366 */
typedef enum snn_nt_kinetics {
    SNN_NT_APPROXIMATE = 0,       /* :165-205 */
    SNN_NT_DESTEXHE = 1,          /* :125-159 */
    SNN_NT_DISCRETE_SPIKE = 2,    /* :294-322 */
    SNN_NT_EXPONENTIAL_DECAY = 3  /* :329-366 */
} snn_nt_kinetics_t;

/* ReceptorKinetics impls, iterate_and_spike/mod.rs:391-533 */
typedef enum snn_receptor_kinetics {
    SNN_RC_APPROXIMATE = 0,       /* :430-446 */
    SNN_RC_DESTEXHE = 1,          /* :394-425 */
    SNN_RC_EXPONENTIAL_DECAY = 2  /* :501-533 */
} snn_receptor_kinetics_t;

/* SpikeTrain impls, spike_train/mod.rs */
typedef enum snn_spike_train {
    SNN_TRAIN_POISSON = 0,  /* :253-371  */
    SNN_TRAIN_RATE = 1,     /* :980-1033 */
    SNN_TRAIN_PRESET = 2    /* :752-828  */
} snn_spike_train_t;

/* NeuralRefractoriness impls, spike_train/mod.rs:37-180 */
typedef enum snn_refractoriness {
    SNN_REFRACT_DELTA_DIRAC = 0,
    SNN_REFRACT_EXPONENTIAL_DECAY = 1
} snn_refractoriness_t;

typedef enum snn_dtype { SNN_F32 = 0, SNN_U32 = 1, SNN_I32 = 2 } snn_dtype_t;

/* neurotransmitter type slots (IonotropicNeurotransmitterType, iterate_and_spike/mod.rs:1068-1073) */
#define SNN_NUM_NT_TYPES 3
#define SNN_NT_AMPA 0
#define SNN_NT_NMDA 1
#define SNN_NT_GABA 2

/* public bool / scalar members of Lattice (neuron/mod.rs:556-587) and
 * LatticeNetwork (neuron/mod.rs:1554-1563) */
typedef enum snn_option {
    SNN_OPT_ELECTRICAL_SYNAPSE = 0,   /* default 1 */
    SNN_OPT_CHEMICAL_SYNAPSE = 1,     /* default 0 */
    SNN_OPT_DO_PLASTICITY = 2,        /* default 0 (per lattice) */
    SNN_OPT_UPDATE_GRID_HISTORY = 3,  /* default 0 (per lattice): GridVoltageHistory, neuron/mod.rs:286-301 */
    SNN_OPT_UPDATE_SPIKE_HISTORY = 4, /* default 0 (per lattice): SpikeHistory raster, neuron/mod.rs:324-378 */
    SNN_OPT_INTERNAL_CLOCK = 5,       /* usize clock, persists across run calls */
    SNN_OPT_PARALLEL = 6,             /* accepted for API parity; the device path is always parallel */
    SNN_OPT_RNG_SEED = 7,             /* Philox key for Poisson spike trains (reference: unseeded thread_rng).  Default: a distinct key per
                                         handle; the counter is (train, per-handle draw number) and is NOT reset by reset_timing, so repeated
                                         presentations see fresh noise */
    SNN_OPT_UPDATE_AVERAGE_HISTORY = 8, /* AverageVoltageHistory, neuron/mod.rs:303-322 */
    SNN_OPT_STEPS_PER_GRAPH = 9,      /* timesteps per kernel launch for lattices / networks that the one-launch-per-step kernels leave
                                         launch-bound (whole-GPU handles below ~10^6 neurons that are not stepped by the TMA-staged
                                         kernels): 0 (default) = a whole run (or history chunk) per cooperative launch with a grid-wide
                                         barrier between timesteps, 1 = one launch per timestep, k = at most k.  Results are
                                         bit-identical for every value. */
    SNN_OPT_UPDATE_EEG_HISTORY = 10,  /* default 0 (per lattice): EEGHistory, neuron/mod.rs:231-284 */
    SNN_OPT_GENERAL_PARTITION = 12,   /* partitioned handles: the next snn_lattice_set_graph_csr builds gather-list ghosts (general-graph
                                         partition) even if this rank's edges happen to stay inside the strip halo — set it on EVERY
                                         rank when any rank's graph reaches further (the mode must be the same on all ranks) */
    SNN_OPT_HALO_TIMEOUT_MS = 11,     /* partitioned handles: bound of one in-kernel wait for a neighbouring strip (default 30000);
                                         run() first meets the neighbours on the host (4x this bound) before any step is enqueued */
    SNN_OPT_UPDATE_GRAPH_HISTORY = 13,  /* default 0 (per lattice): Graph::update_history of the lattice's own graph (graph/mod.rs:278-284),
                                           one record per step, read with snn_lattice_get_graph_history / snn_network_get_graph_history */
    SNN_OPT_UPDATE_CONNECTING_GRAPH_HISTORY = 14, /* default 0 (network-wide): LatticeNetwork::update_connecting_graph_history, one
                                                     record per step of every connecting block (pre_id != post_id) */
    SNN_OPT_UPDATE_SPIKE_EVENTS = 15, /* default 0 (per lattice, spike-train lattices included): one record per step of the cells that
                                         spiked, compacted on the device; read with snn_lattice_get_spike_events /
                                         snn_network_get_spike_events.  Independent of SNN_OPT_UPDATE_SPIKE_HISTORY */
    SNN_OPT_STEP_PATH = 16,           /* read-only: the step path of the handle's last run / run_timed / run_with_rewards, path + 16 * multi.
                                         path: 0 nothing run yet, 1 general (one thread per neuron), 2 wide (one CTA per slice),
                                         3 wide split (per-edge terms pass, then ordered sums), 4 TMA-staged persistent kernel,
                                         5 window-staged persistent kernel (radius-1 stencils).  multi: 1 when whole chunks of
                                         timesteps ran in one cooperative launch (SNN_OPT_STEPS_PER_GRAPH) */
    SNN_OPT_UNIFORM_TILES = 17,       /* read-only: of the 256-neuron tiles of the handle's last run on the window-staged kernel, those
                                         whose neurons all have the bit patterns of the tile's first neuron in every parameter the step
                                         reads (these tiles read one copy of them instead of one per neuron); 0 on every other path */
    SNN_OPT_STENCIL_TILES = 18        /* read-only: of the 256-neuron tiles of the handle's last run on the window-staged kernel, those
                                         that derived their in-edge indices from the radius-1 stencil instead of reading the edge table's
                                         index words: every tile when every tile reads its parameter row and every index word of the table
                                         is the stencil's, bit for bit (type bits included); else 0, as on every other path */
} snn_option_t;

/* STDP, backend/src/neuron/plasticity/mod.rs:14-39 (defaults 2, 2, 4.5, 4.5, 0.1) */
typedef struct snn_stdp {
    float a_plus;
    float a_minus;
    float tau_plus;
    float tau_minus;
    float dt;
} snn_stdp_t;

/* BCM, backend/src/neuron/plasticity/mod.rs:80-97 (defaults 0.1, 0.1, 0.1) */
typedef struct snn_bcm {
    float decay;
    float average_scalar;
    float dt;
} snn_bcm_t;

/* RewardModulatedSTDP, backend/src/neuron/plasticity/mod.rs:155-189 (defaults 0, 20, 0.0001, 2, 2, 4.5, 4.5, 0.1).  Its weights
 * are TraceRSTDP values {counter, dw, weight, c} (:121-136): `weight` is the ordinary edge weight of the graph calls, the other
 * three members are read with snn_lattice_get_connection_traces. */
typedef struct snn_rstdp {
    float dopamine;
    float tau_d;
    float tau_c;
    float a_plus;
    float a_minus;
    float tau_plus;
    float tau_minus;
    float dt;
} snn_rstdp_t;

typedef struct snn_lattice_desc {
    uint32_t struct_size;       /* = sizeof(snn_lattice_desc_t) */
    int32_t model;              /* snn_model_t */
    int32_t nt_kinetics;        /* snn_nt_kinetics_t */
    int32_t receptor_kinetics;  /* snn_receptor_kinetics_t */
    uint32_t rows;
    uint32_t cols;
    int32_t device;             /* CUDA ordinal; -1 = current device */
    /* multi-GPU row-strip partition (SURVEY §8e); world = 1 for a whole lattice.
     * rows/cols are the GLOBAL grid; this handle owns rows
     * [snn_partition_begin(rows, world, rank), snn_partition_begin(rows, world, rank+1)). */
    int32_t part_rank;
    int32_t part_world;
} snn_lattice_desc_t;

typedef struct snn_lattice snn_lattice_t;
typedef struct snn_network snn_network_t;

/* ---------------------------------------------------------------- library */
SNN_API int32_t snn_abi_version(void);
SNN_API const char *snn_status_string(int32_t status);
/* last error text recorded on this handle (or the thread's last create() failure when h == NULL) */
SNN_API const char *snn_lattice_last_error(const snn_lattice_t *h);
SNN_API const char *snn_network_last_error(const snn_network_t *h);
/* number of CUDA devices visible; returns SNN_GPU_GET_DEVICE_FAILURE when there is none */
SNN_API int32_t snn_device_count(int32_t *count);

/* ---------------------------------------------------------------- lattice
 * Replaces LatticeGPU (gpu_lattices/mod.rs:327-511) + its RunLattice impl (:1081-1100). */

/* LatticeGPU::try_default + populate(base_neuron, rows, cols) (gpu_lattices/mod.rs:395-408):
 * every field of every neuron starts at the model's Default (e.g. IzhikevichNeuron::default,
 * integrate_and_fire/mod.rs:1198-1220); nodes are added row-major so graph index == i*cols+j. */
SNN_API int32_t snn_lattice_create(const snn_lattice_desc_t *desc, snn_lattice_t **out);
SNN_API int32_t snn_lattice_destroy(snn_lattice_t *h);

SNN_API int32_t snn_lattice_rows(const snn_lattice_t *h, uint32_t *rows_local, uint32_t *cols);
/* number of neurons this handle owns (rows_local*cols) */
SNN_API int32_t snn_lattice_size(const snn_lattice_t *h, uint64_t *n);

/* field directory: the reference's HashMap<String, BufferGPU> keys for the lattice's neuron type */
SNN_API int32_t snn_lattice_field_count(const snn_lattice_t *h, uint32_t *count);
SNN_API int32_t snn_lattice_field_info(const snn_lattice_t *h, uint32_t index, const char **name,
                                       int32_t *dtype, uint32_t *per_neuron);

/* write one named SoA field for all owned neurons (convert_to_gpu, integrate_and_fire/mod.rs:729-773).
 * count must be n*per_neuron.  Equivalent of Lattice::apply / set_cell_grid for that field. */
SNN_API int32_t snn_lattice_set_field(snn_lattice_t *h, const char *name, const void *data,
                                      uint64_t count, int32_t dtype);
/* broadcast one scalar to the whole field (populate with a modified base neuron) */
SNN_API int32_t snn_lattice_fill_field_f32(snn_lattice_t *h, const char *name, float value);
SNN_API int32_t snn_lattice_fill_field_u32(snn_lattice_t *h, const char *name, uint32_t value);
SNN_API int32_t snn_lattice_fill_field_i32(snn_lattice_t *h, const char *name, int32_t value);
/* read one named field back (convert_to_cpu, integrate_and_fire/mod.rs:776-917) */
SNN_API int32_t snn_lattice_get_field(snn_lattice_t *h, const char *name, void *out, uint64_t count,
                                      int32_t dtype);

/* Graph ingestion.  `n` is the number of graph nodes and must equal the lattice size.
 * dense = the reference's GraphGPU layout (graph/mod.rs:88-93, 300-361): connections[pre*n+post] in
 * {0,1}, weights[pre*n+post], index_to_position[n] graph index -> flat cell index (NULL = identity). */
SNN_API int32_t snn_lattice_set_graph_dense(snn_lattice_t *h, const uint32_t *connections,
                                            const float *weights, const uint32_t *index_to_position,
                                            uint32_t n);
/* CSR by postsynaptic neuron: in-edges of post p are pre[row_ptr[p]..row_ptr[p+1]).  For a
 * partitioned handle rows are the owned neurons and pre holds GLOBAL flat indices. */
SNN_API int32_t snn_lattice_set_graph_csr(snn_lattice_t *h, const uint64_t *row_ptr, const uint32_t *pre,
                                          const float *weights, uint64_t n, uint64_t nnz);
/* structured generator for `connect` predicates of the form max(|dr|,|dc|) <= radius && x != y
 * (Moore neighbourhood, non-periodic), every weight = `weight` (connect(.., None) gives 1.0,
 * neuron/mod.rs:1134-1157).  Built on the device; the only way to reach 10^7 neurons. */
SNN_API int32_t snn_lattice_set_graph_grid(snn_lattice_t *h, uint32_t radius, float weight);
SNN_API int32_t snn_lattice_graph_nnz(snn_lattice_t *h, uint64_t *nnz);
/* canonical CSR (pre ascending inside each row) with the current weights; any pointer may be NULL */
SNN_API int32_t snn_lattice_get_graph_csr(snn_lattice_t *h, uint64_t *row_ptr, uint32_t *pre, float *weights,
                                          uint64_t n, uint64_t nnz);
SNN_API int32_t snn_lattice_get_graph_dense(snn_lattice_t *h, uint32_t *connections, float *weights, uint32_t n);
/* Graph::lookup_weight on flat indices (graph/mod.rs:196-206); *connected = 0 for None.  Reads one row of the device table. */
SNN_API int32_t snn_lattice_lookup_weight(snn_lattice_t *h, uint64_t pre, uint64_t post, float *weight,
                                          int32_t *connected);
/* Graph::edit_weight(pre, post, Option<f32>) (graph/mod.rs:208-226): connected = 0 is None (the edge is removed), else
 * Some(weight).  Same error order as the reference (postsynaptic position first).  Some(w) over an existing edge is one word
 * written on the device; adding or removing an edge edits the host CSR and the device table is rebuilt at the next run
 * (whole-lattice handles only). */
SNN_API int32_t snn_lattice_edit_weight(snn_lattice_t *h, uint64_t pre, uint64_t post, int32_t connected, float weight);
/* Graph::get_incoming_connections over the postsynaptic positions [row_begin, row_end) (graph/mod.rs:228-256), with the current
 * weights: CSR decoded from the device table without downloading the whole graph.  row_ptr has row_end - row_begin + 1
 * entries; pre / weights hold up to `capacity` edges (either may be NULL to count only); *nnz = edges in the range. */
SNN_API int32_t snn_lattice_get_graph_rows(snn_lattice_t *h, uint64_t row_begin, uint64_t row_end, uint64_t *row_ptr, uint32_t *pre,
                                           float *weights, uint64_t capacity, uint64_t *nnz);

SNN_API int32_t snn_lattice_set_option(snn_lattice_t *h, int32_t option, int64_t value);
SNN_API int32_t snn_lattice_get_option(const snn_lattice_t *h, int32_t option, int64_t *value);
SNN_API int32_t snn_lattice_set_plasticity(snn_lattice_t *h, const snn_stdp_t *stdp);
SNN_API int32_t snn_lattice_get_plasticity(const snn_lattice_t *h, snn_stdp_t *stdp);
/* Lattice::set_dt (neuron/mod.rs:649-652): every neuron's dt and the plasticity rule's dt */
SNN_API int32_t snn_lattice_set_dt(snn_lattice_t *h, float dt);
/* Lattice::reset_timing (neuron/mod.rs:405-420): clock = 0, every last_firing_time = None */
SNN_API int32_t snn_lattice_reset_timing(snn_lattice_t *h);

/* RunLattice::run_lattice (neuron/mod.rs:1209-1219 / gpu_lattices/mod.rs:1088-1099). Blocks. */
SNN_API int32_t snn_lattice_run(snn_lattice_t *h, uint64_t iterations);
/* same, additionally returns the device time of the step loop measured with CUDA events on the
 * engine's own stream, and the number of kernels launched inside it */
SNN_API int32_t snn_lattice_run_timed(snn_lattice_t *h, uint64_t iterations, float *elapsed_ms,
                                      uint64_t *kernel_launches);

/* Lattice<BCMIzhikevichNeuron, ..., BCM, ...>: the plasticity rule of the lattice becomes BCM (plasticity/mod.rs:99-111, triggered
 * by spiking neurons like STDP: every in-edge and out-edge of a neuron that spiked, using the BCMActivity values of both
 * ends).  SNN_OPT_DO_PLASTICITY keeps switching plasticity on and off.  SNN_MODEL_BCM_IZHIKEVICH `Lattice` handles: whole lattices,
 * row strips and general-graph partitions (an edge whose presynaptic neuron lives on another rank is updated by the rank that owns
 * its postsynaptic row, from that neuron's spike time and current_activity exported after every step).  May be called before or
 * after the partition is attached.  A reward modulator, when enabled, takes precedence. */
SNN_API int32_t snn_lattice_set_bcm_plasticity(snn_lattice_t *h, int32_t enable, const snn_bcm_t *bcm);

/* RewardModulatedLattice (neuron/mod.rs:2717-3416).  set_reward_modulator(enable = 1) turns the handle into a reward-modulated
 * lattice: the graph's weights become TraceRSTDP values and, while `do_modulation` is on, EVERY edge is updated twice per
 * timestep by RewardModulatedSTDP::update_weight (once from each end, plasticity/mod.rs:197-233; do_update is always true).
 * snn_lattice_run then is RunLattice::run_lattice (:3361-3374, no reward signal) and snn_lattice_run_with_rewards runs one
 * timestep per entry of `rewards`, each preceded by RewardModulatedSTDP::update(reward) (run_lattice_with_reward, :3250-3257).
 * Single-lattice handles (whole or row-strip partitioned).  Traces are reset when the graph is rebuilt. */
SNN_API int32_t snn_lattice_set_reward_modulator(snn_lattice_t *h, int32_t enable, int32_t do_modulation, const snn_rstdp_t *modulator);
SNN_API int32_t snn_lattice_get_reward_modulator(const snn_lattice_t *h, snn_rstdp_t *modulator);
SNN_API int32_t snn_lattice_run_with_rewards(snn_lattice_t *h, const float *rewards, uint64_t n_rewards);
/* TraceRSTDP members of every edge in the order of snn_lattice_get_graph_csr (counter as u32); any pointer may be NULL */
SNN_API int32_t snn_lattice_get_connection_traces(snn_lattice_t *h, uint32_t *counter, float *dw, float *c, uint64_t nnz);
/* Graph::edit_weight with whole TraceRSTDP values on every existing edge (same order; NULL = leave that member alone):
 * overwrites in place, the adjacency and the other members are kept */
SNN_API int32_t snn_lattice_set_connection_traces(snn_lattice_t *h, const float *weight, const uint32_t *counter, const float *dw,
                                                  const float *c, uint64_t nnz);

/* histories recorded on the device during run when the matching option is on.
 * grid: steps x n f32 (GridVoltageHistory); spikes: steps x n u8 (SpikeHistory);
 * average: steps f32 (AverageVoltageHistory). `steps` recorded so far via history_len. */
SNN_API int32_t snn_lattice_history_len(const snn_lattice_t *h, uint64_t *steps);
SNN_API int32_t snn_lattice_get_grid_history(snn_lattice_t *h, float *out, uint64_t capacity_floats);
SNN_API int32_t snn_lattice_get_spike_history(snn_lattice_t *h, uint8_t *out, uint64_t capacity_bytes);
SNN_API int32_t snn_lattice_get_average_history(snn_lattice_t *h, float *out, uint64_t capacity_floats);
/* SpikeHistory::aggregate (neuron/mod.rs:335-359): per neuron, the number of recorded steps in which it spiked (isize).  Counted
 * on the device from the staged raster while SNN_OPT_UPDATE_SPIKE_HISTORY is on; reset by reset_history. */
SNN_API int32_t snn_lattice_get_spike_aggregate(snn_lattice_t *h, int64_t *out, uint64_t capacity);
/* EEGHistory (neuron/mod.rs:231-284): one value per step, (1 / (4 pi conductivity distance)) * sum(V - reference_voltage).
 * Defaults 0.007 mV, 0.8 mm, 251 S/mm (EEGHistory::default, :243-252). */
SNN_API int32_t snn_lattice_set_eeg_parameters(snn_lattice_t *h, float reference_voltage, float distance, float conductivity);
SNN_API int32_t snn_lattice_get_eeg_history(snn_lattice_t *h, float *out, uint64_t capacity_floats);
SNN_API int32_t snn_lattice_reset_history(snn_lattice_t *h);
/* graph history (SNN_OPT_UPDATE_GRAPH_HISTORY): `steps` records of `nnz` f32 weights each, every record in the edge order of
 * snn_lattice_get_graph_csr.  Record k holds the weights after step k's plasticity (Lattice::iterate pushes the history at the
 * end of the step, neuron/mod.rs:973-979), so with STDP the last record equals snn_lattice_get_graph_csr after the run.  Recorded
 * on the device and drained between history chunks; while it is on, every timestep is its own launch (SNN_OPT_STEPS_PER_GRAPH = 1).
 * Cleared by reset_history (not by reset_timing).  SNN_UNSUPPORTED from run: partitioned handles and reward-modulated lattices
 * (TraceRSTDP weights); from set_graph_* and edge-adding/removing edit_weight: while the history holds records, since the
 * records assume one adjacency (edit_weight of an existing edge is allowed; reset_history lifts the restriction). */
SNN_API int32_t snn_lattice_graph_history_len(snn_lattice_t *h, uint64_t *steps, uint64_t *nnz);
SNN_API int32_t snn_lattice_get_graph_history(snn_lattice_t *h, float *out, uint64_t capacity_floats);
/* spike events (SNN_OPT_UPDATE_SPIKE_EVENTS): `steps` records, record k being the cells that spiked in the k-th recorded step (the
 * same step as row k of the spike history when both are on), `n_events` cell indices in all.  Records ascend by step and indices
 * ascend inside a record.  Indices are flat cell indices i*cols+j; a row-strip or general-graph partition records the GLOBAL flat
 * indices of its own rows.  The compaction runs on the device once per history chunk (popcount per raster word, scan, scatter);
 * only the per-record counts and the events are copied to the host.  Cleared by reset_history (not by reset_timing). */
SNN_API int32_t snn_lattice_spike_event_count(const snn_lattice_t *h, uint64_t *steps, uint64_t *n_events);
/* step_ptr: steps + 1 entries (CSR by step: record k is neuron[step_ptr[k] .. step_ptr[k+1])); neuron: up to `capacity` indices,
 * SNN_SIZE_MISMATCH when n_events exceeds it.  Either pointer may be NULL. */
SNN_API int32_t snn_lattice_get_spike_events(snn_lattice_t *h, uint64_t *step_ptr, uint32_t *neuron, uint64_t capacity);

/* ---- multi-GPU row strips (one process per GPU; plumbing by the caller, e.g. torch.distributed) */
/* first global row of `rank`'s strip; rank == world gives `rows` */
SNN_API uint32_t snn_partition_begin(uint32_t rows, int32_t world, int32_t rank);
/* bytes of the opaque blob below */
SNN_API uint32_t snn_lattice_ipc_blob_size(void);
/* export this strip's halo-visible device slab (CUDA IPC handle + layout) */
SNN_API int32_t snn_lattice_ipc_export(snn_lattice_t *h, void *blob);
/* attach the neighbouring strip: direction -1 = rank-1 (rows above), +1 = rank+1 (rows below) */
SNN_API int32_t snn_lattice_ipc_attach(snn_lattice_t *h, int32_t direction, const void *blob);
/* the same for a neighbouring strip whose handle lives in THIS process (same device, or a device with peer access): no CUDA IPC.
 * Both handles attach each other; they are then stepped concurrently from separate host threads with the same iteration
 * counts.  On a single device the strips must be small enough for their step kernels to be resident together (boundary warps
 * spin on the neighbour's progress) — meant for tests and for one process driving several GPUs. */
SNN_API int32_t snn_lattice_attach_local(snn_lattice_t *h, int32_t direction, snn_lattice_t *neighbour);

/* ---- multi-GPU, general graphs (SURVEY 8e): the same contiguous node ranges (whole rows) per rank, but in-edges from ANY node of
 * any rank.  snn_lattice_set_graph_csr with global presynaptic indices switches a partitioned handle to this mode as soon as an
 * edge reaches beyond the strip's halo rows: the ghosts then are gather lists of exactly the remote nodes the rank's rows read.
 * Set-up, per pair of ranks (the caller moves the lists and blobs, e.g. torch.distributed.all_gather_object):
 *   1. r: gpart_wants(q, idx, cap, &n, &slot)   the nodes of q that r reads (ascending global indices) and the node slot in r's
 *                                               arrays where the first of them lives
 *   2. q: gpart_set_exports(r, idx, n, slot)    q will write those nodes into r's slots after every step
 *   3. both: gpart_attach(peer, blob of snn_lattice_ipc_export) or gpart_attach_local(peer, handle in this process)
 * Every step a rank waits, where a slice reads ghosts or exports, until all its peers have completed the previous step, and
 * raises its own completion counter at every peer when its last warp is done: ranks are never more than one step apart. */
SNN_API int32_t snn_lattice_gpart_wants(snn_lattice_t *h, int32_t peer, uint32_t *global_idx, uint64_t capacity, uint64_t *n,
                                        uint32_t *first_slot);
SNN_API int32_t snn_lattice_gpart_set_exports(snn_lattice_t *h, int32_t peer, const uint32_t *global_idx, uint64_t n,
                                              uint32_t first_slot_at_peer);
SNN_API int32_t snn_lattice_gpart_attach(snn_lattice_t *h, int32_t peer, const void *blob);
SNN_API int32_t snn_lattice_gpart_attach_local(snn_lattice_t *h, int32_t peer, snn_lattice_t *peer_handle);

/* ---------------------------------------------------------------- network
 * Replaces LatticeNetworkGPU (gpu_lattices/mod.rs:1560-1656) + RunNetwork (:3183-3212); semantics
 * follow the CPU LatticeNetwork (neuron/mod.rs:1538-2675). All lattices share one neuron model and
 * all spike-train lattices one spike-train type, as the Rust generics force. */
typedef struct snn_network_desc {
    uint32_t struct_size;
    int32_t model;
    int32_t nt_kinetics;
    int32_t receptor_kinetics;
    int32_t spike_train;        /* snn_spike_train_t */
    int32_t refractoriness;     /* snn_refractoriness_t */
    int32_t device;
} snn_network_desc_t;

SNN_API int32_t snn_network_create(const snn_network_desc_t *desc, snn_network_t **out);
SNN_API int32_t snn_network_destroy(snn_network_t *h);
/* LatticeNetwork::add_lattice / add_spike_train_lattice (neuron/mod.rs:1663-1698); ids are unique */
SNN_API int32_t snn_network_add_lattice(snn_network_t *h, uint64_t id, uint32_t rows, uint32_t cols);
SNN_API int32_t snn_network_add_spike_train_lattice(snn_network_t *h, uint64_t id, uint32_t rows, uint32_t cols);
SNN_API int32_t snn_network_lattice_size(const snn_network_t *h, uint64_t id, uint64_t *n);

SNN_API int32_t snn_network_field_count(const snn_network_t *h, uint64_t id, uint32_t *count);
SNN_API int32_t snn_network_field_info(const snn_network_t *h, uint64_t id, uint32_t index, const char **name,
                                       int32_t *dtype, uint32_t *per_neuron);
SNN_API int32_t snn_network_set_field(snn_network_t *h, uint64_t id, const char *name, const void *data,
                                      uint64_t count, int32_t dtype);
SNN_API int32_t snn_network_fill_field_f32(snn_network_t *h, uint64_t id, const char *name, float value);
SNN_API int32_t snn_network_fill_field_u32(snn_network_t *h, uint64_t id, const char *name, uint32_t value);
SNN_API int32_t snn_network_fill_field_i32(snn_network_t *h, uint64_t id, const char *name, int32_t value);
SNN_API int32_t snn_network_get_field(snn_network_t *h, uint64_t id, const char *name, void *out, uint64_t count,
                                      int32_t dtype);
/* PresetSpikeTrain::firing_times (spike_train/mod.rs:768): ragged per-train lists, CSR-packed */
SNN_API int32_t snn_network_set_preset_firing_times(snn_network_t *h, uint64_t id, const uint64_t *offsets,
                                                    const float *times, uint64_t n_trains, uint64_t n_times);

/* LatticeNetwork::connect(pre_id, post_id, ..) (neuron/mod.rs:1845-1930): overwrites every
 * pre->post pair between the two lattices. pre_id == post_id sets the lattice's internal graph.
 * dense layout [pre*n_post + post]. */
SNN_API int32_t snn_network_connect_dense(snn_network_t *h, uint64_t pre_id, uint64_t post_id,
                                          const uint32_t *connections, const float *weights,
                                          uint64_t n_pre, uint64_t n_post);
/* CSR by post over the post lattice's neurons; pre = flat index inside the pre lattice */
SNN_API int32_t snn_network_connect_csr(snn_network_t *h, uint64_t pre_id, uint64_t post_id,
                                        const uint64_t *row_ptr, const uint32_t *pre, const float *weights,
                                        uint64_t n_post, uint64_t nnz);
SNN_API int32_t snn_network_connection_nnz(snn_network_t *h, uint64_t pre_id, uint64_t post_id, uint64_t *nnz);
SNN_API int32_t snn_network_get_connection_dense(snn_network_t *h, uint64_t pre_id, uint64_t post_id,
                                                 uint32_t *connections, float *weights, uint64_t n_pre,
                                                 uint64_t n_post);
/* the block in the layout of snn_network_connect_csr (row_ptr: n_post + 1 entries; nnz from snn_network_connection_nnz) */
SNN_API int32_t snn_network_get_connection_csr(snn_network_t *h, uint64_t pre_id, uint64_t post_id, uint64_t *row_ptr,
                                               uint32_t *pre, float *weights, uint64_t n_post, uint64_t nnz);

/* Graph::lookup_weight / edit_weight between two lattices of the network (or inside one when pre_id == post_id) on flat
 * indices: LatticeNetwork::connect's id errors first (neuron/mod.rs:1852-1862), then GraphError as for the lattice calls */
SNN_API int32_t snn_network_lookup_weight(snn_network_t *h, uint64_t pre_id, uint64_t post_id, uint64_t pre, uint64_t post,
                                          float *weight, int32_t *connected);
SNN_API int32_t snn_network_edit_weight(snn_network_t *h, uint64_t pre_id, uint64_t post_id, uint64_t pre, uint64_t post,
                                        int32_t connected, float weight);

/* network-wide: ELECTRICAL_SYNAPSE, CHEMICAL_SYNAPSE, INTERNAL_CLOCK, RNG_SEED, PARALLEL, UPDATE_CONNECTING_GRAPH_HISTORY */
SNN_API int32_t snn_network_set_option(snn_network_t *h, int32_t option, int64_t value);
SNN_API int32_t snn_network_get_option(const snn_network_t *h, int32_t option, int64_t *value);
/* per lattice: DO_PLASTICITY, UPDATE_GRID_HISTORY, UPDATE_SPIKE_HISTORY, UPDATE_GRAPH_HISTORY, INTERNAL_CLOCK (spike-train lattices) */
SNN_API int32_t snn_network_set_lattice_option(snn_network_t *h, uint64_t id, int32_t option, int64_t value);
SNN_API int32_t snn_network_get_lattice_option(const snn_network_t *h, uint64_t id, int32_t option, int64_t *value);
SNN_API int32_t snn_network_set_plasticity(snn_network_t *h, uint64_t id, const snn_stdp_t *stdp);
SNN_API int32_t snn_network_set_dt(snn_network_t *h, float dt);           /* neuron/mod.rs:1655-1660 */
SNN_API int32_t snn_network_reset_timing(snn_network_t *h);                /* neuron/mod.rs:1710-1717 */

/* RunNetwork::run_lattices (neuron/mod.rs:2667-2674). Blocks. */
SNN_API int32_t snn_network_run(snn_network_t *h, uint64_t iterations);

/* RewardModulatedLatticeNetwork (neuron/mod.rs:3455-5455): a network handle that also holds reward-modulated lattices.
 *  - add_reward_modulated_lattice (:3615-3634): a lattice whose own graph carries TraceRSTDP weights and whose plasticity is a
 *    RewardModulatedSTDP (`do_modulation` defaults to 1, :2772; modulator defaults as snn_rstdp_t above);
 *  - set_connection_reward_modulated: the block pre_id -> post_id of the connecting graph, built with the snn_network_connect_*
 *    calls, holds RewardModulatedConnection::RewardModulatedWeight values (connect_with_reward_modulation, :4076-4209) instead
 *    of ::Weight (connect, :3836-3947); connecting the block again makes it a Weight block again;
 *  - snn_network_run is RunNetwork::run_lattices (:5411-5426, no reward signal); snn_network_run_with_rewards runs one timestep
 *    per entry, every modulator taking the reward first (run_lattices_with_reward, :5385-5392 -> :5280-5297).
 * After all neurons of a timestep have stepped (post_neuron_update_step, :5030-5062) every neuron of a reward-modulated lattice
 * with do_modulation updates: the edges of the lattice's own graph, twice (as in-edge of one end and out-edge of the other);
 * incoming RewardModulatedWeight edges once with that lattice's modulator; incoming Weight edges from plain lattices with the
 * INPUT lattice's STDP parameters (:4868-4884).  Plain lattices keep LatticeNetwork's STDP.  The reference looks OUTGOING
 * connecting edges up with their end points swapped and panics (:4760-4763, 4931-4934): run returns SNN_UNSUPPORTED for connecting
 * edges out of a reward-modulated lattice with do_modulation or out of a plain lattice with do_plasticity, and for the incoming
 * arms that unwrap a missing lattice kind (:4727-4731, 4741-4747).  Single-GPU handles. */
SNN_API int32_t snn_network_add_reward_modulated_lattice(snn_network_t *h, uint64_t id, uint32_t rows, uint32_t cols);
SNN_API int32_t snn_network_set_reward_modulator(snn_network_t *h, uint64_t id, int32_t do_modulation, const snn_rstdp_t *modulator);
SNN_API int32_t snn_network_get_reward_modulator(snn_network_t *h, uint64_t id, int32_t *do_modulation, snn_rstdp_t *modulator);
SNN_API int32_t snn_network_set_connection_reward_modulated(snn_network_t *h, uint64_t pre_id, uint64_t post_id, int32_t reward_modulated);
SNN_API int32_t snn_network_run_with_rewards(snn_network_t *h, const float *rewards, uint64_t n_rewards);
/* TraceRSTDP members of the edges of one block in the order of snn_network_get_connection_csr (see the snn_lattice_ calls) */
SNN_API int32_t snn_network_get_connection_traces(snn_network_t *h, uint64_t pre_id, uint64_t post_id, uint32_t *counter, float *dw,
                                                  float *c, uint64_t nnz);
SNN_API int32_t snn_network_set_connection_traces(snn_network_t *h, uint64_t pre_id, uint64_t post_id, const float *weight,
                                                  const uint32_t *counter, const float *dw, const float *c, uint64_t nnz);
SNN_API int32_t snn_network_run_timed(snn_network_t *h, uint64_t iterations, float *elapsed_ms,
                                      uint64_t *kernel_launches);

SNN_API int32_t snn_network_history_len(const snn_network_t *h, uint64_t id, uint64_t *steps);
SNN_API int32_t snn_network_get_grid_history(snn_network_t *h, uint64_t id, float *out, uint64_t capacity_floats);
SNN_API int32_t snn_network_get_spike_history(snn_network_t *h, uint64_t id, uint8_t *out, uint64_t capacity_bytes);
SNN_API int32_t snn_network_get_spike_aggregate(snn_network_t *h, uint64_t id, int64_t *out, uint64_t capacity);
SNN_API int32_t snn_network_get_average_history(snn_network_t *h, uint64_t id, float *out, uint64_t capacity_floats);
SNN_API int32_t snn_network_set_eeg_parameters(snn_network_t *h, uint64_t id, float reference_voltage, float distance, float conductivity);
SNN_API int32_t snn_network_get_eeg_history(snn_network_t *h, uint64_t id, float *out, uint64_t capacity_floats);
SNN_API int32_t snn_network_reset_history(snn_network_t *h);
/* graph history of the block pre_id -> post_id: a lattice's own graph (pre_id == post_id, SNN_OPT_UPDATE_GRAPH_HISTORY through
 * snn_network_set_lattice_option) or a connecting block (SNN_OPT_UPDATE_CONNECTING_GRAPH_HISTORY).  Record k holds the weights
 * step k's input gather used: LatticeNetwork::iterate pushes the histories before that step's STDP (neuron/mod.rs:2565-2576), so
 * record 0 is the weights before the run.  Edge order of snn_network_get_connection_csr(pre_id, post_id); a block never recorded
 * (or without edges) reports steps = nnz = 0.  Same restrictions as the lattice calls (reward-modulated networks: SNN_UNSUPPORTED). */
SNN_API int32_t snn_network_graph_history_len(snn_network_t *h, uint64_t pre_id, uint64_t post_id, uint64_t *steps, uint64_t *nnz);
SNN_API int32_t snn_network_get_graph_history(snn_network_t *h, uint64_t pre_id, uint64_t post_id, float *out, uint64_t capacity_floats);
/* spike events of lattice `id` (a neuron or spike-train lattice), indices inside that lattice; see the snn_lattice_ calls */
SNN_API int32_t snn_network_spike_event_count(const snn_network_t *h, uint64_t id, uint64_t *steps, uint64_t *n_events);
SNN_API int32_t snn_network_get_spike_events(snn_network_t *h, uint64_t id, uint64_t *step_ptr, uint32_t *neuron, uint64_t capacity);

#ifdef __cplusplus
}
#endif
#endif /* SNN_B200_H */
