/* lmcma_b200.h — C ABI of the B200-native LM-CMA trajectory optimiser (liblmcma_b200.so).
 *
 * This is the drop-in boundary for the hot path of behnamasadi/lmcma_path_planner:
 *   - the LM-CMA optimiser class  (reference: lmcma_path_planner/src/lmcma.hpp:41-144)
 *   - the grid-map cost-model pieces (reference: sample_based_optimisation_based_path_planner/src/
 *     sample_based_optimisation_based_path_planner.cpp:587-690), assembled into a batched
 *     per-trajectory cost evaluator (the reference evaluates one OMPL state at a time).
 * Every entry point cites the reference interface it replaces.  Plain pointers and sizes only;
 * no C++ / torch types.  All functions return LMCMA_B200_OK (0) or a negative error code;
 * lmcma_b200_last_error() returns a thread-local description of the last failure.
 * There is NO CPU fallback: every compute entry point fails with LMCMA_B200_ERR_CUDA when no
 * sm_100 device is usable.
 *
 * Host buffers may be pageable or pinned.  "_dev" variants take device pointers (resident in HBM)
 * and a cudaStream_t passed as void*.
 *
 * Thread / stream contract.  An optimiser handle (lmcma_b200_opt) is NOT re-entrant, like the reference object: one
 * host thread at a time per handle; different handles are independent.  A map handle may be shared by any number of
 * optimiser handles and host threads: lmcma_b200_cost_evaluate_dev may be called concurrently from several threads and
 * on several streams for different queries (the end points travel by value with each launch; no per-map device state is
 * written); lmcma_b200_cost_evaluate and lmcma_b200_cost_trace (host buffers) serialise on a per-map lock because they
 * share the map's staging buffers and private stream.  lmcma_b200_map_set_l2_persist, lmcma_b200_map_update_occupancy and
 * lmcma_b200_map_destroy must not race with evaluations on the same map.  lmcma_b200_tell_all_dev enqueues on the
 * handle's stream only and returns without waiting: the caller's cost, and every later call on the handle, are ordered
 * after it by that stream (call lmcma_b200_set_stream with the stream the cost runs on, never NULL).
 *
 * Environment knobs (LMCMA_B200_*, experiments / debugging only) are read once when a handle is created, never on a
 * launch path.  The overlapped single-query generation (a forked CUDA graph whose branches must run concurrently) is
 * enabled only after a per-device probe has seen two graph branches co-scheduled (so profilers / sanitizers that
 * serialise kernels get the linear graph automatically; LMCMA_B200_OVERLAP=0 forces it).  If co-scheduling is lost
 * later, no kernel traps: the next synchronising call returns LMCMA_B200_ERR_CUDA once, the handle falls back to the
 * linear graph, and the generation in flight is void (restore the state with set_* or recreate the handle).
 */
#ifndef LMCMA_B200_H
#define LMCMA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LMCMA_B200_ABI_VERSION 1

enum {
    LMCMA_B200_OK = 0,
    LMCMA_B200_ERR_ARG = -1,      /* bad argument (null pointer, size mismatch, unsupported shape) */
    LMCMA_B200_ERR_CUDA = -2,     /* CUDA runtime failure or no usable device */
    LMCMA_B200_ERR_STATE = -3,    /* call out of protocol order (e.g. tell before ask) */
    LMCMA_B200_ERR_NOMEM = -4
};

/* where the N(0,1) deviates of sample() come from (reference: CMABase::sampleStandardNormal, lmcma.cpp:212-218) */
enum {
    LMCMA_B200_RNG_PHILOX = 0,   /* device counter-based Philox4x32-10 + Box-Muller (throughput runs) */
    LMCMA_B200_RNG_HANSEN = 1,   /* host replay of the reference's serial generator (lmcma.cpp:14-82), uploaded per
                                    generation: reproduces the reference's stream for a given seed (batch must be 1) */
    LMCMA_B200_RNG_INJECT = 2    /* caller supplies Z through lmcma_b200_inject_z before every sample (parity runs) */
};

enum { LMCMA_B200_MAP_F32 = 0, LMCMA_B200_MAP_U8 = 1 };

typedef struct lmcma_b200_opt lmcma_b200_opt;   /* a batch of B independent optimiser instances of one shape */
typedef struct lmcma_b200_map lmcma_b200_map;   /* a 2-D / 3-D distance map resident in HBM */

/* ---------------------------------------------------------------- library / device ------------ */
int lmcma_b200_abi_version(void);
const char* lmcma_b200_last_error(void);
int lmcma_b200_device_count(int* count_out);
/* SM count, L2 bytes, total HBM bytes, compute capability (major*10+minor) of `device` */
int lmcma_b200_device_info(int device, int* sm_count, int64_t* l2_bytes, int64_t* hbm_bytes, int* cc);

/* ---------------------------------------------------------------- cost map -------------------- */
/* Replaces the global `Eigen::MatrixXd EDT_Matrix` (planner.cpp:37) and its loaders (planner.cpp:354-395,
 * 777-818).  dist_host: distance to the nearest obstacle in cells, 0 on obstacles, row-major
 * [ny][nx] (dims == 2, row = y, col = x as in planner.cpp:597-602) or [nz][ny][nx] (dims == 3).
 * storage F32: the device keeps sign-tagged reciprocal clearance 1/max(E, c_min) (negative on
 *              obstacles), 4 B/cell.
 * storage U8 : the device keeps q = E > 0 ? clamp(floor(E / u8_scale), 1, 255) : 0, 1 B/cell; the
 *              evaluator sees E_q = q * u8_scale (use lmcma_b200_map_dequantized to obtain E_q).
 * c_min: floor on the clearance used in the state cost 1/clearance (planner.cpp:667). */
int lmcma_b200_map_create(int device, int dims, const int32_t* shape_xyz, const float* dist_host,
                          int storage, float u8_scale, float c_min, lmcma_b200_map** map_out);
/* Occupancy grid (1 = obstacle; row-major [ny][nx] / [nz][ny][nx]) -> exact Euclidean distance field in cells, on the
 * device (separable, integer-exact; k_edt.cuh).  Replaces the reference's ways of obtaining EDT_Matrix from a map:
 * the in-file 8SSEDT on a fixed 100 x 100 grid (planner.cpp:403-490) and dynamicEDT3D (planner.cpp:81-87, 305-307).
 * clamp > 0 limits the distance (dynamicEDT3D's maxdist); clamp <= 0 leaves it unbounded.  A grid without any obstacle
 * gives the clamp everywhere, or FLT_MAX when unclamped.  Every axis must be at most 32767 cells long (else
 * LMCMA_B200_ERR_ARG); the distances are exact for every such grid. */
int lmcma_b200_edt(int device, int dims, const int32_t* shape_xyz, const uint8_t* occ_host, float clamp, float* dist_host_out);
/* map_create fed by an occupancy grid: distance transform + conversion to the map storage, all on the device */
int lmcma_b200_map_create_from_occupancy(int device, int dims, const int32_t* shape_xyz, const uint8_t* occ_host, float clamp,
                                         int storage, float u8_scale, float c_min, lmcma_b200_map** map_out);
/* Replace the occupancy of the box [lo, lo + size) (cells, x y [z]; occ_box row-major [sz][sy][sx], non-zero = obstacle)
 * of a map built by lmcma_b200_map_create_from_occupancy, and bring its storage up to date on the device.  Afterwards the
 * map holds, bit for bit, what map_create_from_occupancy of the edited grid with the same clamp / storage / u8_scale /
 * c_min would hold.  Synchronous.  Must not race with evaluations of this map (like map_destroy).  Optimiser handles
 * attached to the map, including their captured graphs, read the new contents on their next launch: no re-attach.
 * With clamp > 0 only the cells closer than the clamp to the box are recomputed, from a window of the grid around them;
 * with clamp <= 0 the whole grid is (one obstacle removed can change any distance), from the occupancy the map storage
 * encodes, so only the box crosses PCIe either way.
 * LMCMA_B200_ERR_STATE: a map made by lmcma_b200_map_create (a caller's distance field has no occupancy behind it).
 * LMCMA_B200_ERR_ARG: a null pointer, a size below 1, or a box not inside the grid.  A refused call changes nothing. */
int lmcma_b200_map_update_occupancy(lmcma_b200_map* map, const int32_t* lo_xyz, const int32_t* size_xyz, const uint8_t* occ_box_host);
int lmcma_b200_map_destroy(lmcma_b200_map* map);
/* the distance field the evaluator effectively uses, back on the host: U8 storage gives E_q = q * u8_scale; F32 storage
 * gives 1 / (1 / max(E, c_min)) in FP32, i.e. the clearance with the c_min floor (up to the rounding of the two
 * reciprocals), and 0 on obstacles */
int lmcma_b200_map_dequantized(const lmcma_b200_map* map, float* dist_host_out);
/* pin the map in L2 (cudaAccessPolicyWindow, persisting) for the launches of this library.  An optimiser handle attached
 * to several maps (lmcma_b200_attach_cost_maps) sets no window: one window covers one address range */
int lmcma_b200_map_set_l2_persist(lmcma_b200_map* map, int enable);

/* A planning query: fixed end points (planner.cpp:701-711) and the objective weights
 * (shortrisky = {100, 1}, longsafe = {1, 1000}; planner.cpp:677-690) plus the collision penalty. */
typedef struct {
    float start[3];
    float goal[3];
} lmcma_b200_endpoints;

typedef struct {
    int32_t waypoints;   /* W interior waypoints; n = dims * W, dimension-major x[d*W + w] (lmcma.cpp:786-791) */
    float w_len;         /* weight of the path length            (PathLengthOptimizationObjective, planner.cpp:638) */
    float w_clr;         /* weight of the integral of 1/clearance (ClearanceObjective, planner.cpp:648-669) */
    float w_col;         /* penalty per colliding sample          (negation of ValidityChecker::isValid, planner.cpp:591-603) */
} lmcma_b200_objective;

/* Batched trajectory cost: replaces per-state ValidityChecker::isValid / clearance /
 * ClearanceObjective::stateCost (planner.cpp:591-669) + OMPL's path integration.
 * X_host: count x n FP32 candidates, dense.  Outputs (each may be NULL except f): fitness,
 * number of colliding samples (bit-exact contract) and number of map samples visited.
 * Page-locked buffers (cudaHostAlloc / cudaHostRegister) are read and written by the kernel
 * directly (no staging copy); pageable buffers are staged through device memory. */
int lmcma_b200_cost_evaluate(lmcma_b200_map* map, const lmcma_b200_objective* obj, const lmcma_b200_endpoints* ends,
                             const float* X_host, int32_t count, float* f_host, int32_t* ncoll_host,
                             int32_t* nsamp_host);
/* device-resident variant: X_dev is count x n with row stride `ld` floats (ld >= n). */
int lmcma_b200_cost_evaluate_dev(lmcma_b200_map* map, const lmcma_b200_objective* obj, const lmcma_b200_endpoints* ends,
                                 const float* X_dev, int64_t ld, int32_t count, float* f_dev, int32_t* ncoll_dev,
                                 int32_t* nsamp_dev, void* cuda_stream);
/* debug / parity: linear cell index ((z*ny + y)*nx + x, -1 = outside the map) of every sample of ONE
 * trajectory in visiting order; *n_cells_out receives the true number of samples. */
int lmcma_b200_cost_trace(lmcma_b200_map* map, const lmcma_b200_objective* obj, const lmcma_b200_endpoints* ends,
                          const float* x_host, int64_t* cells_host, int64_t max_cells, int64_t* n_cells_out);

/* ---------------------------------------------------------------- optimiser ------------------- */
typedef struct {
    int32_t n;            /* problem dimension (CMABase::init(N), lmcma.cpp:130) */
    int32_t lambda;       /* population; < 1 -> 4 + int(3 ln n) (lmcma.cpp:134-135) */
    int32_t m;            /* stored direction pairs; < 1 -> lambda (the reference's rule, lmcma.cpp:266) */
    int32_t batch;        /* B independent instances advanced in lock-step (>= 1) */
    double sigma0;        /* initial step size (LMCMA ctor `sigma`, lmcma.hpp:131-133) */
    int64_t seed;         /* `inseed`; PHILOX key / HANSEN seed (>= 1 for the reference's determinism) */
    int32_t rng;          /* LMCMA_B200_RNG_* */
    int32_t device;       /* CUDA ordinal */
    int32_t record_z;     /* keep the deviates of the last sample() readable (LMCMA_B200_F32_Z) */
    /* split-population mode (one population over several GPUs): this handle samples and evaluates the
     * offspring rows [pop_offset, pop_offset + pop_count) of lambda.  pop_count < 1 -> all rows. */
    int32_t pop_offset;
    int32_t pop_count;
    int32_t reserved[5];
} lmcma_b200_config;

/* LMCMA::LMCMA + LMCMA::init (lmcma.hpp:131-135, lmcma.cpp:233-299).  x0: batch x n initial means
 * (`initialParams`; NULL -> uniform(0,1) start, lmcma.cpp:161-163, HANSEN rng only).  lo/hi: n box bounds
 * shared by the batch or NULL (lmcma.cpp:220-230).  Unlike the reference the arrays are COPIED.
 * Builds the first population unless rng == INJECT (then the first inject_z does). */
int lmcma_b200_create(const lmcma_b200_config* cfg, const double* x0, const double* lo, const double* hi,
                      lmcma_b200_opt** opt_out);
/* Same with the reference's `covariance` constructor argument (lmcma.hpp:131-133): a fixed n x n symmetric positive
 * definite prior (e.g. lmcma_b200_covariance).  It is factored once (cholesky, lmcma.cpp:165-169, 844-855) and every
 * deviate vector becomes z <- L z before computeAz (sampleStandardNormal + applyCovL, lmcma.cpp:212-218, 857-864):
 * on the device one FP32 contraction [batch * pop_count x n] x [n x n] per generation.  covariance == NULL -> no prior. */
int lmcma_b200_create_with_prior(const lmcma_b200_config* cfg, const double* x0, const double* lo, const double* hi,
                                 const double* covariance, lmcma_b200_opt** opt_out);
int lmcma_b200_destroy(lmcma_b200_opt* opt);

/* run this handle's work on the caller's stream (void* cudaStream_t; NULL -> the handle's own
 * non-blocking stream).  Lets a host framework order its own events / collectives with the kernels. */
int lmcma_b200_set_stream(lmcma_b200_opt* opt, void* cuda_stream);

/* resolved shape: [n, lambda, mu, m, batch, pop_offset, pop_count, row stride (floats)] */
int lmcma_b200_shape(const lmcma_b200_opt* opt, int32_t* out8);

/* Reference protocol, one candidate at a time (batch == 1):
 *   ask_one  = CMABase::getNextParameterVector (lmcma.cpp:172-182; does not advance)
 *   tell_one = CMABase::setEvaluationFeedback  (lmcma.cpp:184-205; the lambda-th call runs update(); sample()) */
int lmcma_b200_ask_one(lmcma_b200_opt* opt, double* params, int32_t n);
int lmcma_b200_tell_one(lmcma_b200_opt* opt, const double* feedbacks, int32_t num_feedbacks);

/* Batched protocol: the whole population (batch x pop_count x n, FP32, dense) out, all fitnesses in.
 * tell_all runs LMCMA::update (lmcma.cpp:313-424) and LMCMA::sample (lmcma.cpp:301-311) on the device; it returns when the
 * next population is ready.  For one query with the device RNG the fitness-independent part of the update runs beside
 * the fitness copy and the ranking (one forked CUDA graph per call; same bits as the serial order). */
int lmcma_b200_ask_all(lmcma_b200_opt* opt, float* X_host);
int lmcma_b200_tell_all(lmcma_b200_opt* opt, const float* f_host);

/* Zero-copy ask for the host-buffer protocol.  *X_host_view receives a READ-ONLY pointer to the handle's page-locked
 * mirror of the current population (batch x pop_count rows, row stride *ld_out floats >= n; valid until the next
 * tell / run / destroy).  Once this has been called, the sampler of every following tell_all writes the candidates into
 * the mirror itself while it runs (posted PCIe writes overlapping the sampling), so this call only waits for the
 * stream; lmcma_b200_cost_evaluate recognises a pointer into the mirror and evaluates the device copy it mirrors (no
 * H2D of the candidates).  Same contents as lmcma_b200_ask_all. */
int lmcma_b200_ask_all_view(lmcma_b200_opt* opt, const float** X_host_view, int64_t* ld_out);

/* Device-resident batched protocol, for a cost the caller computes on the GPU.
 * X_dev: the current population, batch x pop_count rows of n FP32, row stride *ld_out floats (>= n).  Read-only.
 * f_dev: the handle's fitness buffer, batch x lambda FP32, dense.  The caller writes it, then calls tell_all_dev.
 * Both pointers stay valid and unchanged for the handle's lifetime.  Any handle may call this.  Nothing is allocated, so
 * a stream capture may begin right after it. */
int lmcma_b200_device_buffers(lmcma_b200_opt* opt, const float** X_dev, int64_t* ld_out, float** f_dev);
/* update() + sample() from the fitness in f_dev, enqueued on the handle's stream (lmcma_b200_set_stream).  Returns without
 * waiting.  Later work on that stream sees the next population in X_dev.  The same bits as lmcma_b200_tell_all given the
 * same fitness.  Capturable into the caller's stream capture (torch.cuda.graph, cudaStreamBeginCapture): under a capture
 * it enqueues the stream-ordered generation, builds and replays no graph of its own, allocates nothing and never waits.
 * Uncaptured, one query with the overlapped generation replays tell_all's forked graph without its fitness copy; other
 * handles enqueue the stream-ordered generation.  A lost co-scheduling is reported by the next synchronising call.
 * The handle's stream must be one the caller's cost is ordered with: set_stream with the cost's own stream.  NULL selects
 * the handle's private non-blocking stream, which neither the caller's streams nor the legacy default stream wait for.
 * Replays of a caller's graph advance the state without this library seeing them: once a generation has been recorded,
 * ask_all_view and ask_one always read the population from the device, and the setters of V, P, NJ, LJ, T and VEC
 * rebuild the pair mirror the sampler reads at once.  Order the replays with later calls on the handle (replay on the
 * handle's stream, or synchronise).
 * LMCMA_B200_ERR_STATE: rng != PHILOX, a split-population handle. */
int lmcma_b200_tell_all_dev(lmcma_b200_opt* opt);

/* Restart chosen instances of a live batch in place, for a planning service or a restart policy whose queries finish at
 * different times.  Each reset instance gets exactly what lmcma_b200_create leaves for a start x0 and step size sigma0 (mean
 * x0, every path, direction pair, slot, fitness and best-so-far cleared, itr = counteval = 0), with its deviate stream moved
 * on by one epoch (LMCMA_B200_I32_EPOCH), so a restart from the same start does not repeat the earlier run; then its first
 * population is drawn.  The other instances, the handle's CUDA graphs and its kernel configuration are untouched: the
 * next run / tell replays the graphs it has.  The cost's launch shape stays what attach_cost chose from the end points
 * of instance 0; it only sizes k_cost's launch, so longer trajectories of reset instances take more rounds and stay
 * correct.
 *
 * Host: synchronous.  idx: count distinct instance indices; x0: count x n; sigma0: count, or NULL for cfg.sigma0; ends:
 * count new end-point pairs, or NULL to keep them (needs an attached cost).  count == 0 does nothing.  The flagged rows of
 * the host mirror (ask_all_view) are rewritten, so the mirror stays as current as it was.
 * LMCMA_B200_ERR_ARG: an index out of range or repeated, a null idx / x0, a non-finite x0, a sigma0 not finite or <= 0,
 * count < 0.  LMCMA_B200_ERR_STATE: rng HANSEN or INJECT, a split-population handle, ends without an attached cost.  A
 * refused call changes nothing. */
int lmcma_b200_reset_instances(lmcma_b200_opt* opt, int32_t count, const int32_t* idx, const double* x0,
                               const double* sigma0, const lmcma_b200_endpoints* ends);
/* Device: the same reset from flags the caller computed on the device.  flags_dev: batch int32, non-zero = reset;
 * x0_dev: batch x n FP64 dense (rows of unflagged instances are not read); sigma0_dev: batch FP64 or NULL (cfg.sigma0);
 * ends_dev: batch x 6 FP32 {start xyz, goal xyz} or NULL (keep); best_x_out_dev: batch x n FP32 and best_f_out_dev: batch
 * FP64, or NULL: the retiring instance's best_x and best_f (as stored) before the reset, written for flagged rows only.
 * Enqueued on the handle's stream (as lmcma_b200_tell_all_dev, set_stream with the stream the flags are computed on);
 * never waits and allocates nothing.  Capturable: under the caller's stream capture it records into that capture, and its
 * kernels are not counted by lmcma_b200_launch_count.  The inputs are trusted as tell_all_dev trusts f_dev: values are not
 * checked (sigma0 > 0, finite x0 are the caller's part).  The host mirror is stale afterwards (ask_all_view copies).
 * LMCMA_B200_ERR_ARG: a null flags_dev / x0_dev.  LMCMA_B200_ERR_STATE: as the host variant. */
int lmcma_b200_reset_instances_dev(lmcma_b200_opt* opt, const int32_t* flags_dev, const double* x0_dev,
                                   const double* sigma0_dev, const float* ends_dev, float* best_x_out_dev,
                                   double* best_f_out_dev);

/* deviates for the NEXT sample(): batch x pop_count x n FP32 (rng == INJECT).  The first call after
 * create builds the first population immediately; later calls are consumed by the next tell. */
int lmcma_b200_inject_z(lmcma_b200_opt* opt, const float* Z_host);

/* re-run LMCMA::sample (lmcma.cpp:301-311) from the CURRENT state with the deviates already on the device
 * (INJECT: the last injected Z; PHILOX: regenerated from the counter).  Used after set_* (teacher forcing). */
int lmcma_b200_resample(lmcma_b200_opt* opt);

/* LMCMA::isBehaviorLearningDone (lmcma.cpp:426-429): done[b] = sigma[b] < 1e-20 */
int lmcma_b200_is_done(lmcma_b200_opt* opt, int32_t* done_host);

/* ---- fused on-device planning: cost evaluation attached to the optimiser ---- */
/* ends: batch end-point pairs (one query per instance).  The map must live on the same device. */
int lmcma_b200_attach_cost(lmcma_b200_opt* opt, lmcma_b200_map* map, const lmcma_b200_objective* obj,
                           const lmcma_b200_endpoints* ends);
/* One handle on several maps (several floors or sites, a coarse map beside a fine one), so that one batch and one launch
 * of each kernel serve queries on all of them: instance b is evaluated on maps[map_of[b]] (map_of: batch entries).  Every
 * map must live on the handle's device and share dims and storage; shape, u8_scale, c_min and clamp may differ.  One
 * objective for the whole handle; the end points stay per instance.  The box bounds stay per handle: samples of an
 * instance that leave its map are collisions, so maps padded to one shape give every instance a tight box.
 * map_of is per-instance state: LMCMA_B200_I32_MAP_OF (get / set) and lmcma_b200_instance_maps_dev change it without
 * rebuilding a graph, and reset_instances leaves it alone.  The maps must outlive the attachment, as with attach_cost, and
 * an occupancy update of any of them is seen by the next launch.  L2 persistence (lmcma_b200_map_set_l2_persist) is not
 * applied on a handle with several maps: an access-policy window covers one address range.  map_count == 1 attaches
 * maps[0] exactly as lmcma_b200_attach_cost does.
 * LMCMA_B200_ERR_ARG: a null pointer, map_count < 1, maps of different devices / dims / storage, dims * waypoints != n, a
 * map_of entry outside [0, map_count).  LMCMA_B200_ERR_STATE: a split-population handle (the mg_* entry points take one
 * map).  A refused call changes nothing. */
int lmcma_b200_attach_cost_maps(lmcma_b200_opt* opt, int32_t map_count, lmcma_b200_map* const* maps,
                                const int32_t* map_of /* batch */, const lmcma_b200_objective* obj,
                                const lmcma_b200_endpoints* ends /* batch */);
/* The handle's device copy of map_of (batch int32), stable for the handle's lifetime.  The caller may write it on the
 * handle's stream, also inside its stream capture, as it writes f_dev of lmcma_b200_device_buffers; the next cost launch
 * reads it.  Values are trusted, with one exception: k_cost gives an instance whose entry lies outside [0, map_count)
 * f = +inf and ncoll = nsamp = 0 and reads no map for it.  LMCMA_B200_ERR_STATE on a handle not attached to several
 * maps. */
int lmcma_b200_instance_maps_dev(lmcma_b200_opt* opt, int32_t** map_of_dev);
/* `generations` x [cost -> rank -> update -> sample] replayed from a CUDA graph with no
 * host round trip (the loop of example_lmcma.cpp:49-55 with the cost on the device). Asynchronous. */
int lmcma_b200_run(lmcma_b200_opt* opt, int32_t generations);
int lmcma_b200_sync(lmcma_b200_opt* opt);
/* number of kernels this library has launched so far (all handles, this process).  A replay of one of its CUDA graphs
 * (lmcma_b200_run, lmcma_b200_tell_all, lmcma_b200_tell_all_dev) counts the kernels the graph holds; building a graph
 * counts none.  Kernels lmcma_b200_tell_all_dev enqueues into the caller's stream capture count none either: they run
 * when the caller replays its graph, which this library does not see. */
int64_t lmcma_b200_launch_count(void);
/* CUDA-event timing of everything enqueued by the last lmcma_b200_run on this handle (ms) */
int lmcma_b200_last_run_ms(lmcma_b200_opt* opt, float* ms_out);
/* per-kernel CUDA-event timing: runs `generations` un-graphed generations with an event pair around
 * each of the 4 kernels; ms_out4 = mean ms per launch of {cost, rank (+ recombination partial sums), update, sample} */
int lmcma_b200_profile_kernels(lmcma_b200_opt* opt, int32_t generations, float* ms_out4);

/* best evaluated candidate so far per instance (the reference keeps only BestF, lmcma.cpp:192-194) */
int lmcma_b200_best(lmcma_b200_opt* opt, float* x_best_host /* batch x n */, float* f_best_host /* batch */);
/* Re-evaluate each instance's best-so-far candidate (lmcma_b200_best) on the attached map as it is now, and make its
 * cost the new best_f.  Needed after a map update: otherwise a stale best_f from the old map keeps a path that now
 * collides as "best" for good.  Instances with no evaluation yet are left as they are.  best_x and counteval do not
 * change; PREV_FIT keeps the previous generation's fitness on the old map, which the next update compares once in its
 * step-size rule (the reference has no notion of a changing cost).  Synchronous.
 * LMCMA_B200_ERR_STATE without an attached cost, and on a split-population handle (best_x may hold a peer's row there). */
int lmcma_b200_rescore_best(lmcma_b200_opt* opt);

/* ---- state access (parity / teacher forcing / checkpointing) ---- */
enum {
    LMCMA_B200_F64_XMEAN = 0,      /* batch x n            (CMABase::xmean) */
    LMCMA_B200_F64_SIGMA = 1,      /* batch                (LMCMA::sigma) */
    LMCMA_B200_F64_S = 2,          /* batch                (LMCMA::s) */
    LMCMA_B200_F64_BESTF = 3,      /* batch                (CMABase::BestF) */
    LMCMA_B200_F64_CONSTS = 4,     /* [c1, cc, cs, val_target, K, M, mueff]  (lmcma.cpp:144-156, 238, 268-272) */
    LMCMA_B200_F64_WEIGHTS = 5,    /* mu                   (CMABase::weights) */
    LMCMA_B200_F64_NJ = 6,         /* batch x m            (LMCMA::Nj_arr) */
    LMCMA_B200_F64_LJ = 7          /* batch x m            (LMCMA::Lj_arr) */
};
enum {
    LMCMA_B200_F32_X = 0,          /* batch x pop_count x n (CMABase::arx) */
    LMCMA_B200_F32_PC = 1,         /* batch x n            (LMCMA::pc) */
    LMCMA_B200_F32_V = 2,          /* batch x m x n        (LMCMA::v_arr, slot-indexed) */
    LMCMA_B200_F32_P = 3,          /* batch x m x n        (LMCMA::pc_arr, slot-indexed) */
    LMCMA_B200_F32_FIT = 4,        /* batch x lambda       fitness as told (unsorted) */
    LMCMA_B200_F32_FIT_SORTED = 5, /* batch x lambda       (CMABase::arfitness after myqsort) */
    LMCMA_B200_F32_PREV_FIT = 6,   /* batch x lambda       (LMCMA::prev_arfitness) */
    LMCMA_B200_F32_Z = 7           /* batch x pop_count x n deviates of the last sample() (record_z or INJECT) */
};
enum {
    LMCMA_B200_I32_T = 0,          /* batch x m   (LMCMA::t, slot order oldest -> newest) */
    LMCMA_B200_I32_VEC = 1,        /* batch x m   (LMCMA::vec, generation stamp per slot) */
    LMCMA_B200_I32_ARINDEX = 2,    /* batch x lambda (LMCMA::arindex) */
    LMCMA_B200_I32_RANK = 3,       /* batch x lambda inverse of ARINDEX */
    LMCMA_B200_I32_ITR = 4,        /* batch       (CMABase::itr) */
    LMCMA_B200_I32_LIVE = 5,       /* batch       (LMCMA::iterator_sz) */
    LMCMA_B200_I32_COUNTEVAL = 6,  /* batch       (CMABase::counteval) */
    LMCMA_B200_I32_NCOLL = 7,      /* batch x pop_count colliding samples of the last evaluated population */
    LMCMA_B200_I32_NSAMP = 8,      /* batch x pop_count map samples of the last evaluated population */
    LMCMA_B200_I32_LAUNCH = 9,     /* LMCMA_B200_LAUNCH_FIELDS values per HANDLE (not per instance), read-only: the launch
                                      configuration chosen at create, indexed by LMCMA_B200_LAUNCH_* below */
    LMCMA_B200_I32_EPOCH = 10,     /* batch      deviate stream of the instance: 0 at create, + 1 per reset_instances.  The
                                      PHILOX key is (lo32(seed), hi32(seed) + epoch) mod 2^32, so seed s at epoch e draws what
                                      seed s + e 2^32 draws at epoch 0.  A checkpoint that restores ITR restores this too */
    LMCMA_B200_I32_MAP_OF = 11     /* batch       map of the instance (lmcma_b200_attach_cost_maps); all zeros on a handle on one
                                      map.  Settable with entries in [0, map_count); no graph is rebuilt */
};
/* fields of LMCMA_B200_I32_LAUNCH.  Sampler kernels: 0 = k_sample<NV> (narrow), 1 = k_sample_wide<RBW> (a row split over CW
 * column-warps, R row groups per CTA), 2 = k_sample_rows<QW, RL> (rows on lanes).  KC / STAGES are those of the chosen
 * sampler.  The update is k_update<NVB, RMAX, ROWS_IN_SMEM, OVERLAP, WARPS>, or with GRAM the Gram-matrix recompute whose
 * k_coef keeps COEF_ELEMS elements per lane (0 without GRAM).  The overlapped k_update build is the one of the fused
 * generations and of tell_all when OVERLAP is 1.  Two fields no longer vary and keep their place: SMP_SPEC is always 1
 * (the NV = 4 narrow sampler runs full groups of pairs without per-pair predicates), and SWEEP_WARPS equals UPD_WARPS
 * (every warp of k_update's CTA owns rows of the register sweep). */
enum {
    LMCMA_B200_LAUNCH_SAMPLER = 0, LMCMA_B200_LAUNCH_SMP_NV, LMCMA_B200_LAUNCH_SMP_SPEC, LMCMA_B200_LAUNCH_SMP_THREADS,
    LMCMA_B200_LAUNCH_SMP_RBW, LMCMA_B200_LAUNCH_SMP_CW, LMCMA_B200_LAUNCH_SMP_R, LMCMA_B200_LAUNCH_SMP_ROWS_QW,
    LMCMA_B200_LAUNCH_SMP_ROWS_RL, LMCMA_B200_LAUNCH_SMP_KC, LMCMA_B200_LAUNCH_SMP_STAGES,
    LMCMA_B200_LAUNCH_UPD_NVB, LMCMA_B200_LAUNCH_UPD_RMAX, LMCMA_B200_LAUNCH_UPD_ROWS_IN_SMEM, LMCMA_B200_LAUNCH_UPD_GRAM,
    LMCMA_B200_LAUNCH_UPD_WARPS, LMCMA_B200_LAUNCH_UPD_SWEEP_WARPS, LMCMA_B200_LAUNCH_COEF_ELEMS,
    LMCMA_B200_LAUNCH_RANK_THREADS, LMCMA_B200_LAUNCH_RANK_FTILE, LMCMA_B200_LAUNCH_RANK_TILE_SORTED,
    LMCMA_B200_LAUNCH_PROGRESSIVE, LMCMA_B200_LAUNCH_OVERLAP,
    LMCMA_B200_LAUNCH_FIELDS
};
int lmcma_b200_get_f64(lmcma_b200_opt* opt, int32_t which, double* out, int64_t capacity);
int lmcma_b200_get_f32(lmcma_b200_opt* opt, int32_t which, float* out, int64_t capacity);
int lmcma_b200_get_i32(lmcma_b200_opt* opt, int32_t which, int32_t* out, int64_t capacity);
/* teacher forcing: overwrite optimiser state (same `which` / layouts as the getters; XMEAN, SIGMA, S,
 * NJ, LJ | PC, V, P, PREV_FIT | T, VEC, ITR, LIVE, EPOCH, MAP_OF are settable) */
int lmcma_b200_set_f64(lmcma_b200_opt* opt, int32_t which, const double* in, int64_t count);
int lmcma_b200_set_f32(lmcma_b200_opt* opt, int32_t which, const float* in, int64_t count);
int lmcma_b200_set_i32(lmcma_b200_opt* opt, int32_t which, const int32_t* in, int64_t count);

/* ---- split-population mode (one population over G GPUs; SURVEY.md section 8e) ---- */
/* Each rank owns rows [pop_offset, pop_offset+pop_count) (batch must be 1).  Per generation:
 *   mg_evaluate  : cost of the local rows -> f_local_dev (pop_count FP32, caller-owned device buffer)
 *   (caller all-gathers the fitness into f_all: lambda FP32 in rank order)
 *   mg_rank      : ranks of the local rows against all lambda + local weighted partial sums ->
 *                  payload_dev (mg_payload_floats() FP32, caller-owned device buffer)
 *   (caller all-gathers the payloads: G x mg_payload_floats())
 *   mg_update    : update() from the G payloads + sample() of the local rows for the next generation
 * All enqueue on `cuda_stream` (void* cudaStream_t, NULL -> the handle's stream) so the caller's
 * collectives (NCCL through torch.distributed, or ncclAllGather from C++) are ordered with them. */
int lmcma_b200_mg_payload_floats(lmcma_b200_opt* opt, int32_t* floats_out);
int lmcma_b200_mg_evaluate(lmcma_b200_opt* opt, float* f_local_dev, void* cuda_stream);
int lmcma_b200_mg_rank(lmcma_b200_opt* opt, const float* f_all_dev, float* payload_dev, void* cuda_stream);
int lmcma_b200_mg_update(lmcma_b200_opt* opt, const float* payload_all_dev, int32_t world, void* cuda_stream);

/* ---------------------------------------------------------------- host-side reference pieces -- */
/* The reference's serial generator (random_init/random_Gauss, lmcma.cpp:14-82) for callers that
 * want the reference's stream: fills out[count] with N(0,1) after skipping `skip` deviates. */
int lmcma_b200_hansen_gauss(int64_t seed, int64_t skip, int64_t count, double* out);
int lmcma_b200_hansen_uniform(int64_t seed, int64_t count, double* out);
/* Smoothness prior (covariance(), lmcma.cpp:769-810): host-side, heap-allocated (the reference's stack
 * arrays overflow for n >~ 720).  out: (dims*waypoints)^2 doubles, row-major. */
int lmcma_b200_covariance(int32_t dims, int32_t waypoints, double* out);
/* cholesky() (lmcma.cpp:844-855): lower factor of a symmetric positive definite n x n matrix, row-major, zero above
 * the diagonal (the reference takes Eigen's LLT; this is plain Cholesky-Banachiewicz in FP64). */
int lmcma_b200_cholesky(int32_t n, const double* C, double* L_out);

/* The remaining free functions of the reference header (lmcma.hpp:32-38, 248-254), host-side FP64, so that code written
 * against them keeps compiling through include/lmcma.hpp:
 * differentiationMatrix (lmcma.cpp:812-834): centred 7-tap rule of `order` 0..3 into the top-left block of a row-major
 * matrix with row stride row_len (< 0 -> num_time_steps). */
int lmcma_b200_differentiation_matrix(int32_t num_time_steps, int32_t order, double dt, double* diff_matrix, int32_t row_len);
/* invert (lmcma.cpp:836-842; Eigen's inverse there, Gauss-Jordan with partial pivoting here).  A != Ainv. */
int lmcma_b200_invert(const double* A, double* Ainv, int32_t n);
/* applyCovL (lmcma.cpp:857-864): z <- L z with L COLUMN-major n x n, the layout the reference's cholesky() writes. */
int lmcma_b200_apply_cov_l(const double* L_colmajor, double* z, int32_t n);
/* myqsort (lmcma.cpp:84-104): ascending stable order; the sorted values overwrite arfitness, ids go to arindex. */
int lmcma_b200_myqsort(int32_t sz, double* arfitness_inout, int32_t* arindex_out);
/* random_t + random_init / random_Uniform / random_Gauss / random_exit (lmcma.cpp:9-82) as an opaque stream object */
typedef struct lmcma_b200_rng lmcma_b200_rng;
int lmcma_b200_rng_create(int64_t seed, lmcma_b200_rng** rng_out);
int lmcma_b200_rng_destroy(lmcma_b200_rng* rng);
double lmcma_b200_rng_uniform(lmcma_b200_rng* rng);
double lmcma_b200_rng_gauss(lmcma_b200_rng* rng);

/* ---------------------------------------------------------------- map ingest (host-side file parsing) ---------- */
/* All four: pass out == NULL to query the size first.
 * BMP (24/32-bit, uncompressed): occupancy with the reference's rule g < 128 -> obstacle (Signed_Distance_Fields_test,
 * planner.cpp:505-523); rows top to bottom, occ_out[y * width + x]. */
int lmcma_b200_load_bmp(const char* path, uint8_t* occ_out, int64_t capacity, int32_t* width, int32_t* height);
/* binvox run-length voxel grid (format as read by binvox2bt.cpp:164-285; files under .../files/mesh_files):
 * occ_out[(z * ny + y) * nx + x], shape_xyz = {nx, ny, nz}; translate / scale from the header (nullable). */
int lmcma_b200_load_binvox(const char* path, uint8_t* occ_out, int64_t capacity, int32_t* shape_xyz, double* translate_xyz,
                           double* scale);
/* OctoMap binary tree (.bt: what binvox2bt.cpp:287-300 writes and planner.cpp:152-163 reads with OcTree::readBinary;
 * files .../files/mesh_files/{Dude,room}.binvox.bt): dense occupancy of the bounding box of the occupied leaves,
 * occ_out[(z * ny + y) * nx + x] (1 = occupied, 0 = free or unknown), pruned leaves expanded; origin_key_xyz = key of
 * the first cell per axis (cell k spans [(k - 32768) res, (k - 32767) res)), res = leaf size (both nullable). */
int lmcma_b200_load_bt(const char* path, uint8_t* occ_out, int64_t capacity, int32_t* shape_xyz, int32_t* origin_key_xyz, double* res);
/* comma-separated matrix, one row per line: the file populate_EDT_Matrix_old reads into EDT_Matrix (planner.cpp:777-818) */
int lmcma_b200_load_text_matrix(const char* path, double* out, int64_t capacity, int32_t* rows, int32_t* cols);

#ifdef __cplusplus
}
#endif
#endif /* LMCMA_B200_H */
