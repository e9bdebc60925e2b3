// lmcma_b200.hpp — header-only C++ façade over the C ABI (lmcma_b200.h) with the shape of the reference's
// optimiser class, so that code written against lmcma_path_planner/src/lmcma.hpp:89-144 compiles against
// this header unchanged (see INTEGRATION.md).  Plain C++11, no CUDA / torch headers; link with
// -llmcma_b200.  Nothing in here computes: every method forwards to the device library, and every failure
// of the library throws lmcma_b200::Error (the reference has no error path at all; a silent CPU fallback
// does not exist).
//
//   reference                                              this header
//   LMCMA::LMCMA(...)            lmcma.hpp:131-133          lmcma_b200::LMCMA::LMCMA(...) — same 8 arguments (+ m)
//   LMCMA::init(N)               lmcma.cpp:262-299          LMCMA::init(N)            -> lmcma_b200_create (HANSEN rng)
//   getNextParameterVector       lmcma.cpp:172-182          LMCMA::getNextParameterVector -> lmcma_b200_ask_one
//   setEvaluationFeedback        lmcma.cpp:184-205          LMCMA::setEvaluationFeedback  -> lmcma_b200_tell_one
//   isBehaviorLearningDone       lmcma.cpp:426-429          LMCMA::isBehaviorLearningDone -> lmcma_b200_is_done
//   counteval, BestF             lmcma.hpp:64-65            public members, maintained identically (lmcma.cpp:189-198)
//   class CMABase                lmcma.hpp:41-81            lmcma_b200::CMABase (public surface; the hooks live on the device)
//   covariance, differentiationMatrix, invert, cholesky, applyCovL, random_*, myqsort, compare
//                                lmcma.hpp:26-38, 248-254   same names in namespace lmcma_b200 (global through include/lmcma.hpp)
//   EDT_Matrix + ValidityChecker + ClearanceObjective       lmcma_b200::CostMap (batched evaluate)
//                                planner.cpp:37, 587-690
//   optimal_palnning_without_setting_path planner.cpp:694   lmcma_b200::plan(...) — the fused on-device planner
#ifndef LMCMA_B200_HPP
#define LMCMA_B200_HPP

#include <cfloat>
#include <cstddef>
#include <iostream>
#include <stdexcept>
#include <string>
#include <vector>

#include "lmcma_b200.h"

namespace lmcma_b200 {

struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string& what) : std::runtime_error(what), code(c) {}
};
inline void check(int rc) {
    if (rc != LMCMA_B200_OK) throw Error(rc, std::string("lmcma_b200: ") + lmcma_b200_last_error());
}

// objective weights of the reference (planner.cpp:677-690)
struct Weights { float w_len, w_clr; };
static const Weights kShortRisky = {100.0f, 1.0f};
static const Weights kLongSafe = {1.0f, 1000.0f};

// ---------------------------------------------------------------------------------------------------
// The reference's optimiser class.  Differences, all deliberate and documented in INTEGRATION.md:
//  * pointer arguments are read in init() and COPIED (the reference keeps borrowing lo/hi on every
//    sample(), lmcma.cpp:222-229);
//  * inseed < 1 means seed 1, not wall-clock (lmcma.cpp:40-45), so runs are reproducible;
//  * a `covariance` prior is factored on the host (plain Cholesky instead of Eigen's LLT) and applied on the device;
//  * arithmetic on the device is FP32 for the bulk arrays (FP64 for sigma, s, xmean, Nj, Lj).
// ---------------------------------------------------------------------------------------------------
// The reference's abstract base (lmcma.hpp:41-81): constructor arguments, the public ask / tell protocol and the public
// counters.  The reference's protected members (arx, xmean, weights, ... and the update() / sample() hooks) live on the
// device behind the C ABI here, so a subclass supplies the handle instead of the two hooks; code that only uses the
// public surface (every caller in the reference tree) compiles unchanged.
class CMABase {
public:
    int counteval;
    double BestF;

    CMABase(double* initialParams, int lambda, double* loBounds, double* hiBounds, double* covariance, int inseed,
            bool verbose = false)
        : counteval(0), BestF(DBL_MAX), x0_(initialParams), lo_(loBounds), hi_(hiBounds), cov_(covariance), lambda_(lambda),
          seed_(inseed), verbose_(verbose), n_(0), h_(0) {}
    virtual ~CMABase() { lmcma_b200_destroy(h_); }
    CMABase(const CMABase&) = delete;
    CMABase& operator=(const CMABase&) = delete;

    virtual void init(int N) = 0;
    void getNextParameterVector(double* params, int N) { check(lmcma_b200_ask_one(handle(), params, N)); }
    // lmcma.cpp:184-205.  The fitness crosses the boundary as FP32 (the device ranks FP32 values): |f| beyond FLT_MAX is
    // clamped by the library, costs closer than one FP32 ulp tie and then rank by index.  counteval / BestF are updated
    // only after the library has accepted the value, so host and device protocol state cannot diverge on an error.
    void setEvaluationFeedback(double* feedbacks, int numFeedbacks) {
        check(lmcma_b200_tell_one(handle(), feedbacks, numFeedbacks));
        double f = 0.0;
        for (int i = 0; i < numFeedbacks; ++i) f += feedbacks[i];
        ++counteval;
        if (f < BestF || counteval == 1) {
            BestF = f;
            if (verbose_) std::cout << "Functions evaluation #" << counteval << ", value: " << f << std::endl;
        }
    }
    virtual bool isBehaviorLearningDone() { return false; }      // lmcma.cpp:207-210
    // the batched protocol and the state getters of the C ABI stay reachable
    lmcma_b200_opt* handle() const {
        if (!h_) throw Error(LMCMA_B200_ERR_STATE, "lmcma_b200: init(N) has not been called");
        return h_;
    }

protected:
    double *x0_, *lo_, *hi_, *cov_;
    int lambda_, seed_;
    bool verbose_;
    int n_;
    lmcma_b200_opt* h_;
};

class LMCMA : public CMABase {
public:
    LMCMA(double* initialParams, int lambda = 0, double* loBounds = 0, double* hiBounds = 0, double sigma = 1.0,
          double* covariance = 0, int inseed = 0, bool verbose = false, int m = 0, int device = 0)
        : CMABase(initialParams, lambda, loBounds, hiBounds, covariance, inseed, verbose), m_(m), device_(device), sigma_(sigma) {}

    void init(int N) {
        lmcma_b200_destroy(h_);
        h_ = 0;
        lmcma_b200_config cfg = lmcma_b200_config();
        cfg.n = N; cfg.lambda = lambda_; cfg.m = m_; cfg.batch = 1; cfg.sigma0 = sigma_;
        cfg.seed = seed_ < 1 ? 1 : seed_; cfg.rng = LMCMA_B200_RNG_HANSEN; cfg.device = device_;
        check(lmcma_b200_create_with_prior(&cfg, x0_, lo_, hi_, cov_, &h_));
        n_ = N; counteval = 0; BestF = DBL_MAX;
    }
    bool isBehaviorLearningDone() {                               // lmcma.cpp:426-429
        int32_t done = 0;
        check(lmcma_b200_is_done(handle(), &done));
        return done != 0;
    }

private:
    int m_, device_;
    double sigma_;
};

// ---------------------------------------------------------------------------------------------------
// The free functions of the reference header (lmcma.hpp:4-38, 248-254), same names, argument meaning and array
// layouts, forwarding to the host-side entry points of the C ABI.  include/lmcma.hpp brings them (and LMCMA / CMABase)
// into the global namespace so that a translation unit written against the reference header compiles unchanged.
// ---------------------------------------------------------------------------------------------------
typedef struct { double value; int id; } sortedvals;              // lmcma.hpp:4-8
struct random_t { lmcma_b200_rng* impl; long unsigned startseed; };   // lmcma.hpp:10-24 (the state lives behind the C ABI)

inline long random_Start(random_t* t, long unsigned inseed) {     // lmcma.cpp:14-33
    if (t->impl) lmcma_b200_rng_destroy(t->impl);
    t->impl = 0;
    if (inseed < 1) inseed = 1;
    check(lmcma_b200_rng_create((int64_t)inseed, &t->impl));
    t->startseed = inseed;
    return (long)inseed;
}
inline long random_init(random_t* t, long unsigned inseed) {      // lmcma.cpp:35-47 (inseed < 1: seed 1 here, wall clock there)
    t->impl = 0;
    return random_Start(t, inseed);
}
inline void random_exit(random_t* t) { if (t->impl) lmcma_b200_rng_destroy(t->impl); t->impl = 0; }   // lmcma.cpp:9-12
inline double random_Uniform(random_t* t) { return lmcma_b200_rng_uniform(t->impl); }                 // lmcma.cpp:49-61
inline double random_Gauss(random_t* t) { return lmcma_b200_rng_gauss(t->impl); }                     // lmcma.cpp:63-82
inline int compare(const void* a, const void* b) {                // lmcma.cpp:84-91
    const double x = static_cast<const sortedvals*>(a)->value, y = static_cast<const sortedvals*>(b)->value;
    return x < y ? -1 : (x > y ? 1 : 0);
}
inline void myqsort(int sz, double* arfitness, int* arindex, sortedvals* arr) {   // lmcma.cpp:93-104
    std::vector<int32_t> ids(sz > 0 ? sz : 0);
    check(lmcma_b200_myqsort(sz, arfitness, ids.data()));
    for (int i = 0; i < sz; ++i) { arindex[i] = ids[i]; if (arr) { arr[i].value = arfitness[i]; arr[i].id = ids[i]; } }
}
inline void covariance(int num_dims, int num_waypoints, double* cov) { check(lmcma_b200_covariance(num_dims, num_waypoints, cov)); }   // lmcma.cpp:769-810
inline void differentiationMatrix(int num_time_steps, int order, double dt, double* diff_matrix, int rowLen = -1) {                      // lmcma.cpp:812-834
    check(lmcma_b200_differentiation_matrix(num_time_steps, order, dt, diff_matrix, rowLen));
}
inline void invert(double* A, double* Ainv, int N) { check(lmcma_b200_invert(A, Ainv, N)); }                                            // lmcma.cpp:836-842
// lmcma.cpp:844-855: the reference writes L[m * N + n] = L(n, m), i.e. the lower factor COLUMN-major
inline void cholesky(double* C, double* L, int N) {
    std::vector<double> rowmajor((size_t)N * N);
    check(lmcma_b200_cholesky(N, C, rowmajor.data()));
    for (int r = 0; r < N; ++r)
        for (int c = 0; c < N; ++c) L[(size_t)c * N + r] = rowmajor[(size_t)r * N + c];
}
inline void applyCovL(double* L, double* z, int N) { check(lmcma_b200_apply_cov_l(L, z, N)); }                                          // lmcma.cpp:857-864

// ---------------------------------------------------------------------------------------------------
// Distance map + batched trajectory cost: what the global EDT_Matrix, ValidityChecker::isValid/clearance
// and ClearanceObjective::stateCost provide one state at a time (planner.cpp:37, 587-669).
// dist: row-major [ny][nx] (2-D) or [nz][ny][nx] (3-D), distance in cells, 0 on obstacles.
// ---------------------------------------------------------------------------------------------------
class CostMap {
public:
    CostMap(int dims, const int32_t* shape_xyz, const float* dist, int storage = LMCMA_B200_MAP_F32, float u8_scale = 0.25f,
            float c_min = 0.5f, int device = 0)
        : dims_(dims), h_(0) {
        check(lmcma_b200_map_create(device, dims, shape_xyz, dist, storage, u8_scale, c_min, &h_));
    }
    CostMap(lmcma_b200_map* adopted, int dims) : dims_(dims), h_(adopted) {}   // e.g. from lmcma_b200_map_create_from_occupancy
    ~CostMap() { lmcma_b200_map_destroy(h_); }
    CostMap(const CostMap&) = delete;
    CostMap& operator=(const CostMap&) = delete;
    int dims() const { return dims_; }
    lmcma_b200_map* handle() const { return h_; }

    // X: count x (dims*waypoints) candidates, dimension-major rows; f (and optionally the collision counts) out
    void evaluate(const float* X, int count, int waypoints, const float* start, const float* goal, Weights w, float w_col,
                  float* f, int32_t* ncoll = 0, int32_t* nsamp = 0) const {
        lmcma_b200_objective obj = {waypoints, w.w_len, w.w_clr, w_col};
        lmcma_b200_endpoints e = lmcma_b200_endpoints();
        for (int c = 0; c < dims_; ++c) { e.start[c] = start[c]; e.goal[c] = goal[c]; }
        check(lmcma_b200_cost_evaluate(h_, &obj, &e, X, count, f, ncoll, nsamp));
    }

    // replanning on a changing map built from occupancy: replace the occupancy of the box [lo, lo + size) (occ row-major
    // [sz][sy][sx], non-zero = obstacle); optimiser handles attached to the map see the update on their next run
    void updateOccupancy(const int32_t* lo_xyz, const int32_t* size_xyz, const uint8_t* occ) {
        check(lmcma_b200_map_update_occupancy(h_, lo_xyz, size_xyz, occ));
    }

private:
    int dims_;
    lmcma_b200_map* h_;
};

// ---------------------------------------------------------------------------------------------------
// One planning query solved entirely on the device (the role of optimal_palnning_without_setting_path,
// planner.cpp:694-775, with LM-CMA instead of RRTConnect): straight-line initial mean, box bounds
// [0, size-1] per axis (planner.cpp:696-697), `generations` fused generations, best evaluated path out.
// Returns the best cost; path receives dims*waypoints floats, dimension-major.
// ---------------------------------------------------------------------------------------------------
struct PlanOptions {
    int waypoints, lambda, m, generations;
    double sigma0;
    long long seed;
    Weights weights;
    float w_col;
    int device;
    PlanOptions() : waypoints(20), lambda(0), m(0), generations(200), sigma0(5.0), seed(1), weights(kLongSafe), w_col(1e4f), device(0) {}
};

inline float plan(const CostMap& map, const int32_t* shape_xyz, const float* start, const float* goal, const PlanOptions& po,
                  std::vector<float>* path) {
    const int D = map.dims(), W = po.waypoints, n = D * W;
    std::vector<double> x0(n), lo(n), hi(n);
    for (int d = 0; d < D; ++d)
        for (int w = 0; w < W; ++w) {
            const double t = double(w + 1) / double(W + 1);
            x0[d * W + w] = start[d] + (goal[d] - start[d]) * t;
            lo[d * W + w] = 0.0;
            hi[d * W + w] = double(shape_xyz[d] - 1);
        }
    lmcma_b200_config cfg = lmcma_b200_config();
    cfg.n = n; cfg.lambda = po.lambda; cfg.m = po.m; cfg.batch = 1; cfg.sigma0 = po.sigma0; cfg.seed = po.seed;
    cfg.rng = LMCMA_B200_RNG_PHILOX; cfg.device = po.device;
    lmcma_b200_opt* h = 0;
    check(lmcma_b200_create(&cfg, x0.data(), lo.data(), hi.data(), &h));
    lmcma_b200_objective obj = {W, po.weights.w_len, po.weights.w_clr, po.w_col};
    lmcma_b200_endpoints e = lmcma_b200_endpoints();
    for (int c = 0; c < D; ++c) { e.start[c] = start[c]; e.goal[c] = goal[c]; }
    float best = 0.f;
    int rc = lmcma_b200_attach_cost(h, map.handle(), &obj, &e);
    if (!rc) rc = lmcma_b200_run(h, po.generations);
    if (!rc) rc = lmcma_b200_sync(h);
    if (!rc && path) path->resize(n);
    if (!rc) rc = lmcma_b200_best(h, path ? path->data() : 0, &best);
    std::string err = rc ? lmcma_b200_last_error() : "";
    lmcma_b200_destroy(h);
    if (rc) throw Error(rc, "lmcma_b200: " + err);
    return best;
}

}  // namespace lmcma_b200

#endif  // LMCMA_B200_HPP
