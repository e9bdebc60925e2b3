// lmcma_capi_state.cu — state getters / setters (parity, teacher forcing, checkpointing) and the host-side pieces of the
// reference API (random stream, smoothness prior, the free functions of lmcma.hpp).  Part of liblmcma_b200.so.
#include "lmcma_internal.cuh"

using namespace lmcma;
using namespace lmcma_capi;

extern "C" {
// ---- state access ------------------------------------------------------------------------------
int lmcma_b200_get_f64(lmcma_b200_opt* o, int32_t which, double* out, int64_t cap) {
    ARG(o && out, "null pointer");
    CU(cudaSetDevice(o->cfg.device));
    const OptDev& d = o->d;
    const size_t B = d.B;
    switch (which) {
        case LMCMA_B200_F64_XMEAN:
            ARG(cap >= (int64_t)(B * d.n), "capacity");
            return d2h_rows(out, d.xmean, B, d.n * sizeof(double), d.ns * sizeof(double), o->stream);
        case LMCMA_B200_F64_SIGMA: case LMCMA_B200_F64_S: case LMCMA_B200_F64_BESTF: {
            ARG(cap >= (int64_t)B, "capacity");
            std::vector<Scalars> sc(B);
            CU(cudaMemcpyAsync(sc.data(), d.sc, B * sizeof(Scalars), cudaMemcpyDeviceToHost, o->stream));
            CU(cudaStreamSynchronize(o->stream));
            for (size_t b = 0; b < B; ++b)
                out[b] = which == LMCMA_B200_F64_SIGMA ? sc[b].sigma : (which == LMCMA_B200_F64_S ? sc[b].s : sc[b].best_f);
            return 0;
        }
        case LMCMA_B200_F64_CONSTS:
            ARG(cap >= 7, "capacity");
            out[0] = d.c1; out[1] = d.cc; out[2] = d.cs; out[3] = d.target; out[4] = d.K; out[5] = d.M; out[6] = d.mueff;
            return 0;
        case LMCMA_B200_F64_WEIGHTS:
            ARG(cap >= d.mu, "capacity");
            std::copy(o->weights.begin(), o->weights.end(), out);
            return 0;
        case LMCMA_B200_F64_NJ: case LMCMA_B200_F64_LJ:
            ARG(cap >= (int64_t)(B * d.m), "capacity");
            CU(cudaMemcpyAsync(out, which == LMCMA_B200_F64_NJ ? d.Nj : d.Lj, B * d.m * sizeof(double), cudaMemcpyDeviceToHost, o->stream));
            CU(cudaStreamSynchronize(o->stream));
            return 0;
    }
    return fail(LMCMA_B200_ERR_ARG, "unknown f64 field %d", which);
}

int lmcma_b200_get_f32(lmcma_b200_opt* o, int32_t which, float* out, int64_t cap) {
    ARG(o && out, "null pointer");
    CU(cudaSetDevice(o->cfg.device));
    const OptDev& d = o->d;
    const size_t B = d.B, w = d.n * sizeof(float), p = d.ns * sizeof(float);
    switch (which) {
        case LMCMA_B200_F32_X:
            ARG(cap >= (int64_t)(B * d.pop_count * d.n), "capacity");
            return d2h_rows(out, d.X, B * d.pop_count, w, p, o->stream);
        case LMCMA_B200_F32_Z:
            if (!d.Z) return fail(LMCMA_B200_ERR_STATE, "deviates are not recorded (record_z = 0)");
            ARG(cap >= (int64_t)(B * d.pop_count * d.n), "capacity");
            return d2h_rows(out, d.Z, B * d.pop_count, w, p, o->stream);
        case LMCMA_B200_F32_PC:
            ARG(cap >= (int64_t)(B * d.n), "capacity");
            return d2h_rows(out, d.pc, B, w, p, o->stream);
        case LMCMA_B200_F32_V: case LMCMA_B200_F32_P:
            ARG(cap >= (int64_t)(B * d.m * d.n), "capacity");
            return d2h_rows(out, which == LMCMA_B200_F32_V ? d.V : d.P, B * d.m, w, p, o->stream);
        case LMCMA_B200_F32_FIT: case LMCMA_B200_F32_FIT_SORTED: case LMCMA_B200_F32_PREV_FIT: {
            ARG(cap >= (int64_t)(B * d.lambda), "capacity");
            const float* src = which == LMCMA_B200_F32_FIT ? d.fit : (which == LMCMA_B200_F32_FIT_SORTED ? d.fit_sorted : d.prev_fit);
            CU(cudaMemcpyAsync(out, src, B * d.lambda * sizeof(float), cudaMemcpyDeviceToHost, o->stream));
            CU(cudaStreamSynchronize(o->stream));
            if (which == LMCMA_B200_F32_PREV_FIT)   // the device keeps it in evaluation order; the reference keeps it sorted
                for (size_t b = 0; b < B; ++b) std::sort(out + b * d.lambda, out + (b + 1) * d.lambda);
            return 0;
        }
    }
    return fail(LMCMA_B200_ERR_ARG, "unknown f32 field %d", which);
}

int lmcma_b200_get_i32(lmcma_b200_opt* o, int32_t which, int32_t* out, int64_t cap) {
    ARG(o && out, "null pointer");
    CU(cudaSetDevice(o->cfg.device));
    const OptDev& d = o->d;
    const size_t B = d.B;
    const int* src = nullptr; size_t cnt = 0;
    switch (which) {
        case LMCMA_B200_I32_T: src = d.t; cnt = B * d.m; break;
        case LMCMA_B200_I32_VEC: src = d.vec; cnt = B * d.m; break;
        case LMCMA_B200_I32_ARINDEX: src = d.arindex; cnt = B * d.lambda; break;
        case LMCMA_B200_I32_RANK: src = d.rank; cnt = B * d.lambda; break;
        case LMCMA_B200_I32_NCOLL: src = d.ncoll; cnt = B * d.pop_count; break;
        case LMCMA_B200_I32_NSAMP: src = d.nsamp; cnt = B * d.pop_count; break;
        case LMCMA_B200_I32_ITR: case LMCMA_B200_I32_LIVE: case LMCMA_B200_I32_COUNTEVAL: {
            ARG(cap >= (int64_t)B, "capacity");
            std::vector<Scalars> sc(B);
            CU(cudaMemcpyAsync(sc.data(), d.sc, B * sizeof(Scalars), cudaMemcpyDeviceToHost, o->stream));
            CU(cudaStreamSynchronize(o->stream));
            for (size_t b = 0; b < B; ++b)
                out[b] = which == LMCMA_B200_I32_ITR ? sc[b].itr : (which == LMCMA_B200_I32_LIVE ? sc[b].live : (int)sc[b].counteval);
            return 0;
        }
        case LMCMA_B200_I32_LAUNCH:     // per handle: the launch plan create chose (lmcma_plan.cpp)
            ARG(cap >= LMCMA_B200_LAUNCH_FIELDS, "capacity");
            launch_fields(o->plan, out);
            out[LMCMA_B200_LAUNCH_OVERLAP] = o->overlap ? 1 : 0;   // what the handle runs now, not what the plan allowed
            return 0;
        default: return fail(LMCMA_B200_ERR_ARG, "unknown i32 field %d", which);
    }
    ARG(cap >= (int64_t)cnt, "capacity");
    CU(cudaMemcpyAsync(out, src, cnt * sizeof(int), cudaMemcpyDeviceToHost, o->stream));
    CU(cudaStreamSynchronize(o->stream));
    return 0;
}

int lmcma_b200_set_f64(lmcma_b200_opt* o, int32_t which, const double* in, int64_t count) {
    ARG(o && in, "null pointer");
    o->spec_valid = false;                              // tell_all's speculative update saw the state before this call
    CU(cudaSetDevice(o->cfg.device));
    const OptDev& d = o->d;
    const size_t B = d.B;
    switch (which) {
        case LMCMA_B200_F64_XMEAN:
            ARG(count == (int64_t)(B * d.n), "count");
            return h2d_rows(d.xmean, in, B, d.n * sizeof(double), d.ns * sizeof(double), o->stream);
        case LMCMA_B200_F64_SIGMA: case LMCMA_B200_F64_S: {
            ARG(count == (int64_t)B, "count");
            std::vector<Scalars> sc(B);
            CU(cudaMemcpyAsync(sc.data(), d.sc, B * sizeof(Scalars), cudaMemcpyDeviceToHost, o->stream));
            CU(cudaStreamSynchronize(o->stream));
            for (size_t b = 0; b < B; ++b) (which == LMCMA_B200_F64_SIGMA ? sc[b].sigma : sc[b].s) = in[b];
            CU(cudaMemcpyAsync(d.sc, sc.data(), B * sizeof(Scalars), cudaMemcpyHostToDevice, o->stream));
            CU(cudaStreamSynchronize(o->stream));
            return 0;
        }
        case LMCMA_B200_F64_NJ: case LMCMA_B200_F64_LJ: {
            ARG(count == (int64_t)(B * d.m), "count");
            o->mirror_dirty = true;
            CU(cudaMemcpyAsync(which == LMCMA_B200_F64_NJ ? d.Nj : d.Lj, in, B * d.m * sizeof(double), cudaMemcpyHostToDevice, o->stream));
            if (which == LMCMA_B200_F64_NJ) {
                std::vector<float> f(in, in + B * d.m);
                CU(cudaMemcpyAsync(d.Njf, f.data(), f.size() * sizeof(float), cudaMemcpyHostToDevice, o->stream));
                CU(cudaStreamSynchronize(o->stream));
            }
            CU(cudaStreamSynchronize(o->stream));
            return 0;
        }
    }
    return fail(LMCMA_B200_ERR_ARG, "f64 field %d is not settable", which);
}

int lmcma_b200_set_f32(lmcma_b200_opt* o, int32_t which, const float* in, int64_t count) {
    ARG(o && in, "null pointer");
    o->spec_valid = false;                              // tell_all's speculative update saw the state before this call
    CU(cudaSetDevice(o->cfg.device));
    const OptDev& d = o->d;
    const size_t B = d.B, w = d.n * sizeof(float), p = d.ns * sizeof(float);
    switch (which) {
        case LMCMA_B200_F32_PC:
            ARG(count == (int64_t)(B * d.n), "count");
            return h2d_rows(d.pc, in, B, w, p, o->stream);
        case LMCMA_B200_F32_V: case LMCMA_B200_F32_P:
            ARG(count == (int64_t)(B * d.m * d.n), "count");
            o->mirror_dirty = true;
            return h2d_rows(which == LMCMA_B200_F32_V ? d.V : d.P, in, B * d.m, w, p, o->stream);
        case LMCMA_B200_F32_X: {
            ARG(count == (int64_t)(B * d.pop_count * d.n), "count");
            o->x_cache_valid = false;
            o->xh_fresh = false;
            // keep the offsets d = x - xmean consistent with the overwritten candidates
            std::vector<double> xm(B * d.n);
            int rc = d2h_rows(xm.data(), d.xmean, B, d.n * sizeof(double), d.ns * sizeof(double), o->stream);
            if (rc) return rc;
            std::vector<float> dd((size_t)count);
            for (size_t b = 0; b < B; ++b)
                for (size_t r = 0; r < (size_t)d.pop_count; ++r)
                    for (int k = 0; k < d.n; ++k) {
                        const size_t idx = (b * d.pop_count + r) * d.n + k;
                        dd[idx] = (float)((double)in[idx] - xm[b * d.n + k]);
                    }
            if ((rc = h2d_rows(d.D, dd.data(), B * d.pop_count, w, p, o->stream))) return rc;
            return h2d_rows(d.X, in, B * d.pop_count, w, p, o->stream);
        }
        case LMCMA_B200_F32_PREV_FIT:
            ARG(count == (int64_t)(B * d.lambda), "count");
            CU(cudaMemcpyAsync(d.prev_fit, in, B * d.lambda * sizeof(float), cudaMemcpyHostToDevice, o->stream));
            CU(cudaStreamSynchronize(o->stream));
            if (d.prev_sorted) {                                  // the sorted-tile ranking searches an ascending copy
                std::vector<float> srt(in, in + B * d.lambda);
                for (size_t b = 0; b < B; ++b) std::sort(srt.begin() + b * d.lambda, srt.begin() + (b + 1) * d.lambda);
                CU(cudaMemcpy(d.prev_sorted, srt.data(), srt.size() * sizeof(float), cudaMemcpyHostToDevice));
            }
            return 0;
    }
    return fail(LMCMA_B200_ERR_ARG, "f32 field %d is not settable", which);
}

int lmcma_b200_set_i32(lmcma_b200_opt* o, int32_t which, const int32_t* in, int64_t count) {
    ARG(o && in, "null pointer");
    o->spec_valid = false;                              // tell_all's speculative update saw the state before this call
    CU(cudaSetDevice(o->cfg.device));
    const OptDev& d = o->d;
    const size_t B = d.B;
    switch (which) {
        case LMCMA_B200_I32_T: case LMCMA_B200_I32_VEC:
            ARG(count == (int64_t)(B * d.m), "count");
            o->mirror_dirty = true;
            CU(cudaMemcpyAsync(which == LMCMA_B200_I32_T ? d.t : d.vec, in, B * d.m * sizeof(int), cudaMemcpyHostToDevice, o->stream));
            CU(cudaStreamSynchronize(o->stream));
            return 0;
        case LMCMA_B200_I32_ITR: case LMCMA_B200_I32_LIVE: case LMCMA_B200_I32_COUNTEVAL: {
            ARG(count == (int64_t)B, "count");
            std::vector<Scalars> sc(B);
            CU(cudaMemcpyAsync(sc.data(), d.sc, B * sizeof(Scalars), cudaMemcpyDeviceToHost, o->stream));
            CU(cudaStreamSynchronize(o->stream));
            for (size_t b = 0; b < B; ++b) {
                if (which == LMCMA_B200_I32_ITR) sc[b].itr = in[b];
                else if (which == LMCMA_B200_I32_LIVE) sc[b].live = in[b];
                else sc[b].counteval = in[b];
            }
            CU(cudaMemcpyAsync(d.sc, sc.data(), B * sizeof(Scalars), cudaMemcpyHostToDevice, o->stream));
            CU(cudaStreamSynchronize(o->stream));
            return 0;
        }
    }
    return fail(LMCMA_B200_ERR_ARG, "i32 field %d is not settable", which);
}

// ---- host-side reference pieces ------------------------------------------------------------------
int lmcma_b200_hansen_gauss(int64_t seed, int64_t skip, int64_t count, double* out) {
    ARG(out && count >= 0 && skip >= 0, "bad argument");
    HansenStream r(seed);
    for (int64_t i = 0; i < skip; ++i) (void)r.gauss();
    for (int64_t i = 0; i < count; ++i) out[i] = r.gauss();
    return 0;
}
int lmcma_b200_hansen_uniform(int64_t seed, int64_t count, double* out) {
    ARG(out && count >= 0, "bad argument");
    HansenStream r(seed);
    for (int64_t i = 0; i < count; ++i) out[i] = r.uniform();
    return 0;
}
int lmcma_b200_covariance(int32_t dims, int32_t waypoints, double* out) {
    ARG(out && dims >= 1 && waypoints >= 1, "bad argument");
    if (!smoothness_covariance(dims, waypoints, out)) return fail(LMCMA_B200_ERR_ARG, "singular finite-difference block");
    return 0;
}

int lmcma_b200_differentiation_matrix(int32_t num_time_steps, int32_t order, double dt, double* diff_matrix, int32_t row_len) {
    ARG(diff_matrix && num_time_steps >= 1 && order >= 0 && order <= 3 && dt != 0.0, "bad argument");
    ARG(row_len < 0 || row_len >= num_time_steps, "row_len shorter than the block");
    differentiation_matrix(num_time_steps, order, dt, diff_matrix, row_len);
    return 0;
}
int lmcma_b200_invert(const double* A, double* Ainv, int32_t n) {
    ARG(A && Ainv && n >= 1 && A != Ainv, "bad argument");
    if (!invert_dense(A, n, Ainv)) return fail(LMCMA_B200_ERR_ARG, "matrix is singular");
    return 0;
}
int lmcma_b200_apply_cov_l(const double* L_colmajor, double* z, int32_t n) {
    ARG(L_colmajor && z && n >= 1, "bad argument");
    std::vector<double> out(n, 0.0);
    for (int j = 0; j < n; ++j) {                       // column by column: out += z_j * L(:, j)
        const double zj = z[j];
        const double* col = L_colmajor + (size_t)j * n;
        for (int i = 0; i < n; ++i) out[i] += col[i] * zj;
    }
    std::copy(out.begin(), out.end(), z);
    return 0;
}
int lmcma_b200_myqsort(int32_t sz, double* arfitness_inout, int32_t* arindex_out) {
    ARG(sz >= 0 && (sz == 0 || (arfitness_inout && arindex_out)), "bad argument");
    stable_rank(sz, arfitness_inout, arindex_out);
    return 0;
}
struct lmcma_b200_rng { HansenStream s; explicit lmcma_b200_rng(int64_t seed) : s(seed) {} };
int lmcma_b200_rng_create(int64_t seed, lmcma_b200_rng** out) {
    ARG(out, "null pointer");
    *out = new lmcma_b200_rng(seed);
    return 0;
}
int lmcma_b200_rng_destroy(lmcma_b200_rng* r) { delete r; return 0; }
double lmcma_b200_rng_uniform(lmcma_b200_rng* r) { return r ? r->s.uniform() : 0.0; }
double lmcma_b200_rng_gauss(lmcma_b200_rng* r) { return r ? r->s.gauss() : 0.0; }

int lmcma_b200_cholesky(int32_t n, const double* Cm, double* L_out) {
    ARG(Cm && L_out && n >= 1, "bad argument");
    if (!cholesky_lower(Cm, n, L_out)) return fail(LMCMA_B200_ERR_ARG, "matrix is not symmetric positive definite");
    return 0;
}

}  // extern "C"
