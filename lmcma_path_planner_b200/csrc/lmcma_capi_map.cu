// lmcma_capi_map.cu — cost map handles (bricked storage, device distance transform), the batched trajectory cost evaluator
// and its launch selection.  Part of liblmcma_b200.so (see lmcma_internal.cuh).
#include "lmcma_internal.cuh"
#include "k_cost.cuh"
#include "k_edt.cuh"

using namespace lmcma;
using namespace lmcma_capi;

namespace {
template <int DIMS, int STORAGE, bool TRACE, int MINB = 7>
int launch_cost_t(const MapDev& mp, const CostArgs& a0, int rows, int B, CostShape shape, cudaStream_t st) {
    CostArgs a = a0;
    a.spt = (a.W + 1 + shape.tpt - 1) / shape.tpt;
    a.cb = shape.cb & ~1;                                       // even: k_cost zeroes two block records per store
    // segment records 36 B, sample offsets, per-block records 8 B (k_cost.cuh), 256-entry table (u8 storage)
    // + the candidate row (16-byte aligned)
    const size_t smem = (size_t)36 * (a.W + 1) + sizeof(int) * (a.W + 2) + 28 + (size_t)8 * shape.cb + (STORAGE == 1 ? 1024 : 0) +
                        sizeof(float) * DIMS * ((size_t)a.W + 2) + 16;
    return launch(k_cost<DIMS, STORAGE, TRACE, MINB>, dim3(rows, B), shape.tpt, smem, st, false, mp, a);
}

}  // namespace

namespace lmcma_capi {
int launch_cost(const MapDev& mp, const CostArgs& a, int rows, int B, CostShape shape, bool trace, cudaStream_t st) {
    if (rows <= 0 || B <= 0) return 0;
    if (trace) {
        if (mp.dims == 2) return mp.storage == 0 ? launch_cost_t<2, 0, true>(mp, a, rows, B, shape, st) : launch_cost_t<2, 1, true>(mp, a, rows, B, shape, st);
        return mp.storage == 0 ? launch_cost_t<3, 0, true>(mp, a, rows, B, shape, st) : launch_cost_t<3, 1, true>(mp, a, rows, B, shape, st);
    }
    // seven CTAs per SM (32 registers, 28 / 36 B of spills outside the sample loop) keep a 1024-trajectory population resident in
    // ONE wave.  The 40-register build at six per SM was 7 % faster from four waves on in round 1 (0.280 -> 0.261 ms for 16384
    // trajectories); after round 2's instruction diet of the phases around the loop it is the other way round in 2-D (C3 batch
    // of 262144 trajectories: 3.39 ms at seven per SM, 3.47 ms at six), so 2-D launches always take the seven-per-SM build
    const int minb = shape.minb ? shape.minb : (mp.dims == 3 && (long long)rows * B >= 4LL * 7 * 148 ? 6 : 7);
    if (minb == 6) {
        if (mp.dims == 2) return mp.storage == 0 ? launch_cost_t<2, 0, false, 6>(mp, a, rows, B, shape, st) : launch_cost_t<2, 1, false, 6>(mp, a, rows, B, shape, st);
        return mp.storage == 0 ? launch_cost_t<3, 0, false, 6>(mp, a, rows, B, shape, st) : launch_cost_t<3, 1, false, 6>(mp, a, rows, B, shape, st);
    }
    if (mp.dims == 2) return mp.storage == 0 ? launch_cost_t<2, 0, false>(mp, a, rows, B, shape, st) : launch_cost_t<2, 1, false>(mp, a, rows, B, shape, st);
    return mp.storage == 0 ? launch_cost_t<3, 0, false>(mp, a, rows, B, shape, st) : launch_cost_t<3, 1, false>(mp, a, rows, B, shape, st);
}

// CTA width and per-block record capacity of k_cost from the expected samples per trajectory
CostShape pick_cost_shape(int W, const float* start, const float* goal, int dims, const Tuning& tune) {
    float linf = 0.f;
    if (start && goal)
        for (int c = 0; c < dims; ++c) linf = std::max(linf, std::fabs(goal[c] - start[c]));
    const double est = 2.0 * (W + 1) + linf;     // expected samples per trajectory
    CostShape sh;
    sh.tpt = 32;
    // enough lanes for the samples, and a thread per segment (phase 1 is a chain of dependent loads per segment);
    // k_cost is built for at most 8 warps (COST_MAX_WARPS)
    while (sh.tpt < 256 && (est / sh.tpt > 24.0 || W + 1 > sh.tpt)) sh.tpt <<= 1;
    const int forced = tune.cost_tpt;
    if (forced >= 32 && forced <= 256 && forced % 32 == 0) sh.tpt = forced;
    sh.minb = tune.cost_minb;
    // 32-sample blocks whose records are staged at once (longer trajectories take several rounds): ~3x the estimate
    sh.cb = 64;
    while (sh.cb < 2048 && sh.cb * 32.0 < 3.0 * est) sh.cb <<= 1;
    const int forced_cb = tune.cost_cb;
    if (forced_cb >= 8 && forced_cb <= 4096) sh.cb = forced_cb;
    return sh;
}

}  // namespace lmcma_capi

namespace {
// device-side alias of a page-locked host buffer (unified addressing), or null for pageable / foreign memory
void* mapped_device_pointer(const void* host, int device) {
    cudaPointerAttributes at;
    memset(&at, 0, sizeof(at));
    if (cudaPointerGetAttributes(&at, host) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    if (at.type != cudaMemoryTypeHost || !at.devicePointer) return nullptr;
    (void)device;
    return at.devicePointer;
}

// Page-locked host mirrors of candidate populations handed out by lmcma_b200_ask_all_view: lmcma_b200_cost_evaluate
// recognises a pointer into one of them and evaluates the DEVICE copy it mirrors (no H2D of the candidates).
struct MirrorEntry { const char* host; size_t bytes; const float* dev; long long ld; int device; };
std::mutex g_mirror_mu;
std::vector<MirrorEntry> g_mirrors;
}  // namespace
namespace lmcma_capi {
void register_mirror(const void* host, size_t bytes, const float* dev, long long ld, int device) {
    std::lock_guard<std::mutex> lk(g_mirror_mu);
    g_mirrors.push_back(MirrorEntry{static_cast<const char*>(host), bytes, dev, ld, device});
}
void unregister_mirror(const void* host) {
    std::lock_guard<std::mutex> lk(g_mirror_mu);
    for (size_t i = 0; i < g_mirrors.size(); ++i)
        if (g_mirrors[i].host == host) { g_mirrors.erase(g_mirrors.begin() + i); break; }
}
}  // namespace lmcma_capi
namespace {
// device row pointer + row stride behind a host pointer that lies inside a registered mirror (row-aligned), else null
const float* mirrored_device_rows(const void* host, int device, size_t need_bytes, long long* ld) {
    std::lock_guard<std::mutex> lk(g_mirror_mu);
    const char* p = static_cast<const char*>(host);
    for (const MirrorEntry& m : g_mirrors) {
        if (m.device != device || p < m.host || p + need_bytes > m.host + m.bytes) continue;
        const size_t off = (size_t)(p - m.host);
        if (off % ((size_t)m.ld * sizeof(float)) != 0) continue;
        *ld = m.ld;
        return m.dev + off / sizeof(float);
    }
    return nullptr;
}

}  // namespace

extern "C" {
// =================================================================================================
// cost map
// =================================================================================================
// handle + device buffers + LUT of a cost map (no contents yet)
extern "C" int lmcma_b200_map_destroy(lmcma_b200_map* m);
static int map_alloc(int device, int dims, const int32_t* shape, int storage, float u8_scale, float c_min, lmcma_b200_map** out) {
    ARG(out && shape, "null pointer");
    ARG(dims == 2 || dims == 3, "dims must be 2 or 3");
    ARG(storage == LMCMA_B200_MAP_F32 || storage == LMCMA_B200_MAP_U8, "unknown storage");
    ARG(c_min > 0.f, "c_min must be > 0");
    ARG(storage == LMCMA_B200_MAP_F32 || u8_scale > 0.f, "u8_scale must be > 0");
    for (int c = 0; c < dims; ++c) ARG(shape[c] >= 1, "bad shape");
    DeviceProps* props;
    int rc = query_props(device, &props);
    if (rc) return rc;
    CU(cudaSetDevice(device));
    lmcma_b200_map* m = new lmcma_b200_map();
    m->tune = Tuning::from_env();
    m->device = device; m->storage = storage; m->c_min = c_min; m->scale = u8_scale;
    m->dev.dims = dims; m->dev.nx = shape[0]; m->dev.ny = shape[1]; m->dev.nz = dims == 3 ? shape[2] : 1;
    m->dev.storage = storage; m->dev.g_coll = 1.0f / c_min;
    m->cells = (size_t)m->dev.nx * m->dev.ny * m->dev.nz;
    const BrickShape bs = dims == 2 ? (storage == 0 ? brick_shape<2, 0>() : brick_shape<2, 1>())
                                    : (storage == 0 ? brick_shape<3, 0>() : brick_shape<3, 1>());
    const unsigned nbx = (m->dev.nx + bs.bx - 1) / bs.bx, nby = (m->dev.ny + bs.by - 1) / bs.by,
                   nbz = (m->dev.nz + bs.bz - 1) / bs.bz;
    m->dev.nbx = nbx; m->dev.nby = nby;
    if (dims == 2) { m->dev.py = storage == 0 ? brick_pitch_y<2, 0>(nbx) : brick_pitch_y<2, 1>(nbx); m->dev.pz = 0; }
    else {
        m->dev.py = storage == 0 ? brick_pitch_y<3, 0>(nbx) : brick_pitch_y<3, 1>(nbx);
        m->dev.pz = storage == 0 ? brick_pitch_z<3, 0>(nbx, nby) : brick_pitch_z<3, 1>(nbx, nby);
    }
    m->stored = (size_t)nbx * nby * nbz * bs.bx * bs.by * bs.bz;
    if (m->stored >= ((size_t)1 << 32)) { delete m; return fail(LMCMA_B200_ERR_ARG, "map too large: %zu stored cells (limit 2^32)", m->stored); }
    rc = 0;
    cudaError_t e = cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) rc = fail(LMCMA_B200_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
    if (!rc && storage == LMCMA_B200_MAP_F32) { rc = dmalloc(&m->d_g32, m->stored); m->dev.g32 = m->d_g32; }   // padding cells are never addressed
    if (!rc && storage == LMCMA_B200_MAP_U8) {
        rc = dmalloc(&m->d_q8, m->stored);
        if (!rc) rc = dmalloc(&m->d_lut, 256);
        if (!rc) {
            float lut[256];
            lut[0] = -m->dev.g_coll;
            for (int v = 1; v < 256; ++v) lut[v] = 1.0f / std::max((float)v * u8_scale, c_min);
            e = cudaMemcpy(m->d_lut, lut, sizeof(lut), cudaMemcpyHostToDevice);
            if (e != cudaSuccess) rc = fail(LMCMA_B200_ERR_CUDA, "cudaMemcpy: %s", cudaGetErrorString(e));
        }
        m->dev.q8 = m->d_q8; m->dev.lut = m->d_lut;
    }
    if (rc) { lmcma_b200_map_destroy(m); return rc; }
    *out = m;
    return 0;
}

// row-major distance field on the device -> the bricked storage (values + layout, lmcma_layout.hpp)
static int map_fill_from_dist_dev(lmcma_b200_map* m, const float* d_dist, cudaStream_t st) {
    const MapDev& d = m->dev;
    const unsigned blocks = (unsigned)((m->cells + 255) / 256);
    auto kern = d.dims == 2 ? (m->storage == 0 ? k_brick<2, 0> : k_brick<2, 1>) : (m->storage == 0 ? k_brick<3, 0> : k_brick<3, 1>);
    return launch(kern, blocks, 256, 0, st, false, d_dist, m->d_g32, m->d_q8, d.nx, d.ny, d.nz, d.nbx, d.nby, m->c_min, m->scale);
}

// exact Euclidean distance transform on the device (k_edt.cuh): d_occ (1 = obstacle) -> d_dist, both row-major [z][y][x]
static int edt_device(int dims, const int32_t* shape, const unsigned char* d_occ, float clamp, float* d_dist, cudaStream_t st) {
    const int nx = shape[0], ny = shape[1], nz = dims == 3 ? shape[2] : 1;
    ARG(nx <= 32767 && ny <= 32767 && nz <= 32767, "axis longer than 32767 cells");
    const size_t cells = (size_t)nx * ny * nz;
    unsigned *d2 = nullptr, *gh = nullptr;   // squared distances (k_edt.cuh)
    int *s = nullptr, *t = nullptr;
    int rc = dmalloc(&d2, cells);
    if (!rc) rc = dmalloc(&s, cells);
    if (!rc) rc = dmalloc(&t, cells);
    if (!rc) rc = dmalloc(&gh, cells);
    if (!rc) {
        const long long nlines = (long long)ny * nz, ylines = (long long)nx * nz, zlines = (long long)nx * ny;
        rc = launch(k_edt_x, (unsigned)((nlines + 7) / 8), 256, 0, st, false, d_occ, d2, nx, nlines);
        if (!rc && ny > 1) rc = launch(k_edt_axis, (unsigned)((ylines + 127) / 128), 128, 0, st, false, d2, ny, nx, nx, nz, (long long)nx * ny, s, t, gh);
        if (!rc && nz > 1) rc = launch(k_edt_axis, (unsigned)((zlines + 127) / 128), 128, 0, st, false, d2, nz, (long long)nx * ny, nx * ny, 1, 0, s, t, gh);
        if (!rc) rc = launch(k_edt_finish, (unsigned)((cells + 255) / 256), 256, 0, st, false, d2, d_dist, (long long)cells, clamp);
        cudaError_t e = cudaStreamSynchronize(st);
        if (!rc && e != cudaSuccess) rc = fail(LMCMA_B200_ERR_CUDA, "distance transform: %s", cudaGetErrorString(e));
    }
    cudaFree(d2); cudaFree(s); cudaFree(t); cudaFree(gh);
    return rc;
}

int lmcma_b200_map_create(int device, int dims, const int32_t* shape, const float* dist, int storage, float u8_scale,
                          float c_min, lmcma_b200_map** out) {
    ARG(dist, "null pointer");
    lmcma_b200_map* m = nullptr;
    int rc = map_alloc(device, dims, shape, storage, u8_scale, c_min, &m);
    if (rc) return rc;
    float* d_dist = nullptr;
    rc = dmalloc(&d_dist, m->cells);
    if (!rc) {
        cudaError_t e = cudaMemcpyAsync(d_dist, dist, m->cells * sizeof(float), cudaMemcpyHostToDevice, m->stream);
        if (e != cudaSuccess) rc = fail(LMCMA_B200_ERR_CUDA, "cudaMemcpy: %s", cudaGetErrorString(e));
    }
    if (!rc) rc = map_fill_from_dist_dev(m, d_dist, m->stream);
    if (!rc) { cudaError_t e = cudaStreamSynchronize(m->stream); if (e != cudaSuccess) rc = fail(LMCMA_B200_ERR_CUDA, "map upload: %s", cudaGetErrorString(e)); }
    cudaFree(d_dist);
    if (rc) { lmcma_b200_map_destroy(m); return rc; }
    *out = m;
    return 0;
}

int lmcma_b200_edt(int device, int dims, const int32_t* shape, const uint8_t* occ_host, float clamp, float* dist_host_out) {
    ARG(shape && occ_host && dist_host_out, "null pointer");
    ARG(dims == 2 || dims == 3, "dims must be 2 or 3");
    for (int c = 0; c < dims; ++c) ARG(shape[c] >= 1, "bad shape");
    DeviceProps* props;
    int rc = query_props(device, &props);
    if (rc) return rc;
    CU(cudaSetDevice(device));
    const size_t cells = (size_t)shape[0] * shape[1] * (dims == 3 ? shape[2] : 1);
    unsigned char* d_occ = nullptr; float* d_dist = nullptr;
    rc = dmalloc(&d_occ, cells);
    if (!rc) rc = dmalloc(&d_dist, cells);
    if (!rc) { cudaError_t e = cudaMemcpy(d_occ, occ_host, cells, cudaMemcpyHostToDevice); if (e != cudaSuccess) rc = fail(LMCMA_B200_ERR_CUDA, "cudaMemcpy: %s", cudaGetErrorString(e)); }
    if (!rc) rc = edt_device(dims, shape, d_occ, clamp, d_dist, 0);
    if (!rc) { cudaError_t e = cudaMemcpy(dist_host_out, d_dist, cells * sizeof(float), cudaMemcpyDeviceToHost); if (e != cudaSuccess) rc = fail(LMCMA_B200_ERR_CUDA, "cudaMemcpy: %s", cudaGetErrorString(e)); }
    cudaFree(d_occ); cudaFree(d_dist);
    return rc;
}

int lmcma_b200_map_create_from_occupancy(int device, int dims, const int32_t* shape, const uint8_t* occ_host, float clamp, int storage,
                                         float u8_scale, float c_min, lmcma_b200_map** out) {
    ARG(occ_host, "null pointer");
    lmcma_b200_map* m = nullptr;
    int rc = map_alloc(device, dims, shape, storage, u8_scale, c_min, &m);
    if (rc) return rc;
    unsigned char* d_occ = nullptr; float* d_dist = nullptr;
    rc = dmalloc(&d_occ, m->cells);
    if (!rc) rc = dmalloc(&d_dist, m->cells);
    if (!rc) { cudaError_t e = cudaMemcpy(d_occ, occ_host, m->cells, cudaMemcpyHostToDevice); if (e != cudaSuccess) rc = fail(LMCMA_B200_ERR_CUDA, "cudaMemcpy: %s", cudaGetErrorString(e)); }
    if (!rc) rc = edt_device(dims, shape, d_occ, clamp, d_dist, m->stream);
    if (!rc) rc = map_fill_from_dist_dev(m, d_dist, m->stream);
    if (!rc) { cudaError_t e = cudaStreamSynchronize(m->stream); if (e != cudaSuccess) rc = fail(LMCMA_B200_ERR_CUDA, "map build: %s", cudaGetErrorString(e)); }
    cudaFree(d_occ); cudaFree(d_dist);
    if (rc) { lmcma_b200_map_destroy(m); return rc; }
    *out = m;
    return 0;
}

int lmcma_b200_map_destroy(lmcma_b200_map* m) {
    if (!m) return 0;
    cudaSetDevice(m->device);
    cudaFree(m->d_g32); cudaFree(m->d_q8); cudaFree(m->d_lut); cudaFree(m->d_X); cudaFree(m->d_f);
    cudaFree(m->d_nc); cudaFree(m->d_ns);
    if (m->stream) cudaStreamDestroy(m->stream);
    delete m;
    return 0;
}

int lmcma_b200_map_dequantized(const lmcma_b200_map* m, float* out) {
    ARG(m && out, "null pointer");
    CU(cudaSetDevice(m->device));
    const int dims = m->dev.dims, storage = m->storage;
    const unsigned nbx = m->dev.nbx, nby = m->dev.nby;
    auto offset_of = [&](unsigned x, unsigned y, unsigned z) -> size_t {
        if (dims == 2) return storage == 0 ? brick_offset<2, 0>(x, y, z, nbx, nby) : brick_offset<2, 1>(x, y, z, nbx, nby);
        return storage == 0 ? brick_offset<3, 0>(x, y, z, nbx, nby) : brick_offset<3, 1>(x, y, z, nbx, nby);
    };
    std::vector<float> g; std::vector<unsigned char> q;
    if (storage == LMCMA_B200_MAP_F32) {
        g.resize(m->stored);
        CU(cudaMemcpy(g.data(), m->d_g32, m->stored * sizeof(float), cudaMemcpyDeviceToHost));
    } else {
        q.resize(m->stored);
        CU(cudaMemcpy(q.data(), m->d_q8, m->stored, cudaMemcpyDeviceToHost));
    }
    for (int z = 0; z < m->dev.nz; ++z)
        for (int y = 0; y < m->dev.ny; ++y)
            for (int x = 0; x < m->dev.nx; ++x) {
                const size_t o = offset_of(x, y, z), i = ((size_t)z * m->dev.ny + y) * m->dev.nx + x;
                // F32 stores 1/max(E, c_min): not invertible below c_min, so report the effective clearance
                if (storage == LMCMA_B200_MAP_F32) out[i] = g[o] < 0.f ? 0.f : 1.0f / g[o];
                else out[i] = (float)q[o] * m->scale;
            }
    return 0;
}

int lmcma_b200_map_set_l2_persist(lmcma_b200_map* m, int enable) {
    ARG(m, "null map");
    CU(cudaSetDevice(m->device));
    DeviceProps* props;
    int rc = query_props(m->device, &props);
    if (rc) return rc;
    const size_t bytes = m->storage == LMCMA_B200_MAP_F32 ? m->stored * 4 : m->stored;
    if (enable) CU(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, std::min(bytes, props->persist_max)));
    m->persist = enable != 0;
    return 0;
}

}  // extern "C"
int lmcma_capi::apply_l2_window(lmcma_b200_map* m, cudaStream_t st) {
    if (!m->persist) return 0;
    DeviceProps* props;
    int rc = query_props(m->device, &props);
    if (rc) return rc;
    int max_win = 0;
    CU(cudaDeviceGetAttribute(&max_win, cudaDevAttrMaxAccessPolicyWindowSize, m->device));
    const size_t bytes = m->storage == LMCMA_B200_MAP_F32 ? m->stored * 4 : m->stored;
    cudaStreamAttrValue v;
    memset(&v, 0, sizeof(v));
    v.accessPolicyWindow.base_ptr = m->storage == LMCMA_B200_MAP_F32 ? (void*)m->d_g32 : (void*)m->d_q8;
    v.accessPolicyWindow.num_bytes = std::min(bytes, (size_t)max_win);
    v.accessPolicyWindow.hitRatio = std::min(1.0f, (float)props->persist_max / (float)std::max<size_t>(bytes, 1));
    v.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    v.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    CU(cudaStreamSetAttribute(st, cudaStreamAttributeAccessPolicyWindow, &v));
    return 0;
}

int lmcma_capi::check_obj(const lmcma_b200_map* m, const lmcma_b200_objective* obj) {
    ARG(m && obj, "null pointer");
    ARG(obj->waypoints >= 1 && obj->waypoints <= 8190, "waypoints out of range");
    return 0;
}
extern "C" {

int lmcma_b200_cost_evaluate_dev(lmcma_b200_map* m, const lmcma_b200_objective* obj, const lmcma_b200_endpoints* ends,
                                 const float* X_dev, int64_t ld, int32_t count, float* f_dev, int32_t* ncoll_dev,
                                 int32_t* nsamp_dev, void* stream) {
    int rc = check_obj(m, obj);
    if (rc) return rc;
    ARG(ends && X_dev && f_dev, "null pointer");
    ARG(count >= 0 && ld >= (int64_t)m->dev.dims * obj->waypoints, "bad count / ld");
    if (count == 0) return 0;
    CU(cudaSetDevice(m->device));
    cudaStream_t st = (cudaStream_t)stream;
    CostArgs a;
    memset(&a, 0, sizeof(a));
    a.W = obj->waypoints; a.w_len = obj->w_len; a.w_clr = obj->w_clr; a.w_col = obj->w_col;
    a.X = X_dev; a.ld = ld; a.inst_rows = count; a.ends = nullptr; a.ends_per_instance = 0;
    for (int c = 0; c < 3; ++c) { a.ends0[c] = ends->start[c]; a.ends0[3 + c] = ends->goal[c]; }   // by value: nothing shared between callers
    a.f = f_dev; a.f_stride = count; a.f_offset = 0; a.ncoll = ncoll_dev; a.nsamp = nsamp_dev;
    if ((rc = apply_l2_window(m, st))) return rc;
    return launch_cost(m->dev, a, count, 1, pick_cost_shape(a.W, ends->start, ends->goal, m->dev.dims, m->tune), false, st);
}

int lmcma_b200_cost_evaluate(lmcma_b200_map* m, const lmcma_b200_objective* obj, const lmcma_b200_endpoints* ends,
                             const float* X_host, int32_t count, float* f_host, int32_t* ncoll_host, int32_t* nsamp_host) {
    int rc = check_obj(m, obj);
    if (rc) return rc;
    ARG(ends && X_host && f_host && count >= 0, "null pointer / negative count");
    if (count == 0) return 0;
    std::lock_guard<std::mutex> lock(m->host_path);   // staging buffers + private stream: one host-buffer call per map at a time
    CU(cudaSetDevice(m->device));
    const size_t n = (size_t)m->dev.dims * obj->waypoints;
    // Page-locked caller buffers (cudaHostAlloc / cudaHostRegister) are handed to the kernel as they are: every CTA reads
    // its own candidate row across PCIe once, coalesced, while other CTAs compute (instead of a serial H2D copy in front
    // of the kernel), and the three results per trajectory are stored straight into the caller's arrays.  Pageable
    // buffers are staged through device memory.  LMCMA_B200_ZEROCOPY=0 forces staging.
    const bool zc = m->tune.zerocopy != 0;
    // a pointer into a population mirror handed out by lmcma_b200_ask_all_view: the device already holds these rows
    long long ld_rows = (long long)n;
    const float* X_dev = nullptr;
    if (zc) {
        long long ld_m = 0;
        const float* mir = mirrored_device_rows(X_host, m->device, 1, &ld_m);
        if (mir && ld_m >= (long long)n && mirrored_device_rows(X_host, m->device, ((size_t)(count - 1) * ld_m + n) * sizeof(float), &ld_m)) { X_dev = mir; ld_rows = ld_m; }
    }
    if (!X_dev && zc) X_dev = static_cast<const float*>(mapped_device_pointer(X_host, m->device));
    float* f_dev = zc ? static_cast<float*>(mapped_device_pointer(f_host, m->device)) : nullptr;
    int32_t* nc_dev = (zc && ncoll_host) ? static_cast<int32_t*>(mapped_device_pointer(ncoll_host, m->device)) : nullptr;
    int32_t* ns_dev = (zc && nsamp_host) ? static_cast<int32_t*>(mapped_device_pointer(nsamp_host, m->device)) : nullptr;
    const bool out_direct = f_dev && (!ncoll_host || nc_dev) && (!nsamp_host || ns_dev);
    if (!X_dev) {
        if (m->d_X_cap < (size_t)count * n) {
            cudaFree(m->d_X); m->d_X = nullptr; m->d_X_cap = 0;
            DM(m->d_X, (size_t)count * n);
            m->d_X_cap = (size_t)count * n;
        }
        CU(cudaMemcpyAsync(m->d_X, X_host, (size_t)count * n * sizeof(float), cudaMemcpyHostToDevice, m->stream));
        X_dev = m->d_X;
    }
    if (!out_direct) {
        if (m->d_out_cap < (size_t)count) {
            cudaFree(m->d_f); cudaFree(m->d_nc); cudaFree(m->d_ns);
            m->d_f = nullptr; m->d_nc = nullptr; m->d_ns = nullptr; m->d_out_cap = 0;
            DM(m->d_f, count); DM(m->d_nc, count); DM(m->d_ns, count);
            m->d_out_cap = count;
        }
        f_dev = m->d_f; nc_dev = m->d_nc; ns_dev = m->d_ns;
    }
    rc = lmcma_b200_cost_evaluate_dev(m, obj, ends, X_dev, (int64_t)ld_rows, count, f_dev, ncoll_host ? nc_dev : nullptr,
                                      nsamp_host ? ns_dev : nullptr, m->stream);
    if (rc) return rc;
    if (!out_direct) {
        CU(cudaMemcpyAsync(f_host, m->d_f, count * sizeof(float), cudaMemcpyDeviceToHost, m->stream));
        if (ncoll_host) CU(cudaMemcpyAsync(ncoll_host, m->d_nc, count * sizeof(int), cudaMemcpyDeviceToHost, m->stream));
        if (nsamp_host) CU(cudaMemcpyAsync(nsamp_host, m->d_ns, count * sizeof(int), cudaMemcpyDeviceToHost, m->stream));
    }
    CU(cudaStreamSynchronize(m->stream));
    return 0;
}

int lmcma_b200_cost_trace(lmcma_b200_map* m, const lmcma_b200_objective* obj, const lmcma_b200_endpoints* ends,
                          const float* x_host, int64_t* cells_host, int64_t max_cells, int64_t* n_cells_out) {
    int rc = check_obj(m, obj);
    if (rc) return rc;
    ARG(ends && x_host && cells_host && n_cells_out && max_cells > 0, "null pointer");
    std::lock_guard<std::mutex> lock(m->host_path);
    CU(cudaSetDevice(m->device));
    const size_t n = (size_t)m->dev.dims * obj->waypoints;
    float* dX = nullptr; float* df = nullptr; int* dns = nullptr; long long* dcells = nullptr;
    rc = dmalloc(&dX, n);
    if (!rc) rc = dmalloc(&df, 1);
    if (!rc) rc = dmalloc(&dns, 1);
    if (!rc) rc = dmalloc(&dcells, (size_t)max_cells);
    if (!rc) {
        cudaError_t e = cudaMemset(dcells, 0xff, (size_t)max_cells * sizeof(long long));
        if (e == cudaSuccess) e = cudaMemcpy(dX, x_host, n * sizeof(float), cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaStreamSynchronize(cudaStreamLegacy);   // the kernel runs on the map's non-blocking stream
        if (e != cudaSuccess) rc = fail(LMCMA_B200_ERR_CUDA, "trace staging: %s", cudaGetErrorString(e));
    }
    if (rc) { cudaFree(dX); cudaFree(df); cudaFree(dns); cudaFree(dcells); return rc; }
    CostArgs a;
    memset(&a, 0, sizeof(a));
    a.W = obj->waypoints; a.w_len = obj->w_len; a.w_clr = obj->w_clr; a.w_col = obj->w_col;
    a.X = dX; a.ld = (long long)n; a.inst_rows = 1; a.ends = nullptr; a.ends_per_instance = 0;
    for (int c = 0; c < 3; ++c) { a.ends0[c] = ends->start[c]; a.ends0[3 + c] = ends->goal[c]; }
    a.f = df; a.f_stride = 1; a.nsamp = dns; a.cells = dcells; a.max_cells = max_cells;
    rc = launch_cost(m->dev, a, 1, 1, pick_cost_shape(a.W, ends->start, ends->goal, m->dev.dims, m->tune), true, m->stream);
    if (!rc) {
        cudaError_t e = cudaStreamSynchronize(m->stream);
        if (e != cudaSuccess) rc = fail(LMCMA_B200_ERR_CUDA, "trace kernel: %s", cudaGetErrorString(e));
    }
    int ns = 0;
    if (!rc) {
        cudaMemcpy(&ns, dns, sizeof(int), cudaMemcpyDeviceToHost);
        cudaMemcpy(cells_host, dcells, (size_t)std::min<int64_t>(ns, max_cells) * sizeof(long long), cudaMemcpyDeviceToHost);
        *n_cells_out = ns;
    }
    cudaFree(dX); cudaFree(df); cudaFree(dns); cudaFree(dcells);
    return rc;
}

}  // extern "C"
