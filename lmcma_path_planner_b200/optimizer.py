"""Python host mirror of the reference-facing interface, over the C ABI (include/lmcma_b200.h).

* ``CostMap``     — the distance map + batched trajectory cost (replaces the global ``EDT_Matrix`` and
  ``ValidityChecker`` / ``ClearanceObjective`` pieces, planner.cpp:37, 587-690).
* ``Optimizer``   — a batch of LM-CMA instances on the device (ask/tell, fused on-device generations).
* ``LMCMA``       — the reference class shape (lmcma.hpp:89-144): same constructor arguments, same
  ``init / getNextParameterVector / setEvaluationFeedback / isBehaviorLearningDone`` protocol and the
  public ``counteval`` / ``BestF`` members, so the parity tests read like the reference's own demo
  (example_lmcma.cpp:28-76).

Nothing here computes on the CPU: every method forwards to liblmcma_b200.so.
"""
import ctypes as C

import numpy as np

from . import _capi as K

SHORTRISKY = (100.0, 1.0)    # planner.cpp:677-682
LONGSAFE = (1.0, 1000.0)     # planner.cpp:684-690


def _objective(waypoints, weights, w_col):
    o = K.Objective()
    o.waypoints = int(waypoints)
    o.w_len, o.w_clr, o.w_col = float(weights[0]), float(weights[1]), float(w_col)
    return o


def _endpoints(start, goal):
    e = K.Endpoints()
    for i in range(3):
        e.start[i] = float(start[i]) if i < len(start) else 0.0
        e.goal[i] = float(goal[i]) if i < len(goal) else 0.0
    return e


class CostMap:
    """dist: float32 [ny, nx] or [nz, ny, nx]; distance (cells) to the nearest obstacle, 0 on obstacles."""

    def __init__(self, dist, storage="f32", u8_scale=0.25, c_min=0.5, device=0):
        d = K.f32c(dist)
        assert d.ndim in (2, 3)
        self.dims = d.ndim
        self.shape = d.shape
        shp = np.array(d.shape[::-1], np.int32)
        self.storage = {"f32": K.MAP_F32, "u8": K.MAP_U8}[storage]
        self.c_min = float(c_min)
        self.device = device
        h = C.c_void_p()
        K.check(K.lib().lmcma_b200_map_create(device, self.dims, K.iptr(shp), K.fptr(d), self.storage,
                                             float(u8_scale), float(c_min), C.byref(h)))
        self._h = h
        self.bytes_per_cell = 4 if self.storage == K.MAP_F32 else 1

    @classmethod
    def from_occupancy(cls, occ, clamp=0.0, storage="f32", u8_scale=0.25, c_min=0.5, device=0):
        """Occupancy grid (non-zero = obstacle) -> distance transform + map storage, all on the device."""
        o = np.ascontiguousarray(np.asarray(occ) != 0, np.uint8)
        self = cls.__new__(cls)
        self.dims, self.shape = o.ndim, o.shape
        self.storage = {"f32": K.MAP_F32, "u8": K.MAP_U8}[storage]
        self.c_min, self.device = float(c_min), device
        shp = np.array(o.shape[::-1], np.int32)
        h = C.c_void_p()
        K.check(K.lib().lmcma_b200_map_create_from_occupancy(device, o.ndim, K.iptr(shp), o.ctypes.data_as(C.POINTER(C.c_uint8)),
                                                             float(clamp), self.storage, float(u8_scale), float(c_min), C.byref(h)))
        self._h = h
        self.bytes_per_cell = 4 if self.storage == K.MAP_F32 else 1
        return self

    def close(self):
        if getattr(self, "_h", None):
            K.lib().lmcma_b200_map_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def dequantized(self):
        out = np.zeros(self.shape, np.float32)
        K.check(K.lib().lmcma_b200_map_dequantized(self._h, K.fptr(out)))
        return out

    def set_l2_persist(self, enable=True):
        K.check(K.lib().lmcma_b200_map_set_l2_persist(self._h, int(enable)))

    def evaluate(self, X, start, goal, waypoints, weights=LONGSAFE, w_col=1e4):
        """Host buffers in, host buffers out (H2D + kernel + D2H)."""
        n = self.dims * waypoints
        X = K.f32c(X).reshape(-1, n)
        cnt = X.shape[0]
        f = np.zeros(cnt, np.float32)
        nc = np.zeros(cnt, np.int32)
        ns = np.zeros(cnt, np.int32)
        obj, ends = _objective(waypoints, weights, w_col), _endpoints(start, goal)
        K.check(K.lib().lmcma_b200_cost_evaluate(self._h, C.byref(obj), C.byref(ends), K.fptr(X), cnt, K.fptr(f),
                                                K.iptr(nc), K.iptr(ns)))
        return {"f": f, "ncoll": nc, "nsamp": ns}

    def evaluate_dev(self, X_ptr, ld, count, f_ptr, start, goal, waypoints, weights=LONGSAFE, w_col=1e4,
                     ncoll_ptr=None, nsamp_ptr=None, stream=None):
        """Device pointers (ints) in / out; enqueues on `stream` (int cudaStream_t, None = legacy default)."""
        obj, ends = _objective(waypoints, weights, w_col), _endpoints(start, goal)
        K.check(K.lib().lmcma_b200_cost_evaluate_dev(self._h, C.byref(obj), C.byref(ends), X_ptr, ld, count, f_ptr,
                                                    ncoll_ptr, nsamp_ptr, stream))

    def trace(self, x, start, goal, waypoints, max_cells=1 << 22):
        x = K.f32c(x)
        cells = np.zeros(max_cells, np.int64)
        n_out = C.c_int64(0)
        obj, ends = _objective(waypoints, LONGSAFE, 0.0), _endpoints(start, goal)
        K.check(K.lib().lmcma_b200_cost_trace(self._h, C.byref(obj), C.byref(ends), K.fptr(x), K.lptr(cells), max_cells,
                                             C.byref(n_out)))
        return cells[:min(n_out.value, max_cells)].copy()


class Optimizer:
    """B independent LM-CMA instances of one shape on one device."""

    def __init__(self, n, x0=None, lam=0, m=0, batch=1, lo=None, hi=None, sigma0=1.0, seed=1, rng="philox",
                 device=0, record_z=False, pop_offset=0, pop_count=0, covariance=None):
        cfg = K.Config()
        cfg.n, cfg.lambda_, cfg.m, cfg.batch = int(n), int(lam), int(m), int(batch)
        cfg.sigma0, cfg.seed = float(sigma0), int(seed)
        cfg.rng = {"philox": K.RNG_PHILOX, "hansen": K.RNG_HANSEN, "inject": K.RNG_INJECT}[rng]
        cfg.device, cfg.record_z = int(device), int(bool(record_z))
        cfg.pop_offset, cfg.pop_count = int(pop_offset), int(pop_count)
        x0a = None if x0 is None else K.f64c(np.broadcast_to(np.asarray(x0, np.float64), (batch, n)) if np.ndim(x0) == 1 else x0)
        loa = None if lo is None else K.f64c(lo)
        hia = None if hi is None else K.f64c(hi)
        cva = None if covariance is None else K.f64c(np.asarray(covariance, np.float64).reshape(n, n))
        h = C.c_void_p()
        K.check(K.lib().lmcma_b200_create_with_prior(C.byref(cfg), None if x0a is None else K.dptr(x0a),
                                                    None if loa is None else K.dptr(loa), None if hia is None else K.dptr(hia),
                                                    None if cva is None else K.dptr(cva), C.byref(h)))
        self._h = h
        shp = np.zeros(8, np.int32)
        K.check(K.lib().lmcma_b200_shape(h, K.iptr(shp)))
        self.n, self.lam, self.mu, self.m, self.batch, self.pop_offset, self.pop_count, self.ld = (int(v) for v in shp)
        self._map = None

    def close(self):
        if getattr(self, "_h", None):
            K.lib().lmcma_b200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- protocol ----
    def ask_all(self):
        X = np.zeros((self.batch, self.pop_count, self.n), np.float32)
        K.check(K.lib().lmcma_b200_ask_all(self._h, K.fptr(X)))
        return X

    def ask_all_view(self):
        """Read-only numpy view [batch, pop_count, n] of the library's page-locked mirror of the population (no copy)."""
        xp, ld = C.POINTER(C.c_float)(), C.c_int64(0)
        K.check(K.lib().lmcma_b200_ask_all_view(self._h, C.byref(xp), C.byref(ld)))
        a = np.ctypeslib.as_array(xp, shape=(self.batch, self.pop_count, int(ld.value)))
        a.flags.writeable = False
        return a[:, :, :self.n]

    def tell_all(self, f):
        f = K.f32c(f).reshape(self.batch, self.lam)
        K.check(K.lib().lmcma_b200_tell_all(self._h, K.fptr(f)))

    def ask_one(self):
        x = np.zeros(self.n, np.float64)
        K.check(K.lib().lmcma_b200_ask_one(self._h, K.dptr(x), self.n))
        return x

    def tell_one(self, feedbacks):
        fb = K.f64c(np.atleast_1d(feedbacks))
        K.check(K.lib().lmcma_b200_tell_one(self._h, K.dptr(fb), len(fb)))

    def inject_z(self, Z):
        Z = K.f32c(Z).reshape(self.batch, self.pop_count, self.n)
        K.check(K.lib().lmcma_b200_inject_z(self._h, K.fptr(Z)))

    def resample(self):
        K.check(K.lib().lmcma_b200_resample(self._h))

    def is_done(self):
        d = np.zeros(self.batch, np.int32)
        K.check(K.lib().lmcma_b200_is_done(self._h, K.iptr(d)))
        return d.astype(bool)

    # ---- fused planning ----
    def attach_cost(self, cmap, starts, goals, waypoints, weights=LONGSAFE, w_col=1e4):
        starts = np.asarray(starts, np.float32).reshape(-1, cmap.dims)
        goals = np.asarray(goals, np.float32).reshape(-1, cmap.dims)
        if starts.shape[0] == 1 and self.batch > 1:
            starts = np.repeat(starts, self.batch, 0)
            goals = np.repeat(goals, self.batch, 0)
        assert starts.shape[0] == self.batch
        ends = (K.Endpoints * self.batch)()
        for b in range(self.batch):
            for c in range(cmap.dims):
                ends[b].start[c] = float(starts[b, c])
                ends[b].goal[c] = float(goals[b, c])
        obj = _objective(waypoints, weights, w_col)
        K.check(K.lib().lmcma_b200_attach_cost(self._h, cmap._h, C.byref(obj), ends))
        self._map = cmap   # keep alive

    def run(self, generations, sync=True):
        K.check(K.lib().lmcma_b200_run(self._h, int(generations)))
        if sync:
            self.sync()

    def sync(self):
        K.check(K.lib().lmcma_b200_sync(self._h))

    def set_stream(self, stream):
        K.check(K.lib().lmcma_b200_set_stream(self._h, stream))

    def last_run_ms(self):
        ms = C.c_float(0)
        K.check(K.lib().lmcma_b200_last_run_ms(self._h, C.byref(ms)))
        return ms.value

    def profile_kernels(self, generations):
        ms = np.zeros(4, np.float32)
        K.check(K.lib().lmcma_b200_profile_kernels(self._h, int(generations), K.fptr(ms)))
        return dict(zip(("cost", "rank", "update", "sample"), (float(v) for v in ms)))

    def best(self):
        x = np.zeros((self.batch, self.n), np.float32)
        f = np.zeros(self.batch, np.float32)
        K.check(K.lib().lmcma_b200_best(self._h, K.fptr(x), K.fptr(f)))
        return x, f

    # ---- state ----
    def _shape_of(self, name):
        B, n, m, lam, pc, mu = self.batch, self.n, self.m, self.lam, self.pop_count, self.mu
        return {"xmean": (B, n), "sigma": (B,), "s": (B,), "best_f": (B,), "consts": (7,), "weights": (mu,),
                "Nj": (B, m), "Lj": (B, m), "X": (B, pc, n), "Z": (B, pc, n), "pc": (B, n), "V": (B, m, n),
                "P": (B, m, n), "fit": (B, lam), "fit_sorted": (B, lam), "prev_fit": (B, lam), "t": (B, m),
                "vec": (B, m), "arindex": (B, lam), "rank": (B, lam), "itr": (B,), "live": (B,),
                "counteval": (B,), "ncoll": (B, pc), "nsamp": (B, pc)}[name]

    def get(self, name):
        shp = self._shape_of(name)
        if name in K.F64:
            out = np.zeros(shp, np.float64)
            K.check(K.lib().lmcma_b200_get_f64(self._h, K.F64[name], K.dptr(out), out.size))
        elif name in K.F32:
            out = np.zeros(shp, np.float32)
            K.check(K.lib().lmcma_b200_get_f32(self._h, K.F32[name], K.fptr(out), out.size))
        else:
            out = np.zeros(shp, np.int32)
            K.check(K.lib().lmcma_b200_get_i32(self._h, K.I32[name], K.iptr(out), out.size))
        return out

    def set(self, name, value):
        shp = self._shape_of(name)
        if name in K.F64:
            a = K.f64c(np.broadcast_to(np.asarray(value, np.float64), shp))
            K.check(K.lib().lmcma_b200_set_f64(self._h, K.F64[name], K.dptr(a), a.size))
        elif name in K.F32:
            a = K.f32c(np.broadcast_to(np.asarray(value, np.float32), shp))
            K.check(K.lib().lmcma_b200_set_f32(self._h, K.F32[name], K.fptr(a), a.size))
        else:
            a = np.ascontiguousarray(np.broadcast_to(np.asarray(value, np.int32), shp))
            K.check(K.lib().lmcma_b200_set_i32(self._h, K.I32[name], K.iptr(a), a.size))

    def launch(self):
        """The kernel configuration this handle's launches use (chosen at create from n, lambda, m, batch and the device):
        a dict over _capi.LAUNCH_FIELDS; "sampler" is "narrow", "wide" or "rows"."""
        v = np.zeros(len(K.LAUNCH_FIELDS), np.int32)
        K.check(K.lib().lmcma_b200_get_i32(self._h, K.I32_LAUNCH, K.iptr(v), v.size))
        out = dict(zip(K.LAUNCH_FIELDS, (int(x) for x in v)))
        out["sampler"] = K.SAMPLERS[out["sampler"]]
        return out

    def load_state(self, st):
        """Teacher forcing: load a state dict as produced by oracle.pyoracle._Base.state()."""
        self.set("xmean", st["xmean"]); self.set("sigma", st["sigma"]); self.set("s", st["s"])
        self.set("pc", st["pc"]); self.set("V", st["V"]); self.set("P", st["P"])
        self.set("Nj", st["Nj"]); self.set("Lj", st["Lj"]); self.set("prev_fit", st["prev_fit"])
        self.set("t", st["t"]); self.set("vec", st["vec"]); self.set("itr", st["itr"]); self.set("live", st["live"])

    # ---- split-population plumbing (device pointers as ints) ----
    def mg_payload_floats(self):
        v = C.c_int32(0)
        K.check(K.lib().lmcma_b200_mg_payload_floats(self._h, C.byref(v)))
        return v.value

    def mg_evaluate(self, f_local_ptr, stream=None):
        K.check(K.lib().lmcma_b200_mg_evaluate(self._h, f_local_ptr, stream))

    def mg_rank(self, f_all_ptr, payload_ptr, stream=None):
        K.check(K.lib().lmcma_b200_mg_rank(self._h, f_all_ptr, payload_ptr, stream))

    def mg_update(self, payload_all_ptr, world, stream=None):
        K.check(K.lib().lmcma_b200_mg_update(self._h, payload_all_ptr, int(world), stream))


class LMCMA:
    """The reference's class shape (lmcma.hpp:131-138).  Differences, all deliberate:
    arrays are copied at construction (the reference borrows the pointers, lmcma.cpp:109-110);
    ``inseed < 1`` means seed 1, not wall-clock (lmcma.cpp:40-45), so runs are reproducible;
    ``covariance`` (n x n, symmetric positive definite) enables the smoothness-prior sampling path."""

    def __init__(self, initialParams, lambda_=0, loBounds=None, hiBounds=None, sigma=1.0, covariance=None,
                 inseed=0, verbose=False, m=0, device=0):
        self._args = dict(x0=initialParams, lam=lambda_, m=m, lo=loBounds, hi=hiBounds, sigma0=sigma,
                          seed=max(1, int(inseed)), device=device, covariance=covariance)
        self.verbose = verbose
        self.counteval = 0
        self.BestF = np.finfo(np.float64).max
        self._opt = None

    def init(self, N):
        self._opt = Optimizer(N, rng="hansen", batch=1, **self._args)
        self.N = N

    def getNextParameterVector(self, params=None, N=None):
        x = self._opt.ask_one()
        if params is not None:
            params[:len(x)] = x
        return x

    def setEvaluationFeedback(self, feedbacks, numFeedbacks=None):
        fb = np.atleast_1d(np.asarray(feedbacks, np.float64))
        if numFeedbacks is not None:
            fb = fb[:numFeedbacks]
        f = float(fb.sum())
        self.counteval += 1
        if f < self.BestF or self.counteval == 1:          # lmcma.cpp:192-198
            self.BestF = f
            if self.verbose:
                print("Functions evaluation #%d, value: %g" % (self.counteval, f))
        self._opt.tell_one(fb)

    def isBehaviorLearningDone(self):
        return bool(self._opt.is_done()[0])
