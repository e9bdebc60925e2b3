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

    def update_occupancy(self, lo_xyz, occ_box):
        """Replace the occupancy of a box of a map built by from_occupancy (non-zero = obstacle): occ_box is [sz, sy, sx]
        or [sy, sx] like the grid, lo_xyz its first cell (x, y[, z]).  Afterwards the map holds what from_occupancy of the
        edited grid would hold; optimisers attached to it see the new map on their next run.  Synchronise them first."""
        o = np.ascontiguousarray(np.asarray(occ_box) != 0, np.uint8)
        if o.ndim != self.dims:
            raise ValueError("occ_box has %d dimensions, the map %d" % (o.ndim, self.dims))
        lo = np.array(lo_xyz, np.int32).reshape(self.dims)
        size = np.array(o.shape[::-1], np.int32)
        K.check(K.lib().lmcma_b200_map_update_occupancy(self._h, K.iptr(lo), K.iptr(size), o.ctypes.data_as(C.POINTER(C.c_uint8))))

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


class _DeviceBuffer:
    """One of an optimiser's device buffers as a __cuda_array_interface__ (FP32, or typestr).  A tensor made from it holds a
    reference to it, and through `owner` to the optimiser, so garbage collection cannot free the memory under it (close()
    still does).  torch takes no read-only flag: that
    X must not be written is the caller's part (device_tensors)."""

    def __init__(self, owner, ptr, shape, strides, typestr="<f4"):
        self.owner = owner
        self.__cuda_array_interface__ = {"shape": shape, "strides": strides, "typestr": typestr, "data": (ptr, False),
                                         "version": 2}


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
        self.device = int(device)
        self._map = None
        self._stream = None          # set_stream: None = the handle's own non-blocking stream

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

    def device_tensors(self):
        """torch views (X [batch, pop_count, n], F [batch, lambda]) over the handle's device buffers, for a cost computed on
        the GPU: read the population from X, write every fitness into F, then call tell_all_dev.  X is READ-ONLY (its rows
        have stride ld floats); F must be fully written before each tell.  The views keep this optimiser from being garbage
        collected, but close() frees the buffers under them: do not use them after close().

        The handle's work must be ordered with the cost's: run the cost on a torch.cuda.Stream() (not the default stream)
        and put the handle on it first, set_stream(s.cuda_stream).  The default stream's cuda_stream is 0, which selects the
        handle's own non-blocking stream, and nothing torch enqueues is ordered with that one; tell_all_dev refuses it.
        Nothing is allocated, so a torch.cuda.graph capture may follow at once."""
        import torch                                             # only this method needs torch
        xp, fp, ld = C.c_void_p(), C.c_void_p(), C.c_int64(0)
        K.check(K.lib().lmcma_b200_device_buffers(self._h, C.byref(xp), C.byref(ld), C.byref(fp)))
        ld = int(ld.value)
        X = _DeviceBuffer(self, xp.value, (self.batch, self.pop_count, self.n), (self.pop_count * ld * 4, ld * 4, 4))
        F = _DeviceBuffer(self, fp.value, (self.batch, self.lam), (self.lam * 4, 4))
        dev = torch.device("cuda", self.device)
        return torch.as_tensor(X, device=dev), torch.as_tensor(F, device=dev)

    def tell_all_dev(self):
        """update() + sample() from the fitness in device_tensors()'s F, enqueued on the handle's stream; returns without
        waiting.  Same bits as tell_all with the same fitness.  Capturable in torch.cuda.graph (with the handle on the
        capture stream).  PHILOX handles of one unsplit population only.

        Raises (ERR_STATE, nothing enqueued) while the handle runs on its own stream: Python code cannot enqueue a cost on
        that stream, so the tell could not be ordered after it (see device_tensors)."""
        if self._stream is None:
            raise K.LmcmaError(K.ERR_STATE, "tell_all_dev on the handle's own stream: no cost can be ordered before it; "
                               "set_stream(s.cuda_stream) with the (non-default) torch stream the cost runs on")
        K.check(K.lib().lmcma_b200_tell_all_dev(self._h))

    def reset_instances(self, idx, x0, sigma0=None, starts=None, goals=None):
        """Restart the instances idx in place, as a fresh create would start them from x0 [len(idx), n] (or one row for
        all) with step size sigma0 (per instance, one value, or None for the handle's sigma0), on a new deviate stream.
        starts / goals: new end points, one row per instance or one for all (needs an attached cost), or None to keep
        them.  Synchronous; the other instances and the handle's graphs are untouched."""
        idx = np.ascontiguousarray(np.atleast_1d(np.asarray(idx)), np.int32)
        count = len(idx)
        x0a = K.f64c(np.broadcast_to(np.asarray(x0, np.float64), (count, self.n)) if np.ndim(x0) == 1 else x0)
        sg = None if sigma0 is None else K.f64c(np.broadcast_to(np.asarray(sigma0, np.float64), (count,)))
        ends = None
        if starts is not None or goals is not None:
            starts = np.asarray(starts, np.float32).reshape(-1, np.shape(starts)[-1])
            goals = np.asarray(goals, np.float32).reshape(-1, np.shape(goals)[-1])
            if starts.shape[0] == 1 and count > 1:
                starts = np.repeat(starts, count, 0)
                goals = np.repeat(goals, count, 0)
            assert starts.shape[0] == count and goals.shape[0] == count
            ends = (K.Endpoints * count)(*[_endpoints(starts[i], goals[i]) for i in range(count)])
        K.check(K.lib().lmcma_b200_reset_instances(self._h, count, K.iptr(idx), K.dptr(x0a),
                                                   None if sg is None else K.dptr(sg), ends))

    def reset_instances_dev(self, flags, x0, sigma0=None, ends=None, best_x_out=None, best_f_out=None):
        """The reset from flags computed on the device, enqueued on the handle's stream without waiting (capturable in
        torch.cuda.graph, like tell_all_dev).  torch CUDA tensors on this handle's device, contiguous: flags int32 [batch]
        (non-zero = reset), x0 float64 [batch, n] (rows of unflagged instances unused), sigma0 float64 [batch] or None,
        ends float32 [batch, 6] (start xyz, goal xyz) or None; best_x_out float32 [batch, n] / best_f_out float64 [batch]
        or None receive each reset instance's best before the reset.  The library trusts the values (finite x0,
        sigma0 > 0); this method checks dtypes, shapes, devices and contiguity only, without a synchronise."""
        import torch                                             # only the device path needs torch
        if self._stream is None:
            raise K.LmcmaError(K.ERR_STATE, "reset_instances_dev on the handle's own stream: nothing torch enqueues is ordered "
                               "with it; set_stream(s.cuda_stream) with the (non-default) torch stream the flags come from")
        B, n = self.batch, self.n
        want = dict(flags=(torch.int32, (B,)), x0=(torch.float64, (B, n)), sigma0=(torch.float64, (B,)),
                    ends=(torch.float32, (B, 6)), best_x_out=(torch.float32, (B, n)), best_f_out=(torch.float64, (B,)))
        given = dict(flags=flags, x0=x0, sigma0=sigma0, ends=ends, best_x_out=best_x_out, best_f_out=best_f_out)
        ptr = {}
        for name, t in given.items():
            if t is None:
                if name in ("flags", "x0"):
                    raise ValueError("%s is required" % name)
                ptr[name] = None
                continue
            dtype, shape = want[name]
            if not isinstance(t, torch.Tensor) or t.dtype != dtype or tuple(t.shape) != shape:
                raise ValueError("%s must be a %s tensor of shape %s" % (name, dtype, shape))
            if t.device != torch.device("cuda", self.device) or not t.is_contiguous():
                raise ValueError("%s must be contiguous on cuda:%d" % (name, self.device))
            ptr[name] = t.data_ptr()
        K.check(K.lib().lmcma_b200_reset_instances_dev(self._h, ptr["flags"], ptr["x0"], ptr["sigma0"], ptr["ends"],
                                                       ptr["best_x_out"], ptr["best_f_out"]))

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
    def attach_cost(self, cmap_or_maps, starts, goals, waypoints, weights=LONGSAFE, w_col=1e4, map_of=None):
        """The fused generations' cost: one CostMap, or a sequence of CostMaps of one dims and storage with map_of [batch]
        naming each instance's map (lmcma_b200_attach_cost_maps; map_of may be omitted for a single map).  starts / goals:
        one row per instance or one for all.  The handle keeps its maps alive."""
        several = not isinstance(cmap_or_maps, CostMap)
        cmaps = list(cmap_or_maps) if several else [cmap_or_maps]
        if not cmaps:
            raise ValueError("attach_cost needs at least one map")
        dims = cmaps[0].dims
        starts = np.asarray(starts, np.float32).reshape(-1, dims)
        goals = np.asarray(goals, np.float32).reshape(-1, dims)
        if starts.shape[0] == 1 and self.batch > 1:
            starts = np.repeat(starts, self.batch, 0)
            goals = np.repeat(goals, self.batch, 0)
        assert starts.shape[0] == self.batch
        ends = (K.Endpoints * self.batch)()
        for b in range(self.batch):
            for c in range(dims):
                ends[b].start[c] = float(starts[b, c])
                ends[b].goal[c] = float(goals[b, c])
        obj = _objective(waypoints, weights, w_col)
        if not several:
            if map_of is not None and np.any(np.asarray(map_of) != 0):
                raise ValueError("map_of names maps other than the one given")
            K.check(K.lib().lmcma_b200_attach_cost(self._h, cmap_or_maps._h, C.byref(obj), ends))
        else:
            if map_of is None:
                if len(cmaps) > 1:
                    raise ValueError("map_of is required with several maps")
                map_of = 0
            mo = np.ascontiguousarray(np.broadcast_to(np.asarray(map_of, np.int32), (self.batch,)))
            hs = (C.c_void_p * len(cmaps))(*[m._h for m in cmaps])
            K.check(K.lib().lmcma_b200_attach_cost_maps(self._h, len(cmaps), hs, K.iptr(mo), C.byref(obj), ends))
        self._map = cmaps[0] if not several else cmaps   # keep alive

    def device_map_index(self):
        """torch int32 view [batch] over the handle's map index of every instance (a handle attached to several maps): write
        it on the handle's stream, also inside a torch.cuda.graph capture, and the next cost launch evaluates each instance
        on its new map.  Values must lie in [0, number of maps); an instance whose entry does not gets f = +inf.  Same
        ownership rules as device_tensors."""
        import torch                                             # only this method needs torch
        p = C.c_void_p()
        K.check(K.lib().lmcma_b200_instance_maps_dev(self._h, C.byref(p)))
        buf = _DeviceBuffer(self, p.value, (self.batch,), (4,), "<i4")
        return torch.as_tensor(buf, device=torch.device("cuda", self.device))

    def run(self, generations, sync=True):
        K.check(K.lib().lmcma_b200_run(self._h, int(generations)))
        if sync:
            self.sync()

    def sync(self):
        K.check(K.lib().lmcma_b200_sync(self._h))

    def set_stream(self, stream):
        """int cudaStream_t to run on; None or 0 = the handle's own non-blocking stream"""
        K.check(K.lib().lmcma_b200_set_stream(self._h, stream))
        self._stream = stream or None

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

    def rescore_best(self):
        """best_f <- the cost of best_x on the attached map as it is now (after CostMap.update_occupancy), for every
        instance evaluated at least once; on a handle with several maps each instance's own map."""
        K.check(K.lib().lmcma_b200_rescore_best(self._h))

    # ---- state ----
    def _shape_of(self, name):
        B, n, m, lam, pc, mu = self.batch, self.n, self.m, self.lam, self.pop_count, self.mu
        return {"xmean": (B, n), "sigma": (B,), "s": (B,), "best_f": (B,), "consts": (7,), "weights": (mu,),
                "Nj": (B, m), "Lj": (B, m), "X": (B, pc, n), "Z": (B, pc, n), "pc": (B, n), "V": (B, m, n),
                "P": (B, m, n), "fit": (B, lam), "fit_sorted": (B, lam), "prev_fit": (B, lam), "t": (B, m),
                "vec": (B, m), "arindex": (B, lam), "rank": (B, lam), "itr": (B,), "live": (B,),
                "counteval": (B,), "ncoll": (B, pc), "nsamp": (B, pc), "epoch": (B,), "map_of": (B,)}[name]

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
