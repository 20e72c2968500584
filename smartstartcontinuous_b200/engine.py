"""Python host side of the C ABI: one ``Engine`` = one ``ss_ctx`` = one GPU.

The two seams of the reference map to two methods:

  Engine.select_start(...)  -> smartexplorationcontinuous.py:260-280 (KDE + UCB + argmax)
  Engine.plan(...)          -> NND_MB_agent.get_best_sim_actions, NND_MB_agent.py:498-520

Error codes of the library are mapped to the exception classes the reference raises
(ValueError / numpy.linalg.LinAlgError / AssertionError-like ValueError); a missing
library or GPU raises -- nothing here computes on the CPU.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import (PENALTY_PER_SAMPLE, PENALTY_REFERENCE, PRECISION_AUTO, PRECISION_BF16_TC,
                   PRECISION_FP32, PRECISION_FP64)

_PENALTY = {"reference": PENALTY_REFERENCE, "per_sample": PENALTY_PER_SAMPLE,
            PENALTY_REFERENCE: PENALTY_REFERENCE, PENALTY_PER_SAMPLE: PENALTY_PER_SAMPLE}
_PRECISION = {"fp32": PRECISION_FP32, "bf16_tc": PRECISION_BF16_TC, "auto": PRECISION_AUTO, "fp64": PRECISION_FP64,
              PRECISION_FP32: PRECISION_FP32, PRECISION_BF16_TC: PRECISION_BF16_TC,
              PRECISION_AUTO: PRECISION_AUTO, PRECISION_FP64: PRECISION_FP64}


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


class _NumpyGlobalMT:
    """Direct access to the MT19937 state struct of numpy's global legacy generator (the one behind
    np.random.uniform): BitGenerator.ctypes.state_address points at {uint32 key[624]; int pos}.  The library
    then reads and advances numpy's state in place -- np.random.get_state() / set_state() cost 50-150 us per
    round trip, more than a small decision.  Verified against get_state() once per generator object; any
    surprise (another bit generator, another layout) disables it and the caller uses get_state / set_state."""

    _checked = {}

    @classmethod
    def address(cls):
        try:
            bg = np.random.mtrand._rand._bit_generator
            ok = cls._checked.get(id(bg))
            if ok is None:
                ok = False
                if type(bg).__name__ == "MT19937":
                    addr = bg.ctypes.state_address
                    addr = addr if isinstance(addr, int) else C.cast(addr, C.c_void_p).value
                    st = np.random.get_state()
                    key = np.ctypeslib.as_array((C.c_uint32 * 624).from_address(addr))
                    if st[0] == "MT19937" and np.array_equal(key, st[1]) and \
                            C.c_int.from_address(addr + 2496).value == st[2]:
                        ok = (bg, addr)                 # keep the object alive with its address
                cls._checked[id(bg)] = ok
            if not ok or ok[0] is not bg:
                return None
            return ok[1]
        except Exception:
            return None


class _DevicePointer(int):
    """A device address handed to the library in place of a host array."""


def _ptr(a):
    """Address for a c_void_p argument (an int: ndarray.ctypes.data_as costs twice as much per argument)."""
    if a is None:
        return None
    if isinstance(a, _DevicePointer):
        return int(a)
    return a.ctypes.data


def _bounds(v, da):
    """Action bound as contiguous float64 [da] (no copy when it already is one)."""
    if v is None:
        return None
    if isinstance(v, np.ndarray) and v.dtype == np.float64 and v.shape == (da,) and v.flags.c_contiguous:
        return v
    return _f64(np.broadcast_to(np.asarray(v, dtype=np.float64), (da,)))


class Engine:
    def __init__(self, device=0):
        self._lib = _lib.load()
        h = C.c_void_p()
        rc = self._lib.ss_create(C.byref(h), int(device))
        if rc != 0:
            msg = self._lib.ss_last_error(None).decode()
            raise RuntimeError("ss_create(device=%d) failed (%d): %s" % (device, rc, msg))
        self._h = h
        self.device = int(device)
        self._model_shape = None
        self._keepalive = []

    # ------------------------------------------------------------------ plumbing
    def close(self):
        if getattr(self, "_h", None):
            self._lib.ss_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc == 0:
            return
        msg = self._lib.ss_last_error(self._h).decode()
        if rc == _lib.SS_ESINGULAR:
            raise np.linalg.LinAlgError(msg)
        if rc in (_lib.SS_EINVAL, _lib.SS_EUNSUPPORTED):
            raise ValueError(msg)
        raise RuntimeError("libss_b200 error %d: %s" % (rc, msg))

    def set_stream(self, cuda_stream_handle):
        self._check(self._lib.ss_set_stream(self._h, C.c_void_p(int(cuda_stream_handle))))

    def device_info(self):
        v = [C.c_int() for _ in range(4)]
        self._check(self._lib.ss_device_info(self._h, *[C.byref(x) for x in v]))
        return dict(sm_count=v[0].value, cc=(v[1].value, v[2].value), sm_clock_khz=v[3].value)

    def last_timings(self):
        ms = (C.c_float * 8)()
        names = (C.c_char_p * 8)()
        n = self._lib.ss_last_timings(self._h, ms, names, 8)
        return [(names[i].decode(), float(ms[i])) for i in range(n)]

    def set_timing(self, enabled):
        """Per-phase CUDA events (last_timings) on / off.  Off by default: the events between the kernels cost
        ~30 us per call (a third of a K = 4096 decision)."""
        self._check(self._lib.ss_set_timing(self._h, 1 if enabled else 0))

    def launch_count(self):
        return int(self._lib.ss_launch_count(self._h))

    # ------------------------------------------------------------------ stage 1
    def select_start(self, all_states, queries, values, n_transitions, volume=1.0, alpha=1.0,
                     beta=2.0, want_density=False, want_ucb=False):
        """KDE + UCB + argmax.  Returns (best_j, best_ucb, densities | None, ucb | None)."""
        data = _f64(all_states)
        q = _f64(queries)
        if data.ndim != 2 or q.ndim != 2 or data.shape[1] != q.shape[1]:
            raise ValueError("all_states [n+1, d] and queries [m, d] must be 2-D with the same d")
        v = None if values is None else np.ascontiguousarray(np.asarray(values).reshape(-1), dtype=np.float32)
        if v is not None and v.shape[0] != q.shape[0]:
            raise ValueError("values must have one entry per query")
        dens = np.empty(q.shape[0]) if want_density else None
        ucb = np.empty(q.shape[0]) if want_ucb else None
        best = C.c_int64(-1)
        best_ucb = C.c_double(0.0)
        self._check(self._lib.ss_kde_ucb_argmax(
            self._h, _ptr(data), data.shape[0], data.shape[1], _ptr(q), q.shape[0], _ptr(v),
            int(n_transitions), float(volume), float(alpha), float(beta), _ptr(dens), _ptr(ucb),
            C.byref(best), C.byref(best_ucb)))
        return int(best.value), float(best_ucb.value), dens, ucb

    def kde_set_precision(self, precision):
        """Arithmetic of select_start / select_start_mirror / select_start_dev: "fp32" (default; densities to
        ~1e-5) or "fp64" (scipy.stats.gaussian_kde's float64 evaluation operation for operation, alpha * values in
        float32 like numpy: densities to ~1e-13, scipy's choice whenever the top-two UCB gap is larger).  Setting
        the current value costs nothing."""
        codes = {"fp32": PRECISION_FP32, "fp64": PRECISION_FP64}
        if precision not in codes:
            raise ValueError("selection precision must be 'fp32' or 'fp64', got %r" % (precision,))
        self._check(self._lib.ss_kde_set_precision(self._h, codes[precision]))

    # NVLink peer-memory exchange for sharded batches (one process per GPU)
    def peer_setup(self, group=None):
        """Open the peer-memory exchange between the Engines of a torch.distributed group (one node,
        <= 8 ranks): CUDA IPC handles are all-gathered once; afterwards sharded decisions exchange
        their projection sums and winner packages inside the kernels (csrc/peer.cu)."""
        import torch
        import torch.distributed as dist
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        handle = (C.c_ubyte * 64)()
        self._check(self._lib.ss_peer_init(self._h, rank, world, handle))
        dev = torch.device("cuda", self.device) if dist.get_backend(group) == "nccl" else torch.device("cpu")
        mine = torch.tensor(list(bytes(handle)), dtype=torch.uint8, device=dev)
        gathered = torch.empty(64 * world, dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(gathered, mine, group=group)
        blob = bytes(gathered.cpu().numpy().tobytes())
        self._check(self._lib.ss_peer_open(self._h, blob, world))
        dist.barrier(group)

    def peer_setup_single(self):
        """A one-rank exchange (this GPU only): the fused kernels then write to and read from their own
        slots -- used by the single-GPU tests to exercise the exchange kernels."""
        handle = (C.c_ubyte * 64)()
        self._check(self._lib.ss_peer_init(self._h, 0, 1, handle))
        self._check(self._lib.ss_peer_open(self._h, bytes(handle), 1))

    @property
    def peer_ready(self):
        return bool(self._lib.ss_peer_ready(self._h))

    def peer_argmax_merge(self, value, index):
        """np.argmax-ordered pick over every rank's (value, global index) through the peer exchange."""
        v, k = C.c_double(0.0), C.c_int64(-1)
        self._check(self._lib.ss_peer_argmax_merge(self._h, float(value), int(index), C.byref(v), C.byref(k)))
        return float(v.value), int(k.value)

    def peer_close(self):
        self._check(self._lib.ss_peer_close(self._h))

    # critic value net in front of the UCB (SURVEY 8f row f4)
    def set_value_net(self, net):
        """net: dict with 'actor' = [(W1, b1), (W2, b2), (W3, b3)], 'critic' = same (critic W2 is
        [(h1 + da), h2]), optional 'actor_ln' / 'critic_ln' = [(gamma1, beta1), (gamma2, beta2)],
        'last_layer_tanh', 'obs_mean' / 'obs_std' / 'obs_clip', 'ret_mean' / 'ret_std' / 'ret_clip'
        (models_editted.py:22-100, ddpg_editted.py:106-131).  None clears it.  With a net set,
        select_start / select_start_mirror accept values=None and compute them on the device."""
        from ._lib import ValueNetStruct
        if net is None:
            self._check(self._lib.ss_value_net_set(self._h, None))
            self._value_net_keep = None
            return
        f32 = lambda a: np.ascontiguousarray(np.asarray(a, dtype=np.float32))
        keep = []

        def ptr(a):
            a = f32(a)
            keep.append(a)
            return a.ctypes.data_as(C.c_void_p)

        (aW1, ab1), (aW2, ab2), (aW3, ab3) = net["actor"]
        (cW1, cb1), (cW2, cb2), (cW3, cb3) = net["critic"]
        st = ValueNetStruct()
        st.d, st.h1a = np.shape(aW1)
        st.h2a, st.da = np.shape(aW3)
        st.h1c, st.h2c = np.shape(cW1)[1], np.shape(cW3)[0]
        if np.shape(cW2) != (st.h1c + st.da, st.h2c) or np.shape(aW2) != (st.h1a, st.h2a) or np.shape(cW1)[0] != st.d:
            raise ValueError("value net: inconsistent layer shapes")
        ln = net.get("actor_ln") is not None
        st.layer_norm, st.last_layer_tanh = int(ln), int(bool(net.get("last_layer_tanh", False)))
        for name, arr in (("aW1", aW1), ("ab1", ab1), ("aW2", aW2), ("ab2", ab2), ("aW3", aW3), ("ab3", ab3),
                          ("cW1", cW1), ("cb1", cb1), ("cW2", cW2), ("cb2", cb2), ("cW3", cW3), ("cb3", cb3)):
            setattr(st, name, ptr(arr))
        if ln:
            (ag1, abe1), (ag2, abe2) = net["actor_ln"]
            (cg1, cbe1), (cg2, cbe2) = net["critic_ln"]
            for name, arr in (("ag1", ag1), ("abe1", abe1), ("ag2", ag2), ("abe2", abe2),
                              ("cg1", cg1), ("cbe1", cbe1), ("cg2", cg2), ("cbe2", cbe2)):
                setattr(st, name, ptr(arr))
        if net.get("obs_mean") is not None:
            om, os_ = _f64(net["obs_mean"]).reshape(-1), _f64(net["obs_std"]).reshape(-1)
            keep += [om, os_]
            st.obs_mean, st.obs_std = _ptr(om), _ptr(os_)
        # both clips are unconditional in the reference graph (ddpg_editted.py:106-109, 130-131);
        # defaults = baselines' observation_range / return_range
        st.obs_clip_lo, st.obs_clip_hi = [float(v) for v in net.get("obs_clip", (-5.0, 5.0))]
        st.ret_clip_lo, st.ret_clip_hi = [float(v) for v in net.get("ret_clip", (-np.inf, np.inf))]
        if net.get("ret_mean") is not None:
            st.has_ret_norm = 1
            st.ret_mean, st.ret_std = float(net["ret_mean"]), float(net["ret_std"])
        self._check(self._lib.ss_value_net_set(self._h, C.byref(st)))
        self._value_net_keep = keep

    def state_values(self, queries):
        """agent.get_state_value(queries) of the value net set with set_value_net: [m] float32."""
        q = _f64(queries)
        out = np.empty(q.shape[0], dtype=np.float32)
        self._check(self._lib.ss_value_net_eval(self._h, _ptr(q), q.shape[0], q.shape[1], _ptr(out)))
        return out

    # device-resident mirror of the replay buffer's state ring (SURVEY 8f row f2)
    def mirror_sync(self, ring):
        """Upload the (s, s2) rows written to ``ring`` (replay_buffer._StateRing) since the last
        call: at most two contiguous H2D copies per array; a new ring object is uploaded whole."""
        state = getattr(self, "_mirror_state", None)
        if state is None or state[0] is not ring or ring.pushes < state[1]:
            state = (ring, 0)
            self._check(self._lib.ss_mirror_reset(self._h))
        done = state[1]
        cap, d = ring.capacity, ring.dim
        todo = ring.pushes - done
        if todo >= ring.count:                       # everything in use changed (or first sync)
            spans = [(0, ring.count)] if ring.count else []
        else:
            r0 = done % cap
            spans = [(r0, min(todo, cap - r0))]
            if todo > cap - r0:
                spans.append((0, todo - (cap - r0)))
        for which, arr in ((0, ring.s), (1, ring.s2)):
            for r0, cnt in spans:
                if cnt > 0:
                    rows = np.ascontiguousarray(arr[r0:r0 + cnt], dtype=np.float64)
                    self._check(self._lib.ss_mirror_write(self._h, which, int(cap), int(d), int(r0), int(cnt), _ptr(rows)))
        self._mirror_state = (ring, ring.pushes)

    def select_start_mirror(self, ring, buffer_indices, values, n_transitions, volume=1.0, alpha=1.0, beta=2.0,
                            want_density=False, want_ucb=False):
        """select_start with the data set and the candidate states taken from the device mirror of
        ``ring``: data = every s + the newest s2, queries = s2 of ``buffer_indices`` (logical buffer
        indices).  Only the m row indices and values are uploaded."""
        self.mirror_sync(ring)
        rows = np.ascontiguousarray(ring.physical_rows(buffer_indices), dtype=np.int64)
        last = int(ring.physical_rows([ring.count - 1])[0])
        v = None if values is None else np.ascontiguousarray(np.asarray(values).reshape(-1), dtype=np.float32)
        if v is not None and v.shape[0] != rows.shape[0]:
            raise ValueError("values must have one entry per query")
        dens = np.empty(rows.shape[0]) if want_density else None
        ucb = np.empty(rows.shape[0]) if want_ucb else None
        best = C.c_int64(-1)
        best_ucb = C.c_double(0.0)
        self._check(self._lib.ss_kde_ucb_argmax_mirror(
            self._h, int(ring.count), last, _ptr(rows), rows.shape[0], _ptr(v), int(n_transitions), float(volume),
            float(alpha), float(beta), _ptr(dens), _ptr(ucb), C.byref(best), C.byref(best_ucb)))
        return int(best.value), float(best_ucb.value), dens, ucb

    def select_start_dev(self, data_ptr, n_pts, d, queries_ptr, m, values_ptr, n_transitions,
                         volume=1.0, alpha=1.0, beta=2.0, density_ptr=None, ucb_ptr=None):
        """Same with device pointers (e.g. torch tensors' data_ptr()); returns (best_j, best_ucb)."""
        best = C.c_int64(-1)
        best_ucb = C.c_double(0.0)
        self._check(self._lib.ss_kde_ucb_argmax_dev(
            self._h, C.c_void_p(data_ptr), int(n_pts), int(d), C.c_void_p(queries_ptr), int(m),
            C.c_void_p(values_ptr), int(n_transitions), float(volume), float(alpha), float(beta),
            C.c_void_p(density_ptr) if density_ptr else None,
            C.c_void_p(ucb_ptr) if ucb_ptr else None, C.byref(best), C.byref(best_ucb)))
        return int(best.value), float(best_ucb.value)

    # ------------------------------------------------------------------ plan set-up geometry
    def path_close_pairs(self, path, radii, theta):
        """Pairs (s, e), e >= s + 2, of path states within theta of each other in the elliptical
        metric, in np.argwhere order: the O(P^2) half of path_shortcutter (numerical.py:226-246)."""
        p = _f64(path)
        r = _f64(radii).reshape(-1)
        if p.ndim != 2 or r.shape[0] != p.shape[1]:
            raise ValueError("path [P, d] and radii [d] expected")
        cap = max(1024, 4 * p.shape[0])
        while True:
            out = np.empty((cap, 2), dtype=np.int32)
            cnt = C.c_int64(0)
            self._check(self._lib.ss_path_close_pairs(self._h, _ptr(p), p.shape[0], p.shape[1], _ptr(r), float(theta),
                                                      _ptr(out), cap, C.byref(cnt)))
            if cnt.value <= cap:
                return out[:cnt.value]
            cap = int(cnt.value)

    def path_shortcut(self, path, radii, theta):
        """Indices of the path states path_shortcutter (numerical.py:226-246) keeps: pair mask and
        interval-scheduling DP both on the device."""
        p = _f64(path)
        r = _f64(radii).reshape(-1)
        if p.ndim != 2 or r.shape[0] != p.shape[1]:
            raise ValueError("path [P, d] and radii [d] expected")
        keep = np.empty(p.shape[0], dtype=np.int32)
        cnt = C.c_int(0)
        self._check(self._lib.ss_path_shortcut(self._h, _ptr(p), p.shape[0], p.shape[1], _ptr(r), float(theta),
                                               _ptr(keep), C.byref(cnt)))
        return keep[:cnt.value]

    # ------------------------------------------------------------------ stage 2
    def set_model(self, weights, biases, norm):
        """weights[l] [in, out] (y = x W + b), biases[l] [out]; norm: dict mean_x std_x mean_y
        std_y mean_z std_z (NND_MB_agent.py:302-315)."""
        ws = [_f64(w) for w in weights]
        bs = [_f64(b).reshape(-1) for b in biases]
        L = len(ws) - 1
        if L < 1 or len(bs) != len(ws):
            raise ValueError("need num_fc_layers + 1 weight matrices and as many biases")
        d = ws[-1].shape[1]
        da = ws[0].shape[0] - d
        h = ws[0].shape[1]
        for l, (w, b) in enumerate(zip(ws, bs)):
            exp_in = d + da if l == 0 else h
            exp_out = d if l == L else h
            if w.shape != (exp_in, exp_out) or b.shape != (exp_out,):
                raise ValueError("layer %d has shape %s / %s, expected (%d, %d)"
                                 % (l, w.shape, b.shape, exp_in, exp_out))
        n = {k: _f64(np.asarray(norm[k]).reshape(-1)) for k in
             ("mean_x", "std_x", "mean_y", "std_y", "mean_z", "std_z")}
        if n["mean_x"].size != d or n["mean_y"].size != da or n["mean_z"].size != d:
            raise ValueError("normalisation statistics do not match the model's d / da")
        wp = (C.c_void_p * len(ws))(*[w.ctypes.data for w in ws])
        bp = (C.c_void_p * len(bs))(*[b.ctypes.data for b in bs])
        self._check(self._lib.ss_mpc_set_model(
            self._h, d, da, L, h, wp, bp, _ptr(n["mean_x"]), _ptr(n["std_x"]), _ptr(n["mean_y"]),
            _ptr(n["std_y"]), _ptr(n["mean_z"]), _ptr(n["std_z"])))
        self._model_shape = (d, da, L, h)

    # ------------------------------------------------------------------ dynamics-model training (row f1)
    def dyn_set_data(self, which, X, Z):
        """Upload a training set (which = 0: initial / "old", 1: aggregated / "new"): X [n, d + da]
        normalised inputs, Z [n, d] normalised state deltas."""
        X, Z = _f64(X), _f64(Z)
        n = X.shape[0] if X.ndim == 2 else 0
        if n and (X.ndim != 2 or Z.ndim != 2 or Z.shape[0] != n):
            raise ValueError("X [n, d + da] and Z [n, d] expected")
        self._check(self._lib.ss_dyn_set_data(self._h, int(which), _ptr(X) if n else None, _ptr(Z) if n else None, n))

    def dyn_train_batches(self, idx_old, idx_new, lr, want_losses=True):
        """Adam steps over explicit batches (row i of idx_old / idx_new = one batch); returns the
        per-batch losses (before each update) or None."""
        io = np.ascontiguousarray(idx_old, dtype=np.int32)
        inw = np.ascontiguousarray(idx_new, dtype=np.int32)
        nb = io.shape[0] if io.size else inw.shape[0]
        n_old = io.shape[1] if io.size else 0
        n_new = inw.shape[1] if inw.size else 0
        losses = np.empty(nb) if want_losses else None
        self._check(self._lib.ss_dyn_train_batches(self._h, _ptr(io) if io.size else None, _ptr(inw) if inw.size else None,
                                                   int(nb), int(n_old), int(n_new), float(lr), _ptr(losses)))
        return losses

    def dyn_eval_loss(self, which, batchsize):
        """(mean batch MSE over the consecutive full batches of data set `which`, number of batches)."""
        out = C.c_double(0.0)
        nb = C.c_int(0)
        self._check(self._lib.ss_dyn_eval_loss(self._h, int(which), int(batchsize), C.byref(out), C.byref(nb)))
        return float(out.value), int(nb.value)

    def dyn_commit(self):
        """Hand the trained parameters to the rollout kernels (device-side re-packing)."""
        self._check(self._lib.ss_dyn_commit(self._h))

    def dyn_reset_optimizer(self):
        self._check(self._lib.ss_dyn_reset_optimizer(self._h))

    def dyn_set_precision(self, precision):
        """Arithmetic of the device trainer: "fp32" (default) or "fp64" (float64 data, masters, moments
        and steps, like the reference's graph).  A change discards the trainer state: training restarts
        from the parameters of the last set_model with fresh Adam moments, and both data sets must be
        uploaded again."""
        codes = {"fp32": PRECISION_FP32, "fp64": PRECISION_FP64}
        if precision not in codes:
            raise ValueError("trainer precision must be 'fp32' or 'fp64', got %r" % (precision,))
        self._check(self._lib.ss_dyn_set_precision(self._h, codes[precision]))

    def dyn_get_params(self):
        """(weights, biases) of the model as float64 numpy ([in, out] / [out])."""
        d, da, L, h = self._model_shape
        sizes = [d + da] + [h] * L + [d]
        ws = [np.empty((i, o)) for i, o in zip(sizes[:-1], sizes[1:])]
        bs = [np.empty(o) for o in sizes[1:]]
        wp = (C.c_void_p * len(ws))(*[w.ctypes.data for w in ws])
        bp = (C.c_void_p * len(bs))(*[b.ctypes.data for b in bs])
        self._check(self._lib.ss_dyn_get_params(self._h, wp, bp))
        return ws, bs

    def tc_supported(self):
        return bool(self._lib.ss_mpc_tc_supported(self._h))

    def last_rollout_kernel(self):
        """Name of the rollout kernel the last decision ran on."""
        return {0: "mpc_rollout_simt_kernel", 1: "mpc_rollout_tc_kernel", 2: "mpc_rollout_tc_quad_kernel",
                3: "mpc_rollout_thread_kernel", 4: "mpc_rollout_fp64_kernel"}.get(
            int(self._lib.ss_mpc_last_kernel(self._h)))

    def set_plan(self, desired_states, distances_left, radii):
        ds = _f64(desired_states)
        dl = _f64(distances_left).reshape(-1)
        r = _f64(radii).reshape(-1)
        if ds.ndim != 2 or dl.shape[0] != ds.shape[0] or r.shape[0] != ds.shape[1]:
            raise ValueError("desired_states [W, d], distances_left [W], radii [d] expected")
        self._check(self._lib.ss_mpc_set_plan(self._h, _ptr(ds), ds.shape[0], _ptr(dl), _ptr(r),
                                              ds.shape[1]))

    def _plan_args(self, state, actions, K, H, act_low, act_high):
        d, da, _, _ = self._model_shape
        st = _f64(state).reshape(-1)
        if st.size != d:
            raise ValueError("state has %d entries, model expects %d" % (st.size, d))
        if isinstance(actions, _DevicePointer):
            pass                                   # [K, H, da] float64 already on the device
        elif actions is not None:
            actions = _f64(actions)
            if actions.ndim != 3 or actions.shape[2] != da:
                raise ValueError("actions must be [K, H, da]")
            K, H = actions.shape[0], actions.shape[1]
        return st, actions, int(K), int(H), _bounds(act_low, da), _bounds(act_high, da)

    def plan(self, state, wp_index, *, actions=None, K=None, H=None, seed=0, act_low=None,
             act_high=None, gamma=.75, horizontal_penalty_factor=.5, penalty_mode="reference",
             precision="auto", want_scores=False, want_path=True, k_offset=0, K_global=None, actions_dev=None,
             rng_state=None):
        """One MPC decision on this GPU.  Returns dict(best_k, best_score, best_sequence [H,da],
        best_path [H+1,d], scores [K] | None).  actions_dev: device address of [K, H, da] float64
        samples (mt19937_uniform) instead of a host array; K and H must then be given."""
        if self._model_shape is None:
            raise RuntimeError("set_model() first")
        d, da, _, _ = self._model_shape
        if isinstance(rng_state, int):
            # the reference's draw + the decision + the generator state written back in place, in one call
            # (rng_state = the address of numpy's state struct, global_rng_address())
            st = _f64(state).reshape(-1)
            if st.size != d:
                raise ValueError("state has %d entries, model expects %d" % (st.size, d))
            K, H = int(K), int(H)
            Kg = K if K_global is None else int(K_global)
            scores = np.empty(K) if want_scores else None
            seq = np.empty((H, da)) if want_path else None
            path = np.empty((H + 1, d)) if want_path else None
            best = C.c_int64(-1)
            best_score = C.c_double(0.0)
            self._last = (K, H)
            self._check(self._lib.ss_mpc_plan_mt19937(
                self._h, _ptr(st), int(wp_index), K, int(k_offset), Kg, H, rng_state, rng_state + 2496,
                _ptr(_bounds(act_low, da)), _ptr(_bounds(act_high, da)), float(gamma), float(horizontal_penalty_factor),
                _PENALTY[penalty_mode], _PRECISION[precision], C.byref(best), C.byref(best_score), _ptr(seq), _ptr(path),
                _ptr(scores)))
            return dict(best_k=int(best.value), best_score=float(best_score.value), best_sequence=seq,
                        best_path=path, scores=scores)
        if rng_state is not None:
            # the reference's draw, npr.uniform(low, high, (K, H, da)) of NND_MB_agent.py:500-501, made on
            # the device from the host generator's state; the advanced state comes back in the result
            K_global = int(K) if K_global is None else int(K_global)
            actions_dev = self.mt19937_uniform(rng_state, K_global * int(H) * da, act_low, act_high,
                                               first=int(k_offset) * int(H) * da, count=int(K) * int(H) * da)
        if actions_dev is not None:
            actions = _DevicePointer(actions_dev)
        st, actions, K, H, lo, hi = self._plan_args(state, actions, K, H, act_low, act_high)
        K_global = K if K_global is None else int(K_global)
        scores = np.empty(K) if want_scores else None
        seq = np.empty((H, da)) if want_path else None
        path = np.empty((H + 1, d)) if want_path else None
        best = C.c_int64(-1)
        best_score = C.c_double(0.0)
        self._last = (K, H)
        self._check(self._lib.ss_mpc_plan(
            self._h, _ptr(st), int(wp_index), K, int(k_offset), K_global, H, _ptr(actions),
            C.c_uint64(int(seed)), _ptr(lo), _ptr(hi), float(gamma),
            float(horizontal_penalty_factor), _PENALTY[penalty_mode], _PRECISION[precision],
            C.byref(best), C.byref(best_score), _ptr(seq), _ptr(path), _ptr(scores)))
        res = dict(best_k=int(best.value), best_score=float(best_score.value), best_sequence=seq,
                   best_path=path, scores=scores)
        if rng_state is not None:
            res["rng_state"] = self.mt19937_state()
        return res

    @staticmethod
    def global_rng_address():
        """Address of the state struct of numpy's global legacy generator, or None (then use get_state())."""
        return _NumpyGlobalMT.address()

    # three-call form (multi-GPU reference penalty): rollout -> all-reduce sums -> finish
    def rollout(self, state, wp_index, *, actions=None, K=None, H=None, seed=0, act_low=None,
                act_high=None, gamma=.75, horizontal_penalty_factor=.5, penalty_mode="reference",
                precision="auto", k_offset=0, K_global=None, actions_dev=None, rng_state=None):
        if rng_state is not None:
            da = self._model_shape[1]
            Kg = int(K) if K_global is None else int(K_global)
            actions_dev = self.mt19937_uniform(rng_state, Kg * int(H) * da, act_low, act_high,
                                               first=int(k_offset) * int(H) * da, count=int(K) * int(H) * da)
        if actions_dev is not None:
            actions = _DevicePointer(actions_dev)
        st, actions, K, H, lo, hi = self._plan_args(state, actions, K, H, act_low, act_high)
        K_global = K if K_global is None else int(K_global)
        self._check(self._lib.ss_mpc_rollout(
            self._h, _ptr(st), int(wp_index), K, int(k_offset), K_global, H, _ptr(actions),
            C.c_uint64(int(seed)), _ptr(lo), _ptr(hi), float(gamma),
            float(horizontal_penalty_factor), _PENALTY[penalty_mode], _PRECISION[precision]))
        self._last = (K, H)

    def projection_sums_ptr(self):
        """(device pointer, count) of the float64 per-time-step sums to all-reduce, or (0, 0)."""
        p = C.c_void_p()
        n = C.c_int()
        self._check(self._lib.ss_mpc_projection_sums(self._h, C.byref(p), C.byref(n)))
        return (p.value or 0), n.value

    def finish(self, want_scores=False):
        K, _ = self._last
        scores = np.empty(K) if want_scores else None
        best = C.c_int64(-1)
        best_score = C.c_double(0.0)
        self._check(self._lib.ss_mpc_finish(self._h, C.byref(best), C.byref(best_score), _ptr(scores)))
        return int(best.value), float(best_score.value), scores

    def finish_package(self, want_path=True):
        """Phase B + arg-max + the local winner's sequence and path, left on the device as one
        float64 package [score, k_global, sequence (H*da), path ((H+1)*d)]: (device ptr, count)."""
        p = C.c_void_p()
        n = C.c_int()
        self._check(self._lib.ss_mpc_finish_package(self._h, 1 if want_path else 0, C.byref(p), C.byref(n)))
        return (p.value or 0), n.value

    def read_package(self, count):
        out = np.empty(count)
        self._check(self._lib.ss_mpc_read_package(self._h, _ptr(out), int(count)))
        return out

    def get_states(self):
        """[H+1, K, d] trajectories of the last reference-mode rollout."""
        d = self._model_shape[0]
        K, H = self._last
        out = np.empty((H + 1, K, d))
        self._check(self._lib.ss_mpc_get_states(self._h, _ptr(out)))
        return out

    def forward_sim(self, state, actions=None, precision="fp32", *, actions_dev=None, K=None, H=None):
        """Dyn_Model.do_forward_sim(many_in_parallel=True) on the GPU (ss_mpc_forward_sim): states [H+1, K, d].
        state [d] starts every sequence there; [K, d] starts sequence k at row k.  actions [K, H, da], or
        actions_dev = the device address of such samples (mt19937_uniform) with K and H given.  precision as in
        plan ("fp64": the reference's float64 arithmetic).  Needs set_model only; the plan is neither needed nor
        changed, and finish / replay / projection_sums_ptr refuse until the next rollout or plan."""
        if self._model_shape is None:
            raise RuntimeError("set_model() first")
        d, da, _, _ = self._model_shape
        st = _f64(state)
        if st.ndim == 1 and st.shape[0] == d:
            n_starts = 1
        elif st.ndim == 2 and st.shape[1] == d:
            n_starts = st.shape[0]
        else:
            raise ValueError("state must be [d] or [K, d] with d = %d, got shape %s" % (d, st.shape))
        if actions_dev is not None:
            actions = _DevicePointer(actions_dev)
        elif actions is None:
            raise ValueError("actions [K, H, da] or actions_dev are needed")
        else:
            actions = _f64(actions)
            if actions.ndim != 3 or actions.shape[2] != da:
                raise ValueError("actions must be [K, H, da]")
            K, H = actions.shape[0], actions.shape[1]
        K, H = int(K), int(H)
        out = np.empty((H + 1, K, d))
        self._check(self._lib.ss_mpc_forward_sim(self._h, _ptr(st), n_starts, K, H, _ptr(actions),
                                                 _PRECISION[precision], _ptr(out)))
        self._last = (K, H)
        return out

    def replay(self, k_global):
        d, da, _, _ = self._model_shape
        _, H = self._last
        seq = np.empty((H, da))
        path = np.empty((H + 1, d))
        self._check(self._lib.ss_mpc_replay(self._h, int(k_global), _ptr(seq), _ptr(path)))
        return seq, path

    # numpy's legacy RandomState stream on the device (csrc/mt19937.cu)
    def mt19937_uniform(self, rng_state, n_total, low, high, first=0, count=None):
        """Elements [first, first + count) of what np.random.uniform(low, high, (n_total // da, da))
        would draw from ``rng_state`` (np.random.get_state() / RandomState.get_state(), or the address of
        numpy's global state struct, see global_rng_address), generated on
        the GPU bit for bit and left there: returns the device pointer (pass it to plan / rollout as
        ``actions_dev``).  The state after the whole draw comes from mt19937_state()."""
        lo = low if isinstance(low, np.ndarray) and low.dtype == np.float64 and low.ndim == 1 and low.flags.c_contiguous \
            else _f64(np.asarray(low, dtype=np.float64).reshape(-1))
        hi = high if isinstance(high, np.ndarray) and high.dtype == np.float64 and high.ndim == 1 and high.flags.c_contiguous \
            else _f64(np.asarray(high, dtype=np.float64).reshape(-1))
        count = int(n_total) - int(first) if count is None else int(count)
        out = C.c_void_p()
        if isinstance(rng_state, int):
            # address of numpy's own state struct {uint32 key[624]; int pos} (_NumpyGlobalMT): read in place
            key_ptr, pos = rng_state, C.c_int.from_address(rng_state + 2496).value
            self._mt_rest = None
        else:
            if rng_state[0] != "MT19937":
                raise ValueError("legacy MT19937 state expected")
            key = np.ascontiguousarray(rng_state[1], dtype=np.uint32)
            key_ptr, pos = _ptr(key), int(rng_state[2])
            self._mt_rest = tuple(rng_state[3:])
        self._check(self._lib.ss_mt19937_uniform(self._h, key_ptr, pos, int(n_total), int(first),
                                                 count, lo.shape[0], _ptr(lo), _ptr(hi), C.byref(out)))
        return out.value

    def mt19937_warm(self, n_total, low, high, first=0, count=None):
        """Build (and cache) the jump-ahead plan of a draw shape ahead of time: the polynomials of a large shape
        take ~0.1 s of host arithmetic, which would otherwise land in the first decision."""
        st = np.random.RandomState(0).get_state()
        self.mt19937_uniform(st, n_total, low, high, first=first, count=count)
        self.mt19937_state()

    def mt19937_state_into(self, address):
        """Write the generator state after the last mt19937_uniform draw straight into numpy's state struct."""
        self._check(self._lib.ss_mt19937_state(self._h, C.c_void_p(address),
                                               C.cast(C.c_void_p(address + 2496), C.POINTER(C.c_int))))

    def mt19937_state(self):
        """Generator state after the last mt19937_uniform draw, in np.random.set_state's format."""
        key = np.empty(624, dtype=np.uint32)
        pos = C.c_int(0)
        self._check(self._lib.ss_mt19937_state(self._h, _ptr(key), C.byref(pos)))
        return ("MT19937", key, int(pos.value)) + self._mt_rest

    def read_device_doubles(self, dev_ptr, count):
        """Copy ``count`` float64 from device memory (tests / debugging)."""
        out = np.empty(int(count))
        self._check(self._lib.ss_memcpy_d2h(self._h, _ptr(out), C.c_void_p(int(dev_ptr)), int(count) * 8))
        return out

    def sample_actions(self, K, H, da, seed, act_low, act_high, k_offset=0):
        lo = _f64(np.broadcast_to(np.asarray(act_low, dtype=np.float64), (da,)))
        hi = _f64(np.broadcast_to(np.asarray(act_high, dtype=np.float64), (da,)))
        out = np.empty((K, H, da))
        self._check(self._lib.ss_mpc_sample_actions(self._h, int(K), int(k_offset), int(H), int(da),
                                                    C.c_uint64(int(seed)), _ptr(lo), _ptr(hi),
                                                    _ptr(out)))
        return out
