"""ctypes binding of libsbr_b200.so (include/sbr_b200.h) -- the only way the host code reaches
the device.  There is NO CPU fallback: importing this module without the built library raises
ImportError, and creating an Engine without a CUDA device raises RuntimeError (SBR_E_NOGPU).

The Engine methods mirror the three callables the reference compiles with theano.function
(neural_networks/rnn_base.py:175-213): train_function / test_function / predict_function, and
lasagne's get/set_all_param_values (rnn_base.py:476,515).
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# SBR_B200_LIB selects another build of the same library (e.g. the --timeline profiling build)
LIB_PATH = os.environ.get("SBR_B200_LIB") or os.path.join(_HERE, "libsbr_b200.so")

SBR_MAX_LAYERS = 8
SBR_NCCL_ID_BYTES = 128
SBR_N_STAGES = 9

CELLS = {"LSTM": 0, "GRU": 1, "Vanilla": 2}
LOSSES = {"CCE": 0, "BPR": 1, "BPRI": 2, "TOP1": 3, "Blackout": 4, "hinge": 5, "logit": 6, "logsig": 7}
UPDATERS = {"adam": 0, "adagrad": 1, "adadelta": 2, "rmsprop": 3, "nesterov": 4}
CLUSTER_TYPES = {"softmax": 0, "mix": 1, "sigmoid": 2}
CLUSTER_LOSSES = {"Blackout": 0, "CCE": 1, "BPR": 2, "TOP1": 3, "BPRelu": 4, "lin": 5}
STATUS = {0: "SBR_OK", -1: "SBR_E_ARG", -2: "SBR_E_CUDA", -3: "SBR_E_NCCL", -4: "SBR_E_MASK",
          -5: "SBR_E_RANGE", -6: "SBR_E_NOGPU"}


class SbrError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("%s: %s" % (STATUS.get(code, code), msg))
        self.code = code


class SbrConfig(C.Structure):
    _fields_ = [
        ("struct_size", C.c_int32), ("cell", C.c_int32), ("n_layers", C.c_int32),
        ("layers", C.c_int32 * SBR_MAX_LAYERS), ("n_items", C.c_int32), ("n_extra_ids", C.c_int32),
        ("ids_per_step", C.c_int32), ("embedding", C.c_int32), ("max_length", C.c_int32),
        ("batch_size", C.c_int32), ("loss", C.c_int32), ("n_samples", C.c_int32),
        ("last_layer_tanh", C.c_int32), ("updater", C.c_int32),
        ("lr", C.c_float), ("rho", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float),
        ("grad_clip", C.c_float), ("regularization", C.c_float),
        ("math_mode", C.c_int32), ("device", C.c_int32), ("n_ranks", C.c_int32), ("rank", C.c_int32),
        ("global_batch", C.c_int32), ("n_slots", C.c_int32), ("bidirectional", C.c_int32),
        ("nccl_id", C.c_uint8 * SBR_NCCL_ID_BYTES),
    ]


class SbrClusterConfig(C.Structure):
    _fields_ = [("struct_size", C.c_int32), ("n_clusters", C.c_int32), ("cluster_type", C.c_int32), ("loss", C.c_int32),
                ("n_cluster_samples", C.c_int32)]


class SbrScanPlan(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("family", "G", "BT", "MT", "JU", "wsmem", "splitk", "C", "Hs", "launches",
                                         "tiles_per_launch")]


SCAN_FAMILIES = {0: "tc_cluster", 1: "persistent", 2: "step", 3: "ffma"}


_P = C.c_void_p
_i32p = C.POINTER(C.c_int32)
_f32p = C.POINTER(C.c_float)

# name -> (restype, argtypes); kept in one table so tests can check it against the header
SIGNATURES = {
    "sbr_abi_version": (C.c_int, []),
    "sbr_device_count": (C.c_int, []),
    "sbr_nccl_unique_id": (C.c_int, [C.POINTER(C.c_uint8)]),
    "sbr_create": (C.c_int, [C.POINTER(SbrConfig), C.POINTER(_P)]),
    "sbr_destroy": (None, [_P]),
    "sbr_last_error": (C.c_char_p, [_P]),
    "sbr_param_count": (C.c_int, [_P]),
    "sbr_param_info": (C.c_int, [_P, C.c_int, C.c_char_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int64)]),
    "sbr_get_param": (C.c_int, [_P, C.c_int, _f32p]),
    "sbr_set_param": (C.c_int, [_P, C.c_int, _f32p]),
    "sbr_get_grad": (C.c_int, [_P, C.c_int, _f32p]),
    "sbr_total_params": (C.c_int64, [_P]),
    "sbr_reset_optimizer": (C.c_int, [_P]),
    "sbr_set_skip_update": (C.c_int, [_P, C.c_int]),
    "sbr_train_step_cce": (C.c_int, [_P, _i32p, _f32p, _i32p, _f32p, C.c_int, _f32p]),
    "sbr_train_step_sampled": (C.c_int, [_P, _i32p, _f32p, _i32p, C.c_int, C.c_int, _i32p, C.c_int, _f32p, C.c_int, _f32p]),
    "sbr_train_step_margin_dense": (C.c_int, [_P, _i32p, _f32p, _f32p, _f32p, C.c_int, _f32p]),
    "sbr_train_step_margin": (C.c_int, [_P, _i32p, _f32p, _i32p, _i32p, _f32p, _f32p, C.c_int, C.c_int, _f32p]),
    "sbr_dataset_upload": (C.c_int, [_P, C.c_int, _i32p, _i32p]),
    "sbr_train_step_cce_rows": (C.c_int, [_P, _i32p, _i32p, _i32p, _i32p, _f32p, C.c_int, _f32p]),
    "sbr_stage_cce": (C.c_int, [_P, C.c_int, _i32p, _f32p, _i32p, _f32p, C.c_int]),
    "sbr_train_step_staged": (C.c_int, [_P, C.c_int, _f32p]),
    "sbr_synchronize": (C.c_int, [_P, _f32p]),
    "sbr_scores": (C.c_int, [_P, _i32p, _f32p, C.c_int, C.c_int, _f32p]),
    "sbr_topk": (C.c_int, [_P, _i32p, _f32p, C.c_int, _i32p, _i32p, C.c_int, C.c_int, _i32p]),
    "sbr_create_cluster": (C.c_int, [C.POINTER(SbrConfig), C.POINTER(SbrClusterConfig), C.POINTER(_P)]),
    "sbr_train_step_cluster": (C.c_int, [_P, _i32p, _f32p, _i32p, C.c_int, C.c_int, _i32p, C.c_int, _i32p, C.c_int, _f32p,
                                         C.c_float, C.c_int, _f32p, _f32p]),
    "sbr_cluster_test_topk": (C.c_int, [_P, _i32p, _f32p, C.c_int, _i32p, _i32p, C.c_int, _i32p, _i32p, _i32p, _f32p]),
    "sbr_cluster_build": (C.c_int, [_P, _i32p]),
    "sbr_cluster_topk": (C.c_int, [_P, _i32p, _f32p, C.c_int, _i32p, _i32p, C.c_int, _i32p, _i32p, _i32p, C.c_int]),
    "sbr_stage_name": (C.c_char_p, [C.c_int]),
    "sbr_set_profiling": (C.c_int, [_P, C.c_int]),
    "sbr_stage_times": (C.c_int, [_P, _f32p]),
    "sbr_kernel_launches": (C.c_int64, [_P]),
    "sbr_plan_scan_tiles": (C.c_int, [_i32p, C.c_int, C.c_int, C.c_int, C.c_float, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                      C.POINTER(C.c_int), C.POINTER(C.c_ubyte)]),
    "sbr_plan_layer_scan": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _i32p, C.c_int, C.c_int, C.c_int, _i32p, C.c_int,
                                      C.POINTER(SbrScanPlan)]),
    "sbr_scan_launches": (C.c_int64, [_P]),
    "sbr_debug_gemm": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _f32p, C.c_int, _f32p, C.c_int,
                                 _f32p, C.c_int, C.c_float, C.c_float, _f32p, C.c_int, _f32p]),
    "sbr_timer_start": (C.c_int, [_P]),
    "sbr_timer_stop": (C.c_int, [_P, _f32p]),
}

_lib = None


def load_library():
    """dlopen the in-tree library; loud failure when it was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("libsbr_b200.so is missing (%s). Build it with `python -c 'import __graft_entry__ as g; "
                          "g.build()'` or `python sequence-based-recommendations_b200/build.py`; there is no CPU "
                          "fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.sbr_abi_version() != 2:
        raise ImportError("libsbr_b200.so ABI %d, binding expects 2" % lib.sbr_abi_version())
    _lib = lib
    return lib


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _ptr(a, typ):
    return a.ctypes.data_as(typ)


def _plan_dict(p):
    d = {n: int(getattr(p, n)) for n, _ in SbrScanPlan._fields_}
    d["family"] = SCAN_FAMILIES[d["family"]]
    return d


def plan_layer_scan(cell, H, B, backward, lens=None, t_max=None, n_sm=148, tc_slots=(148, 74, 37, 15), splitk_slots=37,
                    handle=None):
    """The scan variant the launchers pick for one layer and direction (sbr_plan_layer_scan), as a dict.  Without a
    handle the device is described by n_sm, tc_slots (co-resident tcgen05 scan clusters of 1, 2, 4, 8 CTAs) and
    splitk_slots, and the SBR_* switches are read from the environment; returns None when no scan takes the layer."""
    lib = load_library()
    lp = None
    if lens is not None:
        lens = _i32(lens)
        lp = _ptr(lens, _i32p)
    if t_max is None:
        t_max = int(max(lens)) if lens is not None else 1
    slots = _i32(tc_slots)
    out = SbrScanPlan()
    rc = lib.sbr_plan_layer_scan(handle, CELLS[cell], int(H), int(B), lp, int(t_max), int(bool(backward)), int(n_sm),
                                 _ptr(slots, _i32p), int(splitk_slots), C.byref(out))
    if rc == -1:
        return None
    if rc != 0:
        raise SbrError(rc, "sbr_plan_layer_scan")
    return _plan_dict(out)


def nccl_unique_id():
    lib = load_library()
    buf = (C.c_uint8 * SBR_NCCL_ID_BYTES)()
    rc = lib.sbr_nccl_unique_id(buf)
    if rc != 0:
        raise SbrError(rc, lib.sbr_last_error(None).decode())
    return bytes(buf)


class Engine(object):
    """One sbr_model handle (one GPU rank)."""

    def __init__(self, n_items, cell="GRU", layers=(50,), loss="CCE", max_length=30, batch_size=16,
                 embedding=0, n_extra_ids=0, ids_per_step=1, n_samples=32, last_layer_tanh=False,
                 updater="adam", lr=1e-3, rho=0.9, beta1=0.9, beta2=0.999, grad_clip=100.0,
                 regularization=0.0, device=0, n_ranks=1, rank=0, nccl_id=None, global_batch=0,
                 n_slots=1, math_mode=0, bidirectional=False, clusters=None):
        """clusters: None, or dict(n_clusters, cluster_type, loss, n_cluster_samples) for an RNNCluster handle
        (sbr_create_cluster); `loss` is then ignored."""
        self.lib = load_library()
        cfg = SbrConfig()
        cfg.struct_size = C.sizeof(SbrConfig)
        cfg.cell = CELLS[cell]
        layers = list(layers)
        if len(layers) > SBR_MAX_LAYERS:
            raise ValueError("at most %d recurrent layers" % SBR_MAX_LAYERS)
        cfg.n_layers = len(layers)
        for i, h in enumerate(layers):
            cfg.layers[i] = int(h)
        cfg.n_items, cfg.n_extra_ids, cfg.ids_per_step = int(n_items), int(n_extra_ids), int(ids_per_step)
        cfg.embedding, cfg.max_length, cfg.batch_size = int(embedding), int(max_length), int(batch_size)
        cfg.loss = LOSSES["Blackout"] if clusters else LOSSES[loss]
        cfg.n_samples, cfg.last_layer_tanh = int(n_samples), int(bool(last_layer_tanh))
        cfg.updater = UPDATERS[updater]
        cfg.lr, cfg.rho, cfg.beta1, cfg.beta2 = lr, rho, beta1, beta2
        cfg.grad_clip, cfg.regularization = grad_clip, regularization
        cfg.math_mode, cfg.device, cfg.n_ranks, cfg.rank = int(math_mode), int(device), int(n_ranks), int(rank)
        cfg.global_batch, cfg.n_slots = int(global_batch), int(n_slots)
        cfg.bidirectional = int(bool(bidirectional))
        if n_ranks > 1:
            if nccl_id is None or len(nccl_id) != SBR_NCCL_ID_BYTES:
                raise ValueError("n_ranks > 1 needs the 128-byte nccl_id made by nccl_unique_id() on rank 0")
            for i, b in enumerate(nccl_id):
                cfg.nccl_id[i] = b
        self.cfg = cfg
        self.loss = loss
        self.n_items, self.max_length, self.batch_size = int(n_items), int(max_length), int(batch_size)
        self.ids_per_step = int(ids_per_step)
        self.n_samples = int(n_samples)
        self._h = _P()
        self.n_clusters = 0
        if clusters:
            cc = SbrClusterConfig()
            cc.struct_size = C.sizeof(SbrClusterConfig)
            cc.n_clusters = int(clusters["n_clusters"])
            cc.cluster_type = CLUSTER_TYPES[clusters.get("cluster_type", "mix")]
            cc.loss = CLUSTER_LOSSES[clusters.get("loss", "Blackout")]
            cc.n_cluster_samples = max(0, int(clusters.get("n_cluster_samples", 0)))
            self.n_clusters = int(cc.n_clusters)
            self.ccfg = cc
            rc = self.lib.sbr_create_cluster(C.byref(cfg), C.byref(cc), C.byref(self._h))
        else:
            rc = self.lib.sbr_create(C.byref(cfg), C.byref(self._h))
        if rc != 0:
            self._h = None
            raise SbrError(rc, self.lib.sbr_last_error(None).decode())
        self._infos = None

    # -- plumbing -------------------------------------------------------------------------------
    def _check(self, rc):
        if rc != 0:
            raise SbrError(rc, self.lib.sbr_last_error(self._h).decode())

    def close(self):
        if getattr(self, "_h", None):
            self.lib.sbr_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _xm(self, X, mask):
        X = _i32(X)
        if X.ndim == 2:
            X = X[:, :, None]
        B = X.shape[0]
        if X.shape[1:] != (self.max_length, self.ids_per_step):
            raise ValueError("X must be [B, %d, %d], got %s" % (self.max_length, self.ids_per_step, X.shape))
        mask = _f32(mask)
        if mask.shape != (B, self.max_length):
            raise ValueError("mask must be [B, %d]" % self.max_length)
        return np.ascontiguousarray(X), mask, B

    # -- parameters -----------------------------------------------------------------------------
    def param_infos(self):
        """[(name, shape)] in lasagne.layers.get_all_params order (rnn_base.py:476)."""
        if self._infos is None:
            out = []
            for i in range(self.lib.sbr_param_count(self._h)):
                name = C.create_string_buffer(128)
                nd = C.c_int(0)
                shp = (C.c_int64 * 4)()
                self._check(self.lib.sbr_param_info(self._h, i, name, 128, C.byref(nd), shp))
                out.append((name.value.decode(), tuple(int(shp[k]) for k in range(nd.value))))
            self._infos = out
        return self._infos

    def get_all_param_values(self):
        vals = []
        for i, (_, shape) in enumerate(self.param_infos()):
            a = np.empty(shape, dtype=np.float32)
            self._check(self.lib.sbr_get_param(self._h, i, _ptr(a, _f32p)))
            vals.append(a)
        return vals

    def set_all_param_values(self, values):
        infos = self.param_infos()
        if len(values) != len(infos):
            raise ValueError("expected %d parameter arrays, got %d" % (len(infos), len(values)))
        for i, ((name, shape), v) in enumerate(zip(infos, values)):
            a = _f32(v)
            if a.shape != shape:
                raise ValueError("parameter %d (%s): shape %s, expected %s" % (i, name, a.shape, shape))
            self._check(self.lib.sbr_set_param(self._h, i, _ptr(a, _f32p)))

    def get_all_grads(self):
        vals = []
        for i, (_, shape) in enumerate(self.param_infos()):
            a = np.empty(shape, dtype=np.float32)
            self._check(self.lib.sbr_get_grad(self._h, i, _ptr(a, _f32p)))
            vals.append(a)
        return vals

    def total_params(self):
        return int(self.lib.sbr_total_params(self._h))

    def reset_optimizer(self):
        self._check(self.lib.sbr_reset_optimizer(self._h))

    def set_skip_update(self, flag):
        self._check(self.lib.sbr_set_skip_update(self._h, int(bool(flag))))

    # -- train_function -------------------------------------------------------------------------
    def train_step_cce(self, X, mask, Y, pop):
        X, mask, B = self._xm(X, mask)
        Y, pop = _i32(Y), _f32(pop)
        cost = C.c_float(0)
        self._check(self.lib.sbr_train_step_cce(self._h, _ptr(X, _i32p), _ptr(mask, _f32p), _ptr(Y, _i32p),
                                                _ptr(pop, _f32p), B, C.byref(cost)))
        return np.float32(cost.value)

    def train_step_sampled(self, X, mask, Y, samples, pop, Y_all=None, row_offset=0):
        X, mask, B = self._xm(X, mask)
        Y_all = _i32(Y if Y_all is None else Y_all)
        samples, pop = _i32(samples), _f32(pop)
        cost = C.c_float(0)
        self._check(self.lib.sbr_train_step_sampled(self._h, _ptr(X, _i32p), _ptr(mask, _f32p), _ptr(Y_all, _i32p),
                                                    len(Y_all), int(row_offset), _ptr(samples, _i32p), len(samples),
                                                    _ptr(pop, _f32p), B, C.byref(cost)))
        return np.float32(cost.value)

    def train_step_cluster(self, X, mask, Y, samples, cluster_samples=None, noise=None, scale=1.0, Y_all=None,
                           row_offset=0):
        """RNNCluster step; returns (cost, cluster_cost).  noise: [B, n_clusters] of this rank's rows, or None."""
        X, mask, B = self._xm(X, mask)
        Y_all = _i32(Y if Y_all is None else Y_all)
        samples = _i32(samples)
        cs = None if cluster_samples is None else _i32(cluster_samples)
        nz = None if noise is None else _f32(noise)
        if nz is not None and nz.shape != (B, self.n_clusters):
            raise ValueError("noise must be [B, %d]" % self.n_clusters)
        cost, ccost = C.c_float(0), C.c_float(0)
        self._check(self.lib.sbr_train_step_cluster(
            self._h, _ptr(X, _i32p), _ptr(mask, _f32p), _ptr(Y_all, _i32p), len(Y_all), int(row_offset),
            _ptr(samples, _i32p), len(samples), None if cs is None else _ptr(cs, _i32p), 0 if cs is None else len(cs),
            None if nz is None else _ptr(nz, _f32p), float(scale), B, C.byref(cost), C.byref(ccost)))
        return np.float32(cost.value), np.float32(ccost.value)

    def train_step_margin_dense(self, X, mask, Ymat, weight):
        X, mask, B = self._xm(X, mask)
        Ymat, weight = _f32(Ymat), _f32(weight)
        cost = C.c_float(0)
        self._check(self.lib.sbr_train_step_margin_dense(self._h, _ptr(X, _i32p), _ptr(mask, _f32p),
                                                         _ptr(Ymat, _f32p), _ptr(weight, _f32p), B, C.byref(cost)))
        return np.float32(cost.value)

    def train_step_margin(self, X, mask, target_offsets, target_ids, w_neg, default_target=None, exclude_seen=True):
        X, mask, B = self._xm(X, mask)
        off, ids, w = _i32(target_offsets), _i32(target_ids), _f32(w_neg)
        if ids.size == 0:
            ids = np.zeros(1, dtype=np.int32)
        dt = None if default_target is None else _f32(default_target)
        cost = C.c_float(0)
        self._check(self.lib.sbr_train_step_margin(self._h, _ptr(X, _i32p), _ptr(mask, _f32p), _ptr(off, _i32p),
                                                   _ptr(ids, _i32p), _ptr(w, _f32p),
                                                   None if dt is None else _ptr(dt, _f32p),
                                                   int(bool(exclude_seen)), B, C.byref(cost)))
        return np.float32(cost.value)

    # -- device-side batch assembly ---------------------------------------------------------------
    def dataset_upload(self, offsets, ids):
        """The training sequences as a CSR of ids: offsets [n+1], ids [total, ids_per_step]."""
        off = _i32(offsets)
        ids = _i32(ids).reshape(-1, self.ids_per_step)
        if ids.shape[0] != off[-1]:
            raise ValueError("ids has %d rows, offsets end at %d" % (ids.shape[0], off[-1]))
        if ids.size == 0:
            ids = np.zeros((1, self.ids_per_step), dtype=np.int32)
        self._check(self.lib.sbr_dataset_upload(self._h, len(off) - 1, _ptr(off, _i32p), _ptr(np.ascontiguousarray(ids), _i32p)))

    def train_step_cce_rows(self, seq, start, length, Y, pop):
        seq, start, length, Y, pop = _i32(seq), _i32(start), _i32(length), _i32(Y), _f32(pop)
        cost = C.c_float(0)
        self._check(self.lib.sbr_train_step_cce_rows(self._h, _ptr(seq, _i32p), _ptr(start, _i32p), _ptr(length, _i32p),
                                                     _ptr(Y, _i32p), _ptr(pop, _f32p), len(seq), C.byref(cost)))
        return np.float32(cost.value)

    # -- device-resident batches ----------------------------------------------------------------
    def stage_cce(self, slot, X, mask, Y, pop):
        X, mask, B = self._xm(X, mask)
        Y, pop = _i32(Y), _f32(pop)
        self._check(self.lib.sbr_stage_cce(self._h, int(slot), _ptr(X, _i32p), _ptr(mask, _f32p), _ptr(Y, _i32p),
                                           _ptr(pop, _f32p), B))

    def train_step_staged(self, slot, want_cost=True):
        if want_cost:
            cost = C.c_float(0)
            self._check(self.lib.sbr_train_step_staged(self._h, int(slot), C.byref(cost)))
            return np.float32(cost.value)
        self._check(self.lib.sbr_train_step_staged(self._h, int(slot), None))
        return None

    def synchronize(self, want_cost=False):
        cost = C.c_float(0)
        self._check(self.lib.sbr_synchronize(self._h, C.byref(cost) if want_cost else None))
        return np.float32(cost.value) if want_cost else None

    # -- predict / test -------------------------------------------------------------------------
    def scores(self, X, mask, softmax=False):
        X, mask, B = self._xm(X, mask)
        out = np.empty((B, self.n_items), dtype=np.float32)
        self._check(self.lib.sbr_scores(self._h, _ptr(X, _i32p), _ptr(mask, _f32p), B, int(bool(softmax)),
                                        _ptr(out, _f32p)))
        return out

    def topk(self, X, mask, k=10, exclude=None, softmax=False, neg_inf=False):
        """exclude: list (per row) of id lists, or None."""
        X, mask, B = self._xm(X, mask)
        out = np.empty((B, k), dtype=np.int32)
        mode = (1 if softmax else 0) | (2 if neg_inf else 0)
        if exclude is None:
            off_p = ids_p = None
        else:
            off = np.zeros(B + 1, dtype=np.int32)
            off[1:] = np.cumsum([len(e) for e in exclude])
            flat = [i for e in exclude for i in e]
            ids = _i32(flat if flat else [0])
            off_p, ids_p = _ptr(off, _i32p), _ptr(ids, _i32p)
        self._check(self.lib.sbr_topk(self._h, _ptr(X, _i32p), _ptr(mask, _f32p), B, off_p, ids_p, int(k), mode,
                                      _ptr(out, _i32p)))
        return out

    @staticmethod
    def _ragged(exclude, B):
        if exclude is None:
            return None, None, None
        off = np.zeros(B + 1, dtype=np.int32)
        off[1:] = np.cumsum([len(e) for e in exclude])
        flat = [i for e in exclude for i in e]
        ids = _i32(flat if flat else [0])
        return (off, ids), _ptr(off, _i32p), _ptr(ids, _i32p)

    def cluster_test_topk(self, X, mask, k=10, exclude=None):
        """Validation test function of RNNCluster: (ids_full [B,k], ids_cluster [B,k], selected [B], n_used [B])."""
        X, mask, B = self._xm(X, mask)
        keep, off_p, ids_p = self._ragged(exclude, B)
        full = np.empty((B, k), dtype=np.int32)
        clus = np.empty((B, k), dtype=np.int32)
        sel = np.empty(B, dtype=np.int32)
        used = np.empty(B, dtype=np.float32)
        self._check(self.lib.sbr_cluster_test_topk(self._h, _ptr(X, _i32p), _ptr(mask, _f32p), B, off_p, ids_p, int(k),
                                                   _ptr(full, _i32p), _ptr(clus, _i32p), _ptr(sel, _i32p),
                                                   _ptr(used, _f32p)))
        return full, clus, sel, used

    def cluster_build(self):
        """Hard clusters from cluster.R on the device; returns the cluster sizes."""
        sizes = np.empty(self.n_clusters, dtype=np.int32)
        self._check(self.lib.sbr_cluster_build(self._h, _ptr(sizes, _i32p)))
        return sizes

    def cluster_topk(self, X, mask, k=10, exclude=None, use_clusters=True):
        """(ids [B,k] with -1 past min(k, |cluster|), n [B], selected [B])."""
        X, mask, B = self._xm(X, mask)
        keep, off_p, ids_p = self._ragged(exclude, B)
        ids = np.empty((B, k), dtype=np.int32)
        n = np.empty(B, dtype=np.int32)
        sel = np.empty(B, dtype=np.int32)
        self._check(self.lib.sbr_cluster_topk(self._h, _ptr(X, _i32p), _ptr(mask, _f32p), B, off_p, ids_p, int(k),
                                              _ptr(ids, _i32p), _ptr(n, _i32p), _ptr(sel, _i32p), int(bool(use_clusters))))
        return ids, n, sel

    # -- measurement ----------------------------------------------------------------------------
    def set_profiling(self, on):
        self._check(self.lib.sbr_set_profiling(self._h, int(bool(on))))

    def stage_times(self):
        ms = (C.c_float * SBR_N_STAGES)()
        self._check(self.lib.sbr_stage_times(self._h, ms))
        return {self.lib.sbr_stage_name(i).decode(): float(ms[i]) for i in range(SBR_N_STAGES)}

    def kernel_launches(self):
        return int(self.lib.sbr_kernel_launches(self._h))

    def scan_launches(self):
        return int(self.lib.sbr_scan_launches(self._h))

    def plan_layer_scan(self, cell, H, B, backward, lens=None, t_max=None):
        """The live plan of this handle (its switches, SM count and co-resident cluster counts)."""
        return plan_layer_scan(cell, H, B, backward, lens, t_max, handle=self._h)

    def debug_gemm(self, A, B, ta=False, tb=False, C0=None, alpha=1.0, beta=0.0, bias=None, engine=1, reps=1):
        """op(A) @ op(B) through one of the library's GEMM kernels (diagnostics / tests); returns (C, ms)."""
        A, B = _f32(A), _f32(B)
        M, K = (A.shape[1], A.shape[0]) if ta else A.shape
        N = B.shape[0] if tb else B.shape[1]
        assert (B.shape[1] if tb else B.shape[0]) == K
        Cm = np.zeros((M, N), dtype=np.float32) if C0 is None else _f32(C0).copy()
        bp = None if bias is None else _ptr(_f32(bias), _f32p)
        bias_keep = None if bias is None else _f32(bias)
        if bias_keep is not None:
            bp = _ptr(bias_keep, _f32p)
        ms = C.c_float(0)
        self._check(self.lib.sbr_debug_gemm(self._h, int(engine), int(ta), int(tb), M, N, K, _ptr(A, _f32p), A.shape[1],
                                            _ptr(B, _f32p), B.shape[1], _ptr(Cm, _f32p), N, float(alpha), float(beta), bp,
                                            int(reps), C.byref(ms)))
        return Cm, float(ms.value)

    def timer_start(self):
        self._check(self.lib.sbr_timer_start(self._h))

    def timer_stop(self):
        ms = C.c_float(0)
        self._check(self.lib.sbr_timer_stop(self._h, C.byref(ms)))
        return float(ms.value)
