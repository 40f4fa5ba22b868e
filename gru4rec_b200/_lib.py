"""ctypes binding of libg4r.so (include/g4r.h).  There is no CPU path: loading fails loudly if the
library is missing, and creating a handle fails loudly if no CUDA device is visible."""
import ctypes as C
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libg4r.so')
G4R_MAX_LAYERS = 8

G4R_OK, G4R_ERR_INVALID, G4R_ERR_INDEX, G4R_ERR_CUDA, G4R_ERR_NAN, G4R_ERR_STATE = 0, -1, -2, -3, -4, -5
LOSS = {'cross-entropy': 0, 'bpr-max': 1, 'top1-max': 2, 'bpr': 3, 'top1': 4, 'xe_logit': 5}
ACT = {'linear': 0, 'relu': 1, 'tanh': 2, 'leaky': 3, 'elu': 4, 'selu': 5, 'softmax': 6, 'softmax_logit': 7}
ADAPT = {None: 0, 'adagrad': 1, 'rmsprop': 2, 'adadelta': 3, 'adam': 4}


class G4RConfig(C.Structure):
    _fields_ = [
        ('n_items', C.c_int32), ('n_layers', C.c_int32), ('layers', C.c_int32 * G4R_MAX_LAYERS), ('batch_size', C.c_int32),
        ('embedding', C.c_int32), ('constrained_embedding', C.c_int32), ('loss', C.c_int32),
        ('final_act', C.c_int32), ('final_act_p1', C.c_float), ('final_act_p2', C.c_float),
        ('hidden_act', C.c_int32), ('hidden_act_p1', C.c_float), ('hidden_act_p2', C.c_float),
        ('dropout_p_hidden', C.c_float), ('dropout_p_embed', C.c_float),
        ('learning_rate', C.c_float), ('momentum', C.c_float), ('lmbd', C.c_float),
        ('n_sample', C.c_int32), ('sample_alpha', C.c_float),
        ('smoothing', C.c_float), ('bpreg', C.c_float), ('logq', C.c_float),
        ('adapt', C.c_int32), ('sample_store', C.c_int32), ('dropout_seed', C.c_uint32), ('mrg_seed', C.c_uint32),
        ('max_resident_steps', C.c_int32), ('device', C.c_int32), ('world_size', C.c_int32), ('rank', C.c_int32),
        ('eval_batch_size', C.c_int32), ('step_mode', C.c_int32), ('mg_replicated', C.c_int32), ('eval_tc', C.c_int32),
        ('adapt_p1', C.c_float), ('adapt_p1c', C.c_float), ('adapt_p2', C.c_float), ('adapt_p2c', C.c_float), ('grad_cap', C.c_float),
    ]


EXPORTS = [
    'g4r_version', 'g4r_workspace_bytes', 'g4r_create', 'g4r_destroy', 'g4r_last_error', 'g4r_stream',
    'g4r_tensor_shape', 'g4r_set_tensor', 'g4r_get_tensor', 'g4r_reset_hidden',
    'g4r_set_sampling_cdf', 'g4r_set_logq_support', 'g4r_generate_samples', 'g4r_generate_samples_from_uniform',
    'g4r_set_sample_store', 'g4r_get_sample_store', 'g4r_sample_store_rows', 'g4r_set_sample_pointer', 'g4r_get_sample_pointer',
    'g4r_mrg_uniform', 'g4r_searchsorted', 'g4r_gather_rows',
    'g4r_schedule_build', 'g4r_schedule_free', 'g4r_schedule_steps', 'g4r_schedule_events', 'g4r_schedule_export',
    'g4r_train_step', 'g4r_train_steps', 'g4r_upload_steps', 'g4r_run_uploaded', 'g4r_kernel_launches',
    'g4r_profile_uploaded', 'g4r_phase_name', 'g4r_phase_count', 'g4r_persistent_stamps', 'g4r_fast_windows', 'g4r_uses_tensor_cores', 'g4r_mg_unique_id', 'g4r_mg_init',
    'g4r_mg_sharded', 'g4r_mg_ipc_handle', 'g4r_mg_ipc_open', 'g4r_mg_owner', 'g4r_mg_local_row', 'g4r_mg_shard_rows', 'g4r_mg_segment_bytes',
    'g4r_eval_schedule', 'g4r_set_eval_items', 'g4r_predict', 'g4r_reset_eval_hidden',
    'g4r_predict_topk',
]

_lib = None


def load():
    """Load libg4r.so (built in-tree by gru4rec_b200/csrc/build.sh / __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError('libg4r.so not found at %s: build it with gru4rec_b200/csrc/build.sh '
                           '(there is no CPU fallback)' % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, f32p = C.c_void_p, C.c_int32, C.c_int64, C.POINTER(C.c_float)
    lib.g4r_version.restype = C.c_int
    lib.g4r_workspace_bytes.argtypes = [C.POINTER(G4RConfig), C.POINTER(C.c_size_t)]
    lib.g4r_create.argtypes = [C.POINTER(G4RConfig), vp, C.c_size_t, C.POINTER(vp)]
    lib.g4r_destroy.argtypes = [vp]
    lib.g4r_last_error.argtypes = [vp]; lib.g4r_last_error.restype = C.c_char_p
    lib.g4r_stream.argtypes = [vp]; lib.g4r_stream.restype = vp
    lib.g4r_tensor_shape.argtypes = [vp, C.c_char_p, C.POINTER(i64), C.POINTER(i64)]
    lib.g4r_set_tensor.argtypes = [vp, C.c_char_p, vp, i64, i64]
    lib.g4r_get_tensor.argtypes = [vp, C.c_char_p, vp, i64, i64]
    lib.g4r_reset_hidden.argtypes = [vp]
    lib.g4r_set_sampling_cdf.argtypes = [vp, vp, i64]
    lib.g4r_set_logq_support.argtypes = [vp, vp, i64]
    lib.g4r_generate_samples.argtypes = [vp]
    lib.g4r_generate_samples_from_uniform.argtypes = [vp, vp, i64]
    lib.g4r_set_sample_store.argtypes = [vp, vp, i64]
    lib.g4r_get_sample_store.argtypes = [vp, vp, i64]
    lib.g4r_sample_store_rows.argtypes = [vp]
    lib.g4r_set_sample_pointer.argtypes = [vp, i64]
    lib.g4r_get_sample_pointer.argtypes = [vp]; lib.g4r_get_sample_pointer.restype = i64
    lib.g4r_mrg_uniform.argtypes = [vp, vp, i64]
    lib.g4r_searchsorted.argtypes = [vp, vp, i64, vp, i64, vp]
    lib.g4r_gather_rows.argtypes = [vp, vp, i64, i64, vp, i64, vp]
    lib.g4r_schedule_build.argtypes = [vp, i64, vp, i64, vp, i32, i32, i32, C.POINTER(vp)]
    lib.g4r_schedule_free.argtypes = [vp]
    lib.g4r_schedule_steps.argtypes = [vp]; lib.g4r_schedule_steps.restype = i64
    lib.g4r_schedule_events.argtypes = [vp]; lib.g4r_schedule_events.restype = i64
    lib.g4r_schedule_export.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.g4r_train_step.argtypes = [vp, vp, vp, i32, vp, C.POINTER(C.c_float)]
    lib.g4r_train_steps.argtypes = [vp, vp, i64, i64, vp, C.POINTER(i64)]
    lib.g4r_upload_steps.argtypes = [vp, vp, i64, i64]
    lib.g4r_run_uploaded.argtypes = [vp, vp, C.POINTER(C.c_float)]
    lib.g4r_kernel_launches.argtypes = [vp]; lib.g4r_kernel_launches.restype = i64
    lib.g4r_profile_uploaded.argtypes = [vp, vp, vp, i32]
    lib.g4r_phase_name.argtypes = [i32]; lib.g4r_phase_name.restype = C.c_char_p
    lib.g4r_phase_count.restype = C.c_int
    lib.g4r_persistent_stamps.argtypes = [vp, i32, vp, i64]
    lib.g4r_fast_windows.argtypes = [vp, C.POINTER(i64)]; lib.g4r_fast_windows.restype = i64
    lib.g4r_uses_tensor_cores.argtypes = [vp]
    lib.g4r_mg_unique_id.argtypes = [vp]
    lib.g4r_mg_init.argtypes = [vp, vp]
    lib.g4r_mg_sharded.argtypes = [vp]
    lib.g4r_mg_ipc_handle.argtypes = [vp, vp]
    lib.g4r_mg_ipc_open.argtypes = [vp, vp, i32]
    lib.g4r_mg_owner.argtypes = [i64, i32]
    lib.g4r_mg_local_row.argtypes = [i64, i32]; lib.g4r_mg_local_row.restype = i64
    lib.g4r_mg_shard_rows.argtypes = [i64, i32, i32]; lib.g4r_mg_shard_rows.restype = i64
    lib.g4r_mg_segment_bytes.argtypes = [C.POINTER(G4RConfig), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
    lib.g4r_eval_schedule.argtypes = [vp, vp, vp, i32, i32, vp, vp, C.POINTER(i64)]
    lib.g4r_set_eval_items.argtypes = [vp, vp, i64]
    lib.g4r_predict.argtypes = [vp, vp, i32, vp, vp]
    lib.g4r_reset_eval_hidden.argtypes = [vp]
    lib.g4r_predict_topk.argtypes = [vp, vp, i32, vp, vp, i64, i32, vp, vp]
    _lib = lib
    return lib


class NaNError(ArithmeticError):
    def __init__(self, msg, step):
        ArithmeticError.__init__(self, msg)
        self.step = step


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def parse_act(name):
    """'elu-0.5' -> (ACT code, p1, p2)   (gru4rec.py:144-161)."""
    if name in ('linear', 'relu', 'tanh', 'softmax', 'softmax_logit'):
        return ACT[name], 0.0, 0.0
    if name.startswith('leaky-'):
        return ACT['leaky'], float(name.split('-')[1]), 0.0
    if name.startswith('elu-'):
        return ACT['elu'], float(name.split('-')[1]), 0.0
    if name.startswith('selu-'):
        p = [float(x) for x in name.split('-')[1:]]
        return ACT['selu'], p[0], p[1]
    raise NotImplementedError


def set_adapt_params(cfg, adapt, adapt_params, grad_cap):
    """adapt_params as the reference uses them (gru4rec.py:301-304,342-343,368-369); the complements are taken in double like there"""
    ap = [float(x) for x in (adapt_params or [])]
    if adapt in ('rmsprop', 'adadelta') and len(ap) < 1 or adapt == 'adam' and len(ap) < 2:
        raise IndexError('list index out of range')          # what the reference raises when adapt_params is too short
    cfg.adapt_p1 = ap[0] if len(ap) > 0 else 0.0
    cfg.adapt_p1c = (1.0 - ap[0]) if len(ap) > 0 else 0.0
    cfg.adapt_p2 = ap[1] if len(ap) > 1 else 0.0
    cfg.adapt_p2c = (1.0 - ap[1]) if len(ap) > 1 else 0.0
    cfg.grad_cap = float(grad_cap or 0.0)


def make_config(n_items, mk, sample_store=0, eval_lanes=0, max_resident_steps=0, step_mode=0, world_size=1, rank=0, replicated=False, eval_tc=None):
    cfg = G4RConfig()
    layers = mk.get('layers', [100])
    cfg.n_items = n_items
    cfg.n_layers = len(layers)
    for i, l in enumerate(layers):
        cfg.layers[i] = l
    cfg.batch_size = mk.get('batch_size', 32)
    cfg.constrained_embedding = 1 if mk.get('constrained_embedding') else 0
    cfg.embedding = 0 if mk.get('constrained_embedding') else int(mk.get('embedding', 0) or 0)
    cfg.loss = LOSS[mk.get('loss', 'bpr-max')]
    cfg.final_act, cfg.final_act_p1, cfg.final_act_p2 = parse_act(mk.get('final_act', 'linear'))
    cfg.hidden_act, cfg.hidden_act_p1, cfg.hidden_act_p2 = parse_act(mk.get('hidden_act', 'tanh'))
    cfg.dropout_p_hidden = mk.get('dropout_p_hidden', 0.0)
    cfg.dropout_p_embed = mk.get('dropout_p_embed', 0.0)
    cfg.learning_rate = mk.get('learning_rate', 0.1)
    cfg.momentum = mk.get('momentum', 0.0)
    cfg.lmbd = mk.get('lmbd', 0.0)
    cfg.n_sample = mk.get('n_sample', 2048)
    cfg.sample_alpha = mk.get('sample_alpha', 0.75)
    cfg.smoothing = mk.get('smoothing', 0.0)
    cfg.bpreg = mk.get('bpreg', 1.0)
    cfg.logq = mk.get('logq', 0.0)
    cfg.adapt = ADAPT[mk.get('adapt', 'adagrad')]
    cfg.sample_store = sample_store
    cfg.dropout_seed = mk.get('dropout_seed', 0)
    cfg.mrg_seed = 12345
    cfg.max_resident_steps = max_resident_steps
    cfg.world_size, cfg.rank = world_size, rank
    cfg.eval_batch_size = eval_lanes
    cfg.step_mode = step_mode
    cfg.mg_replicated = 1 if replicated else 0     # multi-GPU: replicated tables + NCCL exchange instead of row sharding
    cfg.eval_tc = 0 if eval_tc is None else (2 if eval_tc else 1)   # scoring path: auto / force tcgen05 tiles / force fp32 FFMA tiles
    set_adapt_params(cfg, mk.get('adapt', 'adagrad'), mk.get('adapt_params', []), mk.get('grad_cap', 0.0))
    return cfg



class Schedule(object):
    """Host-side schedule of one epoch (gru4rec.py:594-651 / evaluation.py:90-139), built in C++."""

    def __init__(self, data_items, offset_sessions, session_order, batch_size, n_sample, mode=0):
        lib = load()
        self._lib = lib
        di = np.ascontiguousarray(data_items, dtype=np.int64)
        off = np.ascontiguousarray(offset_sessions, dtype=np.int32)
        order = None if session_order is None else np.ascontiguousarray(session_order, dtype=np.int64)
        h = C.c_void_p()
        # n_sessions = number of sessions this schedule walks: all of them, or the entries of a (possibly sharded) order
        n_sess = len(off) - 1 if order is None else len(order)
        if order is not None and len(order) and (order.min() < 0 or order.max() >= len(off) - 1):
            raise IndexError('session_order refers to a session that does not exist')
        rc = lib.g4r_schedule_build(_ptr(di), len(di), _ptr(off), n_sess, _ptr(order), batch_size, n_sample, mode, C.byref(h))
        if rc == G4R_ERR_INDEX:
            raise IndexError(lib.g4r_last_error(None).decode())
        if rc != 0:
            raise RuntimeError(lib.g4r_last_error(None).decode())
        self.h = h
        self.batch_size = batch_size
        self.n_steps = lib.g4r_schedule_steps(h)
        self.n_events = lib.g4r_schedule_events(h)

    def export(self):
        n, B = self.n_steps, self.batch_size
        X = np.empty((n, B), np.int32); Y = np.empty((n, B), np.int32); F = np.empty((n, B), np.uint8)
        M = np.empty(n, np.int32); S = np.empty((n, B), np.int32)
        self._lib.g4r_schedule_export(self.h, _ptr(X), _ptr(Y), _ptr(F), _ptr(M), _ptr(S))
        return dict(X=X, Y=Y, F=F, M=M, slots=S)

    def batch_sizes(self):
        """M of every mini-batch (the weights of the epoch loss, gru4rec.py:654) without copying the index arrays."""
        M = np.empty(self.n_steps, np.int32)
        self._lib.g4r_schedule_export(self.h, None, None, None, _ptr(M), None)
        return M

    def __del__(self):
        try:
            if self.h:
                self._lib.g4r_schedule_free(self.h)
                self.h = None
        except Exception:
            pass


class Engine(object):
    """Owns one g4r_handle.  Device memory is allocated through torch (used only as an allocator)."""

    def __init__(self, cfg, device=0, use_torch_allocator=True):
        lib = load()
        self.lib = lib
        self.cfg = cfg
        cfg.device = device
        nbytes = C.c_size_t()
        rc = lib.g4r_workspace_bytes(C.byref(cfg), C.byref(nbytes))
        if rc != 0:
            raise NotImplementedError(lib.g4r_last_error(None).decode())
        self._ws = None
        ws_ptr = None
        if use_torch_allocator:
            import torch
            if not torch.cuda.is_available():
                raise RuntimeError('gru4rec_b200 needs a CUDA device (B200 / sm_100a); there is no CPU fallback')
            self._ws = torch.empty(nbytes.value, dtype=torch.uint8, device='cuda:%d' % device)
            ws_ptr = C.c_void_p(self._ws.data_ptr())
        h = C.c_void_p()
        rc = lib.g4r_create(C.byref(cfg), ws_ptr, nbytes.value, C.byref(h))
        if rc != 0:
            msg = lib.g4r_last_error(None).decode()
            if rc == G4R_ERR_INVALID:
                raise NotImplementedError(msg)
            raise RuntimeError('g4r_create failed: ' + msg)
        self.h = h
        self.workspace_bytes = nbytes.value

    def close(self):
        if getattr(self, 'h', None):
            self.lib.g4r_destroy(self.h)
            self.h = None
            self._ws = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, nan_step=None):
        if rc == 0:
            return
        msg = self.lib.g4r_last_error(self.h).decode()
        if rc == G4R_ERR_INDEX:
            raise IndexError(msg)
        if rc == G4R_ERR_INVALID:
            raise NotImplementedError(msg)
        if rc == G4R_ERR_NAN:
            raise NaNError(msg, nan_step)
        raise RuntimeError('libg4r: %s (status %d)' % (msg, rc))

    # ---- tensors ----
    def shape(self, name):
        r, c = C.c_int64(), C.c_int64()
        self._check(self.lib.g4r_tensor_shape(self.h, name.encode(), C.byref(r), C.byref(c)))
        return r.value, c.value

    def set(self, name, arr):
        r, c = self.shape(name)
        a = np.ascontiguousarray(np.asarray(arr, dtype=np.float32).reshape(r, c))
        self._check(self.lib.g4r_set_tensor(self.h, name.encode(), _ptr(a), r, c))

    def get(self, name):
        r, c = self.shape(name)
        if name.split('.')[0] in ('Wy', 'By', 'Wx0'):
            self._quiesce()
        a = np.empty((r, c), dtype=np.float32)
        self._check(self.lib.g4r_get_tensor(self.h, name.encode(), _ptr(a), r, c))
        return a

    def reset_hidden(self):
        self._check(self.lib.g4r_reset_hidden(self.h))

    # ---- sampling ----
    def set_sampling_cdf(self, P):
        P = np.ascontiguousarray(P, dtype=np.float32)
        self._check(self.lib.g4r_set_sampling_cdf(self.h, _ptr(P), len(P)))

    def set_logq_support(self, P0):
        P0 = np.ascontiguousarray(P0, dtype=np.float32)
        self._check(self.lib.g4r_set_logq_support(self.h, _ptr(P0), len(P0)))

    def generate_samples(self):
        self._check(self.lib.g4r_generate_samples(self.h))

    def generate_samples_from_uniform(self, u):
        u = np.ascontiguousarray(u, dtype=np.float32)
        self._check(self.lib.g4r_generate_samples_from_uniform(self.h, _ptr(u), u.size))

    def sample_store_rows(self):
        return self.lib.g4r_sample_store_rows(self.h)

    def set_sample_store(self, st):
        st = np.ascontiguousarray(st, dtype=np.int64)
        self._check(self.lib.g4r_set_sample_store(self.h, _ptr(st), st.shape[0]))

    def get_sample_store(self):
        rows = self.sample_store_rows()
        st = np.empty((rows, self.cfg.n_sample), dtype=np.int64)
        self._check(self.lib.g4r_get_sample_store(self.h, _ptr(st), rows))
        return st

    def set_sample_pointer(self, p):
        self._check(self.lib.g4r_set_sample_pointer(self.h, p))

    def get_sample_pointer(self):
        return self.lib.g4r_get_sample_pointer(self.h)

    def mrg_uniform(self, n):
        out = np.empty(n, dtype=np.float32)
        self._check(self.lib.g4r_mrg_uniform(self.h, _ptr(out), n))
        return out

    # ---- stand-alone ops ----
    def searchsorted(self, d, x):
        d = np.ascontiguousarray(d, dtype=np.float32); x = np.ascontiguousarray(x, dtype=np.float32)
        y = np.empty(x.shape, dtype=np.int64)
        self._check(self.lib.g4r_searchsorted(self.h, _ptr(d), d.size, _ptr(x), x.size, _ptr(y)))
        return y

    def gather_rows(self, table, idx):
        table = np.ascontiguousarray(table, dtype=np.float32); idx = np.ascontiguousarray(idx, dtype=np.int64)
        out = np.empty((idx.size, table.shape[1]), dtype=np.float32)
        self._check(self.lib.g4r_gather_rows(self.h, _ptr(table), table.shape[0], table.shape[1], _ptr(idx), idx.size, _ptr(out)))
        return out

    # ---- training ----
    def train_step(self, X, Y, R=None):
        X = np.ascontiguousarray(X, dtype=np.int32); Y = np.ascontiguousarray(Y, dtype=np.int32)
        Rp = None if R is None else np.ascontiguousarray(np.asarray(R).reshape(-1), dtype=np.int8)
        cost = C.c_float()
        self._check(self.lib.g4r_train_step(self.h, _ptr(X), _ptr(Y), len(X), _ptr(Rp), C.byref(cost)))
        return np.float32(cost.value)

    def train_steps(self, sched, first=0, n=None):
        n = sched.n_steps - first if n is None else n
        if self.cfg.world_size > 1:
            # ranks advance in lock step (one merged update per mini-batch): a different n would dead-lock the collectives
            import torch
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized():
                dev = 'cuda' if dist.get_backend() == 'nccl' else 'cpu'
                t = torch.tensor([n, -n], dtype=torch.int64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MIN)
                if int(t[0]) != n or int(-t[1]) != n:
                    raise ValueError('train_steps: every rank must run the same number of steps (got %d, range %d..%d)' % (n, int(t[0]), int(-t[1])))
        costs = np.empty(n, dtype=np.float32)
        nan_step = C.c_int64(-1)
        rc = self.lib.g4r_train_steps(self.h, sched.h, first, n, _ptr(costs), C.byref(nan_step))
        self._check(rc, nan_step.value)
        return costs

    def upload_steps(self, sched, first, n):
        self._check(self.lib.g4r_upload_steps(self.h, sched.h, first, n))

    def run_uploaded(self, n, want_cost=True):
        costs = np.empty(n, dtype=np.float32) if want_cost else None
        ms = C.c_float()
        self._check(self.lib.g4r_run_uploaded(self.h, _ptr(costs), C.byref(ms)))
        return costs, ms.value

    def profile_uploaded(self):
        """{phase name: (total device ms, launches)} for one pass over the uploaded window."""
        n = self.lib.g4r_phase_count()
        ms = np.zeros(n, dtype=np.float32); cnt = np.zeros(n, dtype=np.int32)
        self._check(self.lib.g4r_profile_uploaded(self.h, _ptr(ms), _ptr(cnt), n))
        return {self.lib.g4r_phase_name(i).decode(): (float(ms[i]), int(cnt[i])) for i in range(n) if cnt[i] > 0}

    def persistent_stamps(self, enable=True, n_steps=0):
        out = np.zeros((n_steps, 16), dtype=np.uint64) if n_steps > 0 else None
        self._check(self.lib.g4r_persistent_stamps(self.h, 1 if enable else 0, _ptr(out), n_steps))
        return out

    def init_multi_gpu(self, dist):
        """Create the NCCL communicator of this handle: rank 0's unique id is broadcast through torch.distributed."""
        import torch
        buf = (C.c_char * 128)()
        if dist.get_rank() == 0:
            rc = self.lib.g4r_mg_unique_id(buf)
            if rc != 0:
                raise RuntimeError('ncclGetUniqueId failed')
        t = torch.tensor(list(bytes(buf)), dtype=torch.uint8, device='cuda' if dist.get_backend() == 'nccl' else 'cpu')
        dist.broadcast(t, 0)
        raw = bytes(t.cpu().tolist())
        idbuf = (C.c_char * 128).from_buffer_copy(raw)
        self._check(self.lib.g4r_mg_init(self.h, idbuf))
        self._dist = dist
        if self.sharded():
            # row-sharded tables: every rank maps the segments of all peers (cudaIpc); the 64-byte handles travel by all-gather
            mh = (C.c_char * 64)()
            self._check(self.lib.g4r_mg_ipc_handle(self.h, mh))
            dev = 'cuda' if dist.get_backend() == 'nccl' else 'cpu'
            mine = torch.tensor(list(bytes(mh)), dtype=torch.uint8, device=dev)
            allh = [torch.empty_like(mine) for _ in range(dist.get_world_size())]
            dist.all_gather(allh, mine)
            raw = b''.join(bytes(t.cpu().tolist()) for t in allh)
            buf2 = (C.c_char * len(raw)).from_buffer_copy(raw)
            self._check(self.lib.g4r_mg_ipc_open(self.h, buf2, dist.get_world_size()))
            dist.barrier()

    def sharded(self):
        return bool(self.lib.g4r_mg_sharded(self.h))

    def _quiesce(self):
        """sharded tensors are assembled from all ranks' memory: every rank must have finished its device work"""
        d = getattr(self, '_dist', None)
        if d is not None and self.sharded():
            import torch
            torch.cuda.synchronize()
            d.barrier()

    def uses_tensor_cores(self):
        return bool(self.lib.g4r_uses_tensor_cores(self.h))

    def fast_windows(self):
        fb = C.c_int64()
        n = self.lib.g4r_fast_windows(self.h, C.byref(fb))
        return n, fb.value

    def kernel_launches(self):
        return self.lib.g4r_kernel_launches(self.h)

    def stream(self):
        return self.lib.g4r_stream(self.h)

    # ---- scoring ----
    def eval_schedule(self, sched, cut_off, mode=0):
        cut = np.ascontiguousarray(cut_off, dtype=np.int32)
        rec = np.zeros(len(cut), dtype=np.float64); mrr = np.zeros(len(cut), dtype=np.float64)
        n = C.c_int64()
        self._check(self.lib.g4r_eval_schedule(self.h, sched.h, _ptr(cut), len(cut), mode, _ptr(rec), _ptr(mrr), C.byref(n)))
        return rec, mrr, n.value

    def set_eval_items(self, items=None):
        """Candidate item indices for eval_schedule (evaluate_gpu(items=...)); None / empty restores the whole catalogue."""
        if items is None or len(items) == 0:
            self._check(self.lib.g4r_set_eval_items(self.h, None, 0))
            return
        it = np.ascontiguousarray(items, dtype=np.int64)
        self._check(self.lib.g4r_set_eval_items(self.h, _ptr(it), it.size))

    def predict(self, X, reset_mask=None):
        X = np.ascontiguousarray(X, dtype=np.int32)
        rm = None if reset_mask is None else np.ascontiguousarray(reset_mask, dtype=np.uint8)
        out = np.empty((len(X), self.cfg.n_items), dtype=np.float32)
        self._check(self.lib.g4r_predict(self.h, _ptr(X), len(X), _ptr(rm), _ptr(out)))
        return out

    def predict_topk(self, X, k, reset_mask=None, cand=None):
        """The k best items of each lane among the scores predict() would return for the same call (the scoring-path hidden state
        advances the same way), selected on the device.  cand: optional item indices (no duplicates) the items compete among;
        softmax-family scores are then normalised over them.  Returns (items int32 [batch, k], scores float32 [batch, k]), each row
        by score descending, ties by item index ascending."""
        X = np.ascontiguousarray(X, dtype=np.int32)
        rm = None if reset_mask is None else np.ascontiguousarray(reset_mask, dtype=np.uint8)
        cd = None if cand is None else np.ascontiguousarray(cand, dtype=np.int64)
        k = int(k)
        items = np.empty((len(X), max(k, 0)), dtype=np.int32)
        scores = np.empty((len(X), max(k, 0)), dtype=np.float32)
        self._check(self.lib.g4r_predict_topk(self.h, _ptr(X), len(X), _ptr(rm), _ptr(cd), 0 if cd is None else cd.size, k,
                                              _ptr(items), _ptr(scores)))
        return items, scores

    def reset_eval_hidden(self):
        self._check(self.lib.g4r_reset_eval_hidden(self.h))
