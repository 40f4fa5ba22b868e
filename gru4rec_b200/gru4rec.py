"""GRU4Rec with the reference's class surface (hidasib/GRU4Rec gru4rec.py:27-781) on the B200 engine.

`run.py -g gru4rec_b200.gru4rec` (or the root-level shim module `gru4rec`) selects this class through the
reference's own plugin seam (run.py:21,39).  Constructor arguments, set_params() coercions and prints,
fit() / predict_next_batch() / savemodel() / loadmodel() signatures and printed lines follow the reference;
the per-mini-batch work runs in libg4r.so (hand-written sm_100a CUDA) through ctypes.  PyTorch is used
only to allocate the device workspace.  There is no CPU fallback.

Interface restatement, stated plainly: `__init__` (argument list, defaults, attribute assignments), `set_params` (the
coercion table and its `SET ... TO ...` / error prints), `init_matrix`, `generate_neg_samples` and the popularity / CDF
preamble of `fit` are the reference's statements almost line for line (gru4rec.py:97-135, 162-187, 254-260, 507-514,
534-556).  That is deliberate and required by the drop-in boundary: keyword names, defaults, coercions, printed lines,
exception types and the NumPy random-stream consumption order are the interface, and
tests/golden/set_params_cases.json + the golden fixtures pin them against the reference class.  Everything below that
surface (schedule, step, optimizers, evaluation, persistence plumbing, multi-GPU) is this repository's own design.
"""
import pickle
import time
import weakref
from collections import OrderedDict  # noqa: F401  (param files use it)

import numpy as np
import pandas as pd

from . import datatools
from . import _lib


class _DeviceParam(object):
    """Stand-in for a Theano shared variable: get_value()/set_value() round-trip through the engine."""

    def __init__(self, owner, name):
        self._owner = weakref.ref(owner)     # no reference cycle: the model (and its device engine) is freed by reference counting
        self.name = name

    def get_value(self, borrow=False):
        return self._owner()._get_param(self.name)

    def set_value(self, value, borrow=False):
        self._owner()._set_param(self.name, value)


class GRU4Rec:
    '''
    GRU4Rec(loss='bpr-max', final_act='elu-1', hidden_act='tanh', layers=[100],
                 n_epochs=10, batch_size=32, dropout_p_hidden=0.0, dropout_p_embed=0.0, learning_rate=0.1, momentum=0.0, lmbd=0.0, embedding=0, n_sample=2048, sample_alpha=0.75, smoothing=0.0, constrained_embedding=False,
                 adapt='adagrad', adapt_params=[], grad_cap=0.0, bpreg=1.0, logq=0.0,
                 sigma=0.0, init_as_normal=False, train_random_order=False, time_sort=True,
                 session_key='SessionId', item_key='ItemId', time_key='Time')
    Same parameters as the reference class (gru4rec.py:28-96), all optimizers (adagrad / rmsprop / adadelta / adam / None),
    grad_cap and smoothing included.  Not on the device path (NotImplementedError when fit() builds the engine): loss /
    final_act pairs other than {cross-entropy+softmax, xe_logit+softmax_logit, pairwise losses + elementwise activations},
    and rmsprop / adadelta / adam together with constrained_embedding.
    '''

    def __init__(self, loss='bpr-max', final_act='linear', hidden_act='tanh', layers=[100],
                 n_epochs=10, batch_size=32, dropout_p_hidden=0.0, dropout_p_embed=0.0, learning_rate=0.1, momentum=0.0, lmbd=0.0, embedding=0, n_sample=2048, sample_alpha=0.75, smoothing=0.0, constrained_embedding=False,
                 adapt='adagrad', adapt_params=[], grad_cap=0.0, bpreg=1.0, logq=0.0,
                 sigma=0.0, init_as_normal=False, train_random_order=False, time_sort=True,
                 session_key='SessionId', item_key='ItemId', time_key='Time'):
        self.layers = layers
        self.n_epochs = n_epochs
        self.batch_size = batch_size
        self.dropout_p_hidden = dropout_p_hidden
        self.dropout_p_embed = dropout_p_embed
        self.learning_rate = learning_rate
        self.adapt_params = adapt_params
        self.momentum = momentum
        self.sigma = sigma
        self.init_as_normal = init_as_normal
        self.session_key = session_key
        self.item_key = item_key
        self.time_key = time_key
        self.grad_cap = grad_cap
        self.bpreg = bpreg
        self.logq = logq
        self.train_random_order = train_random_order
        self.lmbd = lmbd
        if embedding == 'layersize':
            self.embedding = self.layers[0]
        else:
            self.embedding = embedding
        self.constrained_embedding = constrained_embedding
        self.time_sort = time_sort
        self.adapt = adapt
        self.loss = loss
        self.set_loss_function(self.loss)
        self.final_act = final_act
        self.set_final_activation(self.final_act)
        self.hidden_act = hidden_act
        self.set_hidden_activation(self.hidden_act)
        self.n_sample = n_sample
        self.sample_alpha = sample_alpha
        self.smoothing = smoothing
        # engine-side options (not part of the reference surface)
        self.device = 0
        self.dropout_seed = 0
        self.eval_lanes = 512            # run.py evaluates with batch_size=512 (run.py:127)
        self.step_mode = 2               # role-specialised persistent kernel where the shape allows, else generic persistent
        self._engine = None
        self._host = None                # numpy copies of the parameters when no engine is alive


    # ---- names that pickles written by the reference class refer to (gru4rec.py:136-161, 189-248) ----------------------
    # The reference pickles `self` including bound methods (loss_function = self.bpr_max, final_activation =
    # self.Elu(a).execute, ...).  These stubs make such pickles load into this class; the Theano graph builders themselves
    # have no counterpart here (the device kernels are selected from the `loss` / `final_act` / `hidden_act` strings).
    def _make_stub(name):
        def stub(self, *a, **k):
            raise NotImplementedError('Theano graph builders are not part of the B200 implementation')
        stub.__name__ = name            # bound methods are pickled by name: it must be the reference's method name
        stub.__qualname__ = 'GRU4Rec.' + name
        return stub
    cross_entropy = _make_stub('cross_entropy'); cross_entropy_logits = _make_stub('cross_entropy_logits')
    bpr = _make_stub('bpr'); bpr_max = _make_stub('bpr_max'); top1 = _make_stub('top1'); top1_max = _make_stub('top1_max')
    linear = _make_stub('linear'); tanh = _make_stub('tanh'); softmax = _make_stub('softmax'); softmax_logit = _make_stub('softmax_logit')
    softmax_neg = _make_stub('softmax_neg'); relu = _make_stub('relu'); sigmoid = _make_stub('sigmoid')
    del _make_stub

    class Selu:
        def __init__(self, lmbd=1.0, alpha=1.0):
            self.lmbd = lmbd; self.alpha = alpha
        def execute(self, X):
            raise NotImplementedError('Theano graph builders are not part of the B200 implementation')

    class Elu:
        def __init__(self, alpha=1.0):
            self.alpha = alpha
        def execute(self, X):
            raise NotImplementedError('Theano graph builders are not part of the B200 implementation')

    class LeakyReLU:
        def __init__(self, leak=0.0):
            self.leak = leak
        def execute(self, X):
            raise NotImplementedError('Theano graph builders are not part of the B200 implementation')

    # ---- same validation behaviour as the reference setters (gru4rec.py:136-161) ----
    def set_loss_function(self, loss):
        if loss not in ('cross-entropy', 'bpr', 'bpr-max', 'top1', 'top1-max', 'xe_logit'):
            raise NotImplementedError

    def set_final_activation(self, final_act):
        _lib.parse_act(final_act)

    def set_hidden_activation(self, hidden_act):
        if hidden_act in ('softmax', 'softmax_logit'):
            raise NotImplementedError
        _lib.parse_act(hidden_act)

    def set_params(self, **kvargs):
        """gru4rec.py:162-187, including the printed lines."""
        maxk_len = np.max([len(str(x)) for x in kvargs.keys()])
        maxv_len = np.max([len(str(x)) for x in kvargs.values()])
        for k, v in kvargs.items():
            if not hasattr(self, k):
                print('Unkown attribute: {}'.format(k))
                raise NotImplementedError
            else:
                if type(v) == str and k == 'adapt_params': v = [float(l) for l in v.split('/')]
                elif type(v) == str and type(getattr(self, k)) == list: v = [int(l) for l in v.split('/')]
                if type(v) == str and type(getattr(self, k)) == bool:
                    if v == 'True' or v == '1': v = True
                    elif v == 'False' or v == '0': v = False
                    else:
                        print('Invalid value for boolean parameter: {}'.format(v))
                        raise NotImplementedError
                if k == 'embedding' and v == 'layersize':
                    self.embedding = 'layersize'
                setattr(self, k, type(getattr(self, k))(v))
                if k == 'loss': self.set_loss_function(self.loss)
                if k == 'final_act': self.set_final_activation(self.final_act)
                if k == 'hidden_act': self.set_hidden_activation(self.hidden_act)
                print('SET   {}{}TO   {}{}(type: {})'.format(k, ' ' * (maxk_len - len(k) + 3), getattr(self, k), ' ' * (maxv_len - len(str(getattr(self, k))) + 3), type(getattr(self, k))))
        if self.embedding == 'layersize':
            self.embedding = self.layers[0]
            print('SET   {}{}TO   {}{}(type: {})'.format('embedding', ' ' * (maxk_len - len('embedding') + 3), getattr(self, 'embedding'), ' ' * (maxv_len - len(str(getattr(self, 'embedding'))) + 3), type(getattr(self, 'embedding'))))

    # ---- weight initialisation, draw order as in the reference (gru4rec.py:254-294) ----
    def init_matrix(self, shape):
        if self.sigma != 0: sigma = self.sigma
        else: sigma = np.sqrt(6.0 / (shape[0] + shape[1]))
        if self.init_as_normal:
            return np.asarray(np.random.randn(*shape) * sigma, dtype=np.float32)
        else:
            return np.asarray(np.random.rand(*shape) * sigma * 2 - sigma, dtype=np.float32)

    def _init_host_weights(self):
        np.random.seed(42)
        w = {}
        if self.constrained_embedding:
            n_features = self.layers[-1]
        elif self.embedding:
            w['E'] = self.init_matrix((self.n_items, self.embedding))
            n_features = self.embedding
        else:
            n_features = self.n_items
        for i in range(len(self.layers)):
            nin = self.layers[i - 1] if i > 0 else n_features
            m = [self.init_matrix((nin, self.layers[i])) for _ in range(3)]
            w['Wx%d' % i] = np.hstack(m)
            w['Wh%d' % i] = self.init_matrix((self.layers[i], self.layers[i]))
            m2 = [self.init_matrix((self.layers[i], self.layers[i])) for _ in range(2)]
            w['Wrz%d' % i] = np.hstack(m2)
            w['Bh%d' % i] = np.zeros((self.layers[i] * 3,), dtype=np.float32)
        w['Wy'] = self.init_matrix((self.n_items, self.layers[-1]))
        w['By'] = np.zeros((self.n_items, 1), dtype=np.float32)
        return w

    def init(self, data):
        datatools.sort_if_needed(data, [self.session_key, self.time_key])
        offset_sessions = datatools.compute_offset(data, self.session_key)
        self._host = self._init_host_weights()
        return offset_sessions

    # ---- engine management ----
    def _param_names(self):
        names = []
        for i in range(len(self.layers)):
            names += ['Wx%d' % i, 'Wh%d' % i, 'Wrz%d' % i, 'Bh%d' % i]
        names += ['Wy', 'By']
        if self.embedding and not self.constrained_embedding:
            names.append('E')
        return names

    def _make_config(self, sample_store, eval_lanes, training=True, single=False):
        """`training=False`: an engine for the scoring path only (evaluate_gpu / predict_next_batch of a loaded model): the
        optimiser options are irrelevant there, so a model the reference trained with adam / rmsprop / adadelta, grad_cap or
        smoothing can still be scored; fit() with those options raises NotImplementedError (SURVEY section 8 a14)."""
        cfg = _lib.G4RConfig()
        if training and self.adapt not in _lib.ADAPT:
            raise NotImplementedError('adapt=%r is not an optimizer of the reference (gru4rec.py:392-399)' % (self.adapt,))
        cfg.n_items = self.n_items
        cfg.n_layers = len(self.layers)
        for i, l in enumerate(self.layers):
            cfg.layers[i] = l
        cfg.batch_size = self.batch_size
        cfg.constrained_embedding = 1 if self.constrained_embedding else 0
        cfg.embedding = 0 if self.constrained_embedding else int(self.embedding or 0)
        cfg.loss = _lib.LOSS[self.loss]
        cfg.final_act, cfg.final_act_p1, cfg.final_act_p2 = _lib.parse_act(self.final_act)
        cfg.hidden_act, cfg.hidden_act_p1, cfg.hidden_act_p2 = _lib.parse_act(self.hidden_act)
        cfg.dropout_p_hidden = self.dropout_p_hidden
        cfg.dropout_p_embed = self.dropout_p_embed
        cfg.learning_rate = self.learning_rate
        cfg.momentum = self.momentum
        cfg.lmbd = self.lmbd
        cfg.n_sample = self.n_sample
        cfg.sample_alpha = self.sample_alpha
        cfg.smoothing = self.smoothing if training else 0.0
        cfg.bpreg = self.bpreg
        cfg.logq = self.logq
        cfg.adapt = _lib.ADAPT[self.adapt] if training else _lib.ADAPT[None]
        cfg.sample_store = int(sample_store)
        cfg.dropout_seed = self.dropout_seed
        cfg.mrg_seed = 12345
        _lib.set_adapt_params(cfg, self.adapt if training else None, self.adapt_params if training else [], self.grad_cap if training else 0.0)
        cfg.max_resident_steps = 0
        cfg.world_size, cfg.rank = (1, 0) if single else self._world()
        cfg.eval_batch_size = eval_lanes
        cfg.step_mode = self.step_mode
        if self.step_mode == 2 and len(self.layers) == 1 and 120 < self.layers[0] <= 128 and not self.constrained_embedding and not self.embedding and self.batch_size <= 32:
            cfg.step_mode = 3        # the 48-CTA GRU group of step_mode 2 covers 120 hidden units; the cluster variant takes up to 128
        return cfg

    @staticmethod
    def _world():
        """(world_size, rank) of the torch.distributed job this process belongs to, or (1, 0)."""
        try:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
                return dist.get_world_size(), dist.get_rank()
        except Exception:
            pass
        return 1, 0

    def _build_engine(self, sample_store=0, eval_lanes=None, training=True, single=False):
        """`single`: a one-GPU engine even under torchrun (the scoring path of every rank works on a full replica)."""
        eval_lanes = self.eval_lanes if eval_lanes is None else eval_lanes
        host = self._host if self._host is not None else self._pull_host()
        if self._engine is not None:
            self._engine.close()
            self._engine = None
        world, rank = (1, 0) if single else self._world()
        if self._world()[0] > 1:
            import torch
            self.device = torch.cuda.current_device()
        eng = _lib.Engine(self._make_config(sample_store, eval_lanes, training, single=single), device=self.device)
        for name in self._param_names():
            eng.set(name, host[name])
        if world > 1:
            import torch.distributed as dist
            eng.init_multi_gpu(dist)
        self._engine = eng
        self._engine_eval_lanes = eval_lanes
        self._host = None
        self._bind_params()
        return eng

    def _bind_params(self):
        n = len(self.layers)
        self.Wx = [_DeviceParam(self, 'Wx%d' % i) for i in range(n)]
        self.Wh = [_DeviceParam(self, 'Wh%d' % i) for i in range(n)]
        self.Wrz = [_DeviceParam(self, 'Wrz%d' % i) for i in range(n)]
        self.Bh = [_DeviceParam(self, 'Bh%d' % i) for i in range(n)]
        self.H = [_DeviceParam(self, 'H%d' % i) for i in range(n)]
        self.Wy = _DeviceParam(self, 'Wy')
        self.By = _DeviceParam(self, 'By')
        if self.embedding and not self.constrained_embedding:
            self.E = _DeviceParam(self, 'E')

    def _get_param(self, name):
        if self._engine is not None:
            a = self._engine.get(name)
            return a.reshape(-1) if name.startswith('Bh') else a
        return self._host[name]

    def _set_param(self, name, value):
        if self._engine is not None:
            self._engine.set(name, value)
        else:
            self._host[name] = np.asarray(value, dtype=np.float32)

    def _pull_host(self):
        return {name: self._get_param(name) for name in self._param_names()}

    def _ensure_engine(self, eval_lanes):
        """Engine for the scoring path (evaluate_gpu / predict_next_batch).  After a multi-GPU fit() the training engine holds
        1/world of the item tables: the parameters are assembled on the host and every rank scores on its own full replica."""
        if self._engine is None or self._engine_eval_lanes < eval_lanes or int(self._engine.cfg.world_size) > 1:
            self._build_engine(sample_store=0, eval_lanes=max(eval_lanes, self.eval_lanes), training=False, single=True)
        return self._engine

    def generate_neg_samples(self, pop, length):
        """Legacy host-side sampler (store_type='cpu'; gru4rec.py:507-514)."""
        if self.sample_alpha:
            sample = np.searchsorted(pop, np.random.rand(self.n_sample * length))
        else:
            sample = np.random.choice(self.n_items, size=self.n_sample * length)
        if length > 1:
            sample = sample.reshape((length, self.n_sample))
        return sample

    # ---- training (gru4rec.py:515-664) ----
    def fit(self, data, sample_store=10000000, store_type='gpu'):
        '''
        Trains the network.  Same arguments, data-frame side effects ('ItemIdx' column, in-place sort) and
        printed lines as the reference (gru4rec.py:515-664).
        '''
        self.predict = None
        self.error_during_train = False
        # id map in order of first appearance, item index column, supports -- one factorize + one bincount (same values as the
        # reference's unique() / Series lookup / groupby().size() chain, gru4rec.py:534-545)
        codes, itemids = pd.factorize(data[self.item_key].values)
        if (codes < 0).any():
            raise KeyError('missing item id in the training data')
        self.n_items = len(itemids)
        self.itemidmap = pd.Series(data=np.arange(self.n_items), index=itemids, name='ItemIdx')
        data['ItemIdx'] = codes.astype(np.int64)
        offset_sessions = self.init(data)
        pop = pd.Series(np.bincount(data['ItemIdx'].values, minlength=self.n_items), index=self.itemidmap.index.values)
        P0 = None
        if self.logq:
            P0 = pop[self.itemidmap.index.values].values.astype(np.float32)
        generate_length = 0
        use_store = False
        if self.n_sample:
            pop = pop[self.itemidmap.index.values].values ** self.sample_alpha
            pop = pop.cumsum() / pop.sum()
            pop[-1] = 1
            if sample_store:
                generate_length = sample_store // self.n_sample
                if generate_length <= 1:
                    sample_store = 0
                    print('No example store was used')
                elif store_type == 'cpu':
                    use_store = True
                    print('Created sample store with {} batches of samples (type=CPU)'.format(generate_length))
                elif store_type == 'gpu':
                    use_store = True
                else:
                    print('Invalid store type {}'.format(store_type))
                    raise NotImplementedError
            else:
                print('No example store was used')
        per_step_sampling = False
        if self.n_sample and not use_store:
            if store_type == 'cpu':
                # gru4rec.py:612-613: without a store every mini-batch draws its own row on the host (generate_neg_samples(pop, 1))
                per_step_sampling = True
            else:
                # the reference's device path has no per-step sampler: its loop dereferences an undefined sample pointer here
                raise NotImplementedError('n_sample > 0 needs a sample store when store_type is \'gpu\' (sample_store >= 2 * n_sample)')
        if self.adapt == 'adadelta' and self.learning_rate != 1.0:        # gru4rec.py:362-364
            print('Warn: learning_rate is not 1.0 while using adadelta. Setting learning_rate to 1.0')
            self.learning_rate = 1.0
        world, rank = self._world()
        if world > 1 and self.constrained_embedding:
            # the merged update of a shared table interleaves the input rows Wy[X] with the score columns of every rank; the
            # library refuses it too (g4r_mg_init) -- say so before any engine is built, identically on every rank
            raise NotImplementedError('constrained_embedding=True does not train on several GPUs yet: run fit() in one process '
                                      '(evaluate_gpu / predict_next_batch of the trained model do run under torchrun)')
        if world > 1 and store_type == 'cpu':
            # the host-side sampler draws from one NumPy stream and refills at rank-local step counts: the lock-step ranks
            # would diverge (different numbers of collectives) -- only the device store is defined for multi-GPU training
            raise NotImplementedError("store_type='cpu' is not available for multi-GPU training; use the device sample store")
        # the training engine carries no scoring lanes: the step scratch keeps the leading dimension of the mini-batch
        # (the scoring engine with `eval_lanes` lanes is created on the first evaluate_gpu / predict_next_batch call)
        eng = self._build_engine(sample_store=(sample_store if use_store else (2 * self.n_sample if per_step_sampling else 0)), eval_lanes=0)
        if P0 is not None:
            eng.set_logq_support(P0)
        if use_store:
            eng.set_sampling_cdf(pop.astype(np.float32))
            if store_type == 'gpu':
                eng.generate_samples()
                print('Created sample store with {} batches of samples (type=GPU)'.format(generate_length))
            else:
                eng.set_sample_store(self.generate_neg_samples(pop, generate_length))
        # first event time of every session = the time at its offset (the frame is sorted by session, time) -- gru4rec.py:585
        base_order = np.argsort(data[self.time_key].values[offset_sessions[:-1]]) if self.time_sort else np.arange(len(offset_sessions) - 1)
        data_items = data.ItemIdx.values
        # under torchrun: synchronous data parallelism, every rank trains a shard of the sessions
        sched = None
        n_sample_eff = self.n_sample
        for epoch in range(self.n_epochs):
            t0 = time.time()
            eng.reset_hidden()
            session_idx_arr = np.random.permutation(len(offset_sessions) - 1) if self.train_random_order else base_order
            if sched is None or self.train_random_order:
                n_steps = None
                if world > 1:
                    import torch.distributed as dist
                    from .parallel import shard_sessions, common_steps
                    session_idx_arr = shard_sessions(session_idx_arr, rank, world)
                sched = _lib.Schedule(data_items, offset_sessions, session_idx_arr, self.batch_size, n_sample_eff, mode=0)
                n_steps = sched.n_steps if world == 1 else common_steps(sched.n_steps, dist)
                cc = sched.batch_sizes()[:n_steps].astype(np.float64)
            try:
                if per_step_sampling:
                    c = self._train_epoch_per_step_samples(eng, sched, pop)
                elif use_store and store_type == 'cpu':
                    c = self._train_epoch_cpu_store(eng, sched, pop, generate_length)
                else:
                    c = eng.train_steps(sched, 0, n_steps)
            except _lib.NaNError:
                print(str(epoch) + ': NaN error!')
                self.error_during_train = True
                if world > 1:      # the peers find out at their next exchange (time-out -> RuntimeError); nothing collective here
                    self._engine.close(); self._engine = None; self._host = None
                return
            sum_c, sum_e, n_mb = np.sum(c * cc), np.sum(cc), len(c)
            if world > 1:
                # one epoch line for the whole job: event-weighted loss, mini-batches and events of all ranks
                from .parallel import allreduce_sum
                sum_c, sum_e, n_mb = allreduce_sum([sum_c, sum_e, n_mb], dist)
            avgc = sum_c / sum_e
            if np.isnan(avgc):
                print('Epoch {}: NaN error!'.format(str(epoch)))
                self.error_during_train = True
                break
            t1 = time.time()
            dt = t1 - t0
            print('Epoch{} --> loss: {:.6f} \t({:.2f}s) \t[{:.2f} mb/s | {:.0f} e/s]'.format(epoch + 1, avgc, dt, n_mb / dt, sum_e / dt))
        if world > 1:
            self._release_multi_gpu_engine()

    def _release_multi_gpu_engine(self):
        """End of a multi-GPU fit(): every rank assembles the full parameter set on the host (the item tables are row-sharded
        over the ranks' library-owned segments), then all ranks release their training engines together -- no rank frees its
        segment while a peer still reads it.  Scoring / saving afterwards needs no collective (evaluate_gpu, predict_next_batch
        rebuild a single-GPU engine from the host copy; savemodel pickles it)."""
        eng = self._engine
        if eng is None:
            return
        host = self._pull_host()
        eng._quiesce()
        eng.close()
        self._engine = None
        self._host = host

    def _train_epoch_cpu_store(self, eng, sched, pop, generate_length):
        """store_type='cpu' (legacy, gru4rec.py:605-614): samples are drawn by NumPy on the host, one store at a time."""
        costs = []
        done = 0
        while done < sched.n_steps:
            if eng.get_sample_pointer() >= generate_length:
                eng.set_sample_store(self.generate_neg_samples(pop, generate_length))
            n = min(sched.n_steps - done, generate_length - eng.get_sample_pointer())
            costs.append(eng.train_steps(sched, done, n))
            done += n
        return np.concatenate(costs)

    def _train_epoch_per_step_samples(self, eng, sched, pop):
        """store_type='cpu' without a store (gru4rec.py:612-613): one host draw of n_sample items per mini-batch."""
        costs = []
        for k in range(sched.n_steps):
            row = np.asarray(self.generate_neg_samples(pop, 1)).reshape(1, self.n_sample)
            eng.set_sample_store(np.vstack([row, row]))
            eng.set_sample_pointer(0)
            costs.append(eng.train_steps(sched, k, 1))
        return np.concatenate(costs)

    # ---- serving (gru4rec.py:665-728) ----
    def predict_next_batch(self, session_ids, input_item_ids, predict_for_item_ids=None, batch=100):
        '''
        Gives prediction scores for a selected set of items; same contract as the reference
        (gru4rec.py:665-728): hidden state kept per batch coordinate while the session id stays the same.
        Returns a DataFrame, rows = items, columns = events of the batch.
        '''
        if self.error_during_train: raise Exception
        eng = self._ensure_engine(batch)
        if getattr(self, 'predict', None) is None or self.predict_batch != batch:
            self.predict_batch = batch
            eng.reset_eval_hidden()
            self.current_session = np.ones(batch) * -1
            self.predict = True
        session_ids = np.asarray(session_ids)
        reset = (session_ids != self.current_session)
        if reset.any():
            self.current_session = session_ids.copy()
        in_idxs = self.itemidmap[input_item_ids].values
        preds = eng.predict(in_idxs, reset.astype(np.uint8)).T          # items x batch
        if predict_for_item_ids is not None:
            iIdxs = self.itemidmap[predict_for_item_ids].values
            preds = preds[iIdxs]
            if self.final_act in ('softmax', 'softmax_logit'):
                preds = preds / preds.sum(axis=0, keepdims=True)          # softmax over the requested subset
            return pd.DataFrame(data=preds, index=predict_for_item_ids)
        return pd.DataFrame(data=preds, index=self.itemidmap.index)

    def recommend_next_batch(self, session_ids, input_item_ids, k=20, predict_for_item_ids=None, batch=100):
        '''
        The k best next items of every event of the batch, selected on the device: the scores are those predict_next_batch
        returns for the same call, but the items x batch matrix is never built or copied.  The session bookkeeping is the same
        as predict_next_batch's (hidden state kept per batch coordinate while the session id stays the same), so calls of the
        two methods can be interleaved on one model.
        predict_for_item_ids: optional list of distinct item ids the recommendations are drawn from; for softmax / softmax_logit
        the scores are normalised over this list, as predict_next_batch(..., predict_for_item_ids) does.
        Returns (item_ids, scores): original item ids [events x k] and float32 scores [events x k]; row b answers event b,
        sorted by score descending, ties broken by the lower item index.
        '''
        if self.error_during_train: raise Exception
        if isinstance(k, (bool, np.bool_)) or not isinstance(k, (int, np.integer)):
            raise ValueError('k must be an integer, got %r' % (k,))
        cand = None
        if predict_for_item_ids is not None:
            if pd.Index(predict_for_item_ids).has_duplicates:
                raise ValueError('predict_for_item_ids contains duplicates')
            cand = self.itemidmap[predict_for_item_ids].values
        n_cand = self.n_items if cand is None else len(cand)
        if not 1 <= k <= min(256, n_cand):
            raise ValueError('k must be in 1 .. min(256, number of candidate items) = %d, got %d' % (min(256, n_cand), k))
        in_idxs = self.itemidmap[input_item_ids].values
        eng = self._ensure_engine(batch)
        # session bookkeeping of predict_next_batch
        if getattr(self, 'predict', None) is None or self.predict_batch != batch:
            self.predict_batch = batch
            eng.reset_eval_hidden()
            self.current_session = np.ones(batch) * -1
            self.predict = True
        session_ids = np.asarray(session_ids)
        reset = (session_ids != self.current_session)
        if reset.any():
            self.current_session = session_ids.copy()
        idx, scores = eng.predict_topk(in_idxs, int(k), reset.astype(np.uint8), cand)
        return self.itemidmap.index.to_numpy()[idx], scores

    # ---- persistence (gru4rec.py:742-781): pickle of the object with NumPy parameters ----
    def __getstate__(self):
        st = dict(self.__dict__)
        host = self._host if self._engine is None else self._pull_host()
        for k in ('_engine', 'Wx', 'Wh', 'Wrz', 'Bh', 'H', 'Wy', 'By', 'E', '_host'):
            st.pop(k, None)
        n = len(self.layers)
        st['Wx'] = [host['Wx%d' % i] for i in range(n)]
        st['Wh'] = [host['Wh%d' % i] for i in range(n)]
        st['Wrz'] = [host['Wrz%d' % i] for i in range(n)]
        st['Bh'] = [host['Bh%d' % i].reshape(-1) for i in range(n)]
        st['H'] = [np.zeros((self.batch_size, self.layers[i]), dtype=np.float32) for i in range(n)]
        st['Wy'] = host['Wy']
        st['By'] = host['By']
        if 'E' in host:
            st['E'] = host['E']
        # what the reference class needs after unpickling (its __init__ is not run): the bound graph builders, pickled by
        # name (gru4rec.py:136-161) -- with this class registered as gru4rec.GRU4Rec the reference resolves its own methods
        st['loss_function'] = getattr(self, {'cross-entropy': 'cross_entropy', 'bpr': 'bpr', 'bpr-max': 'bpr_max', 'top1': 'top1',
                                             'top1-max': 'top1_max', 'xe_logit': 'cross_entropy_logits'}[self.loss])
        st['final_activation'] = self._act_object(self.final_act)
        st['hidden_activation'] = self._act_object(self.hidden_act)
        for k in ('device', 'dropout_seed', 'eval_lanes', 'step_mode', '_engine_eval_lanes', 'predict', 'predict_batch', 'current_session'):
            st.pop(k, None)
        st['predict'] = None
        return st

    def _act_object(self, name):
        if name.startswith('leaky-'): return self.LeakyReLU(float(name.split('-')[1])).execute
        if name.startswith('elu-'): return self.Elu(float(name.split('-')[1])).execute
        if name.startswith('selu-'): return self.Selu(*[float(x) for x in name.split('-')[1:]]).execute
        return getattr(self, name)

    def __setstate__(self, st):
        st = dict(st)
        for k in ('loss_function', 'final_activation', 'hidden_activation'):   # bound Theano graph builders in reference pickles
            st.pop(k, None)
        self.__dict__.update(st)
        n = len(self.layers)
        host = {}
        for i in range(n):
            host['Wx%d' % i] = np.asarray(self.Wx[i], dtype=np.float32)
            host['Wh%d' % i] = np.asarray(self.Wh[i], dtype=np.float32)
            host['Wrz%d' % i] = np.asarray(self.Wrz[i], dtype=np.float32)
            host['Bh%d' % i] = np.asarray(self.Bh[i], dtype=np.float32).reshape(-1)
        host['Wy'] = np.asarray(self.Wy, dtype=np.float32)
        host['By'] = np.asarray(self.By, dtype=np.float32).reshape(-1, 1)
        if getattr(self, 'embedding', 0) and not getattr(self, 'constrained_embedding', False) and 'E' in st:
            host['E'] = np.asarray(self.E, dtype=np.float32)
        self._host = host
        self._engine = None
        self.predict = None
        for k, v in (('device', 0), ('dropout_seed', 0), ('eval_lanes', 512), ('step_mode', 2)):
            if not hasattr(self, k):
                setattr(self, k, v)

    def savemodel(self, fname):
        with open(fname, 'wb') as f:
            pickle.dump(self, f)

    @classmethod
    def loadmodel(cls, fname):
        return pd.read_pickle(fname)


# Pickles name the class by module path.  The reference's models are `gru4rec.GRU4Rec`; registering this class under the
# same path makes pickles interchangeable in both directions (reference-written pickles load here; pickles written here
# load into the reference class, whose own graph builders are resolved by name).
GRU4Rec.__module__ = 'gru4rec'
GRU4Rec.__qualname__ = 'GRU4Rec'
for _n in ('Selu', 'Elu', 'LeakyReLU'):
    getattr(GRU4Rec, _n).__module__ = 'gru4rec'
    getattr(GRU4Rec, _n).__qualname__ = 'GRU4Rec.' + _n
import sys as _sys
if 'gru4rec' not in _sys.modules:
    import types as _types
    _m = _types.ModuleType('gru4rec')
    _m.GRU4Rec = GRU4Rec
    _sys.modules['gru4rec'] = _m
