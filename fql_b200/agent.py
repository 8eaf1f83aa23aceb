"""FQLAgent: host-side mirror of the reference agent API (agents/fql.py) over the libfql_b200 C ABI.

Same surface as the reference class (`create`, `update`, `sample_actions`, `total_loss`, `compute_flow_actions`,
`target_update` semantics, `network.params / opt_state / step`, `rng`, `config`) and the same parameter layout
(SURVEY 8a), so the training loop of main.py:159-165,216,225,284 runs unchanged.  Differences, all deliberate:
  * state lives in flat device arenas and is updated IN PLACE; `update` returns `(self, info)` so the caller's
    `agent, info = agent.update(batch)` rebind still works (the reference returns a new pytree, fql.py:133);
  * `info` values are fetched lazily from a pinned host ring (like jax's async dispatch: reading a value syncs);
  * noise comes from a device Philox generator keyed by (agent.rng, step); jax threefry streams are not reproduced
    (SURVEY 8c).  Parity tests inject the five noise tensors explicitly via `noise=`.
There is no CPU path: everything below calls CUDA through fql_b200._lib.
"""
from __future__ import annotations

import ctypes as C
import os
import weakref

import numpy as np
import torch

from . import _lib
from .config import get_config  # noqa: F401  (re-export, agents/fql.py:249)

INFO_KEYS = ('critic/critic_loss', 'critic/q_mean', 'critic/q_max', 'critic/q_min', 'actor/actor_loss', 'actor/bc_flow_loss',
             'actor/distill_loss', 'actor/q_loss', 'actor/q', 'actor/mse', 'grad/max', 'grad/min', 'grad/norm')
NOISE_KEYS = ('z_next', 'x0', 't', 'z', 'z_metric')
_BATCH_KEYS = ('observations', 'actions', 'next_observations', 'rewards', 'masks')
_PIN_RING = 4   # pinned staging blocks per batch size
# hyperparameters that may differ between the vectorised seeds (FqlHparams.per_seed); everything else is shared
PER_SEED_KEYS = ('alpha', 'discount', 'tau', 'lr')


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _check_per_seed(per_seed, num_seeds):
    """{key: sequence of num_seeds values} -> {key: tuple of floats}, or None.  Raises ValueError on anything else."""
    if per_seed is None:
        return None
    if not isinstance(per_seed, dict):
        raise ValueError(f'per_seed must be a dict of per-seed sequences (got {type(per_seed).__name__})')
    out = {}
    for k, v in per_seed.items():
        if k not in PER_SEED_KEYS:
            raise ValueError(f'per_seed: {k!r} cannot vary per seed; the keys allowed are {PER_SEED_KEYS}.  Structural keys (network '
                             f'shapes, layer_norm, actor_layer_norm, q_agg, normalize_q_loss, flow_steps, batch_size, encoder) are shared '
                             f'by all seeds')
        a = np.asarray(v, dtype=np.float64)
        if a.shape != (num_seeds,):
            raise ValueError(f'per_seed[{k!r}]: expected {num_seeds} values (one per seed), got shape {a.shape}')
        if not np.isfinite(a).all():
            raise ValueError(f'per_seed[{k!r}]: values must be finite (got {a.tolist()})')
        out[k] = tuple(float(x) for x in a)
    return out or None


class LazyInfo(dict):
    """dict of the 13 training metrics; values materialise (one event sync) on first access."""

    def __init__(self, keys, host_buf, event, seed_index=None):
        super().__init__()
        self._keys, self._buf, self._ev, self._seed = keys, host_buf, event, seed_index
        self._ready = False

    def _fill(self):
        if not self._ready:
            self._ev.synchronize()
            arr = self._buf.numpy().reshape(-1, _lib.NUM_INFO)
            for i, k in enumerate(self._keys):
                dict.__setitem__(self, k, float(arr[0, i]) if arr.shape[0] == 1 else arr[:, i].copy())
            self._ready = True

    def __getitem__(self, k):
        self._fill()
        return dict.__getitem__(self, k)

    def __iter__(self):
        self._fill()
        return dict.__iter__(self)

    def items(self):
        self._fill()
        return dict.items(self)

    def keys(self):
        self._fill()
        return dict.keys(self)

    def values(self):
        self._fill()
        return dict.values(self)

    def __len__(self):
        return len(self._keys)

    def __contains__(self, k):
        return k in self._keys

    def __repr__(self):
        self._fill()
        return dict.__repr__(self)

    def get(self, k, default=None):
        self._fill()
        return dict.get(self, k, default)

    def copy(self):
        self._fill()
        return dict(dict.items(self))

    def pop(self, k, *default):
        self._fill()
        return dict.pop(self, k, *default)

    def __eq__(self, other):
        self._fill()
        return dict.__eq__(self, other)

    __hash__ = None


class TrainStateView:
    """`agent.network`: params / opt_state / step with the reference's nesting (utils/flax_utils.py:53-70)."""

    def __init__(self, agent):
        self._a = agent

    @property
    def params(self):
        return self._a._tree(self._a._params)

    @property
    def opt_state(self):
        a = self._a
        return ({'count': a._count, 'mu': a._tree(a._mu), 'nu': a._tree(a._nu)}, {})

    @property
    def grads(self):
        return self._a._tree(self._a._grads)

    @property
    def step(self):
        return int(self._a._count.item()) + 1  # TrainState.step starts at 1 (flax_utils.py:81), count at 0


class FQLAgent:
    """Flow Q-learning agent on one B200 (or one data-parallel rank)."""

    # ------------------------------------------------------------------ construction (agents/fql.py:173-246)
    @classmethod
    def create(cls, seed, ex_observations, ex_actions, config, *, num_seeds=1, device=None, precision='fp32',
               process_group=None, world_size=None, rank=None, per_seed=None):
        """per_seed: hyperparameter sweeps as vectorised seeds -- a dict from a subset of PER_SEED_KEYS ('alpha', 'discount', 'tau',
        'lr') to sequences of num_seeds values; seed i trains with those values (seed_config(i)), every other key of `config` is
        shared.  The table goes to the device once and every entry point of the step reads it."""
        self = cls.__new__(cls)
        cfg = dict(config)
        ex_observations = np.asarray(ex_observations)
        ex_actions = np.asarray(ex_actions)
        ob_dims = tuple(ex_observations.shape[1:])
        if cfg.get('encoder') is not None:
            if cfg['encoder'] != 'impala_small':
                raise NotImplementedError(f"encoder {cfg['encoder']!r}: only 'impala_small' (BASELINE config 5) is built")
            if len(ob_dims) != 3:
                raise ValueError(f'pixel observations must be [H,W,C] (got ob_dims={ob_dims})')
        elif len(ob_dims) != 1:
            raise ValueError(f'state observations must be vectors (got ob_dims={ob_dims}); set config["encoder"] for pixels')
        ah, vh = tuple(cfg['actor_hidden_dims']), tuple(cfg['value_hidden_dims'])
        if len(set(ah + vh)) != 1 or len(ah) != len(vh):
            raise NotImplementedError('actor/value hidden dims must be one common width and depth')
        cfg['ob_dims'], cfg['action_dim'] = ob_dims, int(ex_actions.shape[-1])
        self.config = cfg
        self.device = torch.device(device if device is not None else f'cuda:{torch.cuda.current_device()}')
        self.num_seeds = int(num_seeds)
        self._per_seed = _check_per_seed(per_seed, self.num_seeds)
        self.pg = process_group
        self.world = 1
        if process_group is not None:
            import torch.distributed as dist
            self.world = dist.get_world_size(process_group)
        if world_size is not None:
            self.world = int(world_size)  # explicit override: the caller drives grads_phase / apply_phase itself
        # 'bf16': every contraction on tcgen05 (pixel configs: implicit-GEMM encoders + layer-by-layer MLPs); 'bf16-enc' (pixel
        # configs only): tcgen05 encoders, the MLPs behind them in fp32; 'fp32-tc' (state observations only): the fp32 schedule with
        # every Dense contraction on tcgen05 as 3xTF32, at the fp32 parity tolerance
        self._precision = {'fp32': _lib.PRECISION_FP32, 'bf16': _lib.PRECISION_BF16_TC, 'bf16-enc': _lib.PRECISION_BF16_ENC,
                           'fp32-tc': _lib.PRECISION_FP32_TC}[precision]
        if self._precision == _lib.PRECISION_FP32_TC and cfg.get('encoder') is not None:
            raise NotImplementedError("precision='fp32-tc' supports state observations only (no tf32 convolutions); "
                                      "use 'fp32' or 'bf16' with encoder='impala_small'")
        self._hidden, self._num_hidden = ah[0], len(ah)
        self._image = ob_dims if cfg.get('encoder') is not None else None
        self._feat = 512 if self._image else ob_dims[0]
        self._lib = _lib.lib()
        ctx = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self._lib.fql_context_create(C.byref(ctx)), 'fql_context_create')
        self._ctx = ctx
        self._hp = _lib.make_hparams(lr=cfg['lr'], discount=cfg['discount'], tau=cfg['tau'], alpha=cfg['alpha'])
        self._hp_table = None
        if self._per_seed is not None:
            # one FqlHparams per seed (make_hparams: 1 - tau in double, as for the shared struct), one host-to-device copy
            rows = [_lib.make_hparams(**{k: self.seed_config(i)[k] for k in PER_SEED_KEYS}) for i in range(self.num_seeds)]
            host = (_lib.FqlHparams * self.num_seeds)(*rows)
            self._hp_table = torch.frombuffer(bytearray(host), dtype=torch.uint8).to(self.device)
            self._hp.per_seed = self._hp_table.data_ptr()
        self._dims_cache = {}
        d = self._dims(int(cfg.get('batch_size', 256)))
        self._leaves, self._arena = _lib.layout(d)
        S = self.num_seeds
        self._params = torch.zeros(S, self._arena, dtype=torch.float32, device=self.device)
        self._mu = torch.zeros_like(self._params)
        self._nu = torch.zeros_like(self._params)
        self._dp_peer = False
        if process_group is not None and self.world > 1 and os.environ.get('FQL_DP_BACKEND', 'peer') != 'nccl':
            self._attach_peer_memory(d, process_group)      # the gradient arena lives in NVLink peer-mapped memory
        else:
            self._grads = torch.zeros_like(self._params)
        self._count = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._shadow = None
        if self._precision == _lib.PRECISION_BF16_TC:
            nb = int(self._lib.fql_shadow_bytes(C.byref(d)))
            if nb == 0:
                raise _lib.FqlError('fql_shadow_bytes: ' + self._lib.fql_last_error().decode())
            self._shadow = torch.zeros(nb, dtype=torch.uint8, device=self.device)
        self._bufs = {}
        self._fwd_cache = {}
        self._ring, self._ring_i = [], 0
        self._host_step = 0          # updates enqueued so far == optax count: the Philox step of the next noise draw
        self.last_h2d_bytes = 0
        self._copy_stream = None     # host batches of update() go up on this stream, under the previous step (two input sets)
        self._overlap_h2d = os.environ.get('FQL_B200_OVERLAP_H2D', '1') != '0'
        self.rank = 0
        if process_group is not None:
            import torch.distributed as dist
            self.rank = dist.get_rank(process_group)
        if rank is not None:
            self.rank = int(rank)
        self._dp_side = None
        self._init_params(seed)
        # agent.rng: a (2,) uint32 key; noise for update k comes from Philox(key, k)
        ss = np.random.SeedSequence(int(seed) if np.ndim(seed) == 0 else [int(x) for x in np.ravel(seed)])
        self.rng = ss.generate_state(2, dtype=np.uint32)
        self.network = TrainStateView(self)
        return self

    @property
    def per_seed(self):
        """The per-seed hyperparameters given to create ({key: tuple of num_seeds floats}), or None when all seeds share `config`."""
        return None if self._per_seed is None else dict(self._per_seed)

    def seed_config(self, i):
        """The config agent (seed) i trains with: `config` with its per-seed values."""
        if not 0 <= i < self.num_seeds:
            raise IndexError(f'seed {i} out of range for {self.num_seeds} seeds')
        cfg = dict(self.config)
        for k, v in (self._per_seed or {}).items():
            cfg[k] = v[i]
        return cfg

    def _attach_peer_memory(self, d, group):
        """Data parallel over NVLink peer memory (include/fql_b200.h, fql_dp_attach): the gradient arena, the metric gather buffer and
        the synchronisation flags of every rank are mapped into every rank (torch's symmetric-memory rendezvous does the CUDA VMM /
        NVLS multicast plumbing), and the library's own kernels reduce the gradient buckets inside the step graph.  No NCCL call
        remains on the step.  FQL_DP_BACKEND=nccl keeps the NCCL all-reduce sequence instead (A/B measurements)."""
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm_mem
        nbytes = int(self._lib.fql_dp_symmetric_bytes(C.byref(d), self.world))
        if nbytes == 0:
            raise _lib.FqlError('fql_dp_symmetric_bytes: ' + self._lib.fql_last_error().decode())
        with torch.cuda.device(self.device):
            buf = symm_mem.empty(nbytes // 4, dtype=torch.float32, device=self.device)
            hdl = symm_mem.rendezvous(buf, group)
            buf.zero_()
            torch.cuda.synchronize(self.device)
            dist.barrier(group)                             # every rank's flags are zero before anyone can signal
        comm = _lib.FqlDpComm()
        comm.rank, comm.world = dist.get_rank(group), self.world
        ptrs = list(hdl.buffer_ptrs)
        if ptrs[comm.rank] != buf.data_ptr():
            raise _lib.FqlError('symmetric memory rendezvous: local buffer pointer mismatch')
        for r in range(self.world):
            comm.base[r] = ptrs[r]
        # NVLS multicast (one multimem.ld_reduce / multimem.st per element whatever the world size) from 4 ranks up; between two
        # ranks plain peer loads / stores move the same bytes faster (measured on 2 x B200: 6.5 MB bucket 30.6 vs 38.4 us alone,
        # 0.281 vs 0.292 ms/step).  FQL_DP_MULTICAST=0/1 forces either.
        want_mc = os.environ.get('FQL_DP_MULTICAST', 'auto')
        use_mc = (self.world > 2) if want_mc == 'auto' else (want_mc != '0')
        mc = int(hdl.multicast_ptr) if use_mc else 0
        comm.base_mc = mc or None
        _lib.check(self._lib.fql_dp_attach(self._ctx, C.byref(d), C.byref(comm)), 'fql_dp_attach')
        self._symm, self._symm_hdl, self._comm = buf, hdl, comm
        self._grads = buf[:self.num_seeds * self._arena].view(self.num_seeds, self._arena)
        self._dp_peer = True
        self.dp_transport = 'nvls-multicast' if mc else 'nvlink-peer'

    def _dims(self, batch):
        if batch not in self._dims_cache:
            c = self.config
            self._dims_cache[batch] = _lib.make_dims(
                batch, self._feat, c['action_dim'], global_batch=batch * self.world, hidden=self._hidden,
                num_hidden=self._num_hidden, critic_layer_norm=c['layer_norm'], actor_layer_norm=c['actor_layer_norm'],
                q_agg=c['q_agg'], normalize_q_loss=c['normalize_q_loss'], flow_steps=c['flow_steps'],
                num_seeds=self.num_seeds, precision=self._precision, image=self._image)
        return self._dims_cache[batch]

    def _init_params(self, seed):
        """default_init = variance_scaling(1,'fan_avg','uniform') (utils/networks.py:9-11); Dense bias 0, LN scale 1 / bias 0;
        target critic <- critic (fql.py:241-242).  Same distribution as Flax, different random stream (SURVEY 7)."""
        rng = np.random.default_rng(np.random.SeedSequence(int(seed)).spawn(1)[0]) if np.ndim(seed) == 0 else np.random.default_rng(0)
        host = np.zeros((self.num_seeds, self._arena), np.float32)
        for lf in self._leaves:
            if lf['net'] == 'target_critic':
                continue
            n = lf['ens'] * lf['rows'] * lf['cols']
            sl = slice(lf['offset'], lf['offset'] + n)
            if lf['is_kernel']:
                # Dense: variance_scaling(1,'fan_avg','uniform'); conv (rows = 9*cin): xavier_uniform with fans 9*cin / 9*cout
                fan_out = lf['cols'] * (9 if lf.get('kind') == 4 else 1)
                lim = np.sqrt(6.0 / (lf['rows'] + fan_out))
                host[:, sl] = rng.uniform(-lim, lim, (self.num_seeds, n)).astype(np.float32)
            elif lf['name'] == 'scale':
                host[:, sl] = 1.0
        self._params.copy_(torch.from_numpy(host))
        self._copy_critic_to_target()
        self.refresh_shadow()

    def refresh_shadow(self):
        """Rebuild the bf16 tensor-core operand copies from the fp32 master parameters (no-op in fp32 mode)."""
        if self._shadow is not None:
            d = self._dims(int(self.config.get('batch_size', 256)))
            with torch.cuda.device(self.device):
                _lib.check(self._lib.fql_refresh_shadow(C.byref(d), _ptr(self._params), _ptr(self._shadow), self._stream()),
                           'fql_refresh_shadow')

    def _net_range(self, net):
        offs = [lf['offset'] for lf in self._leaves if lf['net'] == net]
        nxt = [lf['offset'] for lf in self._leaves if lf['offset'] > max(offs)]
        return min(offs), (min(nxt) if nxt else self._arena)

    def _copy_critic_to_target(self):
        c0, c1 = self._net_range('critic')
        t0, t1 = self._net_range('target_critic')
        self._params[:, t0:t1] = self._params[:, c0:c1]

    def _tree(self, arena):
        """Nested dict of views with the reference layout: modules_<net>/{mlp|value_net}/{Dense_i|LayerNorm_i}/{kernel|bias|scale}."""
        out = {}
        S = self.num_seeds
        for lf in self._leaves:
            path = lf.get('path', (lf['module'],))
            if path[0] == 'encoder' and lf['net'] == 'actor_bc_flow':
                node = out.setdefault('modules_actor_bc_flow_encoder', {})   # fql.py:230-232
                path = path[1:]
            else:
                node = out.setdefault('modules_' + lf['net'], {})
                if path[0] != 'encoder':
                    node = node.setdefault('value_net' if 'critic' in lf['net'] else 'mlp', {})
            for k in path:
                node = node.setdefault(k, {})
            n = lf['ens'] * lf['rows'] * lf['cols']
            shape = lf.get('shape') or ((lf['rows'], lf['cols']) if lf['is_kernel'] else (lf['cols'],))
            if lf['ens'] > 1:
                shape = (lf['ens'],) + shape
            v = arena[:, lf['offset']:lf['offset'] + n]
            node[lf['name']] = v.view((S,) + shape) if S > 1 else v.view(shape)
        return out

    # ------------------------------------------------------------------ state import/export
    def load_tree(self, params=None, mu=None, nu=None, count=None):
        """Copy nested dicts of arrays (numpy/torch, reference layout) into the arenas."""
        for src, dst in ((params, self._params), (mu, self._mu), (nu, self._nu)):
            if src is None:
                continue
            views = self._tree(dst)

            def rec(s, v):
                for k in s:
                    if isinstance(s[k], dict):
                        rec(s[k], v[k])
                    else:
                        v[k].copy_(torch.as_tensor(np.asarray(s[k], dtype=np.float32)))
            rec(src, views)
        if count is not None:
            self._count.fill_(int(count))
            # the noise of update k is Philox(rng, k): a restored run continues the stream instead of replaying it from 0
            # (the reference replaces agent.rng every update, fql.py:125,133; here the key is fixed and the step advances)
            self._host_step = int(count)
        self.refresh_shadow()
        return self

    def export_tree(self, which='params'):
        arena = {'params': self._params, 'mu': self._mu, 'nu': self._nu, 'grads': self._grads}[which]

        def rec(v):
            return {k: rec(x) if isinstance(x, dict) else x.detach().cpu().numpy().copy() for k, x in v.items()}
        return rec(self._tree(arena))

    def state_dict(self):
        """flax.serialization.to_state_dict(agent) nesting (utils/flax_utils.py:171-173; SURVEY 5 checkpoint row)."""
        return {'rng': np.asarray(self.rng, np.uint32).copy(),
                'network': {'step': self.network.step, 'params': self.export_tree('params'),
                            'opt_state': {'0': {'count': int(self._count.item()), 'mu': self.export_tree('mu'),
                                                'nu': self.export_tree('nu')}, '1': {}}}}

    def load_state_dict(self, sd):
        net = sd['network']
        self.load_tree(net['params'], net['opt_state']['0']['mu'], net['opt_state']['0']['nu'], net['opt_state']['0']['count'])
        self.rng = np.asarray(sd['rng'], np.uint32).copy()
        return self

    # ------------------------------------------------------------------ buffers
    def _step_bufs(self, B):
        if B in self._bufs:
            return self._bufs[B]
        d = self._dims(B)
        S, A = self.num_seeds, self.config['action_dim']
        ob = tuple(self.config['ob_dims'])
        shapes = dict(observations=(S, B) + ob, actions=(S, B, A), next_observations=(S, B) + ob, rewards=(S, B), masks=(S, B),
                      z_next=(S, B, A), x0=(S, B, A), t=(S, B, 1), z=(S, B, A), z_metric=(S, B, A))
        dt = lambda k: torch.uint8 if (self._image and k in ('observations', 'next_observations')) else torch.float32
        # One contiguous device block (batch keys first, then the noise keys) and a ring of pinned staging blocks with the same
        # layout: a host batch goes up as ONE copy, and a staging block is only rewritten once the copy that read it has run
        # (the host runs ahead of the GPU by many steps).
        offs, off = {}, 0
        for k, shp in shapes.items():
            nb = int(np.prod(shp)) * (1 if dt(k) == torch.uint8 else 4)
            offs[k] = (off, nb)
            off = (off + nb + 255) // 256 * 256
        view = lambda blk, k: blk[offs[k][0]:offs[k][0] + offs[k][1]].view(dt(k)).view(shapes[k])
        dev_block = torch.empty(off, dtype=torch.uint8, device=self.device)
        dev = {k: view(dev_block, k) for k in shapes}
        pins = []
        for _ in range(_PIN_RING):
            blk = torch.empty(off, dtype=torch.uint8).pin_memory()
            pins.append(dict(block=blk, views={k: view(blk, k) for k in shapes}, event=torch.cuda.Event(), pending=False))
        ws_bytes = int(self._lib.fql_workspace_bytes(C.byref(d)))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=self.device)
        fb = _lib.FqlBatch(*[dev[k].data_ptr() for k in _BATCH_KEYS + NOISE_KEYS])
        st = _lib.FqlState(self._params.data_ptr(), self._mu.data_ptr(), self._nu.data_ptr(), self._grads.data_ptr(),
                           self._count.data_ptr(), self._shadow.data_ptr() if self._shadow is not None else None)
        info = torch.zeros(S, _lib.NUM_INFO, dtype=torch.float32, device=self.device)
        raw = torch.zeros(S, _lib.NUM_RAW, dtype=torch.float32, device=self.device)
        self._bufs[B] = dict(d=d, dev=dev, dev_block=dev_block, pins=pins, pin_i=0, offs=offs, ws=ws, ws_bytes=ws_bytes, fb=fb, st=st,
                             info=info, raw=raw, shapes=shapes, dt=dt, read_done=torch.cuda.Event(), ready=torch.cuda.Event(), flip=0)
        return self._bufs[B]

    def _input_sets(self, base):
        """The two input sets of the overlapped host path (`update(host batch)`): the base buffers and a second device block + pinned
        ring + FqlBatch with everything else (dims, state, workspace, metrics) shared.  While the step graph of one set runs, the next
        batch goes up into the other on the copy stream (the library caches one CUDA graph per argument set, so there are two)."""
        if 'sets' not in base:
            offs, shapes, dt = base['offs'], base['shapes'], base['dt']
            size = base['dev_block'].numel()
            view = lambda blk, k: blk[offs[k][0]:offs[k][0] + offs[k][1]].view(dt(k)).view(shapes[k])
            dev_block = torch.empty(size, dtype=torch.uint8, device=self.device)
            dev = {k: view(dev_block, k) for k in shapes}
            pins = []
            for _ in range(_PIN_RING):
                blk = torch.empty(size, dtype=torch.uint8).pin_memory()
                pins.append(dict(block=blk, views={k: view(blk, k) for k in shapes}, event=torch.cuda.Event(), pending=False))
            alt = dict(base)
            alt.update(dev=dev, dev_block=dev_block, pins=pins, pin_i=0, fb=_lib.FqlBatch(*[dev[k].data_ptr() for k in _BATCH_KEYS + NOISE_KEYS]),
                       read_done=torch.cuda.Event(), ready=torch.cuda.Event())
            alt.pop('sets', None)
            base['sets'] = [base, alt]
        return base['sets']

    def _stage(self, bufs, items):
        """items: [(key, source)], keys in buffer order.  Host sources are packed into the next pinned staging block and sent with
        one copy when they are adjacent in the block (the usual case: all five batch keys, or batch + noise); device tensors are
        copied device to device.  Returns the host-to-device bytes."""
        host = [(k, v) for k, v in items if not (isinstance(v, torch.Tensor) and v.is_cuda)]
        for k, v in items:
            if isinstance(v, torch.Tensor) and v.is_cuda:
                bufs['dev'][k].copy_(v.reshape(bufs['dev'][k].shape), non_blocking=True)
        if not host:
            return 0
        slot = bufs['pins'][bufs['pin_i'] % _PIN_RING]
        bufs['pin_i'] += 1
        if slot['pending']:
            slot['event'].synchronize()
        h2d = 0
        for k, v in host:
            pv = slot['views'][k]
            npdt = np.uint8 if pv.dtype == torch.uint8 else np.float32
            t = v if isinstance(v, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(v, dtype=npdt))
            pv.copy_(t.reshape(pv.shape))
            h2d += bufs['offs'][k][1]
        order = list(bufs['offs'])
        idx = [order.index(k) for k, _ in host]
        if idx == list(range(idx[0], idx[0] + len(idx))):         # adjacent keys: one transfer over the whole span
            lo = bufs['offs'][host[0][0]][0]
            hi = bufs['offs'][host[-1][0]][0] + bufs['offs'][host[-1][0]][1]
            bufs['dev_block'][lo:hi].copy_(slot['block'][lo:hi], non_blocking=True)
        else:
            for k, _ in host:
                bufs['dev'][k].copy_(slot['views'][k], non_blocking=True)
        slot['event'].record(torch.cuda.current_stream(self.device))
        slot['pending'] = True
        return h2d

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _info_out(self, info_dev):
        """Async copy of the metrics into the next slot of a ring of 64 pinned buffers.  A slot is reused only after the LazyInfo that
        still points at it (if the caller kept it, e.g. for periodic logging) has been materialised, so a late read never returns a
        later step's metrics."""
        i = self._ring_i % 64
        if i >= len(self._ring):
            self._ring.append([torch.empty(info_dev.shape, dtype=torch.float32).pin_memory(), torch.cuda.Event(), None])
        slot = self._ring[i]
        host, ev, owner = slot
        prev = owner() if owner is not None else None
        if prev is not None:
            prev._fill()
        self._ring_i += 1
        host.copy_(info_dev, non_blocking=True)
        ev.record(torch.cuda.current_stream(self.device))
        out = LazyInfo(INFO_KEYS, host, ev)
        slot[2] = weakref.ref(out)
        return out

    # ------------------------------------------------------------------ the hot path (agents/fql.py:122-133)
    def update(self, batch, noise=None):
        """One training step.  `batch`: dict of host numpy arrays (main.py:201) or torch tensors, [B,...] (or [S,B,...]
        when num_seeds>1).  Returns (self, info)."""
        if self._overlap_h2d and (self.world == 1 or self._dp_peer) and self._all_host(batch, noise):
            return self, self._update_overlapped(batch, noise)
        bufs = self.stage(batch, noise)
        return self, self.step(bufs, fill_noise=noise is None)

    @staticmethod
    def _all_host(batch, noise):
        vals = [batch[k] for k in _BATCH_KEYS] + ([noise[k] for k in NOISE_KEYS] if noise is not None else [])
        return not any(isinstance(v, torch.Tensor) and v.is_cuda for v in vals)

    def _update_overlapped(self, batch, noise):
        """update(host batch) with the host-to-device copy (and the device noise draw) of THIS step on the copy stream, into the input set
        the previous step is not reading: they run under the previous step's graph instead of in front of this one (main.py:201-204 hands
        a fresh host batch to every update).  FQL_B200_OVERLAP_H2D=0 restores the single-stream path."""
        B = int(np.shape(batch['actions'])[-2])
        base = self._step_bufs(B)
        sets = self._input_sets(base)
        cur = sets[base['flip']]
        base['flip'] ^= 1
        with torch.cuda.device(self.device):
            if self._copy_stream is None:
                self._copy_stream = torch.cuda.Stream(device=self.device)
            cs, main = self._copy_stream, torch.cuda.current_stream(self.device)
            cs.wait_event(cur['read_done'])          # the last consumer of this set (two steps ago) has finished reading it
            items = [(k, batch[k]) for k in _BATCH_KEYS]
            if noise is not None:
                items += [(k, noise[k]) for k in NOISE_KEYS]
            with torch.cuda.stream(cs):
                self.last_h2d_bytes = self._stage(cur, items)
                if noise is None:
                    self._fill_noise(cur, self._host_step)
                cur['ready'].record(cs)
            main.wait_event(cur['ready'])
            return self.step(cur, fill_noise=False)

    def stage(self, batch, noise=None):
        """Copy one batch (and optionally explicit noise) into the static device buffers of its batch size."""
        B = int(np.shape(batch['actions'])[-2])
        bufs = self._step_bufs(B)
        with torch.cuda.device(self.device):
            items = [(k, batch[k]) for k in _BATCH_KEYS]
            if noise is not None:
                items += [(k, noise[k]) for k in NOISE_KEYS]
            self.last_h2d_bytes = self._stage(bufs, items)
        return bufs

    def step(self, bufs, fill_noise=True):
        """Enqueue one update on the staged buffers: [device noise] -> fql_update_step (or the data-parallel split with
        an NCCL all-reduce of the gradient arena in between) -> async copy of the 13 metrics to pinned host memory."""
        with torch.cuda.device(self.device):
            if fill_noise:
                self._fill_noise(bufs, self._host_step)
            self._host_step += 1
            if self.world == 1 or self._dp_peer:
                a = (self._ctx, C.byref(bufs['d']), C.byref(self._hp))
                _lib.check(self._lib.fql_update_step(*a, C.byref(bufs['fb']), C.byref(bufs['st']), _ptr(bufs['info']),
                                                     _ptr(bufs['ws']), bufs['ws_bytes'], self._stream()), 'fql_update_step')
            else:
                self._dp_step(bufs)
            bufs['read_done'].record(torch.cuda.current_stream(self.device))
            return self._info_out(bufs['info'])

    def _dp_step(self, bufs):
        """Data-parallel step: gradients -> NCCL all-reduce of the trainable part of the gradient arena -> all-gather of the 64-byte
        metric accumulators -> identical Adam/Polyak step on every rank.  After two eager steps the whole sequence (library
        kernels and both collectives) is captured once into one CUDA graph per batch size and replayed: a step is then a single
        graph launch instead of two library calls and two process-group calls (the host side was the bottleneck at batch 256)."""
        if not self._dp_graph:
            return self._dp_body(bufs)
        st = bufs.setdefault('dp_graph', {'n': 0, 'graph': None})
        if st['graph'] is not None:
            st['graph'].replay()
            return
        st['n'] += 1
        if st['n'] <= 2:
            return self._dp_body(bufs)
        try:
            g = torch.cuda.CUDAGraph()
            torch.cuda.synchronize(self.device)
            with torch.cuda.graph(g, capture_error_mode='thread_local'):
                self._dp_body(bufs)
            st['graph'] = g
            g.replay()                                   # capture does not execute: this runs the step that was captured
        except Exception as e:                           # keep training on the eager sequence
            import warnings
            warnings.warn(f'fql_b200: data-parallel step could not be captured into a CUDA graph ({e!r}); running it eagerly')
            type(self)._dp_graph = False
            torch.cuda.synchronize(self.device)
            self._dp_body(bufs)

    def release_graphs(self):
        """Drop the captured data-parallel step graphs (call before torch.distributed.destroy_process_group())."""
        torch.cuda.synchronize(self.device)
        for bufs in list(getattr(self, '_bufs', {}).values()):
            if isinstance(bufs, dict) and 'dp_graph' in bufs:
                bufs['dp_graph']['graph'] = None
                bufs.pop('raw_all', None)

    def _dp_body(self, bufs):
        """The data-parallel sequence itself.  With FQL_DP_OVERLAP=1 (eager mode only) the bc-flow + critic prefix of the arena starts
        on a side stream as soon as the library's early event fires, while the one-step actor's backward is still running."""
        import torch.distributed as dist
        from . import dist as fdist
        main = torch.cuda.current_stream(self.device)
        overlap = self._dp_overlap and not self._dp_graph
        if overlap and self._dp_side is None:
            self._dp_side = torch.cuda.Stream(device=self.device)
            self._dp_early = torch.cuda.Event()
            self._dp_early.record(main)                 # materialise the cudaEvent_t
            self._n_early = int(self._lib.fql_early_grads_floats(C.byref(bufs['d'])))
            _lib.check(self._lib.fql_set_early_grads_event(self._ctx, C.c_void_p(self._dp_early.cuda_event)), 'fql_set_early_grads_event')
        self.grads_phase(bufs)
        t0, _ = self._net_range('target_critic')
        if overlap:
            with torch.cuda.stream(self._dp_side):
                self._dp_side.wait_event(self._dp_early)
                w1 = dist.all_reduce(self._grads[:, :self._n_early], op=dist.ReduceOp.SUM, group=self.pg, async_op=True)
            w2 = dist.all_reduce(self._grads[:, self._n_early:t0], op=dist.ReduceOp.SUM, group=self.pg, async_op=True)
            raw_all = fdist.gather_raw(bufs['raw'], group=self.pg)
            w1.wait()
            w2.wait()
        else:
            dist.all_reduce(self._grads[:, :t0], op=dist.ReduceOp.SUM, group=self.pg)
            raw_all = fdist.gather_raw(bufs['raw'], group=self.pg)
        _lib.check(self._lib.fql_step_apply_gathered(self._ctx, C.byref(bufs['d']), C.byref(self._hp), C.byref(bufs['st']), _ptr(raw_all),
                                                     self.world, _ptr(bufs['info']), _ptr(bufs['ws']), bufs['ws_bytes'], self._stream()),
                   'fql_step_apply_gathered')
        bufs['raw_all'] = raw_all                       # keep alive (and at a fixed address for the captured graph)

    _dp_overlap = os.environ.get('FQL_DP_OVERLAP', '0') != '0'
    # opt-in: a captured graph that contains NCCL kernels must be released (FQLAgent.release_graphs) before the process group is
    # destroyed, otherwise teardown deadlocks; the eager sequence has the same device time (the step is not host-bound)
    _dp_graph = os.environ.get('FQL_DP_GRAPH', '0') != '0'

    def grads_phase(self, bufs):
        """Data-parallel half 1 (fql_step_grads): this rank's gradient contribution (already divided by the global batch) into
        the gradient arena and the raw metric accumulators into bufs['raw']."""
        _lib.check(self._lib.fql_step_grads(self._ctx, C.byref(bufs['d']), C.byref(self._hp), C.byref(bufs['fb']), C.byref(bufs['st']),
                                            _ptr(bufs['raw']), _ptr(bufs['ws']), bufs['ws_bytes'], self._stream()), 'fql_step_grads')

    def apply_phase(self, bufs):
        """Data-parallel half 2 (fql_step_apply) on the all-reduced gradients / accumulators: stats + Adam + Polyak + info."""
        _lib.check(self._lib.fql_step_apply(self._ctx, C.byref(bufs['d']), C.byref(self._hp), C.byref(bufs['st']), _ptr(bufs['raw']),
                                            _ptr(bufs['info']), _ptr(bufs['ws']), bufs['ws_bytes'], self._stream()), 'fql_step_apply')

    def _fill_noise(self, bufs, step_for_noise):
        """Philox(agent.rng, step) noise for this rank's rows of the GLOBAL batch (rows [rank*B, (rank+1)*B) of every seed): all
        ranks share the key -- they must, to hold identical parameters -- and differ in the counter range (SURVEY 8e)."""
        dev = bufs['dev']
        seed = int(self.rng[0]) | (int(self.rng[1]) << 32)
        row0 = self.rank * int(bufs['d'].batch) if self.world > 1 else 0
        _lib.check(self._lib.fql_fill_noise_rows(C.byref(bufs['d']), C.c_uint64(seed), C.c_uint64(step_for_noise), C.c_int64(row0),
                                                 _ptr(dev['z_next']), _ptr(dev['x0']), _ptr(dev['t']), _ptr(dev['z']),
                                                 _ptr(dev['z_metric']), self._stream()), 'fql_fill_noise_rows')

    def launch_count(self):
        """Kernels this agent's context has enqueued so far (graph replays count their kernel nodes)."""
        return int(self._lib.fql_launch_count(self._ctx))

    def total_loss(self, batch, grad_params=None, rng=None, noise=None):
        """Forward-only losses (agents/fql.py:94-111 as called by main.py:284): returns (loss, info[10 keys])."""
        if grad_params is not None and grad_params is not self.network.params:
            raise NotImplementedError('total_loss evaluates the stored parameters (grad_params=None, main.py:284); gradients are '
                                      'taken inside update()')
        with torch.cuda.device(self.device):
            bufs = self.stage(batch, noise)
            if noise is None:
                self._fill_noise(bufs, (1 << 62) + self._host_step)
            _lib.check(self._lib.fql_total_loss(self._ctx, C.byref(bufs['d']), C.byref(self._hp), C.byref(bufs['fb']),
                                                C.byref(bufs['st']), _ptr(bufs['info']), _ptr(bufs['ws']), bufs['ws_bytes'],
                                                self._stream()), 'fql_total_loss')
            bufs['read_done'].record(torch.cuda.current_stream(self.device))
            info = self._info_out(bufs['info'])
        vals = {k: info[k] for k in INFO_KEYS[:10]}
        return vals['critic/critic_loss'] + vals['actor/actor_loss'], vals

    def critic_loss(self, batch, grad_params=None, rng=None, noise=None):
        """agents/fql.py:22-44: (critic_loss, {critic_loss, q_mean, q_max, q_min}), forward only -- the gradient of this loss is
        part of `update` (one fused step); `grad_params` is accepted for signature parity and must be None or the stored params."""
        _, info = self.total_loss(batch, grad_params, rng, noise)
        out = {k.split('/', 1)[1]: v for k, v in info.items() if k.startswith('critic/')}
        return out['critic_loss'], out

    def actor_loss(self, batch, grad_params=None, rng=None, noise=None):
        """agents/fql.py:46-92: (actor_loss, {actor_loss, bc_flow_loss, distill_loss, q_loss, q, mse}), forward only."""
        _, info = self.total_loss(batch, grad_params, rng, noise)
        out = {k.split('/', 1)[1]: v for k, v in info.items() if k.startswith('actor/')}
        return out['actor_loss'], out

    def target_update(self, network=None, module_name='critic'):
        """agents/fql.py:113-120: target_critic <- tau * critic + (1 - tau) * target_critic, in place (`update` already does this,
        fused into the optimizer pass; this is the standalone method of the reference's surface)."""
        if module_name != 'critic':
            raise ValueError(f"target_update: FQL only has a target network for 'critic' (got {module_name!r})")
        d = self._dims(int(self.config.get('batch_size', 256)))
        with torch.cuda.device(self.device):
            _lib.check(self._lib.fql_target_update(C.byref(d), C.byref(self._hp), _ptr(self._params), _ptr(self._shadow), self._stream()),
                       'fql_target_update')

    # ------------------------------------------------------------------ agents/fql.py:135-171
    def _fwd_bufs(self, rows):
        """Static buffers of the standalone forward entry points for one row count: device inputs / output / workspace and a
        pinned staging pair, allocated once (the online loop and the evaluator call sample_actions every environment step,
        main.py:225, evaluation.py:98-150)."""
        fb = self._fwd_cache.get(rows)
        if fb is None:
            S, A = self.num_seeds, self.config['action_dim']
            ob = tuple(self.config['ob_dims'])
            odt = torch.uint8 if self._image else torch.float32
            d = self._dims(int(self.config.get('batch_size', 256)))
            wsb = int(self._lib.fql_forward_workspace_bytes(C.byref(d), rows))
            fb = dict(d=d, wsb=wsb, ws=torch.empty(wsb, dtype=torch.uint8, device=self.device),
                      obs=torch.empty((S, rows) + ob, dtype=odt, device=self.device), nz=torch.empty(S, rows, A, device=self.device),
                      out=torch.empty(S, rows, A, device=self.device),
                      obs_pin=torch.empty((S, rows) + ob, dtype=odt).pin_memory(), nz_pin=torch.empty(S, rows, A).pin_memory(),
                      out_pin=torch.empty(S, rows, A).pin_memory())
            if len(self._fwd_cache) >= 8:
                self._fwd_cache.pop(next(iter(self._fwd_cache)))
            self._fwd_cache[rows] = fb
        return fb

    def _fwd_call(self, fn, observations, noises, to_host=True):
        nob = len(self.config['ob_dims'])
        A, S = self.config['action_dim'], self.num_seeds
        lead = tuple(np.shape(observations)[:-nob])
        rows = (int(np.prod(lead)) if lead else 1) // S
        fb = self._fwd_bufs(rows)
        with torch.cuda.device(self.device):
            for src, dev, pin in ((observations, fb['obs'], fb['obs_pin']), (noises, fb['nz'], fb['nz_pin'])):
                if isinstance(src, torch.Tensor) and src.is_cuda:
                    dev.copy_(src.reshape(dev.shape), non_blocking=True)
                else:
                    pin.copy_(torch.as_tensor(np.asarray(src)).reshape(pin.shape))
                    dev.copy_(pin, non_blocking=True)
            _lib.check(fn(self._ctx, C.byref(fb['d']), _ptr(self._params), _ptr(self._shadow), _ptr(fb['obs']), _ptr(fb['nz']), _ptr(fb['out']), rows,
                          _ptr(fb['ws']), fb['wsb'], self._stream()), fn.__name__)
            if not to_host:
                return fb['out'].reshape(lead + (A,))       # a view of the static output buffer (overwritten by the next call)
            fb['out_pin'].copy_(fb['out'], non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
        return fb['out_pin'].numpy().reshape(lead + (A,)).copy()

    def sample_actions(self, observations, seed=None, temperature=1.0, noise=None):
        """clip(actor_onestep_flow(obs, z)), z ~ N(0, I) of shape obs.shape[:-1] + (A,).  `temperature` is accepted and
        ignored exactly like the reference (fql.py:140).  Returns a host numpy array (np.array-able, evaluation.py:150)."""
        lead = tuple(np.shape(observations)[:-len(self.config['ob_dims'])])
        A = self.config['action_dim']
        if noise is None:
            key = np.ravel(np.asarray(seed if seed is not None else self.rng)).astype(np.uint64)
            g = torch.Generator(device='cpu').manual_seed(int(key[0]) ^ (int(key[-1]) << 32) if key.size else 0)
            noise = torch.randn(lead + (A,), generator=g, dtype=torch.float32)
        return self._fwd_call(self._lib.fql_sample_actions, observations, noise)

    def compute_flow_actions(self, observations, noises):
        return self._fwd_call(self._lib.fql_compute_flow_actions, observations, noises)

    def q_values(self, observations, actions, target=False):
        """Q_h(s, a) of both critic heads, [2, rows] (utils/networks.py:178-195 `Value.__call__`; state observations).  Evaluated in
        fp32 from the master parameters (fql_mlp_forward) whatever the training precision: this is the evaluation-side call of
        best-of-N action selection (agents/ifql.py:146-149), not part of the update."""
        if self._image is not None:
            raise NotImplementedError('q_values takes state observations')
        obs = torch.as_tensor(np.asarray(observations), dtype=torch.float32, device=self.device).reshape(-1, self._feat)
        act = torch.as_tensor(np.asarray(actions), dtype=torch.float32, device=self.device).reshape(obs.shape[0], -1)
        rows = int(obs.shape[0])
        d = _lib.FqlDims.from_buffer_copy(self._dims(int(self.config.get('batch_size', 256))))
        d.precision, d.num_seeds = _lib.PRECISION_FP32, 1
        if self.num_seeds != 1:
            raise NotImplementedError('q_values: one agent (num_seeds == 1)')
        x = torch.cat([obs, act], dim=1).contiguous()
        y = torch.empty(2, rows, dtype=torch.float32, device=self.device)
        wsb = int(self._lib.fql_forward_workspace_bytes(C.byref(d), rows))
        ws = torch.empty(wsb, dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.fql_mlp_forward(self._ctx, C.byref(d), _lib.NET_TARGET_CRITIC if target else _lib.NET_CRITIC, _ptr(self._params),
                                                 _ptr(x), _ptr(y), rows, _ptr(ws), wsb, self._stream()), 'fql_mlp_forward')
            torch.cuda.current_stream(self.device).synchronize()
        return y.cpu().numpy()

    def sample_actions_best_of_n(self, observation, num_samples=32, seed=None, noise=None):
        """IFQLAgent.sample_actions (agents/ifql.py:122-149) on this agent's networks -- the reuse of the Euler kernel SURVEY 8(f)4
        names: `num_samples` noises are integrated through the bc-flow velocity field (compute_flow_actions: ONE persistent kernel
        for all samples), clipped, and the action with the largest min-over-heads Q is returned.  `observation`: one state [F]."""
        ob = np.asarray(observation, np.float32).reshape(1, self._feat)
        A = self.config['action_dim']
        if noise is None:
            key = np.ravel(np.asarray(seed if seed is not None else self.rng)).astype(np.uint64)
            noise = np.random.Generator(np.random.Philox(key=int(key[0]) | (int(key[-1]) << 32))).standard_normal((num_samples, A)).astype(np.float32)
        noise = np.asarray(noise, np.float32).reshape(-1, A)
        obs_n = np.repeat(ob, noise.shape[0], axis=0)
        actions = self.compute_flow_actions(obs_n, noise)
        q = self.q_values(obs_n, actions).min(axis=0)
        return actions[int(np.argmax(q))]

    def __del__(self):
        try:
            if getattr(self, '_ctx', None):
                self._lib.fql_context_destroy(self._ctx)
        except Exception:
            pass
