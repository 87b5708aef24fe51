"""B200ImpalaLearner -- the learner side of ImpalaTrainer.learn behind ScaleRL's agent API.

Replaces, for one GPU's shard of the batch, the arithmetic of
``ImpalaTrainer.learn`` (/root/reference scalerl/algorithms/impala/impala_atari.py:270-349) and of
``AtariNet.forward`` (scalerl/algorithms/utils/atari_model.py:77-143, use_lstm=False); implements the
``BaseAgent`` surface (scalerl/algorithms/base.py:68-116): learn / predict / get_weights / set_weights /
save_checkpoint / load_checkpoint.  All math runs in libscalerl_b200.so (C ABI); torch supplies device
memory, streams and (for world_size > 1) the NCCL all-reduce of the flat gradient buffer.

Data parallelism (SURVEY.md §8e): each rank processes B_local columns; gradients are SUM-reduced because
the reference losses are sums over T*B (loss_fn.py:6,13,23); the 40.0 clip applies to the global gradient.
"""
from __future__ import annotations

import ctypes as C
import os
from collections import OrderedDict
from dataclasses import dataclass, asdict
from typing import Dict, Optional

import torch

from . import _lib
from .algorithms.base import BaseAgent

PARAM_NAMES = ('conv1.weight', 'conv1.bias', 'conv2.weight', 'conv2.bias', 'conv3.weight', 'conv3.bias',
               'fc.weight', 'fc.bias', 'policy.weight', 'policy.bias', 'baseline.weight', 'baseline.bias')
LSTM_PARAM_NAMES = tuple(f'rnn_layer.{w}_l{l}' for l in (0, 1) for w in ('weight_ih', 'weight_hh', 'bias_ih', 'bias_hh'))


def reference_param_order(use_lstm: bool = False):
    """names in ``AtariNet.parameters()`` order (atari_model.py:30-59: conv1, conv2, conv3, fc, [rnn_layer], policy,
    baseline) -- the integer keys of ``torch.optim.Optimizer.state_dict()['state']`` in a reference checkpoint"""
    return PARAM_NAMES[:8] + (LSTM_PARAM_NAMES if use_lstm else ()) + PARAM_NAMES[8:]


def _torch_param_groups(hp: 'ImpalaHParams', n: int):
    """param_groups exactly as the installed torch writes them for the reference's optimizer (impala_atari.py:99-105)"""
    dummy = [torch.nn.Parameter(torch.zeros(1)) for _ in range(n)]
    if hp.optimizer == 'rmsprop':
        opt = torch.optim.RMSprop(dummy, lr=hp.learning_rate, momentum=hp.momentum, eps=hp.epsilon, alpha=hp.alpha)
    else:
        opt = torch.optim.Adam(dummy, lr=hp.learning_rate, betas=(hp.adam_beta1, hp.adam_beta2), eps=hp.adam_eps)
    return opt.state_dict()['param_groups']


def to_torch_optimizer_state(hp: 'ImpalaHParams', tensors: Dict[str, Dict[str, torch.Tensor]], step: int) -> dict:
    """``torch.optim.RMSprop(...).state_dict()`` / ``Adam`` layout (what ImpalaTrainer.save_checkpoint stores,
    impala_atari.py:506-511): {'state': {i: {'step', 'square_avg' | 'exp_avg','exp_avg_sq'}}, 'param_groups': [...]},
    i = index in AtariNet.parameters() order.  ``tensors``: kind -> name -> tensor.  No state before the first step,
    as torch (state is created lazily)."""
    order = reference_param_order(hp.use_lstm)
    state = {}
    if step > 0:
        for i, n in enumerate(order):
            st = {'step': torch.tensor(float(step))}
            for kind, d in tensors.items():
                st[kind] = d[n].detach().cpu().clone()
            state[i] = st
    return {'state': state, 'param_groups': _torch_param_groups(hp, len(order))}


def from_torch_optimizer_state(sd: dict, use_lstm: bool):
    """inverse of to_torch_optimizer_state; also accepts round 1's {'step', 'state': {kind: {name: tensor}}} layout.
    -> (step, {kind: {name: tensor}}).  Unknown layouts raise (never silently skipped)."""
    if not sd:
        return 0, {}
    state = sd.get('state', {})
    if 'param_groups' not in sd:                 # legacy layout of this package (round 1)
        kinds = {k: v for k, v in state.items() if k in ('square_avg', 'exp_avg', 'exp_avg_sq')}
        if state and not kinds:
            raise ValueError(f'optimizer_state_dict: unknown layout (keys {list(state)[:4]})')
        return int(sd.get('step', 0)), kinds
    order = reference_param_order(use_lstm)
    if not state:
        return 0, {}
    if sorted(state) != list(range(len(order))):
        raise ValueError(f'optimizer_state_dict: expected state for params 0..{len(order) - 1}, got keys {sorted(state)[:6]}...')
    out: Dict[str, Dict[str, torch.Tensor]] = {}
    steps = set()
    for i, n in enumerate(order):
        for kind, v in state[i].items():
            if kind == 'step':
                steps.add(int(float(v)))
            elif kind in ('square_avg', 'exp_avg', 'exp_avg_sq'):
                out.setdefault(kind, {})[n] = v
            elif kind in ('momentum_buffer', 'grad_avg', 'max_exp_avg_sq'):
                raise ValueError(f"optimizer_state_dict: '{kind}' (momentum / centered / amsgrad) is not supported by the fused optimizer")
            else:
                raise ValueError(f"optimizer_state_dict: unknown per-parameter entry '{kind}'")
    if len(steps) != 1:
        raise ValueError(f'optimizer_state_dict: parameters disagree on the step count: {sorted(steps)}')
    return steps.pop(), out


def param_shapes(num_actions: int, use_lstm: bool = False):
    core = 513 + num_actions
    d = _base_shapes(num_actions)
    if use_lstm:
        for n in LSTM_PARAM_NAMES:
            d[n] = (4 * core, core) if 'weight' in n else (4 * core,)
    return d


def _base_shapes(num_actions: int):
    core = 513 + num_actions
    return OrderedDict([
        ('conv1.weight', (32, 4, 8, 8)), ('conv1.bias', (32,)), ('conv2.weight', (64, 32, 4, 4)), ('conv2.bias', (64,)),
        ('conv3.weight', (64, 64, 3, 3)), ('conv3.bias', (64,)), ('fc.weight', (512, 3136)), ('fc.bias', (512,)),
        ('policy.weight', (num_actions, core)), ('policy.bias', (num_actions,)),
        ('baseline.weight', (1, core)), ('baseline.bias', (1,))])


@dataclass
class ImpalaHParams:
    """Hyper-parameters read by ImpalaTrainer (impala_atari.py:56,72-77,302-328,344) -- the fields the
    reference's RLArguments forgot are added with upstream torchbeast defaults (SURVEY.md §0.3)."""
    rollout_length: int = 20
    batch_size: int = 32                 # columns handled by THIS rank
    num_actions: int = 6
    discounting: float = 0.99
    baseline_cost: float = 0.5
    entropy_cost: float = 0.0006
    reward_clipping: str = 'abs_one'
    clip_rho_threshold: Optional[float] = 1.0
    clip_pg_rho_threshold: Optional[float] = 1.0
    max_grad_norm: float = 40.0          # rl_args.py:108
    learning_rate: float = 1e-4          # rl_args.py:112
    alpha: float = 0.99                  # rl_args.py:114
    momentum: float = 0.0                # rl_args.py:116 (only 0 is supported, as the reference uses)
    epsilon: float = 1e-5                # rl_args.py:117
    optimizer: str = 'rmsprop'           # 'rmsprop' (reference) | 'adam' (north_star)
    adam_beta1: float = 0.9
    adam_beta2: float = 0.999
    adam_eps: float = 1e-8
    precision: str = 'bf16'              # encoder operands: 'bf16' | 'fp32_split' (fp32-accurate hi/lo bf16 pairs; whole-step parity mode)
    use_lstm: bool = False               # AtariNet(use_lstm=True): 2-layer LSTM core (impala_atari.py:56; config 5)

    def to_c(self) -> _lib.SrlConfig:
        if self.reward_clipping not in ('abs_one', 'none'):
            raise ValueError("reward_clipping must be 'abs_one' or 'none'")
        if self.optimizer not in ('rmsprop', 'adam'):
            raise ValueError("optimizer must be 'rmsprop' or 'adam'")
        if self.momentum != 0.0:
            raise ValueError('only momentum=0 is supported (the reference default)')
        c = _lib.SrlConfig()
        c.T, c.B, c.A = self.rollout_length, self.batch_size, self.num_actions
        c.optimizer = 0 if self.optimizer == 'rmsprop' else 1
        c.reward_clip_abs_one = 1 if self.reward_clipping == 'abs_one' else 0
        if self.precision not in ('bf16', 'fp32_split'):
            raise ValueError("precision must be 'bf16' or 'fp32_split'")
        c.precision = 0 if self.precision == 'bf16' else 1
        c.discounting, c.baseline_cost, c.entropy_cost = self.discounting, self.baseline_cost, self.entropy_cost
        c.clip_rho_threshold = -1.0 if self.clip_rho_threshold is None else self.clip_rho_threshold
        c.clip_pg_rho_threshold = -1.0 if self.clip_pg_rho_threshold is None else self.clip_pg_rho_threshold
        c.max_grad_norm = self.max_grad_norm
        c.learning_rate, c.alpha, c.epsilon = self.learning_rate, self.alpha, self.epsilon
        c.adam_beta1, c.adam_beta2, c.adam_eps = self.adam_beta1, self.adam_beta2, self.adam_eps
        c.use_lstm = 1 if self.use_lstm else 0
        return c


class B200ImpalaLearner(BaseAgent):
    """One learner process per GPU.  ``learn(batch)`` consumes the reference's batch dict
    (keys of create_buffers, impala_atari.py:122-151; tensors [T+1, B_local, ...]) and returns the
    reference's stats dict (impala_atari.py:333-340)."""

    def __init__(self, hp: ImpalaHParams, device: Optional[torch.device] = None, process_group=None,
                 init_state_dict: Optional[Dict[str, torch.Tensor]] = None, seed: int = 0, use_graph: bool = True,
                 validate_inputs: bool = False):
        if not torch.cuda.is_available():
            raise RuntimeError('B200ImpalaLearner needs a CUDA device: scalerl_b200 has no CPU fallback')
        super().__init__(hp)                 # BaseAgent keeps the arguments as self.args (algorithms/base.py:14-21)
        self.hp = hp
        self.validate_inputs = validate_inputs      # raise on out-of-range actions like F.one_hot does (one extra sync per step)
        self.device = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
        # process_group: None -> default group when torch.distributed is initialised; False -> never all-reduce
        self.pg = process_group
        dist = torch.distributed
        self._dist = (process_group is not False and dist.is_available() and dist.is_initialized()
                      and dist.get_world_size(process_group or None) > 1)
        self.world_size = dist.get_world_size(process_group or None) if self._dist else 1
        self._L = _lib.lib()
        with torch.cuda.device(self.device):
            self.names = PARAM_NAMES + (LSTM_PARAM_NAMES if hp.use_lstm else ())
            total, self._off, self._cnt = _lib.param_layout(hp.num_actions, hp.use_lstm)
            self.numel = total
            z = lambda: torch.zeros(total, dtype=torch.float32, device=self.device)
            self.flat_params, self.flat_grads, self.opt_state0 = z(), z(), z()
            self._peers = None
            if self._dist and os.environ.get('SRL_DP_FUSED', '1') != '0':
                self._setup_peer_memory(total)       # replaces flat_grads by a symmetric-memory buffer when that works
            self.opt_state1 = z() if hp.optimizer == 'adam' else None
            self.shapes = param_shapes(hp.num_actions, hp.use_lstm)
            self.params = OrderedDict((n, self._view(self.flat_params, i)) for i, n in enumerate(self.names))
            self.grads = OrderedDict((n, self._view(self.flat_grads, i)) for i, n in enumerate(self.names))
            if init_state_dict is None:
                init_state_dict = self._default_init(seed)
            self._cfg = hp.to_c()
            h = C.c_void_p()
            _lib.check(self._L.srl_learner_create(
                C.byref(self._cfg), self.flat_params.data_ptr(), self.flat_grads.data_ptr(), self.opt_state0.data_ptr(),
                self.opt_state1.data_ptr() if self.opt_state1 is not None else None, C.byref(h)), 'srl_learner_create')
            self._h = h
            self.load_state_dict(init_state_dict)
            T, B, A = hp.rollout_length, hp.batch_size, hp.num_actions
            if hp.use_lstm:     # static copies of the initial LSTM state (graph-replay safe addresses)
                self._h0 = torch.zeros(2, B, 513 + A, device=self.device)
                self._c0 = torch.zeros(2, B, 513 + A, device=self.device)
            self._resdev = torch.zeros(8, device=self.device)      # {pg, baseline, entropy, total loss | grad norm, clip coef | pad}: ONE D2H per step
            self._losses = self._resdev[:4]
            self._coef = self._resdev[4:6]
            self._vs = torch.empty(T, B, device=self.device)
            self._pg_adv = torch.empty(T, B, device=self.device)
            self._stats_host = torch.zeros(8, dtype=torch.float32).pin_memory()
        self.global_step = 0
        self.use_graph = use_graph and not os.environ.get('SRL_NO_GRAPH')   # SRL_NO_GRAPH=1: eager launches (for ncu)
        self._graphs = {}       # batch buffer addresses -> captured CUDA graph(s) of the step
        self._seen = set()

    def _setup_peer_memory(self, total):
        """Gradient buffer + 1 KiB control block in symmetric memory (every rank maps every rank's copy): the apply step
        then reduces, clips, updates and gathers in one kernel over NVLink loads (srl_learner_apply_gradients_dp) and the
        step needs no NCCL call.  Any failure (no P2P, > 8 ranks, API missing) leaves the NCCL path in place."""
        dist = torch.distributed
        ok = torch.ones(1, device=self.device)
        peers = None
        try:
            import torch.distributed._symmetric_memory as symm
            group = self.pg or dist.group.WORLD
            world, rank = dist.get_world_size(group), dist.get_rank(group)
            if world > 8:
                raise RuntimeError('more than 8 ranks')
            grads = symm.empty(total, dtype=torch.float32, device=self.device)
            ctl = symm.empty(256, dtype=torch.int32, device=self.device)
            chunk4 = ((total // 4) + world - 1) // world             # float4s per reduced slice
            exch = symm.empty(4 * chunk4 + 4, dtype=torch.float32, device=self.device)
            hg, hc, hx = symm.rendezvous(grads, group), symm.rendezvous(ctl, group), symm.rendezvous(exch, group)
            grads.zero_(); ctl.zero_(); exch.zero_()
            torch.cuda.synchronize(self.device)
            peers = _lib.SrlDpPeers()
            for i in range(world):
                peers.grads[i] = int(hg.buffer_ptrs[i]); peers.ctl[i] = int(hc.buffer_ptrs[i]); peers.exchange[i] = int(hx.buffer_ptrs[i])
            peers.rank, peers.world = rank, world
            if int(hg.buffer_ptrs[rank]) != grads.data_ptr():
                raise RuntimeError('symmetric buffer is not at the tensor address')
            mc = int(getattr(hg, 'multicast_ptr', 0) or 0) if os.environ.get('SRL_DP_NVLS', '1') != '0' else 0
            flag = torch.tensor([1 if mc else 0], device=self.device)          # NVLS only when EVERY rank has the multicast mapping
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.pg or None)
            peers.grads_multicast = mc if bool(flag.item()) else None
            self.dp_path = 'nvls multimem' if peers.grads_multicast else 'peer loads' 
            self._symm_keep = (grads, ctl, hg, hc, exch, hx)
        except Exception as e:         # noqa: BLE001 -- any failure means "use NCCL"
            import warnings
            warnings.warn(f'peer-memory gradient path unavailable ({e!r}); using NCCL all-reduce')
            ok.zero_()
            peers = None
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.pg or None)     # all ranks take the same path (and: a barrier)
        if bool(ok.item()) and peers is not None:
            self.flat_grads = self._symm_keep[0]
            self._peers = peers
        else:
            self._peers = None

    # ------------------------------------------------------------------ parameters
    def _view(self, flat, i):
        n = self.names[i]
        return flat[self._off[i]:self._off[i] + self._cnt[i]].view(self.shapes[n])

    def _default_init(self, seed):
        """torch's default Conv2d/Linear init distribution (U(+-1/sqrt(fan_in))), as AtariNet() would draw."""
        g = torch.Generator().manual_seed(seed)
        sd, fan = OrderedDict(), 1
        H = 513 + self.hp.num_actions
        for n, shp in self.shapes.items():
            if n.startswith('rnn_layer.'):
                fan = H                     # nn.LSTM: U(+-1/sqrt(hidden_size)) for every tensor
            elif n.endswith('.weight'):
                fan = 1
                for d in shp[1:]:
                    fan *= d
            bound = 1.0 / fan ** 0.5
            sd[n] = (torch.rand(shp, generator=g) * 2 - 1) * bound
        return sd

    def state_dict(self) -> 'OrderedDict[str, torch.Tensor]':
        """AtariNet-compatible state_dict (names/layouts of atari_model.py:30-59)."""
        return OrderedDict((n, p.detach().clone()) for n, p in self.params.items())

    def load_state_dict(self, sd: Dict[str, torch.Tensor]) -> None:
        for n in self.names:
            if n not in sd:
                raise KeyError(f'missing key {n} in state_dict')
            if tuple(sd[n].shape) != tuple(self.shapes[n]):
                raise ValueError(f'{n}: shape {tuple(sd[n].shape)} != {tuple(self.shapes[n])}')
            self.params[n].copy_(sd[n].to(self.device, torch.float32))
        _lib.check(self._L.srl_learner_pack_weights(self._h, self._stream()), 'pack_weights')

    def get_weights(self):            # BaseAgent.get_weights (algorithms/base.py:86-92)
        return {k: v.cpu() for k, v in self.state_dict().items()}

    def set_weights(self, weights):   # BaseAgent.set_weights (algorithms/base.py:94-100)
        self.load_state_dict(weights)

    def _opt_tensors(self):
        kinds = ('square_avg',) if self.hp.optimizer == 'rmsprop' else ('exp_avg', 'exp_avg_sq')
        flats = (self.opt_state0,) if self.hp.optimizer == 'rmsprop' else (self.opt_state0, self.opt_state1)
        return {k: OrderedDict((n, self._view(f, i)) for i, n in enumerate(self.names)) for k, f in zip(kinds, flats)}

    def optimizer_state_dict(self):
        """torch.optim state_dict layout of the reference's optimizer (impala_atari.py:99-105,509): loadable by
        ``torch.optim.RMSprop(AtariNet(...).parameters(), ...).load_state_dict`` and back"""
        return to_torch_optimizer_state(self.hp, self._opt_tensors(), self.global_opt_step)

    def load_optimizer_state_dict(self, sd) -> None:
        step, kinds = from_torch_optimizer_state(sd, self.hp.use_lstm)
        mine = self._opt_tensors()
        for kind in kinds:
            if kind not in mine:
                raise ValueError(f"optimizer_state_dict holds '{kind}' but this learner runs {self.hp.optimizer}")
        for kind, views in mine.items():
            if kind in kinds:
                for n, v in views.items():
                    v.copy_(kinds[kind][n])
            elif step > 0:
                raise ValueError(f"optimizer_state_dict lacks '{kind}' for {self.hp.optimizer}")
        self._set_opt_step(step)

    @property
    def global_opt_step(self):
        return getattr(self, '_opt_steps', 0)

    def _set_opt_step(self, step: int) -> None:
        """optimizer step count = Adam's bias-correction t (host copy + the device counter the captured graphs read)"""
        _lib.check(self._L.srl_learner_set_step(self._h, int(step), self._stream()), 'srl_learner_set_step')
        self._opt_steps = int(step)

    def device_opt_step(self) -> int:
        """the step count as the kernels see it (device counter; synchronises)"""
        return int(self._L.srl_learner_get_step(self._h, self._stream()))

    def save_checkpoint(self, path: str) -> None:
        """same dict keys as ImpalaTrainer.save_checkpoint (impala_atari.py:506-511)"""
        torch.save({'model_state_dict': {k: v.cpu() for k, v in self.state_dict().items()},
                    'optimizer_state_dict': self.optimizer_state_dict(), 'hparam': asdict(self.hp)}, path)

    def load_checkpoint(self, path: str) -> None:
        ck = torch.load(path, map_location='cpu', weights_only=False)
        self.load_state_dict(ck['model_state_dict'])
        self.load_optimizer_state_dict(ck.get('optimizer_state_dict', {}))

    # ------------------------------------------------------------------ compute
    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _check_batch(self, batch, rows):
        hp = self.hp
        B, A = hp.batch_size, hp.num_actions
        exp = {'obs': ((rows, B, 4, 84, 84), torch.uint8), 'reward': ((rows, B), torch.float32), 'action': ((rows, B), torch.int64)}
        for k, (shp, dt) in exp.items():
            if k not in batch:
                raise KeyError(f"batch is missing key '{k}'")
            t = batch[k]
            if tuple(t.shape) != shp or t.dtype != dt:
                raise ValueError(f"batch['{k}']: expected {shp} {dt}, got {tuple(t.shape)} {t.dtype}")
            if not t.is_cuda or not t.is_contiguous():
                raise ValueError(f"batch['{k}'] must be a contiguous CUDA tensor")

    def _done_u8(self, batch):
        d = batch['done']
        return d.view(torch.uint8) if d.dtype == torch.bool else d

    def _set_rnn_state(self, state):
        if state is None or len(state) == 0:
            self._h0.zero_(); self._c0.zero_()
        else:
            self._h0.copy_(state[0]); self._c0.copy_(state[1])

    @torch.no_grad()
    def forward(self, batch: Dict[str, torch.Tensor], initial_rnn_state=()):
        """AtariNet.forward (learner path: no action sampling) -> dict(policy_logits [R,B,A], baseline [R,B])."""
        rows = batch['obs'].shape[0]
        self._check_batch(batch, rows)
        hp = self.hp
        logits = torch.empty(rows, hp.batch_size, hp.num_actions, device=self.device)
        baseline = torch.empty(rows, hp.batch_size, device=self.device)
        if hp.use_lstm:
            if rows != hp.rollout_length + 1:
                raise ValueError('the LSTM learner forward needs T+1 rows')
            self._set_rnn_state(initial_rnn_state)
            hT, cT = torch.empty_like(self._h0), torch.empty_like(self._c0)
            _lib.check(self._L.srl_learner_forward_lstm(
                self._h, batch['obs'].data_ptr(), batch['reward'].data_ptr(), self._done_u8(batch).data_ptr(), batch['action'].data_ptr(),
                self._h0.data_ptr(), self._c0.data_ptr(), logits.data_ptr(), baseline.data_ptr(), hT.data_ptr(), cT.data_ptr(), self._stream()),
                'srl_learner_forward_lstm')
            return dict(policy_logits=logits, baseline=baseline), (hT, cT)
        _lib.check(self._L.srl_learner_forward(self._h, batch['obs'].data_ptr(), batch['reward'].data_ptr(), batch['action'].data_ptr(),
                                               rows, logits.data_ptr(), baseline.data_ptr(), self._stream()), 'srl_learner_forward')
        return dict(policy_logits=logits, baseline=baseline)

    # ------------------------------------------------------------------ BaseAgent surface (algorithms/base.py:23-66)
    def _validate(self, batch):
        """what F.one_hot / gather raise on in the reference (atari_model.py:104, vtrace.py:35-40): actions outside [0, A)"""
        a = batch['action']
        if bool(((a < 0) | (a >= self.hp.num_actions)).any()):
            raise RuntimeError(f'Class values must be smaller than num_classes ({self.hp.num_actions}) and non-negative: '
                               f"batch['action'] has min {int(a.min())}, max {int(a.max())}")

    def _policy(self, batch, initial_rnn_state=()):
        out = self.forward(batch, initial_rnn_state)
        return out[0] if isinstance(out, tuple) else out

    @torch.no_grad()
    def get_action(self, batch: Dict[str, torch.Tensor], initial_rnn_state=(), generator=None) -> torch.Tensor:
        """BaseAgent.get_action: exploration-time actions = a multinomial sample of softmax(policy_logits), as
        AtariNet.forward does in training mode (atari_model.py:130-132).  batch: [R, B, ...] rows, R <= T+1."""
        lg = self._policy(batch, initial_rnn_state)['policy_logits']
        R, B, A = lg.shape
        return torch.multinomial(torch.softmax(lg.view(R * B, A), dim=1), num_samples=1, generator=generator).view(R, B)

    @torch.no_grad()
    def predict(self, batch: Dict[str, torch.Tensor], initial_rnn_state=()) -> torch.Tensor:
        """BaseAgent.predict: evaluation-time actions = argmax of the policy logits (AtariNet in eval mode, atari_model.py:133-134)"""
        return torch.argmax(self._policy(batch, initial_rnn_state)['policy_logits'], dim=-1)

    @torch.no_grad()
    def get_value(self, batch: Dict[str, torch.Tensor], initial_rnn_state=()) -> torch.Tensor:
        """BaseAgent.get_value: the baseline head V(s) [R, B]"""
        return self._policy(batch, initial_rnn_state)['baseline']

    def set_option(self, name: str, value: int) -> None:
        """run-time switch of the C context (e.g. 'column_fusion')"""
        _lib.check(self._L.srl_learner_set_option(self._h, name.encode(), int(value)), 'srl_learner_set_option')

    def snapshot_params(self, out: torch.Tensor, only_if_finite: bool = True) -> None:
        """device-to-device copy of the flat fp32 parameters on the current stream (6.75 MB: a few microseconds of HBM
        time): the weight publish reads the snapshot while the next step already updates the live parameters.  With
        ``only_if_finite`` the copy is skipped ON THE DEVICE when the last step's total loss is NaN/Inf (the snapshot keeps
        the last good weights; poisoned parameters never reach the actors)."""
        _lib.check(self._L.srl_learner_snapshot_params(self._h, out.data_ptr(), self._losses.data_ptr() if only_if_finite else None,
                                                       self._stream()), 'srl_learner_snapshot_params')

    # ------------------------------------------------------------------ pipelined step (no host synchronisation)
    def learn_async(self, batch: Dict[str, torch.Tensor], initial_rnn_state=()) -> int:
        """Enqueue one learner step and the D2H read of its result (4 losses, grad norm, clip coefficient and the
        [T,B] episode_return / done rows the stats need) into a pinned result slot; returns a ticket for ``result``.
        Nothing here waits for the GPU: the caller can enqueue the next batch's copies and the weight publish first."""
        hp = self.hp
        if not hasattr(self, '_res'):
            T, B = hp.rollout_length, hp.batch_size
            self._res_depth = 4
            self._res = [dict(scal=torch.zeros(8, dtype=torch.float32).pin_memory(), ep=torch.zeros(T, B, dtype=torch.float32).pin_memory(),
                              done=torch.zeros(T, B, dtype=torch.uint8).pin_memory(), ev=torch.cuda.Event(), has_ep=False)
                         for _ in range(self._res_depth)]
            self._tickets = 0
        self.learn(batch, initial_rnn_state, sync_stats=False)
        k = self._tickets
        r = self._res[k % self._res_depth]
        if self._dist:
            torch.distributed.all_reduce(self._losses, op=torch.distributed.ReduceOp.SUM, group=self.pg or None)
        r['scal'].copy_(self._resdev, non_blocking=True)
        r['has_ep'] = 'episode_return' in batch
        if r['has_ep']:
            r['ep'].copy_(batch['episode_return'][1:], non_blocking=True)
            r['done'].copy_(self._done_u8(batch)[1:], non_blocking=True)
        r['ev'].record(torch.cuda.current_stream(self.device))
        self._tickets = k + 1
        return k

    def result(self, ticket: int) -> Dict[str, object]:
        """block until step ``ticket`` finished; the reference's stats dict (impala_atari.py:332-340) + grad_norm"""
        if not (self._tickets - self._res_depth <= ticket < self._tickets):
            raise ValueError(f'result({ticket}): only the last {self._res_depth} steps are kept (newest ticket {self._tickets - 1})')
        r = self._res[ticket % self._res_depth]
        r['ev'].synchronize()
        h = r['scal']
        ep = r['ep'][r['done'].bool()] if r['has_ep'] else torch.empty(0)
        return {'episode_returns': tuple(ep.numpy()), 'mean_episode_return': float(ep.mean()) if ep.numel() else float('nan'),
                'total_loss': float(h[3]), 'pg_loss': float(h[0]), 'baseline_loss': float(h[1]), 'entropy_loss': float(h[2]),
                'grad_norm': float(h[4])}

    @torch.no_grad()
    def forward_backward(self, batch):
        """enqueue forward + V-trace/loss + backward; gradients (SUM over this rank's columns) land in flat_grads."""
        hp = self.hp
        self._check_batch(batch, hp.rollout_length + 1)
        done = batch['done']
        done_u8 = done.view(torch.uint8) if done.dtype == torch.bool else done
        bl = batch['policy_logits']
        if tuple(bl.shape) != (hp.rollout_length + 1, hp.batch_size, hp.num_actions) or bl.dtype != torch.float32:
            raise ValueError("batch['policy_logits'] must be float32 [T+1, B, A]")
        if hp.use_lstm:
            _lib.check(self._L.srl_learner_forward_backward_lstm(
                self._h, batch['obs'].data_ptr(), batch['reward'].data_ptr(), done_u8.data_ptr(), batch['action'].data_ptr(), bl.data_ptr(),
                self._h0.data_ptr(), self._c0.data_ptr(), self._losses.data_ptr(), self._vs.data_ptr(), self._pg_adv.data_ptr(), self._stream()),
                'srl_learner_forward_backward_lstm')
            return
        _lib.check(self._L.srl_learner_forward_backward(
            self._h, batch['obs'].data_ptr(), batch['reward'].data_ptr(), done_u8.data_ptr(), batch['action'].data_ptr(),
            bl.data_ptr(), self._losses.data_ptr(), self._vs.data_ptr(), self._pg_adv.data_ptr(), self._stream()),
            'srl_learner_forward_backward')

    def all_reduce_gradients(self):
        """SUM (not mean) all-reduce of the whole flat gradient over NCCL (SURVEY.md §8e)."""
        dist = torch.distributed
        dist.all_reduce(self.flat_grads, op=dist.ReduceOp.SUM, group=self.pg or None)

    @torch.no_grad()
    def forward_backward_begin(self, batch):
        """first half of forward_backward: on return (stream order) the fc.weight gradient (95 % of the bytes) is final"""
        hp = self.hp
        self._check_batch(batch, hp.rollout_length + 1)
        done = batch['done']
        done_u8 = done.view(torch.uint8) if done.dtype == torch.bool else done
        _lib.check(self._L.srl_learner_forward_backward_begin(
            self._h, batch['obs'].data_ptr(), batch['reward'].data_ptr(), done_u8.data_ptr(), batch['action'].data_ptr(),
            batch['policy_logits'].data_ptr(), self._losses.data_ptr(), self._vs.data_ptr(), self._pg_adv.data_ptr(), self._stream()),
            'srl_learner_forward_backward_begin')

    @torch.no_grad()
    def backward_finish(self, batch):
        _lib.check(self._L.srl_learner_backward_finish(self._h, batch['obs'].data_ptr(), self._stream()), 'srl_learner_backward_finish')

    @torch.no_grad()
    def apply_gradients(self):
        _lib.check(self._L.srl_learner_apply_gradients(self._h, self._coef.data_ptr(), self._stream()), 'srl_learner_apply_gradients')
        if not torch.cuda.is_current_stream_capturing():     # a capture executes nothing: the replay counts the step
            self._opt_steps = self.global_opt_step + 1

    @torch.no_grad()
    def apply_gradients_dp(self):
        """all ranks: SUM-reduce the gradients over peer memory, clip, optimizer step -- one kernel, no NCCL"""
        _lib.check(self._L.srl_learner_apply_gradients_dp(self._h, C.byref(self._peers), self._coef.data_ptr(), self._stream()),
                   'srl_learner_apply_gradients_dp')
        if not torch.cuda.is_current_stream_capturing():
            self._opt_steps = self.global_opt_step + 1

    def _enqueue_step(self, batch):
        """forward_backward -> apply_gradients on the current stream; with world_size > 1 the fc.weight gradient is
        all-reduced (async, NCCL stream) while the conv layers back-propagate, the small block afterwards."""
        if self._dist and self._peers is not None:
            self.forward_backward(batch)
            self.apply_gradients_dp()
            return
        if not self._dist or self.hp.use_lstm:
            self.forward_backward(batch)
            if self._dist:          # LSTM path: one all-reduce of the whole flat gradient after BPTT
                self.all_reduce_gradients()
            self.apply_gradients()
            return
        self._dp_step(batch, lambda: self.forward_backward_begin(batch), lambda: self.backward_finish(batch), self.apply_gradients)

    def _dp_step(self, batch, begin, finish, apply):
        dist = torch.distributed
        fcw = self.flat_grads[self._off[6]:]
        small = self.flat_grads[:self._off[6]]
        begin()
        work = dist.all_reduce(fcw, op=dist.ReduceOp.SUM, group=self.pg or None, async_op=True)
        finish()
        dist.all_reduce(small, op=dist.ReduceOp.SUM, group=self.pg or None)
        work.wait()
        apply()

    def release_graphs(self):
        """drop the captured CUDA graphs (call before torch.distributed.destroy_process_group)"""
        torch.cuda.synchronize(self.device)
        self._graphs.clear()
        self._seen.clear()

    def _capture_stream(self):
        """The step is captured from a HIGH-priority stream: the kernels of the main chain (forward, dgrads, conv1's wgrad, optimizer) carry
        that priority as graph nodes, the wgrad / re-pack kernels launched on the library's side streams keep the default (lowest) one -- when
        both are ready the block scheduler places the critical chain first (profiles/r02_timeline.md).  SRL_CAPTURE_PRIORITY=0 switches it off."""
        if getattr(self, '_cap_stream', None) is None:
            prio = int(os.environ.get('SRL_CAPTURE_PRIORITY', '-100'))      # clamped to the device's greatest priority
            self._cap_stream = torch.cuda.Stream(device=self.device, priority=prio)
        return self._cap_stream

    def _graph_step(self, batch):
        """Replay the step as CUDA graph(s) keyed by the batch buffers' addresses.  First sight of a buffer set runs
        eagerly (warm-up: sets kernel attributes, allocator state), the second captures, later calls replay.
        With world_size > 1 the NCCL all-reduces stay outside: graph(begin) -> allreduce(fc.weight, async) ->
        graph(finish) -> allreduce(small) -> graph(apply)."""
        key = tuple(batch[k].data_ptr() for k in ('obs', 'reward', 'done', 'action', 'policy_logits'))
        g = self._graphs.get(key)
        if g is None:
            if key not in self._seen:
                self._seen.add(key)
                self._enqueue_step(batch)
                return
            hp = self.hp
            self._check_batch(batch, hp.rollout_length + 1)
            torch.cuda.current_stream(self.device).synchronize()
            if self._dist and self._peers is not None:     # whole DP step in ONE graph: the reduction is inside the apply kernel
                g = (torch.cuda.CUDAGraph(),)
                with torch.cuda.graph(g[0], stream=self._capture_stream()):
                    self.forward_backward(batch)
                    self.apply_gradients_dp()
            elif self._dist and self.hp.use_lstm:
                g = (torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph())
                with torch.cuda.graph(g[0], stream=self._capture_stream()):
                    self.forward_backward(batch)
                with torch.cuda.graph(g[1], stream=self._capture_stream()):
                    self.apply_gradients()
            elif self._dist:
                g = tuple(torch.cuda.CUDAGraph() for _ in range(3))
                with torch.cuda.graph(g[0], stream=self._capture_stream()):
                    self.forward_backward_begin(batch)
                with torch.cuda.graph(g[1], stream=self._capture_stream()):
                    self.backward_finish(batch)
                with torch.cuda.graph(g[2], stream=self._capture_stream()):
                    self.apply_gradients()
            else:
                g = (torch.cuda.CUDAGraph(),)
                with torch.cuda.graph(g[0], stream=self._capture_stream()):
                    self.forward_backward(batch)
                    self.apply_gradients()
            self._graphs[key] = g
        if len(g) == 3:
            self._dp_step(batch, g[0].replay, g[1].replay, g[2].replay)
        elif len(g) == 2:
            g[0].replay()
            self.all_reduce_gradients()
            g[1].replay()
        else:
            g[0].replay()
        self._opt_steps = self.global_opt_step + 1

    @torch.no_grad()
    def learn(self, batch: Dict[str, torch.Tensor], initial_rnn_state=(), sync_stats: bool = True,
              use_graph: Optional[bool] = None) -> Dict[str, object]:
        """One learner step (impala_atari.py:288-346).  Returns the reference's stats dict when sync_stats
        (one D2H read of 6 floats), else {} with everything left enqueued on the stream."""
        if self.validate_inputs:
            self._validate(batch)
        if self.hp.use_lstm:
            self._set_rnn_state(initial_rnn_state)
        if self.use_graph if use_graph is None else use_graph:
            self._graph_step(batch)
        else:
            self._enqueue_step(batch)
        # the reference counts the frames of the GLOBAL batch (impala_atari.py:391); a rank processes B_local columns of it
        self.global_step += self.hp.rollout_length * self.hp.batch_size * self.world_size
        if not sync_stats:
            return {}
        host = self._stats_host
        if self._dist:      # loss scalars are SUMs over the global batch in the reference; reduced only when somebody reads them
            torch.distributed.all_reduce(self._losses, op=torch.distributed.ReduceOp.SUM, group=self.pg or None)
        host[:4].copy_(self._losses, non_blocking=True)
        host[4:6].copy_(self._coef, non_blocking=True)
        done = batch['done'][1:]
        ep = batch['episode_return'][1:][done] if 'episode_return' in batch else torch.empty(0, device=self.device)
        ep_host = ep.cpu()                                  # synchronises the stream (the reference does 6 .item() syncs)
        torch.cuda.current_stream(self.device).synchronize()
        return {'episode_returns': tuple(ep_host.numpy()),
                'mean_episode_return': float(ep_host.mean()) if ep_host.numel() else float('nan'),
                'total_loss': float(host[3]), 'pg_loss': float(host[0]), 'baseline_loss': float(host[1]),
                'entropy_loss': float(host[2]), 'grad_norm': float(host[4])}

    def debug_buffer(self, name: str, dtype=None):
        """copy of an internal activation buffer (tests only)"""
        p, n = C.c_void_p(), C.c_int64()
        _lib.check(self._L.srl_learner_debug_buffer(self._h, name.encode(), C.byref(p), C.byref(n)), 'debug_buffer')
        fp32 = name in ('h', 'logits', 'baseline', 'dlogits', 'dbaseline')      # everything else (xs, a1.., da.., wpack, *_lo) is bf16
        dt = torch.float32 if fp32 else torch.bfloat16
        nbytes = n.value * (4 if fp32 else 2)
        out = torch.empty(n.value, dtype=dt, device=self.device)
        _lib.check(self._L.srl_memcpy_d2d(out.data_ptr(), p.value, nbytes, self._stream()), 'memcpy_d2d')
        torch.cuda.current_stream(self.device).synchronize()
        return out

    def close(self):
        if getattr(self, '_h', None) is not None:
            self._L.srl_learner_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
