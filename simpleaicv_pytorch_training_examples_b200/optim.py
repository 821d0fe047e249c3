"""Fused multi-tensor optimizers (SURVEY.md 8 f2) behind torch.optim's interface.

``FusedSGD`` / ``FusedAdamW`` update ALL parameters of a model with one launch of csrc/capi_optim.cu (torch's foreach
path: 13 / 45 launches per step), refresh the bf16 GEMM-operand copies of the weights in the same pass (the runtime's
separate cast / re-layout kernels: 53 per ResNet-50 step, 49 per ViT-B step) and apply the global-norm gradient clip
without a host sync.  They subclass ``torch.optim.Optimizer``: ``param_groups`` (what ``tools.utils.Scheduler`` rewrites
every iteration), ``state_dict()`` / ``load_state_dict()`` use torch's own keys (``momentum_buffer``; ``step``,
``exp_avg``, ``exp_avg_sq``), so checkpoints interchange with the reference's torch.optim.SGD / AdamW
(reference tools/utils.py:581-600).

Hyper-parameters travel through a pinned ring of RING tables copied to the device at the head of every step; the kernel
picks table (device step counter % RING).  Under CUDA-graph capture that copy is a node of the graph, so
``sync_hyper()`` (a pure host write of slot t % RING, called by graph.GraphedTrainStep before each replay) is all a
per-iteration learning-rate schedule needs, and the host may run RING - 1 steps ahead of the device.
"""
import ctypes
import math

import numpy as np
import torch

from . import _lib

RING = 8   # SAICV_OPT_RING

_TENSOR_DTYPE = np.dtype([('p', '<u8'), ('g', '<u8'), ('s1', '<u8'), ('s2', '<u8'), ('shadow', '<u8'), ('numel', '<i8'),
                          ('group', '<i4'), ('rs', '<i4'), ('c', '<i4'), ('cp', '<i4'), ('kpad', '<i4'), ('pad_', '<i4')])
assert _TENSOR_DTYPE.itemsize == 72   # saicv_opt_tensor (include/saicv_b200.h)


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


class _FusedBase(torch.optim.Optimizer):
    """Shared table building / hyper-parameter plumbing.  Shadows: ``register_shadow(param, bf16_tensor, conv=None)``
    tells the step to keep ``bf16_tensor`` equal to bf16(param) ([N][K] Linear copy, leading rows) or, with
    conv=(c, rs, cp, kpad), to the tap-major conv operand layout of saicv_prep_conv_weight (order 0)."""

    _entry = None       # C-ABI symbol
    _n_state = 1

    def __init__(self, params, defaults):
        super().__init__(params, defaults)
        self._shadows = {}        # id(param) -> (tensor, conv layout or None)
        self._key = None          # identity of the table (pointers of p / grad / shadow)
        self._tab = None
        self._t = 0               # optimizer steps taken (AdamW bias correction)
        self._clip = None
        self._use_clip = False
        self._hyper_host = None   # pinned [RING][groups][8]; slot t % RING holds the table of step t
        self._events = [None] * RING   # recorded after the step that read slot i was launched
        self._pending = None

    # ---- shadows (called by the runtimes: engine/convnet.py, engine/vit.py)
    def register_shadow(self, param, shadow, conv=None, owner=None):
        """owner: the runtime object whose ``w_bf16`` attribute is this copy; when given, the attribute is re-read before
        every step, so a copy the runtime re-allocates (device move) is followed instead of silently going stale."""
        assert shadow.dtype == torch.bfloat16 and shadow.is_contiguous()
        self._shadows[id(param)] = (shadow, conv, owner)
        self._key = None

    def _follow_owners(self):
        for pid, (shadow, conv, owner) in list(self._shadows.items()):
            cur = getattr(owner, 'w_bf16', None) if owner is not None else shadow
            if cur is not None and cur is not shadow:
                self._shadows[pid] = (cur, conv, owner)

    def attach(self, model):
        """Registers the operand copies of every weight of `model`'s runtime (a no-op for plain torch modules)."""
        m = model if hasattr(model, '_runtime') else getattr(model, 'module', model)
        if hasattr(m, '_runtime'):
            from .engine import shadows
            mine = {id(p) for g in self.param_groups for p in g['params']}
            for param, shadow, conv, owner in shadows.collect(m._runtime()):
                if id(param) in mine:
                    self.register_shadow(param, shadow, conv, owner=owner)
        return self

    def load_state_dict(self, state_dict):
        """torch's loader replaces the state tensors (momentum buffers, moments): the device table must be rebuilt."""
        super().load_state_dict(state_dict)
        self._key = None

    # ---- table
    def _params(self):
        out = []
        for gi, g in enumerate(self.param_groups):
            for p in g['params']:
                if p.grad is not None:
                    out.append((gi, p))
        return out

    def _state_tensors(self, p):
        raise NotImplementedError

    def _build(self, plist):
        dev = plist[0][1].device
        chunk = _lib.load().saicv_opt_chunk()
        rows = np.zeros(len(plist), dtype=_TENSOR_DTYPE)
        ct, ci = [], []
        for i, (gi, p) in enumerate(plist):
            assert p.dtype == torch.float32 and p.is_contiguous() and p.grad.dtype == torch.float32 and p.grad.is_contiguous(), \
                'fused optimizers need contiguous fp32 parameters and gradients'
            st = self._state_tensors(p)
            r = rows[i]
            r['p'], r['g'], r['s1'] = p.data_ptr(), p.grad.data_ptr(), st[0].data_ptr()
            r['s2'] = st[1].data_ptr() if len(st) > 1 else 0
            r['numel'], r['group'] = p.numel(), gi
            sh = self._shadows.get(id(p))
            if sh is not None:
                r['shadow'] = sh[0].data_ptr()
                if sh[1] is not None:
                    r['c'], r['rs'], r['cp'], r['kpad'] = sh[1]
                    assert sh[0].numel() >= (p.numel() // (r['c'] * r['rs'])) * r['kpad']
                else:
                    assert sh[0].numel() >= p.numel()
            n = (p.numel() + chunk - 1) // chunk
            ct.extend([i] * n)
            ci.extend(range(n))
        tab = {
            'tensors': torch.from_numpy(rows.view(np.uint8).copy()).to(dev),
            'ct': torch.tensor(ct, dtype=torch.int32).to(dev), 'ci': torch.tensor(ci, dtype=torch.int32).to(dev),
            'n': len(ct), 'partial': torch.empty(len(ct), device=dev), 'dev': dev,
        }
        if self._hyper_host is None or self._hyper_host.shape[1] != len(self.param_groups):
            self._hyper_host = torch.zeros(RING, len(self.param_groups), 8).pin_memory()
            self._hyper_np = self._hyper_host.numpy()
            self._hyper_dev = torch.zeros(RING, len(self.param_groups), 8, device=dev)
            self._clip = torch.ones(2, device=dev)
            self._step_dev = torch.full((1,), self._t, dtype=torch.int32, device=dev)
        return tab

    def _table(self):
        plist = self._params()
        if not plist:
            return None
        self._follow_owners()
        key = tuple((id(p), p.data_ptr(), p.grad.data_ptr(), self._shadows.get(id(p), (None,))[0] is not None and
                     self._shadows[id(p)][0].data_ptr()) for _, p in plist)
        if key != self._key:
            self._tab, self._key = self._build(plist), key
        return self._tab

    # ---- hyper-parameters
    def _hyper_row(self, g, t):
        raise NotImplementedError

    def _publish(self):
        """Host side of step number self._t (0-based): waits until the step that last used its ring slot has been
        launched RING steps ago AND executed, writes the table (AdamW bias corrections are those of update t + 1)."""
        slot = self._t % RING
        if self._events[slot] is not None and not torch.cuda.is_current_stream_capturing():
            self._events[slot].synchronize()
        for gi, g in enumerate(self.param_groups):
            row = self._hyper_row(g, self._t + 1)
            self._hyper_np[slot, gi, :len(row)] = row
        self._t += 1
        return slot

    def _mark(self, slot):
        if self._events[slot] is None:
            self._events[slot] = torch.cuda.Event()
        self._events[slot].record()

    def sync_hyper(self):
        """Before the replay of a CAPTURED step (graph.GraphedTrainStep calls it): host write of the next table."""
        if self._hyper_host is not None:
            self._pending = self._publish()

    def after_replay(self):
        if self._pending is not None:
            self._mark(self._pending)
            self._pending = None

    # ---- gradient clipping fused with the step
    @torch.no_grad()
    def clip_grad_norm(self, max_norm):
        """torch.nn.utils.clip_grad_norm_ without the host sync: the coefficient stays on the device and scales the
        gradients inside the next step().  Returns the (device) total norm."""
        tab = self._table()
        if tab is None:
            return None
        _lib.call('saicv_multi_tensor_clip_coef', _p(tab['tensors']), _p(tab['ct']), _p(tab['ci']), tab['n'],
                  ctypes.c_float(float(max_norm)), _p(tab['partial']), _p(self._clip), _stream())
        self._use_clip = True
        return self._clip[1]

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        tab = self._table()
        if tab is None:
            return loss
        capturing = torch.cuda.is_current_stream_capturing()
        slot = self._publish()
        self._hyper_dev.copy_(self._hyper_host, non_blocking=True)
        _lib.call(self._entry, _p(tab['tensors']), _p(tab['ct']), _p(tab['ci']), tab['n'], _p(self._hyper_dev),
                  len(self.param_groups), _p(self._step_dev), _p(self._clip) if self._use_clip else None, _stream())
        self._use_clip = False
        if capturing:
            self._t -= 1          # recorded, not executed: the first replay publishes this step's table again
        else:
            self._mark(slot)
        # parameters were written through raw pointers: bump the version of the ones whose operand copy was NOT
        # refreshed here, so that the runtimes' prep() re-casts them (the fused ones keep their version and skip it)
        for _, p in self._params():
            if id(p) not in self._shadows:
                torch.autograd.graph.increment_version(p)
        return loss


class FusedSGD(_FusedBase):
    """torch.optim.SGD(params, lr, momentum, weight_decay, nesterov) with dampening 0 (the reference's only use,
    tools/utils.py:581-590)."""
    _entry = 'saicv_multi_tensor_sgd'

    def __init__(self, params, lr=1e-3, momentum=0., weight_decay=0., nesterov=False):
        super().__init__(params, dict(lr=lr, momentum=momentum, weight_decay=weight_decay, nesterov=nesterov, dampening=0.))

    def _state_tensors(self, p):
        st = self.state[p]
        if 'momentum_buffer' not in st or st['momentum_buffer'] is None:
            st['momentum_buffer'] = torch.zeros_like(p, memory_format=torch.preserve_format)   # first step: buf = g
        return (st['momentum_buffer'],)

    def _hyper_row(self, g, t):
        return (g['lr'], g['weight_decay'], g['momentum'], 1. if g['nesterov'] else 0.)


class FusedAdamW(_FusedBase):
    """torch.optim.AdamW(params, lr, betas, eps, weight_decay) (amsgrad / maximize off; tools/utils.py:591-600)."""
    _entry = 'saicv_multi_tensor_adamw'

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2):
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))

    def _state_tensors(self, p):
        st = self.state[p]
        if 'exp_avg' not in st:
            st['step'] = torch.tensor(0.)
            st['exp_avg'] = torch.zeros_like(p, memory_format=torch.preserve_format)
            st['exp_avg_sq'] = torch.zeros_like(p, memory_format=torch.preserve_format)
        return st['exp_avg'], st['exp_avg_sq']

    def _hyper_row(self, g, t):
        b1, b2 = g['betas']
        t = max(t, 1)
        return (g['lr'], g['weight_decay'], b1, b2, g['eps'], 1. - b1 ** t, math.sqrt(1. - b2 ** t))

    def state_dict(self):
        for st in self.state.values():
            if 'step' in st:
                st['step'] = torch.tensor(float(self._t))
        return super().state_dict()

    def load_state_dict(self, state_dict):
        super().load_state_dict(state_dict)
        steps = [float(st['step']) for st in self.state.values() if 'step' in st]
        self._t = int(max(steps)) if steps else 0
        self._key = None
        if self._hyper_host is not None:
            self._step_dev.fill_(self._t)
