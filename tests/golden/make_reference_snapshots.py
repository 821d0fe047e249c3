"""Snapshots of the REFERENCE's own results for the tests that compare with it (tests/test_oracle_vs_reference.py,
test_tools_host_logic.py, test_detr_loss_cpu.py, test_mae_cpu.py, test_distill_cpu.py and, on a GPU,
test_reference_cuda_parity_gpu.py), so that those tests run without the reference.

Every case builds the reference modules exactly as its test builds the module under test, and keeps what the
test compares against:
  * state dicts that must be bit-identical: keys, shapes and a SHA-256 digest of every tensor's bytes;
  * tensors compared with a tolerance: the whole tensor when it has at most K elements, else K elements at
    fixed positions (sample_idx) together with the float64 L2 norm of the whole tensor;
  * host-side values (optimizer groups, learning rates, meters, loss values) as they are.

    python tests/golden/make_reference_snapshots.py            # CPU cases -> reference_snapshots.pts
    python tests/golden/make_reference_snapshots.py --cuda     # GPU cases -> reference_cuda_bs256.pts (needs a GPU)

The reference is imported through baseline/ref_import.py (oracle/install_ref.sh puts it in place).
"""
import hashlib
import importlib.util
import lzma
import os
import pickle
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
CPU_FILE = os.path.join(HERE, 'reference_snapshots.pts')
CUDA_FILE = os.path.join(HERE, 'reference_cuda_bs256.pts')
K = 32                     # elements kept of a tensor that is compared with a tolerance


# ---------------------------------------------------------------------------------------------------- digests
def sample_idx(n, k=K):
    """k distinct positions of a flattened n-element tensor (multiplicative hash with a prime: no RNG involved)."""
    if n <= k:
        return torch.arange(n)
    return (torch.arange(k, dtype=torch.int64) * 2654435761) % n


def take(t, k=K):
    f = t.detach().reshape(-1).cpu()
    return f[sample_idx(f.numel(), k)]


def tensor_hash(t):
    """First 8 bytes of the SHA-256 of a tensor's bytes."""
    t = t.detach().cpu().contiguous().reshape(-1)
    return hashlib.sha256(t.view(torch.uint8).numpy().tobytes()).digest()[:8]


def text_hash(obj):
    return hashlib.sha256(repr(obj).encode()).digest()[:8]


def state_snap(sd):
    return {'keys': text_hash(list(sd)), 'shapes': text_hash([tuple(v.shape) for v in sd.values()]),
            'hash': b''.join(tensor_hash(v) for v in sd.values())}


def close_snap(tensors, k=K):
    """dict name -> tensor  ->  the names, element counts, float64 norms and the concatenated samples."""
    names = list(tensors)
    return {'names': names, 'numel': [tensors[n].numel() for n in names], 'k': k,
            'norm': torch.tensor([tensors[n].detach().double().norm().item() for n in names], dtype=torch.float64),
            'sample': torch.cat([take(tensors[n], k).float() for n in names]) if names else torch.zeros(0)}


def unpack(snap):
    """close_snap -> dict name -> (sample, full-tensor norm)."""
    out, o = {}, 0
    for n, numel, norm in zip(snap['names'], snap['numel'], snap['norm'].tolist()):
        m = min(numel, snap['k'])
        out[n] = (snap['sample'][o:o + m], norm)
        o += m
    return out


# ---------------------------------------------------------------------------------------------------- checks
def check_state(snap, sd, what='state_dict'):
    """sd has the snapshot's keys (in order), shapes and bit-identical values."""
    assert text_hash(list(sd)) == snap['keys'], f'{what}: keys or their order differ'
    assert text_hash([tuple(v.shape) for v in sd.values()]) == snap['shapes'], f'{what}: shapes differ'
    for i, (n, v) in enumerate(sd.items()):
        assert tensor_hash(v) == snap['hash'][8 * i:8 * i + 8], f'{what}: {n} differs from the reference bit for bit'


def check_close(snap, tensors, rtol, atol, names=None):
    """torch.testing.assert_close(tensor, reference, rtol, atol) on the stored elements, and the whole-tensor norm
    within what that bound allows (|a - b| <= atol + rtol |b| elementwise gives | |a| - |b| | <= atol sqrt(n) + rtol |b|)."""
    ref = unpack(snap)
    for n in (names if names is not None else snap['names']):
        s, norm = ref[n]
        t = tensors[n]
        torch.testing.assert_close(take(t, snap['k']).float(), s, rtol=rtol, atol=atol, msg=lambda m: f'{n}: {m}')
        assert abs(t.detach().double().norm().item() - norm) <= atol * t.numel() ** 0.5 + rtol * norm + 1e-12, n


def rel_close(snap, n, t):
    """Relative L2 error of t against the reference tensor n: max of the error on the stored elements and the
    relative difference of the whole-tensor norms (a lower bound of the whole-tensor error)."""
    s, norm = unpack(snap)[n]
    a = take(t, snap['k']).double()
    rel_sample = ((a - s.double()).norm() / s.double().norm().clamp_min(1e-20)).item()
    rel_norm = abs(t.detach().double().norm().item() - norm) / max(norm, 1e-20)
    return max(rel_sample, rel_norm)


def _convert(obj, to_torch):
    if isinstance(obj, dict):
        return {k: _convert(v, to_torch) for k, v in obj.items()}
    if isinstance(obj, list):
        return [_convert(v, to_torch) for v in obj]
    if to_torch and isinstance(obj, np.ndarray):
        return torch.from_numpy(obj)
    if not to_torch and isinstance(obj, torch.Tensor):
        return obj.detach().cpu().numpy()
    return obj


def save(snaps, path):
    """An xz-compressed pickle of plain Python values and numpy arrays (tensors are stored as numpy arrays)."""
    with lzma.open(path, 'wb') as f:
        pickle.dump(_convert(snaps, False), f, protocol=4)


def load(path=CPU_FILE):
    with lzma.open(path, 'rb') as f:
        return _convert(pickle.load(f), True)


# ---------------------------------------------------------------------------------------------------- CPU cases
def _module_from(path, name):
    spec = importlib.util.spec_from_file_location(name, path)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


ORACLE_BITWISE = [('resnet34cifar', 100, (2, 3, 32, 32)), ('resnet50cifar', 10, (2, 3, 32, 32)), ('resnet18', 1000, (2, 3, 64, 64))]
CONSTRUCTORS = ['resnet18', 'resnet50', 'resnet101', 'resnet18cifar', 'resnet152cifar']
VIT_CONSTRUCTORS = [('vit_base_patch16', {'image_size': 64}), ('vit_large_patch16', {'image_size': 32})]
DARKNETS = ['darknettiny', 'darknet19', 'darknet53']
SAM_KW = dict(image_size=160, patch_size=16, embedding_planes=128, block_nums=2, head_nums=2, out_planes=256, window_size=7,
              global_attn_indexes=(1,))
DETR_LOSS_COUNTS = [(1,), (2, 5, 1, 9), (100, 3)]
DISTILL = [('KDLoss', (4.0,)), ('DMLLoss', (2.0,)), ('L2Loss', ()), ('CELoss', ()), ('OneHotLabelCELoss', ())]


def sam_inputs(named_params):
    """The rel-pos tables / pos_embed values and the batch of the SAM-encoder case, drawn in parameter order."""
    g = torch.Generator().manual_seed(9)
    vals = {n: torch.randn(p.shape, generator=g) * 0.2 for n, p in named_params if 'rel_pos' in n or n == 'pos_embed'}
    x = torch.randn(2, 3, 160, 160, generator=g)
    proj = torch.randn(2, 256, 10, 10, generator=g)
    return vals, x, proj


def detr_inputs():
    g = torch.Generator().manual_seed(9)
    x = torch.randn(2, 3, 96, 128, generator=g)
    masks = torch.zeros(2, 96, 128, dtype=torch.bool)
    masks[0, :, 96:] = True
    masks[1, 64:, :] = True
    return x, masks


def _grads(model):
    return {n: p.grad for n, p in model.named_parameters() if p.grad is not None}


def _train_case(ref, x, y):
    ref.train()
    out = ref(x)
    torch.nn.functional.cross_entropy(out.float(), y).backward()
    return {'out': close_snap({'out': out}, k=4096), 'grads': close_snap(_grads(ref)),
            'no_grad': [n for n, p in ref.named_parameters() if p.grad is None]}


def cpu_cases():
    from baseline import ref_import
    torch.set_num_threads(1)
    bb = ref_import.backbones()
    snaps = {}
    # ---- tests/test_oracle_vs_reference.py
    for arch, nc, shape in ORACLE_BITWISE:
        torch.manual_seed(5)
        ref = bb.__dict__[arch](num_classes=nc)
        st = state_snap(ref.state_dict())
        g = torch.Generator().manual_seed(9)
        x = torch.randn(*shape, generator=g)
        y = torch.randint(0, nc, (shape[0],), generator=g)
        snaps[f'oracle_bitwise/{arch}'] = dict(_train_case(ref, x, y), state=st)
    for arch in CONSTRUCTORS:
        torch.manual_seed(0)
        ref = bb.__dict__[arch](num_classes=100)
        snaps[f'constructor/{arch}'] = {'state': state_snap(ref.state_dict()), 'params': text_hash([n for n, _ in ref.named_parameters()])}
    for arch, kw in VIT_CONSTRUCTORS:
        torch.manual_seed(0)
        ref = bb.__dict__[arch](num_classes=7, **kw)
        snaps[f'constructor/{arch}'] = {'state': state_snap(ref.state_dict()), 'params': text_hash([n for n, _ in ref.named_parameters()])}
    for gp in (False, True):
        torch.manual_seed(4)
        ref = bb.vit_base_patch16(image_size=64, global_pool=gp, num_classes=10)
        st = state_snap(ref.state_dict())
        g = torch.Generator().manual_seed(11)
        x = torch.randn(2, 3, 64, 64, generator=g)
        y = torch.randint(0, 10, (2,), generator=g)
        snaps[f'vit/{gp}'] = dict(_train_case(ref, x, y), state=st)
    for arch, seed in [(a, 2) for a in DARKNETS] + [('van_b0', 6)]:
        torch.manual_seed(seed)
        ref = bb.__dict__[arch](num_classes=10)
        st = state_snap(ref.state_dict())
        params = text_hash([n for n, _ in ref.named_parameters()])
        g = torch.Generator().manual_seed(3)
        x = torch.randn(2, 3, 64, 64, generator=g)
        y = torch.randint(0, 10, (2,), generator=g)
        snaps[f'family/{arch}'] = dict(_train_case(ref, x, y), state=st, params=params)
    enc = ref_import.module('SimpleAICV.interactive_segmentation.models.segment_anything.image_encoder')
    torch.manual_seed(3)
    r = enc.ViTImageEncoder(**SAM_KW)
    st = state_snap(r.state_dict())
    vals, x, proj = sam_inputs(list(r.named_parameters()))
    with torch.no_grad():
        for n, p in r.named_parameters():
            if n in vals:
                p.copy_(vals[n])
    r.train()
    out = r(x)
    (out.float() * proj).mean().backward()
    snaps['sam_encoder'] = {'state': st, 'out': close_snap({'out': out}, k=4096), 'grads': close_snap(_grads(r))}
    torch.manual_seed(11)
    r = ref_import.module('SimpleAICV.detection.models').__dict__['resnet18_detr']()
    st = state_snap(r.state_dict())
    for mod in r.modules():
        if isinstance(mod, torch.nn.Dropout):
            mod.p = 0.0
        if isinstance(mod, torch.nn.MultiheadAttention):
            mod.dropout = 0.0
    from oracle import detr as od
    x, masks = detr_inputs()
    r.train()
    cls_r, reg_r = r(x, masks)
    od.surrogate_loss(cls_r, reg_r).backward()
    r.eval()
    with torch.no_grad():
        a = r(x, masks)[0]
        b = r(x, torch.zeros_like(masks))[0]
    snaps['detr'] = {'state': st, 'out': close_snap({'cls': cls_r, 'reg': reg_r, 'eval_cls': a}, k=4096),
                     'grads': close_snap(_grads(r), k=128), 'no_grad': [n for n, p in r.named_parameters() if p.grad is None],
                     'eval_mask_effect': (a - b).abs().max().item()}
    # ---- tests/test_tools_host_logic.py (the reference's tools.utils on the B200 package's models)
    snaps['tools'] = tools_cases(ref_import)
    # ---- tests/test_detr_loss_cpu.py
    mk = _module_from(os.path.join(HERE, 'make_detr_loss_golden.py'), 'mk_detr')
    for counts in DETR_LOSS_COUNTS:
        cls, reg, ann = mk.make_inputs(seed=len(counts), counts=counts)
        losses = ref_import.module('SimpleAICV.detection.losses').DETRLoss()([cls, reg], ann)
        snaps[f'detr_loss/{counts}'] = {k: v.detach().clone() for k, v in losses.items()}
    # ---- tests/test_mae_cpu.py
    gen = _module_from(os.path.join(HERE, 'make_mae_golden.py'), 'mk_mae')
    x, noise = gen.make_inputs()
    model, pred, mask, loss, grads = gen.reference_run(x, noise)
    snaps['mae'] = {'state': state_snap(model.state_dict()), 'mask': mask, 'loss': loss,
                    'pred': close_snap({'pred': pred}, k=4096), 'grads': close_snap(grads)}
    # ---- tests/test_distill_cpu.py
    ref_import._ensure_path()
    from SimpleAICV.distillation import losses as kd
    for name, args in DISTILL:
        stu, other = distill_inputs(name)
        stu.requires_grad_(True)
        a = getattr(kd, name)(*args)(stu, other)
        a.backward()
        snaps[f'distill/{name}'] = {'loss': a.detach().clone(), 'grad': stu.grad.clone()}
    return snaps


def distill_inputs(name):
    g = torch.Generator().manual_seed(0)
    stu = torch.randn(16, 100, generator=g) * 3
    tea = torch.randn(16, 100, generator=g) * 3
    if name == 'CELoss':
        other = torch.randint(0, 100, (16,), generator=g)
    elif name == 'OneHotLabelCELoss':
        other = torch.softmax(torch.randn(16, 100, generator=g), dim=1)
    else:
        other = tea
    return stu, other


def canon_groups(opt, model):
    """Optimizer parameter groups as (weight decay, lr rounded to 1e-15, sorted parameter names), sorted."""
    names = {id(p): n for n, p in model.named_parameters()}
    return sorted((g['weight_decay'], round(g['lr'], 15), sorted(names[id(p)] for p in g['params'])) for g in opt.param_groups)


VIT_EPOCHS = [0.0, 2.5, 5.0, 50.0, 99.5]
R50_EPOCHS = [0.0, 0.5, 0.99, 1.0, 29.9, 30.0, 61.2, 95.0]


def vit_cfg(m):
    class C:
        optimizer = ('AdamW', {'lr': 5e-4, 'global_weight_decay': False, 'weight_decay': 0.05,
                               'no_weight_decay_layer_name_list': ['position_encoding', 'cls_token'],
                               'lr_layer_decay': 0.65, 'lr_layer_decay_block': m.blocks, 'block_name': 'blocks'})
        scheduler = ('CosineLR', {'warm_up_epochs': 5, 'min_lr': 1e-6})
        epochs = 100
    return C


class R50Cfg:
    optimizer = ('SGD', {'lr': 0.1, 'momentum': 0.9, 'global_weight_decay': False, 'weight_decay': 1e-4,
                         'no_weight_decay_layer_name_list': []})
    scheduler = ('MultiStepLR', {'warm_up_epochs': 1, 'gamma': 0.1, 'milestones': [30, 60, 90]})
    epochs = 100


def tools_cases(ref_import):
    from simpleaicv_pytorch_training_examples_b200.classification import backbones
    ref_utils = ref_import.module('tools.utils')
    out = {}
    m = backbones.vit_base_patch16(image_size=32, num_classes=10)
    C = vit_cfg(m)
    ro, _ = ref_utils.build_optimizer(C, m)
    rec = {'groups': canon_groups(ro, m), 'type': type(ro).__name__, 'betas': ro.defaults['betas'], 'eps': ro.defaults['eps'],
           'lr': [], 'groups_after': []}
    rs = ref_utils.Scheduler(C, ro)
    for e in VIT_EPOCHS:
        rs.step(ro, e)
        rec['lr'].append(rs.current_lr)
        rec['groups_after'].append(text_hash(canon_groups(ro, m)))
    out['vit_layer_decay'] = rec
    m = backbones.resnet50cifar(num_classes=10)
    ro, _ = ref_utils.build_optimizer(R50Cfg, m)
    rec = {'groups': canon_groups(ro, m), 'lr': [], 'group_lrs': []}
    rs = ref_utils.Scheduler(R50Cfg, ro)
    for e in R50_EPOCHS:
        rs.step(ro, e)
        rec['lr'].append(rs.current_lr)
        rec['group_lrs'].append(sorted(g['lr'] for g in ro.param_groups))
    out['r50_groups'] = rec
    rc = ref_import.module('SimpleAICV.classification.common')
    a = rc.AverageMeter()
    for v, n in [(1.5, 4), (0.25, 2), (3.0, 1)]:
        a.update(v, n)
    am = rc.AccMeter()
    for c1, c5, n in [(3, 7, 10), (5, 9, 10)]:
        am.update(c1, c5, n)
    am.compute()
    out['meters'] = {'average': (a.avg, a.sum, a.count, a.val), 'acc': (am.acc1, am.acc5)}
    return out


# ---------------------------------------------------------------------------------------------------- GPU cases
CUDA_CASES = [('resnet50', {}, 'CELoss', 256), ('vit_base_patch16', {'image_size': 224, 'global_pool': True}, 'OneHotLabelCELoss', 256)]


def cuda_inputs(loss_name, batch):
    g = torch.Generator().manual_seed(2024)
    x = torch.randn(batch, 3, 224, 224, generator=g)
    lab = torch.randint(0, 1000, (batch,), generator=g)
    if loss_name == 'CELoss':
        return x, lab
    oh = torch.nn.functional.one_hot(lab, 1000).float() * 0.9 + 0.1 / 1000
    return x, 0.5 * oh + 0.5 * oh.roll(1, 0)


def _rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


def cuda_cases():
    """The reference's CUDA path at the benchmarked shape: fp32 and bf16 autocast (tools/scripts.py:153-170)."""
    from baseline import ref_import
    bb = ref_import.backbones()
    ref_l = ref_import.module('SimpleAICV.classification.losses')
    snaps = {'device': torch.cuda.get_device_name(0), 'torch': torch.__version__}
    for arch, kw, loss_name, batch in CUDA_CASES:
        x, y = cuda_inputs(loss_name, batch)
        x, y = x.cuda(), y.cuda()
        torch.manual_seed(0)
        ref = bb.__dict__[arch](num_classes=1000, **kw).cuda().train()
        sd0 = {k: v.clone() for k, v in ref.state_dict().items()}
        crit = ref_l.__dict__[loss_name]().cuda()
        runs = {}
        for autocast in (False, True):
            ref.load_state_dict(sd0)
            ref.zero_grad(set_to_none=True)
            with torch.autocast('cuda', dtype=torch.bfloat16, enabled=autocast):
                out = ref(x)
                loss = crit(out, y)
            loss.backward()
            torch.cuda.synchronize()
            runs[autocast] = (out.detach().float(), loss.detach().float(),
                              {n: p.grad.detach().float().clone() for n, p in ref.named_parameters() if p.grad is not None})
        (lo32, ls32, g32), (lo16, ls16, g16) = runs[False], runs[True]
        stats = {k: v.clone() for k, v in ref.state_dict().items() if 'running_' in k}
        names = list(g16)
        cat = lambda d: torch.cat([d[n].flatten() for n in names])
        snaps[arch] = {
            'state': state_snap(sd0),
            'logits16': close_snap({'logits': lo16}, k=2048), 'logits_scale': lo16.abs().max().item(),
            'logits_noise': (lo16 - lo32).abs().max().item(), 'loss16': ls16.item(), 'loss32': ls32.item(),
            'stats': close_snap(stats, k=16), 'stats_scale': {k: v.abs().max().item() for k, v in stats.items()},
            'g16': close_snap(g16), 'g32': close_snap({n: g32[n] for n in names}),
            'noise': {n: _rel(g16[n], g32[n]) for n in names}, 'whole_noise': _rel(cat(g16), cat(g32)),
        }
        del ref, runs, g16, g32
        torch.cuda.empty_cache()
    return snaps


def main():
    sys.path.insert(0, ROOT)
    if '--cuda' in sys.argv:
        path = sys.argv[sys.argv.index('--cuda') + 1] if len(sys.argv) > sys.argv.index('--cuda') + 1 else CUDA_FILE
        snaps = cuda_cases()
    else:
        path, snaps = CPU_FILE, cpu_cases()
    save(snaps, path)
    print(path, os.path.getsize(path), 'bytes')


if __name__ == '__main__':
    main()
