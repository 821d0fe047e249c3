"""Host-side logic of the tools layer: optimizer parameter groups and LR schedule.

Runs on CPU.  The results are compared with what the reference's own tools/utils.py and classification/common.py
give on the same models (stored in tests/golden/reference_snapshots.pts by tests/golden/make_reference_snapshots.py)."""
import importlib.util
import math
import os

import pytest
import torch

from simpleaicv_pytorch_training_examples_b200.classification import backbones
from simpleaicv_pytorch_training_examples_b200.tools import utils as my_utils

HERE = os.path.dirname(os.path.abspath(__file__))
_spec = importlib.util.spec_from_file_location('make_reference_snapshots', os.path.join(HERE, 'golden', 'make_reference_snapshots.py'))
snap = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(snap)


class _Cfg:
    optimizer = ('SGD', {'lr': 0.1, 'momentum': 0.9, 'global_weight_decay': False, 'weight_decay': 1e-4,
                         'no_weight_decay_layer_name_list': []})
    scheduler = ('MultiStepLR', {'warm_up_epochs': 1, 'gamma': 0.1, 'milestones': [30, 60, 90]})
    epochs = 100


def test_one_dim_params_are_not_decayed():
    m = backbones.resnet18cifar(num_classes=10)
    opt, info = my_utils.build_optimizer(_Cfg, m)
    for g in opt.param_groups:
        nd = {p.ndim for p in g['params']}
        assert (g['weight_decay'] == 0.) == (nd == {1}), (g['weight_decay'], nd)
    assert sum(len(g['params']) for g in opt.param_groups) == len(list(m.parameters()))


@pytest.mark.parametrize('name,params', [('MultiStepLR', {'warm_up_epochs': 2, 'gamma': 0.1, 'milestones': [3, 6]}),
                                         ('CosineLR', {'warm_up_epochs': 1, 'min_lr': 1e-6}),
                                         ('PolyLR', {'warm_up_epochs': 0, 'power': 0.9})])
def test_scheduler_closed_forms(name, params):
    class C(_Cfg):
        scheduler = (name, params)
        epochs = 10
    m = torch.nn.Linear(4, 4)
    opt = torch.optim.SGD(m.parameters(), lr=0.1)
    s = my_utils.Scheduler(C, opt)
    for e in [0.0, 0.5, 1.0, 2.5, 3.0, 6.1, 9.99]:
        s.step(opt, e)
        w = params['warm_up_epochs']
        if e < w:
            exp = e / w * 0.1
        elif name == 'MultiStepLR':
            exp = 0.1 * 0.1 ** len([x for x in params['milestones'] if x <= e])
        elif name == 'CosineLR':
            exp = 0.5 * (math.cos((e - w) / (10 - w) * math.pi) + 1) * (0.1 - 1e-6) + 1e-6
        else:
            exp = (1 - (e - w) / (10 - w)) ** 0.9 * 0.1
        assert abs(opt.param_groups[0]['lr'] - exp) < 1e-12 and abs(s.current_lr - exp) < 1e-12


def _ref_tools():
    return snap.load()['tools']


def test_vit_layer_decay_groups_match_reference_utils():
    """ViT layer-wise lr decay + no-weight-decay name list (tools/utils.py:313-420), the AdamW setting of
    00.classification_training/imagenet/vit_base_patch16_*/train_config.py."""
    ref = _ref_tools()['vit_layer_decay']
    m = backbones.vit_base_patch16(image_size=32, num_classes=10)
    C = snap.vit_cfg(m)
    mo, _ = my_utils.build_optimizer(C, m)
    assert ref['groups'] == snap.canon_groups(mo, m)
    assert ref['type'] == type(mo).__name__ and ref['betas'] == mo.defaults['betas'] and ref['eps'] == mo.defaults['eps']
    ms = my_utils.Scheduler(C, mo)
    for e, lr, groups in zip(snap.VIT_EPOCHS, ref['lr'], ref['groups_after']):
        ms.step(mo, e)
        assert abs(lr - ms.current_lr) < 1e-15
        assert groups == snap.text_hash(snap.canon_groups(mo, m))


def test_groups_and_schedule_match_reference_utils():
    ref = _ref_tools()['r50_groups']
    m = backbones.resnet50cifar(num_classes=10)
    mo, _ = my_utils.build_optimizer(snap.R50Cfg, m)
    assert ref['groups'] == snap.canon_groups(mo, m)
    ms = my_utils.Scheduler(snap.R50Cfg, mo)
    for e, lr, group_lrs in zip(snap.R50_EPOCHS, ref['lr'], ref['group_lrs']):
        ms.step(mo, e)
        assert abs(lr - ms.current_lr) < 1e-12
        assert group_lrs == sorted(g['lr'] for g in mo.param_groups)


def test_checkpoint_key_layout_matches_reference_and_round_trips():
    """latest.pth keeps the reference's DDP key layout ('module.' prefix) at every world size, best.pth has
    none (reference tools/train_classification_model.py:213-229); loading accepts both layouts into wrapped
    and unwrapped models."""
    import torch
    import torch.nn as nn
    from simpleaicv_pytorch_training_examples_b200.tools import utils

    class Wrapper(nn.Module):   # stands in for DistributedDataParallel / B200DataParallel
        def __init__(self, m):
            super().__init__()
            self.module = m

    def net(seed):
        torch.manual_seed(seed)
        return nn.Sequential(nn.Conv2d(3, 4, 3), nn.BatchNorm2d(4))

    src = net(0)
    ref_latest = Wrapper(src).state_dict()                      # what the reference writes
    assert all(k.startswith('module.') for k in ref_latest)
    assert list(utils.checkpoint_model_state(src).keys()) == list(ref_latest.keys())            # unwrapped, world 1
    assert list(utils.checkpoint_model_state(Wrapper(src)).keys()) == list(ref_latest.keys())   # wrapped, world N
    for target in (net(1), Wrapper(net(2))):
        utils.load_model_state(target, ref_latest)               # reference latest.pth
        assert all(torch.equal(a, b) for a, b in zip(utils.unwrap(target).state_dict().values(), src.state_dict().values()))
    for target in (net(3), Wrapper(net(4))):
        utils.load_model_state(target, src.state_dict())         # reference best.pth (no prefix)
        assert all(torch.equal(a, b) for a, b in zip(utils.unwrap(target).state_dict().values(), src.state_dict().values()))


def test_meters_and_amp_type_match_reference():
    """AverageMeter / AccMeter behave like the reference's (classification/common.py:668-709); get_amp_type
    returns bf16 for CPU-resident models (no device to inspect) and has 'B200' in its whitelist."""
    import inspect
    import torch
    from simpleaicv_pytorch_training_examples_b200.classification import common
    ref = _ref_tools()['meters']
    a = common.AverageMeter()
    for v, n in [(1.5, 4), (0.25, 2), (3.0, 1)]:
        a.update(v, n)
    assert abs(a.avg - (1.5 * 4 + 0.5 + 3.0) / 7) < 1e-12 and (a.avg, a.sum, a.count, a.val) == ref['average']
    m = common.AccMeter()
    for c1, c5, n in [(3, 7, 10), (5, 9, 10)]:
        m.update(c1, c5, n)
    m.compute()
    assert (m.acc1, m.acc5) == (0.4, 0.8) and (m.acc1, m.acc5) == ref['acc']
    assert "'B200'" in inspect.getsource(common.get_amp_type)
    assert common.get_amp_type(torch.nn.Linear(2, 2)) == torch.bfloat16


def test_dict_loss_epoch_body_guards_accumulation_and_schedule(monkeypatch):
    """train_epoch_with_loss_terms (the body of train_detection / train_distill_sam_encoder): NaN batches are skipped
    without an optimizer step, gradients accumulate over `accumulation_steps` micro-batches, the scheduler advances once
    per optimizer step with the reference's epoch fraction, and the returned average is the mean total loss
    (reference tools/scripts.py:900-1092).  Host logic only: a torch Linear on CPU stands in for the model."""
    import logging
    from simpleaicv_pytorch_training_examples_b200.tools import scripts, utils as tutils
    monkeypatch.setattr(tutils, 'CudaPrefetcher', lambda loader, **kw: loader)
    torch.manual_seed(0)
    model = torch.nn.Linear(4, 2)
    ref = torch.nn.Linear(4, 2)
    ref.load_state_dict(model.state_dict())
    opt = torch.optim.SGD(model.parameters(), lr=0.1)
    ropt = torch.optim.SGD(ref.parameters(), lr=0.1)
    g = torch.Generator().manual_seed(1)
    batches = [{'image': torch.randn(3, 4, generator=g), 'target': torch.randn(3, 2, generator=g)} for _ in range(6)]
    batches[2]['image'][0, 0] = float('nan')

    class Loader(list):
        dataset = list(range(18))

    class Cfg:
        accumulation_steps, batch_size, print_interval, local_rank, network = 2, 3, 1, 0, 'resnet50_detr'

    class Sched:
        current_lr, calls = 0.1, []

        def step(self, optimizer, epoch):
            self.calls.append(epoch)

    def crit(out, tgt):
        d = out - tgt
        return {'a_loss': d.square().mean(), 'b_loss': d.abs().mean()}

    def compute(data):
        return crit(model(data['image']), data['target']), (data['image'], data['target']), data['image'].size(0)

    sched = Sched()
    avg = scripts.train_epoch_with_loss_terms(Loader(batches), model, crit, opt, sched, 3, logging.getLogger('t'), Cfg, compute)
    # straightforward restatement of the reference semantics
    totals, it = [], 1
    for b in batches:
        if not torch.isfinite(b['image']).all():
            ropt.zero_grad()
            continue                      # note: the reference `continue`s before iter_index += 1
        loss = sum(crit(ref(b['image']), b['target']).values()) / 2
        loss.backward()
        if it % 2 == 0:
            ropt.step()
            ropt.zero_grad()
            totals.append(float(loss))
        it += 1
    for p, q in zip(model.parameters(), ref.parameters()):
        torch.testing.assert_close(p, q)
    assert len(sched.calls) == len(totals) == 2
    assert sched.calls == [2 / 6 + 2, 4 / 6 + 2]
    assert abs(avg - 2 * sum(totals) / len(totals)) < 1e-6


def test_mae_and_distillation_epoch_bodies(monkeypatch):
    """train_mae_self_supervised_learning (reference tools/scripts.py:1774-1934: `outputs, masks = model(images)`,
    `criterion(outputs, labels, masks)`) and train_distill_classification (:291-500: dict of losses, CE on the student - and
    on the teacher only when it is not frozen - every other loss on (student, teacher), each weighted by config.loss_ratio;
    the frozen teacher stays in eval mode).  Host logic only: small torch modules on CPU stand in for the models."""
    import logging
    from simpleaicv_pytorch_training_examples_b200.distillation import losses as kd_losses
    from simpleaicv_pytorch_training_examples_b200.masked_image_modeling import losses as mim_losses
    from simpleaicv_pytorch_training_examples_b200.tools import scripts, utils as tutils
    monkeypatch.setattr(tutils, 'CudaPrefetcher', lambda loader, **kw: loader)
    log = logging.getLogger('t')

    class Loader(list):
        dataset = list(range(12))

    class Sched:
        current_lr = 0.1

        def __init__(self):
            self.calls = []

        def step(self, optimizer, epoch):
            self.calls.append(epoch)

    class Cfg:
        accumulation_steps, batch_size, print_interval, local_rank = 1, 4, 1, 0
        freeze_teacher = True
        loss_ratio = {'CELoss': 1.0, 'KDLoss': 0.5}

    # ---- MAE: model returns (pred, mask)
    class FakeMAE(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.lin = torch.nn.Linear(6, 6)

        def forward(self, x):
            return self.lin(x), (x[..., 0] > 0).float()

    torch.manual_seed(0)
    mae, ref = FakeMAE(), FakeMAE()
    ref.load_state_dict(mae.state_dict())
    g = torch.Generator().manual_seed(2)
    batches = [{'image': torch.randn(4, 5, 6, generator=g), 'label': torch.randn(4, 5, 6, generator=g)} for _ in range(3)]
    opt, ropt = torch.optim.SGD(mae.parameters(), lr=0.1), torch.optim.SGD(ref.parameters(), lr=0.1)
    crit = mim_losses.MSELoss()
    sched = Sched()
    avg = scripts.train_mae_self_supervised_learning(Loader(batches), mae, crit, opt, sched, 1, log, Cfg)
    vals = []
    for b in batches:
        out, mask = ref(b['image'])
        loss = crit(out, b['label'], mask)
        loss.backward()
        ropt.step()
        ropt.zero_grad()
        vals.append(float(loss))
    for p, q in zip(mae.parameters(), ref.parameters()):
        torch.testing.assert_close(p, q)
    assert abs(avg - sum(vals) / 3) < 1e-6 and len(sched.calls) == 3

    # ---- distillation: model returns (teacher logits, student logits)
    class FakeKD(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.teacher, self.student = torch.nn.Linear(6, 5), torch.nn.Linear(6, 5)
            for p in self.teacher.parameters():
                p.requires_grad = False

        def forward(self, x):
            with torch.no_grad():
                t = self.teacher(x)
            return t, self.student(x)

    kd, kref = FakeKD(), FakeKD()
    kref.load_state_dict(kd.state_dict())
    batches = [{'image': torch.randn(4, 6, generator=g), 'label': torch.randint(0, 5, (4,), generator=g)} for _ in range(3)]
    crit = {'CELoss': kd_losses.CELoss(), 'KDLoss': kd_losses.KDLoss(2.0)}
    opt = torch.optim.SGD([p for p in kd.parameters() if p.requires_grad], lr=0.1)
    ropt = torch.optim.SGD([p for p in kref.parameters() if p.requires_grad], lr=0.1)
    avg = scripts.train_distill_classification(Loader(batches), kd, crit, opt, Sched(), 1, log, Cfg)
    assert not kd.teacher.training and kd.student.training
    vals = []
    for b in batches:
        t, s = kref(b['image'])
        loss = crit['CELoss'](s, b['label']) * 1.0 + crit['KDLoss'](s, t) * 0.5
        loss.backward()
        ropt.step()
        ropt.zero_grad()
        vals.append(float(loss))
    for p, q in zip(kd.student.parameters(), kref.student.parameters()):
        torch.testing.assert_close(p, q)
    assert abs(avg - sum(vals) / 3) < 1e-6
