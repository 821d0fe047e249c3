"""Oracle and B200 constructors against the unmodified reference: what the reference computes for each case here is
stored in tests/golden/reference_snapshots.pts (written by tests/golden/make_reference_snapshots.py from the reference
itself): bit-identical seeded state dicts by digest, outputs and gradients by value or at fixed positions plus
whole-tensor norms."""
import importlib.util
import os

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
_spec = importlib.util.spec_from_file_location('make_reference_snapshots', os.path.join(HERE, 'golden', 'make_reference_snapshots.py'))
snap = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(snap)
SNAPS = snap.load()


@pytest.fixture(autouse=True)
def _one_thread():
    """The snapshots were taken with one CPU thread: the same reduction order keeps the comparison at fp32 rounding."""
    n = torch.get_num_threads()
    torch.set_num_threads(1)
    yield
    torch.set_num_threads(n)


def _check_grads(ref, grads, rtol, atol):
    """Every gradient the reference computes, within rtol / atol; the parameters it leaves without one get zero."""
    for n in ref['no_grad']:
        assert grads[n].abs().max() == 0, n
    snap.check_close(ref['grads'], grads, rtol=rtol, atol=atol)


def _check_rel(ref, grads, tol, abs_tol=None):
    for n in ref['no_grad']:
        assert float(grads[n].abs().max()) == 0.0, n
    for n in ref['grads']['names']:
        rel = snap.rel_close(ref['grads'], n, grads[n])
        # fp32 summation order differs between conv2d calls: compare in relative L2
        assert rel < tol or (abs_tol is not None and (snap.take(grads[n]) - snap.unpack(ref['grads'])[n][0]).abs().max().item() < abs_tol), (n, rel)


@pytest.mark.parametrize('arch,nc,shape', [('resnet34cifar', 100, (2, 3, 32, 32)),
                                           ('resnet50cifar', 10, (2, 3, 32, 32)),
                                           ('resnet18', 1000, (2, 3, 64, 64))])
def test_oracle_matches_reference_bitwise(arch, nc, shape):
    from oracle import convnets, train_step
    ref = SNAPS[f'oracle_bitwise/{arch}']
    sd = convnets.init_state(arch, nc, 5)
    snap.check_state(ref['state'], sd)
    g = torch.Generator().manual_seed(9)
    x = torch.randn(*shape, generator=g)
    y = torch.randint(0, nc, (shape[0],), generator=g)
    lo, ls, gr = train_step.loss_and_grads(sd, x, y, arch)
    snap.check_close(ref['out'], {'out': lo}, rtol=1e-5, atol=1e-5)
    _check_grads(ref, gr, rtol=1e-4, atol=1e-6)


@pytest.mark.parametrize('arch', ['resnet18', 'resnet50', 'resnet101', 'resnet18cifar', 'resnet152cifar'])
def test_b200_constructors_match_reference_state_dict(arch):
    """Drop-in contract (SURVEY.md 8b): same keys, shapes and seeded values as the reference."""
    from simpleaicv_pytorch_training_examples_b200.classification import backbones as mine
    ref = SNAPS[f'constructor/{arch}']
    torch.manual_seed(0)
    m = mine.__dict__[arch](num_classes=100)
    snap.check_state(ref['state'], m.state_dict())
    assert snap.text_hash([n for n, _ in m.named_parameters()]) == ref['params']


@pytest.mark.parametrize('global_pool', [False, True])
def test_vit_oracle_matches_reference(global_pool):
    """oracle/vit.py vs SimpleAICV/classification/backbones/vit.py:239-262 (seeded init, logits, every gradient)."""
    from oracle import vit
    ref = SNAPS[f'vit/{global_pool}']
    sd = vit.init_state('vit_base_patch16', 10, 4, image_size=64)
    snap.check_state(ref['state'], sd)
    g = torch.Generator().manual_seed(11)
    x = torch.randn(2, 3, 64, 64, generator=g)
    y = torch.randint(0, 10, (2,), generator=g)
    lo, _, gr = vit.loss_and_grads(sd, x, y, 'vit_base_patch16', global_pool=global_pool)
    snap.check_close(ref['out'], {'out': lo}, rtol=1e-5, atol=1e-6)
    _check_grads(ref, gr, rtol=1e-4, atol=1e-7)     # cls_token has no gradient under global_pool


@pytest.mark.parametrize('arch', ['darknettiny', 'darknet19', 'darknet53'])
def test_darknet_oracle_and_constructors_match_reference(arch):
    """oracle/darknet.py and the B200 constructor shells vs darknet.py:147-432."""
    from oracle import darknet
    from simpleaicv_pytorch_training_examples_b200.classification import backbones as mine
    ref = SNAPS[f'family/{arch}']
    torch.manual_seed(2)
    m = mine.__dict__[arch](num_classes=10)
    sd = darknet.init_state(10, 2, arch=arch)
    snap.check_state(ref['state'], m.state_dict())
    snap.check_state(ref['state'], sd)
    assert snap.text_hash([n for n, _ in m.named_parameters()]) == ref['params']
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, 3, 64, 64, generator=g)
    y = torch.randint(0, 10, (2,), generator=g)
    lo, _, gr = darknet.loss_and_grads(sd, x, y, arch=arch)
    snap.check_close(ref['out'], {'out': lo}, rtol=1e-5, atol=1e-5)
    # gradients of ~1e3 norm: relative L2
    _check_rel(ref, gr, 1e-5)


@pytest.mark.parametrize('arch,kw', [('vit_base_patch16', {'image_size': 64}), ('vit_large_patch16', {'image_size': 32})])
def test_b200_vit_constructors_match_reference_state_dict(arch, kw):
    from simpleaicv_pytorch_training_examples_b200.classification import backbones as mine
    ref = SNAPS[f'constructor/{arch}']
    torch.manual_seed(0)
    m = mine.__dict__[arch](num_classes=7, **kw)
    snap.check_state(ref['state'], m.state_dict())
    assert snap.text_hash([n for n, _ in m.named_parameters()]) == ref['params']


@pytest.mark.parametrize('arch', ['van_b0'])
def test_van_oracle_and_constructor_match_reference(arch):
    """oracle/van.py and the B200 constructor shell vs van.py:211-310 (seeded init, logits, every gradient)."""
    from oracle import van
    from simpleaicv_pytorch_training_examples_b200.classification import backbones as mine
    ref = SNAPS[f'family/{arch}']
    torch.manual_seed(6)
    m = mine.__dict__[arch](num_classes=10)
    sd = van.init_state(arch, 10, 6)
    snap.check_state(ref['state'], m.state_dict())
    snap.check_state(ref['state'], sd)
    assert snap.text_hash([n for n, _ in m.named_parameters()]) == ref['params']
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, 3, 64, 64, generator=g)
    y = torch.randint(0, 10, (2,), generator=g)
    lo, _, gr = van.loss_and_grads(sd, x, y, arch)
    snap.check_close(ref['out'], {'out': lo}, rtol=1e-5, atol=1e-6)
    _check_rel(ref, gr, 1e-4, abs_tol=1e-7)


def test_sam_encoder_oracle_and_constructor_match_reference():
    """oracle/sam_encoder.py and the B200 ViTImageEncoder shell vs segment_anything/image_encoder.py:259-331
    (windowed blocks with padding + a global block; pos_embed / rel-pos tables randomised)."""
    from oracle import sam_encoder as se
    from simpleaicv_pytorch_training_examples_b200.interactive_segmentation.models.segment_anything import image_encoder as mine
    ref = SNAPS['sam_encoder']
    torch.manual_seed(3)
    m = mine.ViTImageEncoder(**snap.SAM_KW)
    sd = se.init_state(3, 160, 16, 128, 2, 2, 4, 256, 7, (1,))
    snap.check_state(ref['state'], m.state_dict())
    snap.check_state(ref['state'], sd)
    vals, x, proj = snap.sam_inputs(list(m.named_parameters()))
    for n, v in vals.items():
        sd[n].copy_(v)
    o, _, gr = se.loss_and_grads(sd, x, proj, 2, 7, (1,))
    snap.check_close(ref['out'], {'out': o}, rtol=1e-4, atol=1e-4)
    _check_rel(dict(ref, no_grad=[]), gr, 1e-4)


def test_detr_oracle_and_constructor_match_reference():
    """oracle/detr.py and the B200 DETR shell vs detection/models/detr.py:273-364 (ResNet-18 body, 6 + 6 layers, padded
    images so that the float key_padding_mask bias matters; dropout zeroed on the reference)."""
    from oracle import detr as od
    from simpleaicv_pytorch_training_examples_b200.detection import models as mine
    ref = SNAPS['detr']
    torch.manual_seed(11)
    m = mine.resnet18_detr()
    sd = od.init_state('resnet18_detr', 11)
    snap.check_state(ref['state'], m.state_dict())
    snap.check_state(ref['state'], sd)
    x, masks = snap.detr_inputs()
    cls_o, reg_o, _, gr = od.loss_and_grads(sd, x, masks, 'resnet18_detr')
    snap.check_close(ref['out'], {'cls': cls_o, 'reg': reg_o}, rtol=1e-4, atol=1e-4, names=['cls', 'reg'])
    _check_rel(ref, gr, 5e-4)      # fp32 summation order in the BN / long-reduction gradients
    # the masked-out keys are NOT excluded by the reference: a bool mask would give a different result
    assert ref['eval_mask_effect'] > 1e-4
    with torch.no_grad():
        a = od.forward(sd, x, masks, 'resnet18_detr', training=False)[0]
        b = od.forward(sd, x, torch.zeros_like(masks), 'resnet18_detr', training=False)[0]
    snap.check_close(ref['out'], {'eval_cls': a}, rtol=1e-4, atol=1e-4, names=['eval_cls'])
    assert (a - b).abs().max() > 1e-4
