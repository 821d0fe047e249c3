"""DETRLoss (detection/losses.py) against the committed reference outputs (tests/golden/detr_loss_b3.ptl, written by
tests/golden/make_detr_loss_golden.py from the reference's DETRLoss) and the reference's loss values on further
inputs (tests/golden/reference_snapshots.pts).  The Hungarian indices are integer work: they must match exactly."""
import importlib.util
import os

import pytest
import torch

from simpleaicv_pytorch_training_examples_b200.detection.losses import DETRLoss, assignment_with_inf

HERE = os.path.dirname(os.path.abspath(__file__))
_spec = importlib.util.spec_from_file_location('mk', os.path.join(HERE, 'golden', 'make_detr_loss_golden.py'))
mk = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(mk)
_spec = importlib.util.spec_from_file_location('make_reference_snapshots', os.path.join(HERE, 'golden', 'make_reference_snapshots.py'))
snap = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(snap)


@pytest.fixture(autouse=True)
def _one_thread():
    """The reference snapshots were taken with one CPU thread: the same reduction order makes bit equality meaningful."""
    n = torch.get_num_threads()
    torch.set_num_threads(1)
    yield
    torch.set_num_threads(n)


def test_detr_loss_reproduces_reference_fixture():
    fix = torch.load(os.path.join(HERE, 'golden', 'detr_loss_b3.ptl'), weights_only=False)
    cls, reg, ann = mk.make_inputs()
    cls.requires_grad_(True)
    reg.requires_grad_(True)
    crit = DETRLoss()
    losses = crit([cls, reg], ann)
    assert list(losses) == list(fix['losses'])
    for k, v in fix['losses'].items():
        torch.testing.assert_close(losses[k], v, rtol=1e-5, atol=1e-6)
    idx = crit.get_matched_pred_target_idxs(cls[-1].detach(), reg[-1].detach().clamp(1e-4, 1 - 1e-4), ann)
    for (a, b), (c, d) in zip(idx, fix['indices']):
        assert a.dtype == torch.int64 and torch.equal(a, c) and torch.equal(b, d)
    sum(losses.values()).backward()
    torch.testing.assert_close(cls.grad.norm(), fix['dcls_norm'], rtol=1e-5, atol=1e-7)
    torch.testing.assert_close(reg.grad.norm(), fix['dreg_norm'], rtol=1e-5, atol=1e-7)
    torch.testing.assert_close(cls.grad.flatten()[:8], fix['dcls_head'], rtol=1e-5, atol=1e-8)


@pytest.mark.parametrize('counts', snap.DETR_LOSS_COUNTS)
def test_detr_loss_matches_reference_live(counts):
    b = snap.load()[f'detr_loss/{counts}']
    cls, reg, ann = mk.make_inputs(seed=len(counts), counts=counts)
    a = DETRLoss()([cls, reg], ann)
    assert list(a) == list(b) and all(torch.equal(a[k], b[k]) for k in b)


def test_assignment_handles_nan_and_infinities():
    import numpy as np
    c = np.array([[1.0, np.inf, 3.0], [np.nan, 0.5, np.inf], [2.0, 2.0, 0.1]])
    rows, cols = assignment_with_inf(c.copy())
    assert list(rows) == [0, 1, 2] and list(cols) == [0, 1, 2]
    with pytest.raises(ValueError):
        assignment_with_inf(np.array([[np.inf, -np.inf], [0.0, 1.0]]))
