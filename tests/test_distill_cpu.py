"""Knowledge-distillation pieces (SURVEY.md 8 f4): the loss tails equal the reference's
(SimpleAICV/distillation/losses.py, its values and gradients on the same logits stored in
tests/golden/reference_snapshots.pts); KDModel has the reference's layout."""
import importlib.util
import os

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
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


@pytest.mark.parametrize('name,args', snap.DISTILL)
def test_distillation_losses_match_reference(name, args):
    from simpleaicv_pytorch_training_examples_b200.distillation import losses
    ref = snap.load()[f'distill/{name}']
    stu2, other = snap.distill_inputs(name)
    stu2.requires_grad_(True)
    b = getattr(losses, name)(*args)(stu2, other)
    b.backward()
    assert torch.equal(ref['loss'], b.detach())
    assert torch.equal(ref['grad'], stu2.grad)


def test_kdmodel_layout_and_frozen_teacher():
    from simpleaicv_pytorch_training_examples_b200.distillation.distillmodel import KDModel
    m = KDModel(teacher_type='resnet34', student_type='resnet18', num_classes=10)
    assert all(not p.requires_grad for p in m.teacher.parameters()) and all(p.requires_grad for p in m.student.parameters())
    keys = list(m.state_dict().keys())
    assert keys[0].startswith('teacher.') and any(k.startswith('student.') for k in keys)
    with pytest.raises(RuntimeError, match='no CPU'):
        m(torch.randn(1, 3, 32, 32))
