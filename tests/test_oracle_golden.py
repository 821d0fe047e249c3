"""The oracle replays the committed reference outputs (tests/golden/*.pt, produced by
tests/golden/make_golden.py from the reference itself) for every model family of the hot path
(ResNet / ResNetCifar, ViT, DarkNet tiny/19/53, VAN).  Runs anywhere: CPU only."""
import glob
import importlib.util
import os

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = sorted(glob.glob(os.path.join(HERE, 'golden', '*.pt')))

_spec = importlib.util.spec_from_file_location('make_golden', os.path.join(HERE, 'golden', 'make_golden.py'))
make_golden = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(make_golden)


def load_fixture(path):
    fix = torch.load(path, weights_only=False)
    fix.setdefault('family', 'resnet')
    fix.setdefault('kwargs', {})
    if 'x' not in fix:  # larger inputs are regenerated from the seed and checked against a digest
        x, _ = make_golden.make_input(tuple(fix['shape']), max(fix['num_classes'], 1), fix['seed'])
        assert abs(float(x.double().sum()) - fix['x_digest'][0]) < 1e-6 and torch.equal(x.flatten()[:4], fix['x_digest'][1])
        fix['x'] = x
    if 'y' not in fix:  # the SAM projection map is regenerated from the seed
        k = fix['kwargs']
        fix['y'] = make_golden.sam_proj(tuple(fix['shape']), k['out_planes'], k['image_size'] // k['patch_size'], fix['seed'])
    return fix


def assert_output_close(fix, name, t, rtol, atol):
    """assert_close against a stored output; a large one is stored at fixed positions with its whole-tensor norm,
    which has to be within what the elementwise bound allows."""
    if name in fix.get('sampled', {}):
        k, norm = fix['sampled'][name]
        assert abs(t.double().norm().item() - norm) <= atol * t.numel() ** 0.5 + rtol * norm, name
        t = make_golden.take(t, k)
    torch.testing.assert_close(t, fix[name], rtol=rtol, atol=atol)


@pytest.mark.parametrize('path', GOLDEN, ids=[os.path.basename(p) for p in GOLDEN])
def test_oracle_reproduces_reference_outputs(path):
    fix = load_fixture(path)
    torch.set_num_threads(1)
    fam, arch, kw = fix['family'], fix['arch'], fix['kwargs']
    sd = make_golden.oracle_init(fam, arch, kw, fix['num_classes'], fix['seed'])
    if fam == 'sam':
        make_golden.sam_randomize(sd, fix['seed'])
    logits, loss, grads = make_golden.oracle_run(fam, arch, kw, sd, fix['x'], fix['y'])
    if fam == 'detr':
        logits, reg = logits
        torch.testing.assert_close(reg, fix['reg'], rtol=1e-5, atol=1e-5)
    # fp32 vs fp32 on CPU: rtol 1e-5 (SURVEY.md 8c); identical torch builds give bit equality
    assert_output_close(fix, 'logits', logits, rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(loss, fix['loss'], rtol=1e-5, atol=1e-6)
    assert set(fix['grad_norm']) <= set(grads)
    for n, g in grads.items():
        if n not in fix['grad_norm']:      # parameters the reference left without a gradient
            assert float(g.abs().max()) == 0.0, n
            continue
        assert abs(g.norm().item() - fix['grad_norm'][n]) <= 1e-4 * max(1.0, fix['grad_norm'][n]), n
        torch.testing.assert_close(g.flatten()[:4], fix['grad_head'][n], rtol=1e-4, atol=1e-6)
    if 'running_mean_conv1' in fix:   # round-1 fixtures
        torch.testing.assert_close(sd['conv1.layer.1.running_mean'], fix['running_mean_conv1'], rtol=1e-5, atol=1e-6)
    for k, v in fix.get('buffers', {}).items():
        torch.testing.assert_close(sd[k], v, rtol=1e-5, atol=1e-6)
    with torch.no_grad():
        ev = make_golden.oracle_run(fam, arch, kw, sd, fix['x'], fix['y'], training=False)
    if fam == 'detr':
        torch.testing.assert_close(ev[1], fix['eval_reg'], rtol=1e-4, atol=1e-4)
        ev = ev[0]
    assert_output_close(fix, 'eval_logits', ev, rtol=1e-4, atol=1e-4)


def test_golden_fixtures_cover_every_built_family():
    fams = {load_fixture(p)['family'] for p in GOLDEN}
    assert {'resnet', 'vit', 'darknet', 'van', 'sam', 'detr'} <= fams, fams
