"""MAE pre-training (SURVEY.md 8 f4): the oracle (oracle/mae.py) replays outputs of the REFERENCE's VITMAEPretrainModel +
MSELoss (tests/golden/mae_b2_64px.ptm, made by tests/golden/make_mae_golden.py), matches the reference's state dict and
gradients (tests/golden/reference_snapshots.pts), and the B200 module shell has the reference's state_dict and seeded initialisation.  CPU only."""
import importlib.util
import os

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ARCH = 'vit_base_patch16_224_mae_pretrain_model'

_spec = importlib.util.spec_from_file_location('make_mae_golden', os.path.join(HERE, 'golden', 'make_mae_golden.py'))
gen = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(gen)
_spec = importlib.util.spec_from_file_location('make_reference_snapshots', os.path.join(HERE, 'golden', 'make_reference_snapshots.py'))
snap = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(snap)


def _fixture():
    return torch.load(os.path.join(HERE, 'golden', 'mae_b2_64px.ptm'), weights_only=False)


def test_oracle_reproduces_reference_mae_outputs():
    from oracle import mae
    fix = _fixture()
    torch.set_num_threads(1)
    sd = mae.init_state(ARCH, fix['seed'], image_size=fix['cfg']['image_size'], enc_depth=2, dec_depth=2)
    assert list(sd.keys()) == fix['state_keys']
    pred, mask, loss, grads = mae.loss_and_grads(sd, fix['x'], fix['noise'], ARCH, enc_depth=2, dec_depth=2)
    assert torch.equal(mask, fix['mask'])                      # index work: bit exact
    assert int(mask.sum()) == fix['x'].shape[0] * 12           # 16 patches, 4 kept per image
    torch.testing.assert_close(pred, fix['pred'], rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(loss, fix['loss'], rtol=1e-5, atol=1e-6)
    assert set(grads) == set(fix['grad_norm'])
    for n, g in grads.items():
        assert abs(g.norm().item() - fix['grad_norm'][n]) <= 1e-4 * max(1.0, fix['grad_norm'][n]), n
        torch.testing.assert_close(g.flatten()[:4], fix['grad_head'][n], rtol=1e-4, atol=1e-6)


def test_oracle_matches_live_reference_mae():
    from oracle import mae
    ref = snap.load()['mae']
    torch.set_num_threads(1)
    x, noise = gen.make_inputs()
    sd = mae.init_state(ARCH, gen.SEED, image_size=gen.CFG['image_size'], enc_depth=2, dec_depth=2)
    snap.check_state(ref['state'], sd)
    opred, omask, oloss, ograds = mae.loss_and_grads(sd, x, noise, ARCH, enc_depth=2, dec_depth=2)
    assert torch.equal(omask, ref['mask'])
    snap.check_close(ref['pred'], {'pred': opred}, rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(oloss, ref['loss'], rtol=1e-5, atol=1e-6)
    snap.check_close(ref['grads'], ograds, rtol=1e-4, atol=1e-6)


@pytest.mark.parametrize('kw', [dict(image_size=64, enc=2, dec=2), dict(image_size=32, enc=1, dec=3)])
def test_b200_mae_constructor_matches_reference_layout_and_seeded_init(kw):
    from oracle import mae
    from simpleaicv_pytorch_training_examples_b200.masked_image_modeling.models import vit_mae
    torch.manual_seed(3)
    m = vit_mae.VITMAEPretrainModel(patch_size=16, image_size=kw['image_size'], encoder_embedding_planes=768,
                                    encoder_block_nums=kw['enc'], encoder_head_nums=12, decoder_embedding_planes=512,
                                    decoder_block_nums=kw['dec'], decoder_head_nums=16)
    sd = mae.init_state(ARCH, 3, image_size=kw['image_size'], enc_depth=kw['enc'], dec_depth=kw['dec'])
    msd = m.state_dict()
    assert list(msd.keys()) == list(sd.keys())
    for k in sd:
        assert torch.equal(msd[k], sd[k]), k
    assert not m.encoder.pos_embed.requires_grad and not m.decoder.pos_embed.requires_grad
    assert set(vit_mae.__all__) == {'vit_base_patch16_224_mae_pretrain_model', 'vit_large_patch16_224_mae_pretrain_model',
                                    'vit_huge_patch14_224_mae_pretrain_model'}
    x = torch.randn(1, 3, kw['image_size'], kw['image_size'])
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        m(x)
    p = m.images_to_patch(x)
    assert torch.equal(m.patch_to_images(p), x)
