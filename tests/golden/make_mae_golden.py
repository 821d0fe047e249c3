"""Generates tests/golden/mae_b2_64px.ptm by running the REFERENCE's VITMAEPretrainModel + MSELoss
(SimpleAICV/masked_image_modeling/models/vit_mae.py, losses.py; imported from the oracle/_ref copy) on a small
seeded case: ViT-B encoder width / decoder width 512 with 2 + 2 blocks, 64 px images (16 patches, 4 kept).  The masking
noise is drawn once here and injected by replacing torch.rand for the duration of the reference forward, so that the
reference's own random_masking code runs on known draws.  Stored: input, noise, prediction, mask, loss, gradient digests.

    python tests/golden/make_mae_golden.py
"""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from baseline import ref_import  # noqa: E402

CFG = dict(patch_size=16, image_size=64, encoder_embedding_planes=768, encoder_block_nums=2, encoder_head_nums=12,
           decoder_embedding_planes=512, decoder_block_nums=2, decoder_head_nums=16)
SEED, BATCH = 5, 2


def reference_run(x, noise):
    ref_import._ensure_path()
    from SimpleAICV.masked_image_modeling.losses import MSELoss
    from SimpleAICV.masked_image_modeling.models.vit_mae import VITMAEPretrainModel
    torch.manual_seed(SEED)
    model = VITMAEPretrainModel(**CFG).train()
    real_rand = torch.rand
    torch.rand = lambda *a, **k: noise.clone()
    try:
        pred, mask = model(x)
    finally:
        torch.rand = real_rand
    loss = MSELoss()(pred, model.images_to_patch(x), mask)
    loss.backward()
    grads = {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None}
    return model, pred.detach(), mask.detach(), loss.detach(), grads


def make_inputs():
    g = torch.Generator().manual_seed(1000 + SEED)
    x = torch.randn(BATCH, 3, CFG['image_size'], CFG['image_size'], generator=g)
    n = (CFG['image_size'] // CFG['patch_size']) ** 2
    noise = torch.rand(BATCH, n, generator=g)
    return x, noise


def main():
    torch.set_num_threads(1)
    x, noise = make_inputs()
    model, pred, mask, loss, grads = reference_run(x, noise)
    from oracle import mae
    sd = mae.init_state('vit_base_patch16_224_mae_pretrain_model', SEED, image_size=CFG['image_size'], enc_depth=2, dec_depth=2)
    ref_sd = model.state_dict()
    assert list(ref_sd.keys()) == list(sd.keys()), 'state_dict key order differs'
    for k in ref_sd:
        assert torch.equal(ref_sd[k], sd[k]), f'seeded init differs at {k}'
    fix = {'cfg': CFG, 'seed': SEED, 'x': x, 'noise': noise, 'pred': pred, 'mask': mask, 'loss': loss,
           'grad_norm': {n: g.norm().item() for n, g in grads.items()}, 'grad_head': {n: g.flatten()[:4].clone() for n, g in grads.items()},
           'state_keys': list(ref_sd.keys())}
    out = os.path.join(HERE, 'mae_b2_64px.ptm')
    torch.save(fix, out)
    print('wrote', out, 'loss', float(loss), 'params with grad', len(grads))


if __name__ == '__main__':
    main()
