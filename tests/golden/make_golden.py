"""Generates tests/golden/*.pt by running the REFERENCE itself (imported from the
oracle/_ref copy, see baseline/ref_import.py).  The fixtures are small: the seeded input
batch (or just its seed + a digest for the larger inputs), the logits / feature digest, the loss and
per-parameter gradient digests (L2 norm + first 4 values); the weights are not stored because the
oracle reproduces the reference's seeded initialisation exactly (checked here, bit for bit).

    python tests/golden/make_golden.py [tag-substring]     # rewrites the (matching) fixtures
"""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
from baseline import ref_import  # noqa: E402
from make_reference_snapshots import take  # noqa: E402

SAMPLED_NUMEL = 65536      # outputs larger than this are stored at SAMPLE_K fixed positions plus their L2 norm (files < 1 MB)
SAMPLE_K = 8192

# (tag, family, arch, kwargs, num_classes, batch shape, seed, store_x)
CASES = [
    ('resnet18cifar_c100_b8', 'resnet', 'resnet18cifar', {}, 100, (8, 3, 32, 32), 0, True),  # BASELINE config #1 shape
    ('resnet50_c1000_b4_64px', 'resnet', 'resnet50', {}, 1000, (4, 3, 64, 64), 0, True),
    ('resnet18_c10_b2_64px', 'resnet', 'resnet18', {}, 10, (2, 3, 64, 64), 3, True),
    ('vit_base_patch16_c10_b2_64px_cls', 'vit', 'vit_base_patch16', {'image_size': 64, 'global_pool': False}, 10, (2, 3, 64, 64), 4, True),
    ('vit_base_patch16_c10_b2_64px_gap', 'vit', 'vit_base_patch16', {'image_size': 64, 'global_pool': True}, 10, (2, 3, 64, 64), 4, True),
    ('vit_base_patch16_c1000_b1_224px_gap', 'vit', 'vit_base_patch16', {'image_size': 224, 'global_pool': True}, 1000, (1, 3, 224, 224), 1, False),
    ('darknet53_c10_b2_64px', 'darknet', 'darknet53', {}, 10, (2, 3, 64, 64), 2, True),
    ('darknet19_c10_b2_64px', 'darknet', 'darknet19', {}, 10, (2, 3, 64, 64), 2, True),
    ('darknettiny_c10_b2_64px', 'darknet', 'darknettiny', {}, 10, (2, 3, 64, 64), 2, True),
    ('van_b0_c10_b2_64px', 'van', 'van_b0', {}, 10, (2, 3, 64, 64), 6, True),
    ('van_b1_c10_b1_64px', 'van', 'van_b1', {}, 10, (1, 3, 64, 64), 7, True),
    # SAM ViT image encoder (windowed 14x14 blocks with padding 20 -> 28, one global block, rel-pos tables and pos_embed
    # randomised with seed 100 + seed so that they matter); num_classes unused; loss = mean(out * proj)
    ('sam_enc_e128_h2_b3_320px', 'sam', 'ViTImageEncoder',
     {'image_size': 320, 'patch_size': 16, 'embedding_planes': 128, 'block_nums': 3, 'head_nums': 2, 'out_planes': 256,
      'window_size': 14, 'global_attn_indexes': (1,)}, 0, (1, 3, 320, 320), 8, False),
    # DETR (detection/models/detr.py): 6 + 6 transformer layers, 100 queries, padded right / bottom borders so that the
    # additive key-padding bias matters; dropout set to 0 on the reference; outputs = (cls, reg), loss = oracle.detr.surrogate_loss
    ('resnet18_detr_b2_128x160', 'detr', 'resnet18_detr', {}, 80, (2, 3, 128, 160), 3, False),
]


def sam_randomize(tensors, seed):
    """Deterministic non-zero values for the zero-initialised pos_embed / rel_pos tables (dict name -> tensor, in place)."""
    g = torch.Generator().manual_seed(100 + seed)
    for n in sorted(tensors):
        if 'rel_pos' in n or n == 'pos_embed':
            tensors[n].copy_(torch.randn(tensors[n].shape, generator=g) * 0.2)


def sam_proj(shape, out_planes, grid, seed):
    return torch.randn(shape[0], out_planes, grid, grid, generator=torch.Generator().manual_seed(500 + seed))


def detr_masks(shape):
    """Deterministic padding masks [B, H, W] (True = padding): image b keeps the top-left (H - 32 b') x (W - 40 b'') part."""
    b, _, h, w = shape
    m = torch.zeros(b, h, w, dtype=torch.bool)
    for i in range(b):
        if i % 2 == 0:
            m[i, :, w - 40:] = True
        else:
            m[i, h - 32:, :] = True
    return m


def detr_disable_dropout(model):
    for mod in model.modules():
        if isinstance(mod, torch.nn.Dropout):
            mod.p = 0.0
        if isinstance(mod, torch.nn.MultiheadAttention):
            mod.dropout = 0.0


def oracle_init(family, arch, kwargs, nc, seed):
    """The oracle's seeded initial state for a fixture (shared with tests/test_oracle_golden.py)."""
    if family == 'resnet':
        from oracle import convnets
        return convnets.init_state(arch, nc, seed)
    if family == 'vit':
        from oracle import vit
        return vit.init_state(arch, nc, seed, image_size=kwargs['image_size'])
    if family == 'darknet':
        from oracle import darknet
        return darknet.init_state(nc, seed, arch=arch)
    if family == 'van':
        from oracle import van
        return van.init_state(arch, nc, seed)
    if family == 'sam':
        from oracle import sam_encoder
        k = kwargs
        sd = sam_encoder.init_state(seed, k['image_size'], k['patch_size'], k['embedding_planes'], k['block_nums'], k['head_nums'], 4,
                                    k['out_planes'], k['window_size'], k['global_attn_indexes'])
        return sd
    if family == 'detr':
        from oracle import detr
        return detr.init_state(arch, seed, num_classes=nc)
    raise KeyError(family)


def oracle_run(family, arch, kwargs, sd, x, y, training=True):
    """(logits, loss, grads) from the oracle in training mode, or eval logits."""
    from oracle import train_step
    if family == 'resnet':
        from oracle import convnets
        if training:
            return train_step.loss_and_grads(sd, x, y, arch)
        return convnets.forward(sd, x, arch, training=False)
    if family == 'vit':
        from oracle import vit
        if training:
            return vit.loss_and_grads(sd, x, y, arch, global_pool=kwargs['global_pool'])
        return vit.forward(sd, x, arch, global_pool=kwargs['global_pool'])
    if family == 'darknet':
        from oracle import darknet
        if training:
            return darknet.loss_and_grads(sd, x, y, arch=arch)
        return darknet.forward(sd, x, training=False, arch=arch)
    if family == 'van':
        from oracle import van
        if training:
            return van.loss_and_grads(sd, x, y, arch)
        return van.forward(sd, x, arch, training=False)
    if family == 'sam':
        from oracle import sam_encoder
        k = kwargs
        if training:
            return sam_encoder.loss_and_grads(sd, x, y, k['head_nums'], k['window_size'], k['global_attn_indexes'], k['patch_size'])
        return sam_encoder.forward(sd, x, k['head_nums'], k['window_size'], k['global_attn_indexes'], k['patch_size'])
    if family == 'detr':
        from oracle import detr
        masks = detr_masks(tuple(x.shape))
        if training:
            cls, reg, loss, grads = detr.loss_and_grads(sd, x, masks, arch)
            return (cls, reg), loss, grads
        return detr.forward(sd, x, masks, arch, training=False)
    raise KeyError(family)


def make_input(shape, nc, seed):
    g = torch.Generator().manual_seed(1000 + seed)
    x = torch.randn(*shape, generator=g)
    y = torch.randint(0, nc, (shape[0],), generator=g)
    return x, y


def main():
    backbones = ref_import.backbones()
    CELoss = ref_import.module('SimpleAICV.classification.losses').CELoss
    only = sys.argv[1] if len(sys.argv) > 1 else ''
    torch.set_num_threads(1)  # fixed reduction order for the recorded numbers
    for tag, family, arch, kwargs, nc, shape, seed, store_x in CASES:
        if only not in tag:
            continue
        try:
            osd = oracle_init(family, arch, kwargs, nc, seed)
        except (ImportError, KeyError, TypeError) as e:
            print(tag, 'skipped (oracle not available yet):', e)
            continue
        torch.manual_seed(seed)
        if family == 'sam':
            enc = ref_import.module('SimpleAICV.interactive_segmentation.models.segment_anything.image_encoder')
            model = enc.ViTImageEncoder(**kwargs)
        elif family == 'detr':
            model = ref_import.module('SimpleAICV.detection.models').__dict__[arch](num_classes=nc, **kwargs)
            detr_disable_dropout(model)
        else:
            model = backbones.__dict__[arch](num_classes=nc, **kwargs)
        sd0 = {k: v.clone() for k, v in model.state_dict().items()}
        assert list(sd0.keys()) == list(osd.keys()), 'oracle state_dict keys != reference'
        assert all(torch.equal(sd0[k], osd[k]) for k in sd0), 'oracle init != reference init'
        x, y = make_input(shape, max(nc, 1), seed)
        model.train()
        if family == 'sam':
            with torch.no_grad():
                sam_randomize(dict(model.named_parameters()), seed)
            y = sam_proj(shape, kwargs['out_planes'], kwargs['image_size'] // kwargs['patch_size'], seed)
            logits = model(x)
            loss = (logits.float() * y).mean()
        elif family == 'detr':
            from oracle import detr as odetr
            logits, reg = model(x, detr_masks(shape))
            loss = odetr.surrogate_loss(logits, reg)
        else:
            logits = model(x)
            loss = CELoss()(logits, y)
        loss.backward()
        fix = {
            'family': family, 'arch': arch, 'kwargs': kwargs, 'num_classes': nc, 'seed': seed, 'shape': shape, 'y': y,
            'x_digest': (float(x.double().sum()), x.flatten()[:4].clone()),
            'logits': logits.detach(), 'loss': loss.detach(),
            'grad_norm': {n: p.grad.norm().item() for n, p in model.named_parameters() if p.grad is not None},
            'grad_head': {n: p.grad.flatten()[:4].clone() for n, p in model.named_parameters() if p.grad is not None},
            'buffers': dict([(k, v.clone()) for k, v in model.state_dict().items() if k.endswith('running_mean')][:2]),
            'torch_version': torch.__version__,
            'reference_commit': '14b1826',
        }
        if store_x:
            fix['x'] = x
        model.eval()
        with torch.no_grad():
            if family == 'detr':
                fix['reg'] = reg.detach()
                fix['eval_logits'], fix['eval_reg'] = [t.clone() for t in model(x, detr_masks(shape))]
            else:
                fix['eval_logits'] = model(x).clone()
        if family == 'sam':
            del fix['y']           # regenerated from the seed (sam_proj)
        for k in ('logits', 'eval_logits'):
            if fix[k].numel() > SAMPLED_NUMEL:
                fix.setdefault('sampled', {})[k] = (SAMPLE_K, fix[k].double().norm().item())
                fix[k] = take(fix[k], SAMPLE_K)
        torch.save(fix, os.path.join(HERE, tag + '.pt'))
        print(tag, 'loss', float(loss), os.path.getsize(os.path.join(HERE, tag + '.pt')), 'bytes')


if __name__ == '__main__':
    main()
