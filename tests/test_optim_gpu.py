"""Fused multi-tensor optimizers (optim.py, csrc/capi_optim.cu) against torch.optim.SGD / AdamW - the optimizers the
reference builds (reference tools/utils.py:581-600) - on identical parameters and gradients: several steps with
per-group learning rates / weight decays that change every step, odd sizes and unaligned gradient views, the fused bf16
operand copies (Linear and conv tap-major layouts), the fused global-norm clip, state_dict interchange and a captured
step with a per-iteration learning rate."""
import pytest
import torch

pytestmark = pytest.mark.gpu

SHAPES = [(64, 64, 3, 3), (256, 64, 1, 1), (1000, 512), (77,), (3, 5, 7), (128, 192, 3, 3), (8192 * 3 + 5,)]


def _make(seed):
    g = torch.Generator(device='cuda').manual_seed(seed)
    ps = [torch.randn(*s, device='cuda', generator=g).requires_grad_(True) for s in SHAPES]
    return ps


def _grads(ps, step, unaligned):
    g = torch.Generator(device='cuda').manual_seed(100 + step)
    flat = torch.randn(sum(p.numel() for p in ps) + 16, device='cuda', generator=g)
    off = 1 if unaligned else 0     # bucket views of the data-parallel wrapper are only 4-byte aligned
    out = []
    for p in ps:
        out.append(flat[off:off + p.numel()].view_as(p))
        off += p.numel()
    return out


def _groups(ps):
    return [{'params': ps[:3], 'weight_decay': 1e-2, 'lr': 0.1}, {'params': ps[3:5], 'weight_decay': 0., 'lr': 0.05},
            {'params': ps[5:], 'weight_decay': 5e-2, 'lr': 0.2}]


@pytest.mark.parametrize('unaligned', [False, True])
@pytest.mark.parametrize('kind', ['sgd', 'sgd_nesterov', 'adamw'])
def test_fused_step_matches_torch(kind, unaligned):
    from simpleaicv_pytorch_training_examples_b200 import optim
    pa, pb = _make(1), _make(1)
    if kind == 'adamw':
        ref = torch.optim.AdamW(_groups(pa), lr=1e-3, betas=(0.9, 0.99), eps=1e-8)
        mine = optim.FusedAdamW(_groups(pb), lr=1e-3, betas=(0.9, 0.99), eps=1e-8)
    else:
        nest = kind == 'sgd_nesterov'
        ref = torch.optim.SGD(_groups(pa), lr=0.1, momentum=0.9, nesterov=nest)
        mine = optim.FusedSGD(_groups(pb), lr=0.1, momentum=0.9, nesterov=nest)
    # bf16 operand copies: Linear-style (padded rows) and conv tap-major with padded channels
    lin_shadow = torch.zeros(1008, 512, device='cuda', dtype=torch.bfloat16)
    mine.register_shadow(pb[2], lin_shadow)
    k, c, r, s = SHAPES[0]
    cp = 128
    conv_shadow = torch.zeros(k, r * s * cp, device='cuda', dtype=torch.bfloat16)
    mine.register_shadow(pb[0], conv_shadow, conv=(c, r * s, cp, r * s * cp))
    versions = [p._version for p in pb]
    for step in range(12):     # more steps than ring slots
        for opt in (ref, mine):
            for gi, g in enumerate(opt.param_groups):
                g['lr'] = (0.1 if kind != 'adamw' else 1e-2) * (1 + gi) * 0.9 ** step
        for p, q, g in zip(pa, pb, _grads(pa, step, unaligned)):
            p.grad, q.grad = g.clone(), g
        ref.step()
        mine.step()
    torch.cuda.synchronize()
    for i, (p, q) in enumerate(zip(pa, pb)):
        err = (p - q).abs().max().item()
        assert err <= 2e-6 * p.abs().max().item() + 1e-7, f'{kind} tensor {i}: max abs diff {err}'
    assert torch.equal(lin_shadow[:1000], pb[2].detach().to(torch.bfloat16)) and not lin_shadow[1000:].any()
    want = torch.zeros(k, r * s, cp, device='cuda')
    want[:, :, :c] = pb[0].detach().permute(0, 2, 3, 1).reshape(k, r * s, c)
    assert torch.equal(conv_shadow.view(k, r * s, cp), want.to(torch.bfloat16))
    # parameters with a fused copy keep their version (the runtime's prep() skips them); the others are bumped
    assert pb[0]._version == versions[0] and pb[2]._version == versions[2]
    assert pb[1]._version > versions[1] and pb[3]._version > versions[3]
    # state interchange with torch.optim
    sd = mine.state_dict()
    ref2 = torch.optim.AdamW(_groups(pa), lr=1e-3, betas=(0.9, 0.99)) if kind == 'adamw' else torch.optim.SGD(_groups(pa), lr=0.1, momentum=0.9)
    ref2.load_state_dict(sd)
    key = 'exp_avg' if kind == 'adamw' else 'momentum_buffer'
    for p, q in zip(pa, pb):
        a, b = ref.state[p][key], mine.state[q][key]
        assert (a - b).abs().max().item() <= 4e-6 * a.abs().max().item() + 1e-7
        assert torch.equal(ref2.state[p][key], mine.state[q][key])
    if kind == 'adamw':
        assert float(ref2.state[pa[0]]['step']) == 12.
    # resume: load torch.optim's state into the fused optimizer in the middle of a run (the loader replaces the state
    # tensors, so the device table must follow) and keep stepping in lockstep
    # (deep copy: torch's loader keeps tensors that already have the parameter's dtype / device, i.e. it would ALIAS the two
    # optimizers' momentum buffers; a checkpoint read with torch.load never aliases)
    import copy
    mine.load_state_dict(copy.deepcopy(ref.state_dict()))
    for step in range(12, 15):
        for opt in (ref, mine):
            for gi, g in enumerate(opt.param_groups):
                g['lr'] = (0.1 if kind != 'adamw' else 1e-2) * (1 + gi) * 0.9 ** step
        for p, q, g in zip(pa, pb, _grads(pa, step, unaligned)):
            p.grad, q.grad = g.clone(), g
        ref.step()
        mine.step()
    torch.cuda.synchronize()
    for i, (p, q) in enumerate(zip(pa, pb)):
        err = (p - q).abs().max().item()
        assert err <= 1e-5 * p.abs().max().item() + 1e-7, f'{kind} after resume, tensor {i}: max abs diff {err}'


def test_fused_clip_matches_clip_grad_norm():
    from simpleaicv_pytorch_training_examples_b200 import optim
    pa, pb = _make(2), _make(2)
    ref = torch.optim.SGD(_groups(pa), lr=0.1, momentum=0.9)
    mine = optim.FusedSGD(_groups(pb), lr=0.1, momentum=0.9)
    for step in range(3):
        for p, q, g in zip(pa, pb, _grads(pa, step, False)):
            p.grad, q.grad = g.clone() * 3, g.clone() * 3
        n_ref = torch.nn.utils.clip_grad_norm_(pa, 0.5)
        n_mine = mine.clip_grad_norm(0.5)
        assert abs(float(n_ref) - float(n_mine)) <= 1e-5 * float(n_ref)
        ref.step()
        mine.step()
    for p, q in zip(pa, pb):
        assert (p - q).abs().max().item() <= 2e-6 * p.abs().max().item() + 1e-7
    # a step without clip after clipped ones uses the raw gradients again
    for p, q, g in zip(pa, pb, _grads(pa, 9, False)):
        p.grad, q.grad = g.clone(), g.clone()
    ref.step()
    mine.step()
    for p, q in zip(pa, pb):
        assert (p - q).abs().max().item() <= 2e-6 * p.abs().max().item() + 1e-7


def test_captured_step_follows_the_learning_rate_schedule():
    """The step is captured ONCE; learning rates rewritten in param_groups between replays (tools.utils.Scheduler does
    that every iteration) reach the kernel through the pinned ring: results equal an eager torch.optim run."""
    from simpleaicv_pytorch_training_examples_b200 import optim
    pa, pb = _make(3), _make(3)
    ref = torch.optim.AdamW(_groups(pa), lr=1e-3)
    mine = optim.FusedAdamW(_groups(pb), lr=1e-3)
    static_g = [torch.zeros_like(p) for p in pb]
    for q, g in zip(pb, static_g):
        q.grad = g
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    lrs = [1e-2 * 0.8 ** i for i in range(14)]

    def set_lr(opt, lr):
        for gi, g in enumerate(opt.param_groups):
            g['lr'] = lr * (1 + gi)

    def feed(step):
        for p, sg, g in zip(pa, static_g, _grads(pa, step, False)):
            p.grad = g.clone()
            sg.copy_(g)

    with torch.cuda.stream(side):   # two eager warm-up steps, like graph.GraphedTrainStep
        for step in range(2):
            set_lr(ref, lrs[step]); set_lr(mine, lrs[step])
            feed(step)
            ref.step(); mine.step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        mine.step()
    for step in range(2, 14):
        set_lr(ref, lrs[step]); set_lr(mine, lrs[step])
        feed(step)
        ref.step()
        mine.sync_hyper()
        graph.replay()
        mine.after_replay()
    torch.cuda.synchronize()
    for i, (p, q) in enumerate(zip(pa, pb)):
        assert (p - q).abs().max().item() <= 3e-6 * p.abs().max().item() + 1e-7, f'tensor {i}'


def test_build_optimizer_fuses_the_runtime_operand_copies():
    """tools.utils.build_optimizer on a CUDA model returns the fused optimizer with the runtime's bf16 weight copies
    attached: after a training step the copies equal a fresh cast of the updated parameters, and the next forward
    launches no cast / re-layout kernel for them."""
    from simpleaicv_pytorch_training_examples_b200 import _lib, optim
    from simpleaicv_pytorch_training_examples_b200.classification import backbones, losses
    from simpleaicv_pytorch_training_examples_b200.tools import utils as tutils

    class Cfg:
        optimizer = ('SGD', {'lr': 0.1, 'momentum': 0.9, 'global_weight_decay': False, 'weight_decay': 1e-4,
                             'no_weight_decay_layer_name_list': []})
    torch.manual_seed(0)
    model = backbones.resnet18cifar(num_classes=10).cuda().train()
    opt, _ = tutils.build_optimizer(Cfg, model)
    assert isinstance(opt, optim.FusedSGD) and len(opt._shadows) >= 20
    x = torch.randn(8, 3, 32, 32, device='cuda')
    y = torch.randint(0, 10, (8,), device='cuda')
    crit = losses.CELoss()
    for _ in range(2):
        crit(model(x), y).backward()
        opt.step()
        opt.zero_grad()
    rt = model._runtime()
    units = [u for u in rt.units() if not u.is_stem]
    for u in units:
        fresh = torch.empty_like(u.w_bf16)
        from simpleaicv_pytorch_training_examples_b200 import ops
        ops.prep_conv_weight(u.conv.weight.detach(), fresh, u.kpad, order=ops.ORDER_RSC, kp=u.kp, cp=u.cp)
        assert torch.equal(fresh, u.w_bf16)
    n0 = _lib.launch_count()
    rt.prep()
    torch.cuda.synchronize()
    assert _lib.launch_count() - n0 <= 2, 'prep() re-cast weights the optimizer had already refreshed'
    # and the fused run equals torch.optim.SGD on the same model / data
    torch.manual_seed(0)
    ref_model = backbones.resnet18cifar(num_classes=10).cuda().train()
    Cfg.optimizer[1]['fused'] = False
    ropt, _ = tutils.build_optimizer(Cfg, ref_model)
    assert isinstance(ropt, torch.optim.SGD)
    for _ in range(2):
        crit(ref_model(x), y).backward()
        ropt.step()
        ropt.zero_grad()
    for (n, p), q in zip(model.named_parameters(), ref_model.parameters()):
        assert (p - q).abs().max().item() <= 1e-5 * q.abs().max().item() + 1e-7, n
