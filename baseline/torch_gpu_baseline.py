"""The target north_star names: the UNMODIFIED reference training loop under torch DDP on this box.

Everything on the timed path is the reference's own code imported from oracle/_ref (oracle/install_ref.sh):
``backbones.__dict__[name]`` builds the model, ``tools.utils.set_seed / build_optimizer / Scheduler /
build_training_mode`` (DistributedDataParallel + GradScaler) prepare it and ``tools.scripts.train_classification``
runs the steps — host syncs, per-step barrier and all (tools/scripts.py:141-270).  Only the data is synthetic
(a list of pinned host batches standing in for the DataLoader, same {'image','label'} contract).

Variants (``--variant``):
  as_shipped  get_amp_type's whitelist lacks 'B200' -> the reference picks fp16 + GradScaler; cudnn.deterministic
  bf16        the one-line whitelist patch (get_amp_type -> bf16), otherwise as shipped         <- the x1.3 target
  tuned       bf16 + cudnn.benchmark + channels_last (NOT the reference's configuration; shown for honesty)

    torchrun --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29533 \
        baseline/torch_gpu_baseline.py --model resnet50 --variant bf16 --steps 20 --warmup 5 [--out file.jsonl]
Prints one JSON line on rank 0 (images/s whole job, device-timed between the first timed batch and the end).
"""
import argparse
import json
import logging
import os
import sys
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from baseline import ref_import  # noqa: E402


class SyntheticLoader:
    """Stands in for the DataLoader: yields the same pinned host batch ``n`` times; records a CUDA event when
    the first timed batch is handed out."""

    def __init__(self, batch, n, warmup, global_batch):
        self.batch, self.n, self.warmup = batch, n, warmup
        self.dataset = range(global_batch * n)       # len(train_loader.dataset) // config.batch_size == n
        self.start = torch.cuda.Event(enable_timing=True)
        self.t0 = None

    def __iter__(self):
        for i in range(self.n):
            if i == self.warmup:
                torch.cuda.synchronize()
                self.t0 = time.perf_counter()
                self.start.record()
            yield self.batch

    def __len__(self):
        return self.n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--model', default='resnet50', choices=['resnet50', 'vit_base_patch16'])
    ap.add_argument('--variant', default='bf16', choices=['as_shipped', 'bf16', 'tuned'])
    ap.add_argument('--batch', type=int, default=256, help='per-GPU batch')
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    rank, world, local = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1)), int(os.environ.get('LOCAL_RANK', 0))
    os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
    os.environ.setdefault('MASTER_PORT', '29533')
    os.environ.setdefault('RANK', '0')
    os.environ.setdefault('WORLD_SIZE', '1')
    torch.cuda.set_device(local)
    dist.init_process_group(backend='nccl', init_method='env://')      # tools/train_classification_model.py:51-53

    backbones = ref_import.backbones()
    ref_losses = ref_import.module('SimpleAICV.classification.losses')
    ref_utils = ref_import.module('tools.utils')
    ref_scripts = ref_import.module('tools.scripts')

    ref_utils.set_seed(0)                                                # cudnn.deterministic=True, benchmark=False
    if a.variant != 'as_shipped':
        ref_scripts.get_amp_type = lambda model: torch.bfloat16         # == adding 'B200' to the whitelist
    if a.variant == 'tuned':
        torch.backends.cudnn.benchmark, torch.backends.cudnn.deterministic = True, False

    class config:
        pass
    config.local_rank, config.gpus_num, config.group = local, world, dist.new_group(list(range(world)))
    config.batch_size = a.batch * world
    config.accumulation_steps, config.print_interval = 1, 10 ** 9
    config.use_amp, config.sync_bn, config.use_ema_model, config.use_compile = True, False, False, False
    config.epochs = 100
    g = torch.Generator().manual_seed(1234 + rank)
    x = torch.randn(a.batch, 3, 224, 224, generator=g)
    if a.model == 'resnet50':
        # 00.classification_training/imagenet/resnet50/train_config.py:29-31,66-91
        model = backbones.resnet50(num_classes=1000)
        criterion = ref_losses.CELoss()
        config.optimizer = ('SGD', {'lr': 0.1, 'momentum': 0.9, 'global_weight_decay': False, 'weight_decay': 1e-4,
                                    'no_weight_decay_layer_name_list': []})
        config.scheduler = ('MultiStepLR', {'warm_up_epochs': 0, 'gamma': 0.1, 'milestones': [30, 60, 90]})
        y = torch.randint(0, 1000, (a.batch,), generator=g)
    else:
        # .../vit_base_patch16_for_self_train_mae_pretrain/train_config.py:26-124 (BASELINE configs[2])
        model = backbones.vit_base_patch16(image_size=224, num_classes=1000, drop_path_prob=0.1, global_pool=True)
        criterion = ref_losses.OneHotLabelCELoss()
        config.optimizer = ('AdamW', {'lr': 5e-4, 'global_weight_decay': False, 'weight_decay': 0.05,
                                      'no_weight_decay_layer_name_list': ['position_encoding', 'cls_token'],
                                      'lr_layer_decay': 0.65, 'lr_layer_decay_block': model.blocks, 'block_name': 'blocks'})
        config.scheduler = ('CosineLR', {'warm_up_epochs': 5, 'min_lr': 1e-6})
        lab = torch.randint(0, 1000, (a.batch,), generator=g)
        oh = torch.nn.functional.one_hot(lab, 1000).float() * 0.9 + 0.1 / 1000
        y = 0.5 * oh + 0.5 * oh.roll(1, 0)
    model = model.cuda()
    criterion = criterion.cuda()
    if a.variant == 'tuned':
        model = model.to(memory_format=torch.channels_last)
        x = x.contiguous(memory_format=torch.channels_last)
    optimizer, _ = ref_utils.build_optimizer(config, model)
    scheduler = ref_utils.Scheduler(config, optimizer)
    model, config.ema_model, config.scaler = ref_utils.build_training_mode(config, model)

    logger = logging.getLogger('baseline')
    logger.addHandler(logging.NullHandler())
    loader = SyntheticLoader({'image': x.pin_memory(), 'label': y.pin_memory()}, a.steps + a.warmup, a.warmup, config.batch_size)
    end = torch.cuda.Event(enable_timing=True)
    loss = ref_scripts.train_classification(loader, model, criterion, optimizer, scheduler, 1, logger, config)
    end.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - loader.t0
    ms = torch.tensor([loader.start.elapsed_time(end) / a.steps], device='cuda')
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    if rank == 0:
        amp = str(ref_scripts.get_amp_type(model))
        line = {'what': 'unmodified reference (oracle/_ref) under torch DDP, its own train_classification loop',
                'model': a.model, 'variant': a.variant, 'amp_type': amp, 'n_gpus': world, 'per_gpu_batch': a.batch,
                'steps': a.steps, 'warmup': a.warmup, 'ms_per_step': float(ms), 'images_per_sec': a.batch * world / float(ms) * 1e3,
                'wall_ms_per_step_rank0': wall / a.steps * 1e3, 'avg_loss': float(loss),
                'cudnn_deterministic': torch.backends.cudnn.deterministic, 'cudnn_benchmark': torch.backends.cudnn.benchmark,
                'h2d_in_timed_region': True, 'torch': torch.__version__, 'gpu': torch.cuda.get_device_name()}
        s = json.dumps(line)
        print(s, flush=True)
        if a.out:
            with open(a.out, 'a') as f:
                f.write(s + '\n')
    dist.destroy_process_group()


if __name__ == '__main__':
    main()
