#!/usr/bin/env python
"""bench.py — images/sec of the SimpleAICV classification training step on B200.

Headline workload (BASELINE.json configs[1]): ResNet-50, 224x224, batch 256 per GPU, synthetic images,
CELoss, SGD(lr 0.1, momentum 0.9, wd 1e-4, 1-D params undecayed) — one "step" is forward + loss +
backward (+ bucketed gradient all-reduce when N > 1) + optimizer step, exactly the work of
tools/scripts.py:141-270 in the reference.  The same JSON line carries a ``vit_base_patch16`` sub-record
(BASELINE configs[2]: ViT-B/16, soft labels, AdamW with layer-wise lr decay) measured the same way.

  python bench.py [--gpus N] [--steps K] [--warmup W]     our arm (sm_100a kernels)
  python bench.py --impl reference ...                    reference arm: the reference's step arithmetic on the
                                                          host cores (the oracle port, fp32)
  python bench.py ... --dump-outputs DIR                  also write what the last timed step computed as DIR/*.npy
Every timed loop runs K steps.  Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for what every key means.
"""
import argparse
import contextlib
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

METRICS = {'resnet50': 'images/sec (ResNet-50 224x224 training step, whole job)',
           'vit_base_patch16': 'images/sec (ViT-B/16 224x224 training step, whole job)',
           'sam_h_encoder': 'images/sec (SAM ViT-H image encoder 1024x1024 training step, whole job)',
           'resnet50_detr': 'images/sec (DETR-R50 1024x1024 training step, whole job)',
           'vit_base_mae': 'images/sec (MAE ViT-B/16 224x224 pre-training step, whole job)'}
WORKLOADS = {'resnet50': 'ResNet-50 224x224 bs256/GPU training step (fwd+CELoss+bwd+grad all-reduce+SGD)',
             'vit_base_patch16': 'ViT-B/16 224x224 bs256/GPU training step (fwd+OneHotLabelCELoss+bwd+grad all-reduce+AdamW)',
             'sam_h_encoder': ('SAM ViT-H image encoder 1024x1024 bs8/GPU training step (encoder fwd + feature MSE against a synthetic '
                               'teacher map, the train_distill_sam_encoder step body + bwd + grad all-reduce + AdamW); prompt encoder / '
                               'mask decoder are outside the built path'),
             'resnet50_detr': ('DETR-R50 1024x1024 bs4/GPU training step (the shipped res50_detr_yoloresize1024 shape; fwd + DETRLoss with the '
                               'Hungarian matcher on the host + bwd + grad all-reduce + AdamW; dropout 0.1 as in the reference constructor)'),
             'vit_base_mae': ('MAE pre-training, vit_base_patch16_224_mae_pretrain_model 224x224 bs256/GPU (75 % of the patches masked: encoder on '
                              '50 tokens, 8-block 512-wide decoder on 197; fwd + MSELoss on removed patches + bwd + grad all-reduce + AdamW)')}
FWD_FLOPS = {'resnet50': 8.178e9, 'vit_base_patch16': 35.13e9, 'sam_h_encoder': 5961e9, 'resnet50_detr': 191.6e9,
             'vit_base_mae': 19.6e9}   # MAE: from the layer shapes (encoder 50 tokens x 12 blocks, decoder 197 tokens x 8 blocks)
FWD_FLOPS_NOTE = 'per image forward (SURVEY.md 8d); a step is 3x'
ALGO_BYTES = {'resnet50': 130e6, 'vit_base_patch16': 3 * 65e6, 'sam_h_encoder': 3 * 3.1e9, 'resnet50_detr': 130e6 * 20.9, 'vit_base_mae': 3 * 40e6}  # per image per step, activations once each way (8d)


def _peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return {'hbm_gbs': d['hbm_gbs'], 'tf_burst': d['bf16_tflops'], 'tf_sustained': d.get('bf16_tflops_sustained', d['bf16_tflops']),
                'source': 'measured'}
    return {'hbm_gbs': 6650.0, 'tf_burst': 1590.0, 'tf_sustained': 1400.0, 'source': 'fallback'}


def _traffic():
    """DRAM traffic per launch of the dominant kernel from the committed ncu --set full capture
    (profiles/r02_traffic.json, written by tests/summarize_profiles.py from the .ncu-rep)."""
    p = os.path.join(ROOT, 'profiles', 'r02_traffic.json')
    return json.load(open(p)) if os.path.exists(p) else None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.path = tempfile.mktemp(suffix='.csv')
        self.proc = None
        self.idx = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.idx), f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-lms', '200'], stdout=open(self.path, 'w'), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], 0, set()
        for line in open(self.path):
            f = [t.strip() for t in line.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx = max(mx, float(f[2]))
            except ValueError:
                continue
            for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[5:9]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': mx or None, 'reasons': sorted(reasons),
                'samples': len(sm)}


def vit_optimizer_cfg(model, capturable=False):
    class _Cfg:
        optimizer = ('AdamW', {'lr': 5e-4, 'global_weight_decay': False, 'weight_decay': 0.05,
                               'no_weight_decay_layer_name_list': ['position_encoding', 'cls_token'],
                               'lr_layer_decay': 0.65, 'lr_layer_decay_block': model.blocks, 'block_name': 'blocks',
                               'capturable': capturable})
    return _Cfg


def r50_optimizer_cfg():
    class _Cfg:
        optimizer = ('SGD', {'lr': 0.1, 'momentum': 0.9, 'global_weight_decay': False, 'weight_decay': 1e-4,
                             'no_weight_decay_layer_name_list': []})
    return _Cfg


def synthetic_batch(model_name, B, rank, pin):
    g = torch.Generator().manual_seed(1234 + rank)
    if model_name == 'resnet50_detr':   # images + [B, 8, 5] boxes (cx, cy, w, h, class) normalised, no padding rows
        x = torch.randn(B, 3, 1024, 1024, generator=g)
        y = torch.cat([torch.rand(B, 8, 2, generator=g) * 0.6 + 0.2, torch.rand(B, 8, 2, generator=g) * 0.3 + 0.05,
                       torch.randint(0, 80, (B, 8, 1), generator=g).float()], dim=2)
        return (x.pin_memory(), y.pin_memory()) if pin else (x, y)
    if model_name == 'sam_h_encoder':   # student image + teacher feature map (train_distill_sam_encoder's tensors)
        x = torch.randn(B, 3, 1024, 1024, generator=g)
        y = torch.randn(B, 256, 64, 64, generator=g)
        return (x.pin_memory(), y.pin_memory()) if pin else (x, y)
    x = torch.randn(B, 3, 224, 224, generator=g)
    if model_name == 'vit_base_mae':   # label = the patchified image (MAESelfSupervisedPretrainCollater's tensors)
        y = torch.einsum('nchpwq->nhwpqc', x.reshape(B, 3, 14, 16, 14, 16)).reshape(B, 196, 768).contiguous()
        return (x.pin_memory(), y.pin_memory()) if pin else (x, y)
    if model_name == 'resnet50':
        y = torch.randint(0, 1000, (B,), generator=g)
    else:  # mixup-style soft labels (SURVEY.md 8d C3)
        lab = torch.randint(0, 1000, (B,), generator=g)
        oh = torch.nn.functional.one_hot(lab, 1000).float() * 0.9 + 0.1 / 1000
        y = 0.5 * oh + 0.5 * oh.roll(1, 0)
    return (x.pin_memory(), y.pin_memory()) if pin else (x, y)


# --------------------------------------------------------------------------------------------
def cpu_reference_step_times(model_name, batch, warmup, steps, threads):
    """The reference's CPU path on the host cores: the oracle port of the reference's model code (oracle/, pinned to
    the reference by tests/golden) driven through the arithmetic of one tools/scripts.py:141-270 step in fp32 (its
    entry points hard-require CUDA/NCCL, SURVEY.md 0.6).  Returns (kind, [seconds per step])."""
    torch.set_num_threads(threads)
    _retain_freed_host_memory()
    x, y = synthetic_batch(model_name, batch, 0, False)
    kind = 'port'
    from oracle import convnets, train_step, vit
    sd = convnets.init_state('resnet50', 1000, 0) if model_name == 'resnet50' else vit.init_state(model_name, 1000, 0)
    buf = {}

    def step():
        if model_name == 'resnet50':
            _, loss, grads = train_step.loss_and_grads(sd, x, y, 'resnet50')
        else:
            _, loss, grads = vit.loss_and_grads(sd, x, y, model_name, global_pool=True)
        train_step.sgd_step(sd, grads, buf, 0.1)
        return float(loss)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        step()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    return kind, times


def _retain_freed_host_memory():
    """glibc returns the multi-GB activation buffers of every CPU step to the kernel and page-faults them
    back in on the next one (round 1: 22x run-to-run spread, most of it system time).  Raising the
    trim / mmap thresholds keeps freed blocks in the process, which makes step times repeatable
    (measured here: 1.5-4.3 s/step -> 1.0-1.3 s/step for ResNet-50 batch 16 on 8 cores)."""
    try:
        import ctypes
        libc = ctypes.CDLL('libc.so.6')
        libc.mallopt(-1, 2 ** 31 - 1)   # M_TRIM_THRESHOLD
        libc.mallopt(-3, 2 ** 31 - 1)   # M_MMAP_THRESHOLD
    except Exception:
        pass


def host_threads():
    """min(32, physical cores): more threads than that made the fp32 CPU step slower and unstable in round 1
    (0.4 .. 9 img/s on 128 logical cores)."""
    try:
        import psutil
        phys = psutil.cpu_count(logical=False) or os.cpu_count() or 1
    except Exception:
        phys = os.cpu_count() or 1
    return max(1, min(32, phys)), phys


def cpu_baseline_record(model_name, batch, warmup, steps):
    threads, phys = host_threads()
    kind, times = cpu_reference_step_times(model_name, batch, warmup, steps, threads)
    med, best = statistics.median(times), min(times)
    return {'value': batch / med, 'unit': 'images/s', 'cores': threads, 'kind': kind,
            'value_best': batch / best, 'sec_per_step_median': med, 'sec_per_step_min': best,
            'sample': (f'{steps} timed steps of batch {batch} after {warmup} warm-ups of the same {model_name} training step '
                       f'(fwd+loss+bwd+optimizer), fp32, oracle port, '
                       f'torch {torch.__version__} CPU, {threads} threads on {phys} physical cores; median reported'),
            'physical_cores': phys}


def run_reference(args, rank):
    """--impl reference: the reference's own CPU implementation of the step (rank 0 only)."""
    if rank != 0:
        return
    batch = 16
    warmup, steps = max(2, min(args.warmup, 3)), args.steps
    cb = cpu_baseline_record(args.model, batch, warmup, steps)
    line = {
        'impl': 'reference', 'metric': METRICS[args.model], 'value': cb['value'], 'unit': 'images/s', 'n_gpus': args.gpus, 'steps': steps,
        'warmup': warmup, 'ms_per_step': cb['sec_per_step_median'] * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': WORKLOADS[args.model] + ' — bounded CPU sample: one process, batch 16 per step',
                   'per_step_batch': batch, 'same_step_arithmetic': True},
        'cpu_baseline': cb,
        'e2e': {'value': cb['value'], 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------
class OpTimer:
    """CUDA-event timing of every C-ABI call (installed around _lib.call for an instrumented pass)."""

    def __init__(self):
        self.records = []

    def install(self):
        from simpleaicv_pytorch_training_examples_b200 import _lib
        import simpleaicv_pytorch_training_examples_b200.ops as ops
        self._lib, self._ops = _lib, ops
        self._orig = _lib.call
        timer = self

        def timed(name, *a):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            rc = timer._orig(name, *a)
            e.record()
            timer.records.append((name, a, s, e))
            return rc

        _lib.call = timed
        ops._lib.call = timed

    def remove(self):
        self._lib.call = self._orig
        self._ops._lib.call = self._orig

    def summarize(self):
        torch.cuda.synchronize()
        out = {}
        for name, a, s, e in self.records:
            key, flops, nbytes = describe(name, a)
            d = out.setdefault(key, {'ms': 0.0, 'calls': 0, 'flops': 0.0, 'bytes': 0.0, 'op': name})
            d['ms'] += s.elapsed_time(e)
            d['calls'] += 1
            d['flops'] += flops
            d['bytes'] += nbytes
        return out


def _cs(a):
    return a._obj if hasattr(a, '_obj') else a


def describe(name, a):
    """(key, algorithmic flops, algorithmic bytes) of one C-ABI call from its arguments."""
    if name in ('saicv_conv_fprop', 'saicv_conv_dgrad', 'saicv_conv_wgrad'):
        cs = next(_cs(v) for v in a if hasattr(v, '_obj'))
        st = cs.stride
        P = (cs.h + 2 * cs.pad - cs.r) // st + 1
        Q = (cs.w + 2 * cs.pad - cs.s) // st + 1
        if name == 'saicv_conv_dgrad':
            P, Q = cs.h, cs.w
        pix = cs.n * P * Q
        flops = 2.0 * pix * cs.k * cs.c * cs.r * cs.s
        x_b, y_b, w_b = cs.n * cs.h * cs.w * cs.c * 2, pix * cs.k * 2, cs.k * cs.c * cs.r * cs.s * 2
        nbytes = x_b + y_b + w_b if name != 'saicv_conv_wgrad' else x_b + y_b + cs.k * cs.c * cs.r * cs.s * 4
        return f'{name[6:]} {cs.r}x{cs.s}/{st} c{cs.c} k{cs.k} {cs.h}x{cs.w}', flops, float(nbytes)
    if name == 'saicv_linear_fwd':      # (..., M, N, K, flags, out_f32, stream)
        M, N, K = a[-6], a[-5], a[-4]
        return f'linear_fwd M{M} N{N} K{K}', 2.0 * M * N * K, 2.0 * (M * K + N * K + M * N)
    if name == 'saicv_linear_dgrad':    # (..., M, N, K, flags, out_f32, stream)
        M, N, K = a[-6], a[-5], a[-4]
        return f'linear_dgrad M{M} N{N} K{K}', 2.0 * M * N * K, 2.0 * (M * K + N * K + M * N)
    if name == 'saicv_linear_wgrad':    # (dy, x, dw, M, N, K, splits, stream)
        M, N, K = a[-5], a[-4], a[-3]
        return f'linear_wgrad M{M} N{N} K{K}', 2.0 * M * N * K, 2.0 * (M * K + M * N) + 4.0 * N * K
    if name in ('saicv_attention_fwd', 'saicv_attention_bwd'):   # (..., b, l, h, d, scale, stream) + optional extras
        b, l, h, d = a[-6], a[-5], a[-4], a[-3]
        mult = 2 if name.endswith('fwd') else 5                  # QK^T, PV | + dP, dQ, dK, dV (S recomputed)
        io = (4 if name.endswith('fwd') else 9) * b * l * h * d * 2
        return f'{name[6:]} B{b} L{l} H{h} D{d}', mult * 2.0 * b * h * l * l * d, float(io)
    if name in ('saicv_attn_fwd', 'saicv_attn_bwd'):             # (byref(args struct), stream)
        st = a[0]._obj
        f = st if name.endswith('fwd') else st.fwd
        bh = f.b * f.h
        # algorithmic work: forward scores + PV; backward S (recomputed), dP, dQ, dK, dV once each (the two-phase
        # kernel recomputes S and dP a second time; that is overhead, not counted)
        macs = bh * f.lq * f.lk * ((f.dqk + f.dv) if name.endswith('fwd') else (3 * f.dqk + 2 * f.dv))
        io = bh * 2 * ((f.lq * (f.dqk + f.dv) + f.lk * (f.dqk + f.dv)) * (1 if name.endswith('fwd') else 3))
        return f'{name[6:]} BH{bh} Lq{f.lq} Lk{f.lk} dqk{f.dqk} dv{f.dv}', 2.0 * macs, float(io)
    return name[6:], 0.0, 0.0


def roofline_from_table(table, peaks, model_name, B, ms_step, dump_path=None):
    """All-launch roofline of the tensor-core engine kernels of one step (gemm_sm100_kernel + the attention
    kernels): every launch is bounded by max(FLOPs / tensor peak, algorithmic bytes / HBM peak); frac =
    sum of those roofline times / sum of the measured CUDA-event times.  The two classes are kept beside it."""
    gemm = {k: v for k, v in table.items() if v['flops'] > 0}
    tf_peak, bw_peak = peaks['tf_sustained'] * 1e12, peaks['hbm_gbs'] * 1e9
    cls = {'tensor': {'work': 0.0, 'ms': 0.0, 'roof_ms': 0.0, 'launches': 0},
           'hbm': {'work': 0.0, 'ms': 0.0, 'roof_ms': 0.0, 'launches': 0}}
    for k, v in gemm.items():
        t_t, t_h = v['flops'] / tf_peak * 1e3, v['bytes'] / bw_peak * 1e3
        c = cls['tensor'] if t_t >= t_h else cls['hbm']
        c['work'] += v['flops'] if t_t >= t_h else v['bytes']
        c['ms'] += v['ms']
        c['roof_ms'] += max(t_t, t_h)
        c['launches'] += v['calls']
        v['roof_frac'] = max(t_t, t_h) / v['ms'] if v['ms'] else 0.0
    gemm_ms = sum(v['ms'] for v in gemm.values())
    all_ms = sum(v['ms'] for v in table.values())
    dom = 'tensor' if cls['tensor']['ms'] >= cls['hbm']['ms'] else 'hbm'
    frac_all = sum(c['roof_ms'] for c in cls.values()) / gemm_ms if gemm_ms else 0.0

    def cls_rec(k):
        c = cls[k]
        if not c['ms']:
            return None
        ach = c['work'] / (c['ms'] / 1e3) / (1e12 if k == 'tensor' else 1e9)
        peak = peaks['tf_sustained'] if k == 'tensor' else peaks['hbm_gbs']
        return {'achieved': ach, 'peak': peak, 'unit': 'TFLOP/s' if k == 'tensor' else 'GB/s', 'frac': ach / peak,
                'launches': c['launches'], 'share_of_engine_time': c['ms'] / gemm_ms}
    d = cls_rec(dom)
    worst = min(gemm, key=lambda k: gemm[k]['roof_frac']) if gemm else None
    top = max(gemm, key=lambda k: gemm[k]['ms']) if gemm else None
    tr = _traffic()
    roof = {'bound': dom, 'achieved': d['achieved'] * frac_all / d['frac'] if d and d['frac'] else None, 'peak': d['peak'] if d else None,
            'unit': d['unit'] if d else None, 'frac': frac_all,
            'traffic': (tr or {}).get(model_name, {}).get('dram_bytes_per_launch'),
            'algorithmic_bytes_per_launch': (sum(v['bytes'] for v in gemm.values()) / max(1, sum(v['calls'] for v in gemm.values()))) if gemm else None,
            'traffic_note': (tr or {}).get(model_name, {}).get('note'),
            'kernel': 'gemm_sm100_kernel (+ attention kernels for ViT)',
            'frac_definition': ('ALL launches of the tensor-core engine in one step: each launch is bounded by max(algorithmic '
                                'FLOPs / sustained bf16 peak, algorithmic bytes / HBM peak) from MEASURED_PEAKS; frac = sum(bound '
                                'times) / sum(CUDA-event times).  achieved/peak/unit restate frac in the units of the class that '
                                'holds most of the time; per-class figures are under classes.'),
            'peak_source': peaks['source'],
            'classes': {k: cls_rec(k) for k in cls},
            'slowest_launch': ({'launch': top, 'ms_per_launch': gemm[top]['ms'] / gemm[top]['calls'],
                                'frac_of_its_roofline': gemm[top]['roof_frac']} if top else None),
            'worst_launch': ({'launch': worst, 'frac_of_its_roofline': gemm[worst]['roof_frac'],
                              'ms_per_step': gemm[worst]['ms']} if worst else None),
            'engine_share_of_step': gemm_ms / all_ms if all_ms else None,
            'step_tensor_tflops': 3 * FWD_FLOPS[model_name] * B / (ms_step / 1e3) / 1e12,
            'step_hbm_gbs_algorithmic': ALGO_BYTES[model_name] * B / (ms_step / 1e3) / 1e9,
            'step_frac_of_network_roofline': max(3 * FWD_FLOPS[model_name] * B / tf_peak, ALGO_BYTES[model_name] * B / bw_peak) * 1e3 / ms_step}
    if dump_path:
        rows = sorted(table.items(), key=lambda kv: -kv[1]['ms'])
        with open(dump_path, 'w') as f:
            f.write('op,calls,ms_per_step,GFLOP,algorithmic_MB,TFLOP/s,GB/s,frac_of_roofline\n')
            for k, v in rows:
                s = v['ms'] / 1e3
                f.write(f"{k},{v['calls']},{v['ms']:.4f},{v['flops'] / 1e9:.2f},{v['bytes'] / 1e6:.2f},"
                        f"{v['flops'] / s / 1e12 if s else 0:.1f},{v['bytes'] / s / 1e9 if s else 0:.1f},{v.get('roof_frac', 0):.3f}\n")
    return roof


def measure_model(model_name, args, rank, world, local_rank, dump_path=None, with_ddp_check=False):
    """Device-timed and end-to-end throughput + the roofline pass for one model.  Returns a dict (rank 0) or None."""
    from simpleaicv_pytorch_training_examples_b200 import _lib
    from simpleaicv_pytorch_training_examples_b200.classification import backbones, losses
    from simpleaicv_pytorch_training_examples_b200.distributed import B200DataParallel, overlap_self_check
    from simpleaicv_pytorch_training_examples_b200.tools import utils as tutils
    dev = torch.device('cuda', local_rank)
    B = {'sam_h_encoder': 8, 'resnet50_detr': 4}.get(model_name, args.batch)
    torch.manual_seed(0)
    x_host, y_host = synthetic_batch(model_name, B, rank, True)
    detr_masks = None
    if model_name == 'resnet50_detr':
        from simpleaicv_pytorch_training_examples_b200.detection import models as det_models
        from simpleaicv_pytorch_training_examples_b200.detection.losses import DETRLoss
        model = det_models.resnet50_detr(num_classes=80).to(dev).train()
        detr_crit = DETRLoss().to(dev)
        detr_masks = torch.zeros(B, 1024, 1024, dtype=torch.bool, device=dev)
        detr_masks[:, :, 896:] = True                              # a padded right border, as the collater produces

        class _DetrNet(torch.nn.Module):                           # (images) -> outputs, so that the generic step applies
            def __init__(self, m):
                super().__init__()
                self.m = m

            def forward(self, x):
                return self.m(x, detr_masks)

        def crit(outs, y):
            return sum(detr_crit(outs, y).values())

        class _Cfg:
            optimizer = ('AdamW', {'lr': 1e-4, 'global_weight_decay': False, 'weight_decay': 1e-4, 'no_weight_decay_layer_name_list': [],
                                   'capturable': True})
        opt, _ = tutils.build_optimizer(_Cfg, model)
    elif model_name == 'sam_h_encoder':
        from simpleaicv_pytorch_training_examples_b200.interactive_segmentation.models.segment_anything import sam
        model = sam.sam_h(image_size=1024, use_gradient_checkpoint=False).image_encoder.to(dev).train()
        crit = torch.nn.MSELoss().to(dev)

        class _Cfg:
            optimizer = ('AdamW', {'lr': 1e-4, 'global_weight_decay': False, 'weight_decay': 0.05,
                                   'no_weight_decay_layer_name_list': [], 'capturable': world == 1 or not args.no_graph_ddp})
        opt, _ = tutils.build_optimizer(_Cfg, model)
    elif model_name == 'vit_base_mae':
        from simpleaicv_pytorch_training_examples_b200.masked_image_modeling import losses as mim_losses
        from simpleaicv_pytorch_training_examples_b200.masked_image_modeling.models import vit_mae
        model = vit_mae.vit_base_patch16_224_mae_pretrain_model().to(dev).train()
        mse = mim_losses.MSELoss().to(dev)

        def crit(outs, y):
            return mse(outs[0], y, outs[1])

        class _Cfg:
            optimizer = ('AdamW', {'lr': 1.5e-4, 'global_weight_decay': False, 'weight_decay': 0.05, 'no_weight_decay_layer_name_list': []})
        opt, _ = tutils.build_optimizer(_Cfg, model)
    elif model_name == 'resnet50':
        model = backbones.resnet50(num_classes=1000).to(dev).train()
        crit = losses.CELoss().to(dev)
        opt, _ = tutils.build_optimizer(r50_optimizer_cfg(), model)
    else:
        model = backbones.vit_base_patch16(image_size=224, num_classes=1000, drop_path_prob=0.1, global_pool=True).to(dev).train()
        crit = losses.OneHotLabelCELoss().to(dev)
        opt, _ = tutils.build_optimizer(vit_optimizer_cfg(model, capturable=(world == 1 or not args.no_graph_ddp)), model)
    ddp = B200DataParallel(model) if world > 1 else None
    net = ddp if ddp is not None else model
    if detr_masks is not None:
        net = _DetrNet(net)
    x_dev, y_dev = x_host.to(dev), y_host.to(dev)

    def step(x, y):
        loss = crit(net(x), y)
        loss.backward()
        opt.step()
        opt.zero_grad()
        return loss

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(k):
            fn()
        e.record()
        barrier()
        ms = torch.tensor([s.elapsed_time(e)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    warm = max(3, args.warmup)
    for _ in range(warm):
        step(x_dev, y_dev)
    ddp_check = None
    if world > 1 and with_ddp_check:
        # bit-exactness of the overlapped bucket all-reduce vs no_sync + reduce_now on the same batch
        # (drop-path masks are reseeded so that both passes draw the same ones)
        def fb():
            torch.manual_seed(77)
            crit(net(x_dev), y_dev).backward()
        ndiff = torch.tensor([overlap_self_check(ddp, fb)], device=dev)
        dist.all_reduce(ndiff, op=dist.ReduceOp.SUM)
        ddp_check = 'ok: overlapped all-reduce bit-identical to no_sync+reduce_now on every rank' if int(ndiff) == 0 \
            else f'FAILED: {int(ndiff)} gradient elements differ'
        opt.zero_grad()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    steps = args.steps
    capturable_step = detr_masks is None     # DETRLoss matches on the host (a sync per step) and DETR trains with dropout
    last = {}                                # the loss of the latest timed step, for --dump-outputs

    def keep(fn):
        return lambda: last.__setitem__('loss', fn())

    l0 = _lib.launch_count()
    ms_total = timed(keep(lambda: step(x_dev, y_dev)), steps)
    launches = _lib.launch_count() - l0
    eager_ms_step = ms_total / steps

    # end to end through the public API: every step's batch comes from pinned host memory through
    # tools.utils.CudaPrefetcher (the loader wrapper train_classification uses: H2D of batch i+1 on a
    # side stream while step i computes) and the loss is read back to the host every step
    # At N = 1 the step is replayed from ONE CUDA graph (graph.GraphedTrainStep, part of the package's API): the host
    # reads every step's loss, so without the graph the ~600 C-ABI launches of the next step could not be issued ahead.
    graphed, graph_note = None, 'eager launches'
    if (world == 1 or not args.no_graph_ddp) and not args.no_graph and capturable_step:
        try:
            torch.cuda.empty_cache()
            from simpleaicv_pytorch_training_examples_b200.graph import GraphedTrainStep
            graphed = GraphedTrainStep(net, crit, opt, x_dev, y_dev)
            graph_note = 'one CUDA graph per step (graph.GraphedTrainStep)' + (', NCCL bucket all-reduces captured' if world > 1 else '')
        except Exception as e:  # pragma: no cover
            graphed, graph_note = None, f'eager (graph capture failed: {type(e).__name__}: {e})'
            torch.cuda.synchronize()

    split = None
    if detr_masks is not None and not args.no_graph and (world == 1 or not args.no_graph_ddp):
        try:   # the criterion needs the host (Hungarian matcher): forward graph + eager criterion + backward/optimizer graph
            from simpleaicv_pytorch_training_examples_b200.graph import GraphedSplitStep
            torch.cuda.empty_cache()
            split = GraphedSplitStep(lambda x: net(x), lambda outs, y: detr_crit(outs, y), opt, [x_dev], y_dev)
            graph_note = 'two CUDA graphs per step around the eager criterion (graph.GraphedSplitStep)' + (', NCCL captured' if world > 1 else '')
        except Exception as e:  # pragma: no cover
            split, graph_note = None, f'eager (graph capture failed: {type(e).__name__}: {e})'
            torch.cuda.synchronize()

    # device-resident throughput: the same graph replayed on resident inputs when there is one, else the eager loop above
    if split is not None:
        split([x_dev], y_dev)
        ms_step = timed(keep(lambda: split([x_dev], y_dev)), steps) / steps
    elif graphed is not None:
        graphed.replay()
        ms_step = timed(keep(graphed.replay), steps) / steps
    else:
        ms_step = eager_ms_step
    value = B * world / (ms_step / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, model_name, last['loss'], model)

    def e2e_loop(k):
        host_batches = ({'image': x_host, 'label': y_host} for _ in range(k))
        for batch in tutils.CudaPrefetcher(host_batches, dev, copy_streams=args.prefetch_streams):
            if split is not None:
                split([batch['image']], batch['label']).item()
            elif graphed is not None:
                graphed(batch['image'], batch['label']).item()
            else:
                step(batch['image'], batch['label']).item()

    e2e_loop(2)
    e2e_ms = timed(lambda: e2e_loop(steps), 1) / steps

    # the same loop with the input-pipeline edge of SURVEY.md 8 f3: the host batch is the decoder's uint8 [B, H, W, 3] pixels
    # (classification.common.Uint8ClassificationCollater), a quarter of the fp32 batch's bytes on the host link; the
    # prefetcher normalises it into the fp32 NCHW batch on the device (csrc/capi_input.cu), then the same step runs
    e2e_u8 = None
    if model_name in ('resnet50', 'vit_base_patch16') and x_host.dim() == 4:
        g8 = torch.Generator().manual_seed(4321 + rank)
        x8 = torch.randint(0, 256, (B, x_host.shape[2], x_host.shape[3], 3), dtype=torch.uint8, generator=g8).pin_memory()
        norm = ((0.485, 0.456, 0.406), (0.229, 0.224, 0.225))

        def e2e_u8_loop(k):
            host_batches = ({'image': x8, 'label': y_host} for _ in range(k))
            for batch in tutils.CudaPrefetcher(host_batches, dev, copy_streams=args.prefetch_streams, normalize=norm):
                if graphed is not None:
                    graphed(batch['image'], batch['label']).item()
                else:
                    step(batch['image'], batch['label']).item()

        e2e_u8_loop(2)
        u8_ms = timed(lambda: e2e_u8_loop(steps), 1) / steps
        e2e_u8 = {'value': B * world / (u8_ms / 1e3), 'unit': 'images/s', 'ms_per_step': u8_ms,
                  'h2d_bytes_per_step': (x8.numel() + y_host.numel() * y_host.element_size()) * world, 'd2h_bytes_per_step': 4 * world,
                  'input': 'uint8 [B,H,W,3] pinned host batch, ToTensor+Normalize+permute on the device (bit-identical to the host pipeline)'}
    graph_ddp_check = None
    if world > 1 and graphed is not None:
        # every rank trained on its own batches: parameters stay identical across ranks only if the captured all-reduces ran
        chk = torch.stack([p.detach().double().abs().sum() for p in model.parameters()]).sum().view(1)
        lo, hi = chk.clone(), chk.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        graph_ddp_check = ('ok: parameters bit-identical on every rank after the captured steps' if float(lo) == float(hi)
                           else f'FAILED: parameter checksums differ across ranks ({float(lo)} .. {float(hi)})')
    clocks = sampler.stop() if rank == 0 else None
    rec = None
    if rank == 0:
        # instrumented pass (not part of any reported throughput): per-op CUDA-event timing
        # (rank 0 only: the gradient exchange is skipped, otherwise the other ranks would be waited for)
        t = OpTimer()
        t.install()
        with (ddp.no_sync() if world > 1 else contextlib.nullcontext()):
            for _ in range(2):
                step(x_dev, y_dev)
        table = t.summarize()
        t.remove()
        for d in table.values():
            d['ms'] /= 2
            d['calls'] //= 2
            d['flops'] /= 2
            d['bytes'] /= 2
        roof = roofline_from_table(table, _peaks(), model_name, B, eager_ms_step, dump_path)
        rec = {'metric': METRICS[model_name], 'value': value, 'unit': 'images/s', 'ms_per_step': ms_step,
               'e2e': {'value': B * world / (e2e_ms / 1e3), 'unit': 'images/s', 'ms_per_step': e2e_ms,
                       'h2d_bytes_per_step': (x_host.numel() * x_host.element_size() + y_host.numel() * y_host.element_size()) * world,
                       'd2h_bytes_per_step': 4 * world, 'mode': graph_note},
               'gpu_launches': int(launches), 'roofline': roof, 'clocks': clocks, 'workload': WORKLOADS[model_name],
               'ddp_check': ddp_check, 'graph_ddp_check': graph_ddp_check, 'eager_ms_per_step': eager_ms_step, 'per_gpu_batch': B, 'timed_steps': steps,
               'value_mode': graph_note, 'e2e_uint8_input': e2e_u8}
    del model, net, opt
    torch.cuda.empty_cache()
    return rec


DUMP_PARAMS = 1 << 21       # parameters kept per model by --dump-outputs (8 MB in float32)
DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, model_name, loss, model):
    """What the last timed step hands its caller: the loss, and the model it trained - the parameters after the
    optimizer step (all of them when there are at most DUMP_PARAMS, else DUMP_PARAMS at positions drawn with a fixed
    seed from the concatenated parameter vector) and, for a model that has them, the floating-point buffers (BatchNorm
    running statistics).  A model without such buffers (ViT) gets no buffers file rather than an empty one."""
    os.makedirs(out_dir, exist_ok=True)
    params = torch.cat([p.detach().float().reshape(-1) for p in model.parameters()])
    if params.numel() > DUMP_PARAMS:
        idx = torch.randperm(params.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_PARAMS].sort().values
        params = params[idx.to(params.device)]
    bufs = [b.detach().double().reshape(-1) for b in model.buffers() if b.is_floating_point()]
    arrays = {'loss': torch.as_tensor(loss).detach().float().reshape(1), 'params': params}
    if bufs:
        arrays['buffers'] = torch.cat(bufs)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f'{model_name}_{name}.npy'), t.cpu().numpy())
    total = sum(os.path.getsize(os.path.join(out_dir, f)) for f in os.listdir(out_dir) if f.endswith('.npy'))
    assert total <= DUMP_LIMIT, f'--dump-outputs wrote {total} bytes (limit {DUMP_LIMIT})'


def run_b200(args, rank, world, local_rank):
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    B = args.batch
    main = measure_model(args.model, args, rank, world, local_rank, args.dump_ops, with_ddp_check=True)
    other = None
    if not args.no_second_model:
        second = 'vit_base_patch16' if args.model == 'resnet50' else 'resnet50'
        other = measure_model(second, args, rank, world, local_rank,
                              args.dump_ops.replace('.csv', f'_{second}.csv') if args.dump_ops else None)
    mae_rec = None
    if args.mae:
        mae_rec = measure_model('vit_base_mae', args, rank, world, local_rank,
                                args.dump_ops.replace('.csv', '_vit_base_mae.csv') if args.dump_ops else None)
    sam_rec = None
    if args.sam:
        sam_rec = measure_model('sam_h_encoder', args, rank, world, local_rank,
                                args.dump_ops.replace('.csv', '_sam_h_encoder.csv') if args.dump_ops else None)
    detr_rec = None
    if args.detr:
        detr_rec = measure_model('resnet50_detr', args, rank, world, local_rank,
                                 args.dump_ops.replace('.csv', '_resnet50_detr.csv') if args.dump_ops else None)
    if rank != 0:
        return
    cpu_base = None
    if world == 1 and not args.no_cpu_baseline:
        cpu_base = cpu_baseline_record(args.model, 16, 2, args.steps)
    line = {
        'metric': main['metric'], 'value': main['value'], 'unit': 'images/s', 'n_gpus': world, 'steps': args.steps,
        'warmup': max(3, args.warmup), 'ms_per_step': main['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
        'config': {'workload': main['workload'], 'per_gpu_batch': B, 'global_batch': B * world, 'parallelism': f'dp{world}',
                   'l2_policy': 'inputs+activations (>10 GB/step) far exceed the 126 MB L2; no explicit flush',
                   'images_per_sec_per_gpu': main['value'] / world},
        'clocks': main['clocks'], 'e2e': main['e2e'], 'gpu_launches': main['gpu_launches'], 'roofline': main['roofline'],
        'cpu_baseline': cpu_base,
    }
    if main.get('ddp_check'):
        line['ddp_check'] = main['ddp_check']
    if main.get('graph_ddp_check'):
        line['graph_ddp_check'] = main['graph_ddp_check']
    SUB = ('metric', 'value', 'unit', 'ms_per_step', 'eager_ms_per_step', 'value_mode', 'e2e', 'e2e_uint8_input', 'gpu_launches', 'roofline',
           'clocks', 'workload', 'per_gpu_batch', 'timed_steps')
    line['eager_ms_per_step'], line['value_mode'] = main['eager_ms_per_step'], main['value_mode']
    line['e2e_uint8_input'] = main.get('e2e_uint8_input')
    if other is not None:
        name = 'vit_base_patch16' if args.model == 'resnet50' else 'resnet50'
        line[name] = {k: other[k] for k in SUB}
        line[name]['images_per_sec_per_gpu'] = other['value'] / world
    if mae_rec is not None:
        line['vit_base_mae'] = {k: mae_rec[k] for k in SUB}
        line['vit_base_mae']['images_per_sec_per_gpu'] = mae_rec['value'] / world
    if sam_rec is not None:
        line['sam_h_encoder'] = {k: sam_rec[k] for k in SUB}
        line['sam_h_encoder']['images_per_sec_per_gpu'] = sam_rec['value'] / world
    if detr_rec is not None:
        line['resnet50_detr'] = {k: detr_rec[k] for k in SUB}
        line['resnet50_detr']['images_per_sec_per_gpu'] = detr_rec['value'] / world
    torch_base = os.path.join(ROOT, 'profiles', 'r02_torch_gpu_baseline.json')
    if os.path.exists(torch_base):
        line['torch_ddp_target'] = {'source': 'profiles/r02_torch_gpu_baseline.json (unmodified reference under torch DDP, same pool)',
                                    'records': json.load(open(torch_base)).get('summary')}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--batch', type=int, default=256, help='per-GPU batch (BASELINE config: 256)')
    ap.add_argument('--model', default='resnet50', choices=['resnet50', 'vit_base_patch16'],
                    help='resnet50 = BASELINE configs[1] (default, the headline); vit_base_patch16 = configs[2]')
    ap.add_argument('--dump-ops', default=None, help='write the per-op timing table (csv) here')
    ap.add_argument('--dump-outputs', default=None, metavar='DIR',
                    help='after the timed steps, write what the last one computed (loss, trained parameters, buffers) as DIR/<model>_<name>.npy')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-second-model', action='store_true', help='skip the sub-record of the other BASELINE model')
    ap.add_argument('--detr', action='store_true', help='add the DETR-R50 sub-record (BASELINE configs[4]; shipped 1024x1024 shape, bs4)')
    ap.add_argument('--mae', action='store_true', help='add the MAE ViT-B/16 pre-training sub-record (SURVEY.md 8 f4)')
    ap.add_argument('--sam', action='store_true', help='add the SAM ViT-H image-encoder sub-record (BASELINE configs[3]: bs8, 1024x1024)')
    ap.add_argument('--no-graph-ddp', action='store_true',
                    help='N > 1: launch the step eagerly instead of capturing it (NCCL bucket all-reduces included) in one CUDA graph')
    ap.add_argument('--prefetch-streams', type=int, default=4, help='copy streams of the end-to-end host prefetcher (tools.utils.CudaPrefetcher)')
    ap.add_argument('--no-graph', action='store_true', help='end-to-end loop without the CUDA graph (eager launches)')
    args = ap.parse_args()
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    if args.impl == 'reference':
        run_reference(args, rank)
        return
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device; the B200 arm has no CPU fallback (use --impl reference for the CPU path)')
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        torch.cuda.set_device(local_rank)
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    try:
        run_b200(args, rank, world, local_rank)
    finally:
        if world > 1:
            dist.destroy_process_group()


if __name__ == '__main__':
    main()
