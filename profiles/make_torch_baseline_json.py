"""Collects gpurun_out/torch_gpu_baseline*.jsonl (written by baseline/torch_gpu_baseline.py on the GPU boxes) into
profiles/r02_torch_gpu_baseline.json (bench.py's torch_ddp_target)."""
import glob
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
recs = []
for f in sorted(glob.glob(os.path.join(ROOT, 'gpurun_out', 'torch_gpu_baseline*.jsonl'))):
    recs += [json.loads(l) for l in open(f) if l.strip()]
summary = {}
for r in recs:
    summary.setdefault(r['model'], {})[f"{r['variant']}_n{r['n_gpus']}"] = {
        'images_per_sec': round(r['images_per_sec'], 1), 'ms_per_step': round(r['ms_per_step'], 2), 'amp_type': r['amp_type'],
        'per_gpu_batch': r['per_gpu_batch']}
out = {'what': ("Unmodified reference modules (oracle/_ref copy of the reference) driven by the reference's own tools/scripts.py "
                'train_classification loop under torch DistributedDataParallel + autocast on the same B200 pool '
                '(baseline/torch_gpu_baseline.py).  Variants: as_shipped = fp16 autocast + GradScaler with cudnn.deterministic (the shipped '
                'config; get_amp_type has no B200 entry); bf16 = the same loop with the amp whitelist forced to bfloat16; tuned = bf16 + '
                'cudnn.benchmark + channels_last (not the reference configuration).  H2D of the batch is inside the timed region (the loop '
                'calls .cuda() per step); synthetic data; whole-job images/s.'),
       'north_star_target': ">= 1.3x the reference's own torch-DDP images/sec", 'summary': summary, 'records': recs}
json.dump(out, open(os.path.join(ROOT, 'profiles', 'r02_torch_gpu_baseline.json'), 'w'), indent=1)
for m, d in summary.items():
    print(m, {k: v['images_per_sec'] for k, v in sorted(d.items())})
