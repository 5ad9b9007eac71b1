"""Step time of the fused training steps in fp16 (with dynamic loss scaling) against bf16, on the two training workloads of bench.py:
CNN:XS at batch 256 and SAUnet:L at batch 25.  The two precisions alternate round by round in one process, so that both see the same
card state; every step is a captured-graph replay, as in bench.py.  The card's name and power limit are printed with the times.

    python tools/bench_fp16_train.py [--rounds 5] [--steps 20] [--warmup 5] [--out profiles/r03_bench_fp16_train.json]

Per workload and precision: the median over rounds of the mean step time (CUDA events around `--steps` steps, synchronised), and the
loss of the last step.  An fp16 step adds one read pass over the flat fp32 gradient (the overflow check) and one single-thread launch (the
scale update) to the bf16 step's work."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def card():
    import torch
    out = {'name': torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'], capture_output=True,
                           text=True, timeout=30)
        out['power_limit'], out['max_sm_clock'] = [v.strip() for v in r.stdout.strip().split(',')][:2]
    except (OSError, ValueError, subprocess.SubprocessError) as e:
        out['power_limit'] = f'unavailable ({e})'
    return out


def make_step(name, precision):
    import bench
    from tests.weights import synth_patches, synth_targets
    spec = bench.WORKLOADS[name]
    model = bench.build_model(name, precision, 'cuda:0').train()
    if spec['cls'].startswith(('basic_cnn', 'deep_cnn')):
        from multipitch_architectures_b200.training import TrainStep as Step
    else:
        from multipitch_architectures_b200.training_unet import UnetTrainStep as Step
    step = Step(model, lr=spec['lr'], weight_decay=0.01, graph=True)
    x, t = synth_patches(spec['batch'], 0).cuda(), synth_targets(spec['batch'], 0).cuda()
    return step, x, t, spec['batch']


def timed(step, x, t, steps):
    import torch
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = step(x, t)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, float(loss.item())


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n\n')[0])
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--workloads', default='train_cnn_xs,train_saunet')
    ap.add_argument('--out', default=None, help='also write the result as JSON to this file')
    args = ap.parse_args()
    import numpy as np
    import torch
    assert torch.cuda.is_available(), 'this measurement needs a GPU'
    torch.cuda.set_device(0)
    res = {'card': card(), 'rounds': args.rounds, 'steps_per_round': args.steps, 'workloads': {}}
    for name in args.workloads.split(','):
        steps = {p: make_step(name, p) for p in ('bf16', 'fp16')}
        for p, (step, x, t, _) in steps.items():
            timed(step, x, t, args.warmup)                         # eager steps 1-2, the capture, warm replays
        ms = {p: [] for p in steps}
        loss = {}
        for _ in range(args.rounds):
            for p, (step, x, t, _) in steps.items():
                v, loss[p] = timed(step, x, t, args.steps)
                ms[p].append(v)
        batch = steps['bf16'][3]
        w = {p: {'ms_per_step_median': float(np.median(v)), 'ms_per_step_rounds': [round(a, 4) for a in v],
                 'patches_per_s': batch / (float(np.median(v)) / 1e3), 'last_loss': loss[p]} for p, v in ms.items()}
        w['fp16']['loss_scale'] = steps['fp16'][0].loss_scale
        w['batch'] = batch
        w['fp16_over_bf16'] = w['fp16']['ms_per_step_median'] / w['bf16']['ms_per_step_median']
        res['workloads'][name] = w
        print(f"{name} (batch {batch}) on {res['card']['name']}, power limit {res['card'].get('power_limit')}: "
              f"bf16 {w['bf16']['ms_per_step_median']:.3f} ms, fp16 {w['fp16']['ms_per_step_median']:.3f} ms per step "
              f"(fp16 / bf16 = {w['fp16_over_bf16']:.3f})", flush=True)
        for step, *_ in steps.values():
            step.release()
        del steps
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
