"""Step time of the fused training steps in fp32, fp16x3 and bf16 on the two training workloads of bench.py: CNN:XS at batch 256 and
SAUnet:L at batch 25.  The precisions alternate round by round in one process after warm-up; every step is a captured-graph replay, as in
bench.py.  The card's name and power limit are recorded with the times.

    python tools/bench_x3_train.py [--rounds 3] [--steps 10] [--warmup 4] [--out profiles/r04_bench_x3_train.json]

Per workload and precision: the median over rounds of the mean step time (CUDA events around `--steps` steps, synchronised)."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'tools')):
    if p not in sys.path:
        sys.path.insert(0, p)

PRECISIONS = ('fp32', 'fp16x3', 'bf16')


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n\n')[0])
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=4)
    ap.add_argument('--workloads', default='train_cnn_xs,train_saunet')
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import numpy as np
    import torch
    from bench_fp16_train import card, make_step, timed
    assert torch.cuda.is_available(), 'this measurement needs a GPU'
    torch.cuda.set_device(0)
    res = {'card': card(), 'rounds': args.rounds, 'steps_per_round': args.steps, 'workloads': {}}
    for name in args.workloads.split(','):
        steps = {p: make_step(name, p) for p in PRECISIONS}
        for step, x, t, _ in steps.values():
            timed(step, x, t, args.warmup)
        ms = {p: [] for p in steps}
        for _ in range(args.rounds):
            for p, (step, x, t, _) in steps.items():
                ms[p].append(timed(step, x, t, args.steps)[0])
        w = {p: {'ms_per_step_median': float(np.median(v)), 'ms_per_step_rounds': [round(a, 4) for a in v]} for p, v in ms.items()}
        w['batch'] = steps['fp32'][3]
        w['fp32_over_fp16x3'] = w['fp32']['ms_per_step_median'] / w['fp16x3']['ms_per_step_median']
        w['fp16x3_over_bf16'] = w['fp16x3']['ms_per_step_median'] / w['bf16']['ms_per_step_median']
        res['workloads'][name] = w
        print(name, {p: round(w[p]['ms_per_step_median'], 3) for p in PRECISIONS}, flush=True)
        for step, *_ in steps.values():
            step.release()
        del steps
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
