"""Times autograd from the activations to the audio: HCQT forward / backward (30 s and 10 min clips, both plans), ops.gather_patches forward /
backward, and engine.audio_vjp for the DRCNN [40,40,30,10]x5 in bf16 on a 30 s clip.  CUDA events, warmed up, the compared calls alternated
within each repetition; medians in ms.  Prints the card and its power limit from the same run and writes JSON into --out.

    python tools/bench_hcqt_grad.py --out /tmp/hcqt_grad [--reps 10]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True, text=True)
        return q.stdout.strip().splitlines()[0]
    except (OSError, IndexError):
        return torch.cuda.get_device_name(0) + ', power limit unknown'


def timed(fns, reps, warmup=2):
    """fns: {name: callable}; -> {name: median ms}, the callables alternated within each repetition."""
    for _ in range(warmup):
        for f in fns.values():
            f()
    torch.cuda.synchronize()
    ts = {k: [] for k in fns}
    for _ in range(reps):
        for k, f in fns.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f()
            e1.record()
            torch.cuda.synchronize()
            ts[k].append(e0.elapsed_time(e1))
    return {k: float(np.median(v)) for k, v in ts.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--reps', type=int, default=10)
    a = ap.parse_args()
    from multipitch_architectures_b200 import engine, ops
    from multipitch_architectures_b200.libdl import nn_models as M
    from tests import hcqt_ref as R
    from tests.synth import synth_clip
    from tests.weights import MODEL_SPECS, fill_state_dict
    torch.cuda.set_device(0)
    dev_line = card()
    print('card:', dev_line)
    res = {'card': dev_line, 'reps': a.reps, 'unit': 'ms (median)'}
    tun = torch.tensor([50], dtype=torch.int32, device='cuda')
    for efficient in (True, False):
        plan = R.make_plan(efficient, 'cuda')
        for seconds in (30, 600):
            y = torch.from_numpy(synth_clip(3, seconds=float(seconds))).cuda()
            yg = y.clone().requires_grad_(True)
            out, _ = plan.run(yg, tun)
            g = torch.randn_like(out)

            def fwd():
                plan.run(y, tun)

            def bwd():
                torch.autograd.grad(out, yg, g, retain_graph=True)
            t = timed({'forward': fwd, 'backward': bwd}, a.reps)
            key = f'hcqt_{"efficient" if efficient else "per_harmonic"}_{seconds}s'
            res[key] = t
            print(key, t, flush=True)
            del out, g, yg
            torch.cuda.empty_cache()
    frames = (torch.rand(6, 1292 + 75, 216, device='cuda') * 0.1).requires_grad_(True)
    patches = ops.gather_patches(frames, 0, 50)
    gp = torch.randn_like(patches)
    res['gather_patches_50x6x75x216'] = t = timed({
        'forward': lambda: ops.gather_patches(frames.detach(), 0, 50),
        'backward': lambda: torch.autograd.grad(patches, frames, gp, retain_graph=True)}, a.reps)
    print('gather_patches', t, flush=True)
    spec = MODEL_SPECS['drcnn']
    m = getattr(M, spec['cls'])(**spec['kw'], precision='bf16')
    m.load_state_dict(fill_state_dict(m.state_dict(), 1))
    m = m.cuda().eval()
    plan = R.make_plan(True, 'cuda')
    y = torch.from_numpy(synth_clip(3, seconds=30.0)).cuda()
    N = plan.n_frames(y.numel())
    g_act = torch.randn(N, 72, device='cuda')
    with torch.no_grad():
        h, _ = plan.run(y, tun)
    res['audio_vjp_drcnn_bf16_30s'] = t = timed({
        'predict_patchwise': lambda: engine.predict_patchwise(m, h, batch=50),
        'audio_vjp': lambda: engine.audio_vjp(m, y, plan, g_act, batch=50, tuning_idx=tun)}, max(3, a.reps // 3), warmup=1)
    print('audio_vjp drcnn bf16 30 s', t, flush=True)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, 'bench_hcqt_grad.json'), 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == '__main__':
    main()
