"""Eval-mode backward (gradients wrt the input, BatchNorm frozen) on the GPU: forward + backward time of CNN:XS (batch 256) and SAUnet:L
(batch 25) in bf16, timed with CUDA events, and the achieved bandwidth of the LayerNorm input-gradient kernels over their algorithmic bytes.
Prints one JSON line (and writes it to --out) with the card's name and power limit read in the same run.

    python tools/bench_eval_backward.py [--iters 20] [--out results/eval_backward.json]"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    r = subprocess.run(['nvidia-smi', '-i', str(torch.cuda.current_device()), '--query-gpu=name,power.limit', '--format=csv,noheader'],
                       capture_output=True, text=True)
    name, _, power = r.stdout.strip().partition(',')
    return {'name': name.strip() or torch.cuda.get_device_name(), 'power_limit': power.strip()}


def time_events(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def model_case(name, B, iters):
    from tests.refshapes import build_model
    from tests.weights import fill_state_dict, synth_patches, synth_targets
    m = build_model(name, precision='bf16')
    m.load_state_dict(fill_state_dict(m.state_dict(), 7, scheme='torch_default'))
    m = m.cuda().eval()
    x, t = synth_patches(B, 7).cuda(), synth_targets(B, 7).cuda()

    def step():
        m.zero_grad(set_to_none=True)
        xr = x.detach().requires_grad_(True)
        torch.nn.functional.binary_cross_entropy(m(xr), t).backward()
    ms = time_events(step, iters)
    with torch.no_grad():
        ms_fwd = time_events(lambda: m(x), iters)
    return {'model': name, 'batch': B, 'eval_fwd_bwd_ms': round(ms, 3), 'patches_per_s': round(B / ms * 1e3, 1),
            'inference_fwd_ms': round(ms_fwd, 3)}


def layernorm_case(B, C, T, F, iters):
    """Algorithmic bytes: x read + dx written (fp32), g read (16-byte CP8 pixels or fp32), the saved rows (8 bytes each) for the CP8 source."""
    from multipitch_architectures_b200 import ops
    x = torch.rand(B, C, T, F, device='cuda')
    w, b = torch.ones(C, F, device='cuda'), torch.zeros(C, F, device='cuda')
    gw, gb = torch.empty(C, F, device='cuda'), torch.empty(C, F, device='cuda')
    dst = ops.CP8(B, C, T, F, device='cuda', fmt=ops.FMT_BF16)
    stats = torch.empty(B * T, 2, device='cuda')
    ops.layernorm_cf_cp8(x, w, b, 1e-5, dst, stats=stats)
    g32 = torch.randn(B, C, T, F, device='cuda')
    n = B * C * T * F
    out = {'shape': [B, C, T, F]}
    for src, fn, nbytes in (('cp8_stats', lambda: ops.layernorm_cf_input_grad(x, dst, w, gw, gb, 1e-5, stats=stats), 8 * n + 16 * B * T * F + 8 * B * T),
                            ('f32', lambda: ops.layernorm_cf_input_grad(x, g32, w, gw, gb, 1e-5), 12 * n)):
        us = time_events(fn, iters * 10) * 1e3
        out[src] = {'us': round(us, 2), 'bytes': nbytes, 'GB_per_s': round(nbytes / us * 1e-3, 1)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('needs a CUDA device (nothing here is measured on the CPU)')
    res = {'card': card(), 'layernorm_input_grad': layernorm_case(256, 6, 75, 216, a.iters),
           'models': [model_case('cnn_xs', 256, a.iters), model_case('saunet_l', 25, a.iters)]}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
