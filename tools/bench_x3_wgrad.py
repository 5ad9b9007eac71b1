"""Time of the tensor-core weight-gradient kernel in split precision (mpa_conv_wgrad_tc_x3) against bf16 (mpa_conv_wgrad_tc), on two
training layers at 75 x 216 patches: the DRCNN's 40 -> 40 15x15 layer (batch 16) and SAUnet:L's 16 -> 128 15x15 layer (upconv4, batch 25).
The formats alternate round by round in one process; the card's name and power limit are recorded with the times.

    python tools/bench_x3_wgrad.py [--rounds 5] [--iters 20] [--out profiles/r04_bench_x3_wgrad.json]

Per layer and format: the median over rounds of the mean kernel time (CUDA events around `--iters` calls of ops.conv_wgrad_tc, which
zeroes gw and then launches the kernel), and the achieved rate of the algorithmic 2 * B*T*F * Cin*Cout*KH*KW FLOP."""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

LAYERS = {'drcnn_40to40_15x15': dict(B=16, Cin=40, Cout=40, K=15), 'saunet_l_16to128_15x15': dict(B=25, Cin=16, Cout=128, K=15)}
T, F = 75, 216


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    import torch
    from multipitch_architectures_b200 import ops
    from bench_fp16_train import card
    torch.manual_seed(0)
    res = {'card': card(), 'T': T, 'F': F, 'layers': {}}
    for name, L in LAYERS.items():
        x = torch.randn(L['B'], L['Cin'], T, F, device='cuda')
        g = torch.randn(L['B'], L['Cout'], T, F, device='cuda') * 1e-2
        gw = torch.empty(L['Cout'], L['Cin'], L['K'], L['K'], device='cuda')
        planes = {fmt: (ops.nchw_to_cp8(x, fmt=f), ops.nchw_to_cp8(g, fmt=f)) for fmt, f in (('bf16', ops.FMT_BF16), ('fp16x3', ops.FMT_F16X3))}
        flop = 2.0 * L['B'] * T * F * L['Cin'] * L['Cout'] * L['K'] ** 2
        times = {fmt: [] for fmt in planes}
        for fmt, (xc, gc) in planes.items():                       # warm-up
            for _ in range(3):
                ops.conv_wgrad_tc(xc, gc, gw, (L['K'], L['K']))
        torch.cuda.synchronize()
        for _ in range(a.rounds):
            for fmt, (xc, gc) in planes.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(a.iters):
                    ops.conv_wgrad_tc(xc, gc, gw, (L['K'], L['K']))
                e1.record()
                e1.synchronize()
                times[fmt].append(e0.elapsed_time(e1) / a.iters)
        r = {'B': L['B'], 'Cin': L['Cin'], 'Cout': L['Cout'], 'K': L['K'], 'gflop': flop / 1e9}
        for fmt, ts in times.items():
            ms = statistics.median(ts)
            r[fmt] = {'ms': round(ms, 4), 'tflops': round(flop / ms / 1e9, 1), 'rounds_ms': [round(t, 4) for t in ts]}
        r['x3_over_bf16'] = round(r['fp16x3']['ms'] / r['bf16']['ms'], 3)
        res['layers'][name] = r
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
