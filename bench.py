#!/usr/bin/env python
"""Benchmark of the hot path: HCQT feature extraction + patch-wise network inference / training (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference|reference-gpu] [--workload ...] [--precision ...] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Default run (what the driver launches): the HEADLINE workload = BASELINE configs[0] at the north star's target size — HCQT + DRCNN
[40,40,30,10]x5 patch-wise inference of one 30 s synthetic 22.05 kHz clip per GPU per step (661,500 samples -> 1,292 HCQT frames -> 1,292
stride-1 patches of 6x75x216 -> 1,292x72 activations), metric audio-seconds per wall second over all ranks — plus, in the SAME JSON line,
a `workloads` dict with short runs of BASELINE configs[1..4] (CNN:XS training, Unet:M and PUnet inference, SAUnet:L data-parallel
training with its NCCL gradient all-reduce inside the timed region) and a `parity` block.

Precision of the headline: `--precision auto` (default) picks the FASTEST tensor-core mode whose activations are within the north
star's 1e-3 of the REFERENCE's outputs on the realistic (trained) weight set over >= 100 patches, with identical thresholded P/R/F —
checked live, outside the timed region, against tests/golden/realistic_golden.npz (made by the unmodified reference classes).  The
other modes are timed as second figures (`other_modes`).

JSON keys (rank 0, one line): value = inputs resident in HBM; e2e = through the public API with pinned HOST audio in and HOST
activations out (H2D + D2H inside the timed region; at N > 1 it ends with the NCCL all-gather of every rank's [n_frames, 72]
activations = the north star's "final gather"); roofline = the dominant kernel (tcgen05 15x15 40->40 convolution) from CUDA events
recorded live in the timed region, per GPU; cpu_baseline = the reference's CPU path on a bounded sample on this box's host cores.

`--impl reference`: the CPU arm alone (rank 0), same metric / config; each step = HCQT + network on a bounded sample of the workload
(>= 200 patches), no extrapolation: value = audio seconds of the sample / measured step time.
`--impl reference-gpu` (informational): the reference's stock PyTorch path (torch conv2d -> cuDNN, batch 50, fp32 and TF32) on cuda:0."""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FPS = 22050 / 512
HCQT_KW = dict(fs=22050, fs_hcqt_target=50, bins_per_octave=36, num_octaves=6, num_harmonics=5, num_subharmonics=1)
GFLOP_PREFILT_LAYER = 11.664      # one 40->40 15x15 layer per patch (SURVEY 8a row N3)
DRAM_BYTES_PER_PATCH_LAYER = (951.8e6 + 938.2e6) / 646     # ncu, fused conv_tc_kernel, 75 rows per patch (profiles/README.md)
REF_ROOT = '/root/reference'
DUMP_BYTES = 64 << 20                   # --dump-outputs writes at most this much

DRCNN_KW = dict(n_chan_input=6, n_chan_layers=[40, 40, 30, 10], n_prefilt_layers=5, residual=True, n_bins_in=216, n_bins_out=72)
CNN_XS_KW = dict(n_chan_input=6, n_chan_layers=[20, 20, 10, 1], n_bins_in=216, n_bins_out=72)
SAUNET_L_KW = dict(n_chan_input=6, n_chan_layers=[128, 80, 50, 30], n_bins_in=216, n_bins_out=72, scalefac=4, embed_dim=128, num_heads=8,
                   mlp_dim=8192, pos_encoding='sinusoidal')
UNET_M_KW = dict(n_chan_input=6, n_chan_layers=[128, 100, 80, 50], n_bins_in=216, n_bins_out=72, scalefac=8)
PUNET_KW = dict(n_chan_input=6, n_chan_layers=[128, 180, 150, 100], n_bins_in=216, n_bins_out=72, scalefac=2, num_polyphony_steps=24)

# SURVEY 8a/8d: 2*MAC of every Conv2d / Linear at T=75 (forward); training = 3x forward
WORKLOADS = {
    'infer_drcnn': dict(kind='infer', cls='deep_cnn_segm_sigmoid', kw=DRCNN_KW, gflop=48.574, realistic='drcnn',
                        label='DRCNN[40,40,30,10]x5 residual (BASELINE configs[0], the north-star target)'),
    'train_cnn_xs': dict(kind='train', cls='basic_cnn_segm_sigmoid', kw=CNN_XS_KW, gflop=0.916, batch=256, lr=1e-3, cpu_batch=64,
                         label='CNN:XS [20,20,10,1] (BASELINE configs[1])'),
    'infer_unet_m': dict(kind='infer', cls='simple_u_net_largekernels', kw=UNET_M_KW, gflop=12.144, realistic='unet_m',
                         label='Unet:M [128,100,80,50] sc=8 (BASELINE configs[2])'),
    'infer_punet': dict(kind='infer', cls='simple_u_net_polyphony_classif_softmax', kw=PUNET_KW, gflop=81.777, realistic=None,
                        label='PUnet [128,180,150,100] sc=2, 24 polyphony steps (BASELINE configs[3])'),
    'train_saunet': dict(kind='train', cls='simple_u_net_doubleselfattn', kw=SAUNET_L_KW, gflop=29.110, batch=25, lr=1e-3, cpu_batch=25,
                         label='SAUnet:L [128,80,50,30] sc=4 E=128 mlp=8192 (BASELINE configs[4]; per-rank batch = the reference batch of 25: '
                               'batch-axis attention and BatchNorm statistics are per batch)'),
}
EXTRA_WORKLOADS = ('train_cnn_xs', 'infer_unet_m', 'infer_punet', 'train_saunet')


def workload_config(name, args):
    """The `config` object: a pure function of the workload and the command line, identical in the product and the reference arm."""
    spec = WORKLOADS[name]
    if spec['kind'] == 'infer':
        return {'workload': f"{spec['label']}: HCQT(6x216, hop 512) + stride-1 patch-wise inference of one {args.seconds:.0f} s 22.05 kHz clip per GPU per step",
                'patches_per_step_per_gpu': int(args.seconds * 22050) // 512 + 1, 'patch': '6x75x216',
                'timing': 'CUDA events; >= 1 GB of activations per step vs 126 MB of L2 (inputs larger than L2)',
                'weights': ('trained on synthetic labelled audio (tests/golden/realistic_weights.npz)' if spec.get('realistic') else
                            'seeded random init (no checkpoint blobs exist)')}
    batch = args.batch if args.batch > 0 else spec['batch']
    return {'workload': f"{spec['label']}: training step (forward + backward + loss + AdamW), synthetic 6x75x216 patches, batch {batch} per GPU",
            'timing': 'CUDA events; the activations of one step exceed L2', 'weights': 'seeded random init', 'dropout': 0.2}


def measured_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get('bf16_tflops_sustained', 1386.1), d.get('hbm_gbs', 6541.5), 'measured (MEASURED_PEAKS.json, sustained)'
    return 1400.0, 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def run(self):
        q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
            'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
        while not self._stop_evt.is_set():
            try:
                r = subprocess.run(['nvidia-smi', '-i', str(self.index), f'--query-gpu={q}', '--format=csv,noheader,nounits'],
                                   capture_output=True, text=True, timeout=5)
                self.rows.append([c.strip() for c in r.stdout.strip().split(',')])
            except Exception:
                pass
            self._stop_evt.wait(0.05)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        sm = sorted(int(r[0]) for r in self.rows if len(r) >= 6 and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) >= 6 and r[1].isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 6 and r[2 + i].lower().startswith('active') for r in self.rows)]
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None, 'reasons': reasons,
                'samples': len(self.rows)}


# ======================================================================================================================= weights
def state_dict_for(name, seed=0):
    """Weights of a workload's model as a plain state_dict (no product class involved): the trained realistic set where one exists,
    else seeded random tensors with the shapes recorded from the reference classes (tests/golden/state_dict_keys.json)."""
    import numpy as np
    import torch
    from tests import realistic as R
    from tests.weights import fill_state_dict
    spec = WORKLOADS[name]
    if spec.get('realistic'):
        return R.state_dict(spec['realistic'])
    key = {'train_cnn_xs': 'cnn_xs', 'infer_punet': 'punet', 'train_saunet': 'saunet_l'}[name]
    keys = json.load(open(os.path.join(ROOT, 'tests', 'golden', 'state_dict_keys.json')))[key]
    shapes = {k: torch.zeros(shape, dtype=getattr(torch, dt)) for k, shape, dt in keys}
    return fill_state_dict(shapes, seed)


# ======================================================================================================================= CPU arms
def _reference_classes():
    """The reference's own libdl.nn_models when /root/reference is mounted (the build container); None on the GPU box."""
    if not os.path.isdir(os.path.join(REF_ROOT, 'libdl')):
        return None
    try:
        sys.dont_write_bytecode = True
        if REF_ROOT not in sys.path:
            sys.path.append(REF_ROOT)
        import importlib
        return importlib.import_module('libdl.nn_models')
    except Exception:
        return None


def cpu_forward_fn(name):
    """-> (callable X -> activations, kind): the unmodified reference class when it can be imported, else the oracle port."""
    import torch
    from oracle import nn_oracle as NO
    spec, sd = WORKLOADS[name], state_dict_for(name)
    ref = _reference_classes()
    if ref is not None and 'pos_encoding' not in spec['kw']:
        m = getattr(ref, spec['cls'])(**spec['kw'])
        m.load_state_dict(sd)
        m.eval()
        return (lambda X: m(X)), 'reference'
    if spec['cls'].startswith(('basic_cnn', 'deep_cnn')):
        return (lambda X: NO.cnn_forward(sd, X, residual=spec['kw'].get('residual', False))), 'port'
    return (lambda X: NO.unet_forward(sd, X)), 'port'


def cpu_infer_step(name, seconds_sample, threads, clip=None, fwd=None):
    """One step of the reference CPU path on a bounded sample: NumPy HCQT of the first `seconds_sample` seconds of the synthetic clip
    + the fp32 network on every stride-1 patch of it (batches of 50, exp126a...py:413-436).  -> (seconds of audio, step seconds)."""
    import numpy as np
    import torch
    from oracle import hcqt_oracle as HO
    from oracle import host_oracle as PO
    torch.set_num_threads(threads)
    y = clip[:int(round(seconds_sample * 22050))]
    t0 = time.perf_counter()
    f, _, _ = HO.compute_efficient_hcqt(y, **HCQT_KW)
    n_frames = f.shape[1]
    ip, _ = PO.pad_for_inference(np.transpose(f, (2, 1, 0)), np.zeros((n_frames, 72)))
    with torch.no_grad():
        for b0 in range(0, n_frames, 50):
            nb = min(50, n_frames - b0)
            X = torch.from_numpy(np.stack([PO.context_item(ip, np.zeros((ip.shape[1], 72)), b0 + i)[0] for i in range(nb)]))
            fwd(X)
    return len(y) / 22050.0, time.perf_counter() - t0, n_frames


def cpu_infer_arm(name, args, threads, steps, warmup, sample_patches):
    """-> dict(value audio-s/s, ms_per_step, sample description, kind)."""
    from tests import synth
    fwd, kind = cpu_forward_fn(name)
    clip = synth.synth_clip(0, seconds=args.seconds)
    sec = min(args.seconds, sample_patches / FPS)
    ts, n_frames, audio = [], 0, 0.0
    for i in range(warmup + steps):
        audio, dt, n_frames = cpu_infer_step(name, sec, threads, clip, fwd)
        if i >= warmup:
            ts.append(dt)
    t = sum(ts) / len(ts)
    src = 'the unmodified reference class (libdl.nn_models)' if kind == 'reference' else 'oracle port of the reference class (torch CPU ops)'
    return {'value': audio / t, 'ms_per_step': 1e3 * t, 'kind': kind,
            'sample': f'each step = NumPy/SciPy restatement of librosa HCQT + fp32 {WORKLOADS[name]["cls"]} [{src}] on the first {audio:.2f} s of the clip '
                      f'= {n_frames} stride-1 patches in batches of 50, measured (no extrapolation): {t:.2f} s per step, mean of {steps} steps after '
                      f'{warmup} warm-up; torch threads={threads}'}


def cpu_train_arm(name, args, threads, steps, warmup):
    """The reference's training step on the host cores: fp32 forward + autograd backward + torch AdamW (reference class when importable)."""
    import torch
    import torch.nn.functional as F
    from oracle import nn_oracle as NO
    from tests.weights import synth_patches, synth_targets
    torch.set_num_threads(threads)
    spec = WORKLOADS[name]
    batch = min(args.batch if args.batch > 0 else spec['batch'], spec['cpu_batch'])
    sd0 = state_dict_for(name)
    x, t = synth_patches(batch, 0), synth_targets(batch, 0)
    ref = _reference_classes()
    cnn = spec['cls'].startswith(('basic_cnn', 'deep_cnn'))
    if ref is not None and 'pos_encoding' not in spec['kw']:
        m = getattr(ref, spec['cls'])(**spec['kw'])
        m.load_state_dict(sd0)
        m.train()
        opt = torch.optim.AdamW(m.parameters(), lr=spec['lr'], weight_decay=0.01)
        fwd, kind = (lambda: m(x)), 'reference'
    else:
        sd = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and 'running_' not in k else v.clone()) for k, v in sd0.items()}
        opt = torch.optim.AdamW([v for v in sd.values() if v.requires_grad], lr=spec['lr'], weight_decay=0.01)
        fwd = (lambda: NO.cnn_forward(sd, x)) if cnn else (lambda: NO.unet_forward(sd, x, train=True, pos_encoding=spec['kw'].get('pos_encoding')))
        kind = 'port'
    ts = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        opt.zero_grad()
        y = fwd()
        if isinstance(y, tuple):
            loss = NO.bce_mean(y[0], t) + F.cross_entropy(y[1], t.sum(-1, keepdim=True).long().squeeze(3)) / 25.0
        else:
            loss = NO.bce_mean(y, t)
        loss.backward()
        opt.step()
        if i >= warmup:
            ts.append(time.perf_counter() - t0)
    dt = sum(ts) / len(ts)
    return {'value': batch / dt, 'ms_per_step': 1e3 * dt, 'kind': kind,
            'sample': f"fp32 {spec['cls']} forward + autograd backward + AdamW ({'reference class' if kind == 'reference' else 'oracle port'}), batch {batch}, "
                      f'mean of {steps} steps after {warmup} warm-up, torch threads={threads}'}


def reference_main(args, rank, cores):
    """`--impl reference`: rank 0 alone times the CPU arm of the selected workload (default: the headline)."""
    if rank != 0:
        return
    name = 'infer_drcnn' if args.workload == 'all' else args.workload
    spec = WORKLOADS[name]
    if spec['kind'] == 'infer':
        # bounded sample: >= 200 patches per step (BASELINE.md 3.3), fewer only when K + W steps would not end within a few minutes
        n = args.cpu_sample if args.steps + args.warmup <= 25 else max(100, args.cpu_sample * 25 // (args.steps + args.warmup))
        r = cpu_infer_arm(name, args, cores, args.steps, args.warmup, n)
        metric, unit = 'audio_seconds_per_second', 'audio-s/s'
    else:
        r = cpu_train_arm(name, args, cores, max(1, min(args.steps, 3)), 1)
        metric, unit = 'train_patches_per_second', 'patches/s'
    print(json.dumps({'impl': 'reference', 'metric': metric, 'value': r['value'], 'unit': unit, 'n_gpus': args.gpus, 'steps': args.steps,
                      'warmup': args.warmup, 'ms_per_step': r['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                      'dtype': 'f32', 'data': 'synthetic', 'config': workload_config(name, args),
                      'cpu_baseline': {'value': r['value'], 'unit': unit, 'cores': cores, 'kind': r['kind'], 'sample': r['sample']},
                      'e2e': {'value': r['value'], 'unit': unit, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}))


def reference_gpu_main(args, cores):
    """Informational: the reference's stock PyTorch path on cuda:0 (torch conv2d -> cuDNN, cudnn.benchmark, batch 50 stride-1 patches,
    fp32 and TF32) — the unmodified reference class when it is importable, else its functional port (the same torch operator calls)."""
    import numpy as np
    import torch
    from oracle import host_oracle as PO
    from oracle import nn_oracle as NO
    from tests import realistic as R
    from multipitch_architectures_b200.libdl.data_preprocessing.hcqt import get_plan, C1_HZ
    from tests import synth
    dev = torch.device('cuda', 0)
    torch.backends.cudnn.benchmark = True
    sd = {k: v.to(dev) for k, v in R.state_dict('drcnn').items()}
    ref = _reference_classes()
    if ref is not None:
        m = ref.deep_cnn_segm_sigmoid(**DRCNN_KW).to(dev).eval()
        m.load_state_dict(sd)
        fwd, kind = (lambda X: m(X)), 'reference'
    else:
        fwd, kind = (lambda X: NO.cnn_forward(sd, X, residual=True)), 'port'
    plan = get_plan(22050, float(C1_HZ / 2 ** ((3 - 1) / (2 * 36))), 512, 36, 6, 5, 1, str(dev))
    y = torch.from_numpy(synth.synth_clip(0, seconds=args.seconds)).to(dev)
    out = {}
    for mode in ('fp32', 'tf32'):
        torch.backends.cudnn.allow_tf32 = mode == 'tf32'
        torch.backends.cuda.matmul.allow_tf32 = mode == 'tf32'

        def step():
            with torch.no_grad():
                hcqt, _ = plan.run(y)                      # feature extraction by this repo's kernels (librosa is not installed anywhere)
                N = hcqt.shape[1]
                ip = torch.nn.functional.pad(hcqt, (0, 0, 37, 38))
                outs = []
                for b0 in range(0, N, 50):
                    nb = min(50, N - b0)
                    X = torch.log(1 + 10 * torch.stack([ip[:, b0 + i:b0 + i + 75] for i in range(nb)]))
                    outs.append(fwd(X).reshape(nb, 72))
                return torch.cat(outs)
        for _ in range(max(1, args.warmup)):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            res = step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / args.steps
        out[mode] = {'value': args.seconds / (ms / 1e3), 'ms_per_step': ms,
                     'max_abs_vs_fp32': None if mode == 'fp32' else float((res - out['fp32']['_res']).abs().max())}
        out[mode]['_res'] = res
    for v in out.values():
        v.pop('_res')
    print(json.dumps({'impl': 'reference-gpu', 'metric': 'audio_seconds_per_second', 'unit': 'audio-s/s', 'value': out['tf32']['value'], 'n_gpus': 1,
                      'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': out['tf32']['ms_per_step'], 'higher_is_better': True,
                      'dtype': 'tf32', 'data': 'synthetic', 'config': workload_config('infer_drcnn', args), 'kind': kind, 'modes': out,
                      'note': 'stock PyTorch path of the reference (torch conv2d -> cuDNN, cudnn.benchmark=True, batches of 50 materialised stride-1 '
                              'patches) on this GPU; HCQT by libmpa (no librosa exists here).  Informational, not the target metric.'}))


# ======================================================================================================================= GPU arms
class Ctx:
    def __init__(self, args, rank, world, local, cores):
        import torch
        self.args, self.rank, self.world, self.local, self.cores = args, rank, world, local, cores
        self.dev = torch.device('cuda', local)

    def barrier(self):
        import torch
        import torch.distributed as dist
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(self, fn, steps):
        """EXACTLY `steps` calls bracketed by barrier + synchronize on both sides, CUDA events, MAX over ranks -> ms."""
        import torch
        import torch.distributed as dist
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        self.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=self.dev)
        if self.world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())


def build_model(name, precision, dev, seed=0):
    from multipitch_architectures_b200.libdl import nn_models as M
    spec = WORKLOADS[name]
    m = getattr(M, spec['cls'])(**spec['kw'], precision=precision)
    m.load_state_dict(state_dict_for(name, seed))
    return m.to(dev)


def gather_outputs(ctx, act, gathered):
    """The north star's final gather: every rank's [n_frames, 72] activations in one NCCL all-gather (inference e2e at N > 1)."""
    import torch.distributed as dist
    if ctx.world == 1:
        return act
    dist.all_gather_into_tensor(gathered, act.contiguous())
    return gathered


def host_arrays(outputs):
    """{name: tensor} -> {name: ndarray}: float64 and integer tensors as float64 (exact), other floating types as float32."""
    import torch
    return {k: (t.double() if t.dtype == torch.float64 or not t.is_floating_point() else t.float()).cpu().numpy() for k, t in outputs.items()}


def write_outputs(path, arrays):
    """Each array as path/<name>.npy.  An array larger than its share of DUMP_BYTES is replaced by a fixed, seeded sample of its rows
    (along the first axis, in order), and the indices of those rows go to path/<name>_rows.npy."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    share = DUMP_BYTES // max(1, len(arrays))
    for name, a in arrays.items():
        if a.nbytes > share:
            row_bytes = a.nbytes // a.shape[0] + 8          # + its float64 index
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], max(1, share // row_bytes), replace=False))
            np.save(os.path.join(path, name + '_rows.npy'), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(path, name + '.npy'), a)


def run_infer(ctx, name, precision, steps, warmup, preload, detail=False, e2e_first=False, outputs=None):
    """HCQT + patch-wise inference of one clip per GPU per step.  DRCNN: streaming engine; U-Nets: batches of materialised patches.
    outputs: a dict that receives, as host arrays, what the last timed device-resident step returned."""
    import torch
    from multipitch_architectures_b200 import _lib
    from multipitch_architectures_b200.engine import CnnStreamEngine, predict_patchwise
    from multipitch_architectures_b200.libdl.data_preprocessing.hcqt import get_plan, C1_HZ
    from tests import synth as HO              # synthetic-clip generator (workload data; the product arm never imports oracle/)
    args, dev, spec = ctx.args, ctx.dev, WORKLOADS[name]
    model = build_model(name, precision, dev).eval()
    cnn = spec['cls'].startswith(('basic_cnn', 'deep_cnn'))
    eng = CnnStreamEngine(model, chunk=args.chunk, fused=not args.plain, ring=args.ring) if cnn else None
    plan = get_plan(22050, float(C1_HZ / 2 ** ((3 - 1) / (2 * 36))), 512, 36, 6, 5, 1, str(dev))
    clips_host = [torch.from_numpy(HO.synth_clip(1000 * ctx.rank + i, seconds=args.seconds)).pin_memory() for i in range(2)]
    clips_dev = [c.to(dev) for c in clips_host]
    n_frames = clips_host[0].numel() // 512 + 1
    out_host = torch.empty(ctx.world if ctx.rank == 0 else 1, n_frames, 72, dtype=torch.float32).pin_memory()
    gathered = torch.empty(ctx.world * n_frames, 72, dtype=torch.float32, device=dev) if ctx.world > 1 else None

    def predict(y):
        """-> {name: tensor}: what a caller of the path receives for the clip y."""
        with torch.no_grad():
            if cnn:
                act, tuning = eng.predict_audio(y, plan)
                return {'activations': act, 'tuning_index': tuning}
            hcqt, _ = plan.run_graph(y)
            out = predict_patchwise(model, hcqt, batch=args.infer_batch)
            return dict(zip(('activations', 'polyphony'), out)) if isinstance(out, tuple) else {'activations': out}

    last = [None]

    def step_resident(i):
        last[0] = predict(clips_dev[i % 2])

    def step_e2e(i):
        act = predict(clips_host[i % 2].to(dev, non_blocking=True))['activations']
        g = gather_outputs(ctx, act, gathered)
        if ctx.rank == 0:
            out_host.view(-1, 72).copy_(g, non_blocking=True)        # rank 0 receives the whole job's activations
        else:
            out_host.view(-1, 72).copy_(act, non_blocking=True)

    for i in range(warmup):
        step_resident(i)
        step_e2e(i)
    sampler = ClockSampler(ctx.local) if (ctx.rank == 0 and detail) else None
    if sampler:
        sampler.start()
    # sustained state: the first timed loop after an idle gap runs 3-5 % faster than the second under the board's power cap
    # (profiles/README.md), so a few untimed steps right before the timed regions put both on the same footing
    for i in range(preload):
        step_resident(i)
    ms_e2e = ctx.timed(step_e2e, steps) if e2e_first else None
    # inside the timed region only the dominant kernel's launches carry events (every event pair costs a few microseconds of stream
    # idle time); the per-stage time shares come from two extra, untimed steps afterwards
    if eng is not None and detail:
        eng.timers, eng.timer_tags = [], {'conv_tc'}
    n0, g0 = _lib.launch_count(), plan.graph_launches
    ms = ctx.timed(step_resident, steps)
    launches = _lib.launch_count() - n0 + (plan.graph_launches - g0)      # host-side counter + the kernel nodes of the replayed HCQT graphs
    if outputs is not None:                 # copied before the untimed steps below reuse the engine's buffers
        outputs.update(host_arrays(last[0]))
    timers, share_timers = [], []
    if eng is not None and detail:
        timers, eng.timers, eng.timer_tags = eng.timers, [], None
        for i in range(2):
            step_resident(i)
        torch.cuda.synchronize()
        share_timers, eng.timers = eng.timers, None
    if ms_e2e is None:
        ms_e2e = ctx.timed(step_e2e, steps)
    clocks = sampler.stop() if sampler else None
    audio_s = args.seconds * steps * ctx.world
    value, e2e_v = audio_s / (ms / 1e3), audio_s / (ms_e2e / 1e3)
    peak_tf, _, peak_src = measured_peaks()
    res = {'value': value, 'ms_per_step': ms / steps, 'dtype': precision, 'gpu_launches': int(launches), 'clocks': clocks,
           'e2e': {'value': e2e_v, 'unit': 'audio-s/s', 'h2d_bytes_per_step': int(clips_host[0].numel() * 4),
                   'd2h_bytes_per_step': int(n_frames * 72 * 4 * (ctx.world if ctx.rank == 0 else 1)), 'ms_per_step': ms_e2e / steps,
                   'final_gather': (f'NCCL all_gather_into_tensor of {ctx.world} x [{n_frames},72] fp32 inside the timed region' if ctx.world > 1 else None)}}
    per_gpu_tf = value / ctx.world * FPS * spec['gflop'] / 1e3
    # patch-wise algorithmic FLOPs (the reference's count: every patch evaluates all its rows) per second per GPU; for the de-duplicated
    # DRCNN schedule this exceeds what the GPU executes (shared rows are computed once), so it is NOT a roofline fraction
    res['patchwise_equivalent_tflops_per_gpu'] = per_gpu_tf
    if eng is not None and detail and ctx.rank == 0:
        by, work = {}, {}
        for tag, a, b, w in timers:
            by.setdefault(tag, []).append(a.elapsed_time(b))
            work[tag] = work.get(tag, 0) + w
        conv = by.get('conv_tc', [])
        # executed algorithmic FLOPs of the 40->40 launches: output rows actually produced x 2*Cin*Cout*KH*KW*F per row (rows shared between
        # overlapping patches are counted ONCE; `patchwise_equivalent_tflops` uses the reference's patch-wise count); this rank's GPU only
        flops_row = GFLOP_PREFILT_LAYER * 1e9 / 75.0
        passes = 3 if precision == 'fp16x3' else 1
        conv_ms = sum(conv)
        achieved = flops_row * work.get('conv_tc', 0) / (conv_ms * 1e-3) / 1e12 if conv else None
        per_launch_rows = work.get('conv_tc', 0) / max(1, len(conv))
        by_all = {}
        for tag, a, b, w in share_timers:
            by_all.setdefault(tag, []).append(a.elapsed_time(b))
        tot_all = sum(sum(v) for v in by_all.values())
        res['roofline'] = {
            'bound': 'tensor', 'kernel': 'conv_tc_kernel (tcgen05 15x15 40->40; bias + LeakyReLU + MaxPool(3,1) + residual epilogue)',
            'achieved': achieved, 'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': (achieved / peak_tf) if achieved else None,
            'traffic': DRAM_BYTES_PER_PATCH_LAYER * per_launch_rows / 75.0 * (2 if precision == 'fp16x3' else 1),
            'traffic_source': 'ncu --set full (profiles/r01_conv_tc_fused_ncu_raw.csv): dram__bytes_read.sum 0.952 GB + dram__bytes_write.sum 0.938 GB per '
                              '646-patch x 75-row launch (algorithmic 0.89 + 0.89 GB), scaled by the rows per launch (x2 planes in fp16x3)',
            'peak_source': peak_src, 'scope': 'one GPU (rank 0): per-GPU achieved rate against one GPU\'s peak', 'launches_timed': len(conv),
            'avg_launch_ms': conv_ms / max(1, len(conv)), 'algorithmic_flops_per_launch': flops_row * per_launch_rows,
            'output_rows_per_launch': per_launch_rows, 'mma_passes_per_product': passes,
            'executed_tensor_tflops': (achieved * passes) if achieved else None,
            'time_share_by_stage': {k: round(sum(v) / tot_all, 4) for k, v in by_all.items()} if tot_all else None,
            'time_share_source': 'events around every stage in two untimed steps after the timed region',
            'schedule': 'fused conv+LReLU+pool3+residual, interior rows shared across patches' if eng.fused else 'plain per-patch'}
    else:
        res['roofline'] = {'bound': 'tensor', 'kernel': 'conv_tc_kernel over all layers (whole step)', 'achieved': per_gpu_tf, 'peak': peak_tf, 'unit': 'TFLOP/s',
                           'frac': per_gpu_tf / peak_tf, 'traffic': None, 'scope': 'per GPU',
                           'note': f"whole-step patch-wise algorithmic FLOPs ({spec['gflop']} GFLOP per patch) / step time, per GPU"}
    del eng, model
    torch.cuda.empty_cache()
    return res


def run_train(ctx, name, precision, steps, warmup, preload, outputs=None):
    """One training step per call: forward + loss + backward (+ NCCL gradient all-reduce at N > 1) + fused AdamW.
    outputs: a dict that receives, as host arrays, the loss of the last timed device-resident step and the parameters it left.  The weight
    gradients are split-K sums finished with fp32 atomicAdd, whose order varies, and AdamW amplifies such last-bit differences, so two runs
    of the same build agree on these to a tolerance only (the headline DRCNN inference outputs repeat bit for bit)."""
    import torch
    from multipitch_architectures_b200 import _lib
    from multipitch_architectures_b200.io import HostPrefetcher
    from tests.weights import synth_patches, synth_targets
    args, dev, spec = ctx.args, ctx.dev, WORKLOADS[name]
    batch = args.batch if args.batch > 0 else spec['batch']
    gflop_step = 3.0 * spec['gflop']
    model = build_model(name, precision, dev).train()
    if spec['cls'].startswith(('basic_cnn', 'deep_cnn')):
        from multipitch_architectures_b200.training import TrainStep as Step
    else:
        from multipitch_architectures_b200.training_unet import UnetTrainStep as Step
    step = Step(model, lr=spec['lr'], weight_decay=0.01, graph=not args.no_train_graph)
    xh, th = synth_patches(batch, ctx.rank).pin_memory(), synth_targets(batch, ctx.rank).pin_memory()
    xd, td = xh.to(dev), th.to(dev)
    loss_host = torch.empty(1).pin_memory()
    last = [None]

    def resident(i):
        last[0] = step(xd, td)

    # end to end: every step's batch travels from pinned host memory inside the timed region, double-buffered on a side stream
    # (io.HostPrefetcher: the copy of batch k+1 overlaps the step on batch k), and the loss is read back
    def host_batches():
        while True:
            yield (xh, th)
    feed = [None]

    def e2e(i):
        if feed[0] is None:
            feed[0] = HostPrefetcher(host_batches(), dev)
        xb, tb = next(feed[0])
        loss_host.copy_(step(xb, tb), non_blocking=True)

    for i in range(warmup):
        resident(i)
        e2e(i)
    for i in range(preload):
        resident(i)
    step.comm_events = [] if ctx.world > 1 else None
    n0, r0 = _lib.launch_count(), getattr(step, 'replays', 0)
    ms = ctx.timed(resident, steps)
    # kernels launched inside the timed region: the host-side counter plus the kernel nodes of every CUDA-graph replay
    launches = _lib.launch_count() - n0 + (getattr(step, 'replays', 0) - r0) * getattr(step, 'launches_per_replay', 0)
    if outputs is not None:                 # copied before the end-to-end steps below train on
        outputs.update(host_arrays({'loss': last[0], 'parameters': step.flat_p}))
    comm = step.comm_events
    step.comm_events = None
    ms_e2e = ctx.timed(e2e, steps)
    n = batch * steps * ctx.world
    value, e2e_v = n / (ms / 1e3), n / (ms_e2e / 1e3)
    tc = precision != 'fp32'
    peak_tf = measured_peaks()[0]
    per_gpu_tf = value / ctx.world * gflop_step / 1e3
    res = {'value': value, 'ms_per_step': ms / steps, 'dtype': 'bf16' if tc else 'f32', 'gpu_launches': int(launches),
           'e2e': {'value': e2e_v, 'unit': 'patches/s', 'h2d_bytes_per_step': int(xh.numel() * 4 + th.numel() * 4), 'd2h_bytes_per_step': 4,
                   'ms_per_step': ms_e2e / steps},
           'roofline': {'bound': 'tensor', 'kernel': ('tcgen05 forward / dgrad / wgrad convolutions + fp32 element-wise kernels' if tc else
                                                      'fp32 CUDA-core training kernels (conv2d_direct / conv_wgrad)') + ': whole step',
                        'achieved': per_gpu_tf, 'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': per_gpu_tf / peak_tf, 'traffic': None, 'scope': 'per GPU',
                        'note': f'whole-step algorithmic FLOPs ({gflop_step:.3f} GFLOP per patch = 3 x forward) / step time, per GPU, against the bf16 tensor peak'},
           'parallelism': f'dp{ctx.world} (replicas of batch {batch}, one flat fp32 NCCL gradient all-reduce per step, then fused AdamW)' if ctx.world > 1 else 'single GPU'}
    if comm:
        torch.cuda.synchronize()
        t = [a.elapsed_time(b) for a, b in comm]
        res['allreduce'] = {'ms_per_step': sum(t) / len(t), 'bytes': int(step.flat_g.numel() * 4), 'calls_timed': len(t),
                            'share_of_step': (sum(t) / len(t)) / (ms / steps),
                            'overlapped_bytes': int((step.flat_g.numel() - getattr(step, 'n_trunk', step.flat_g.numel())) * 4)
                            if getattr(step, 'overlap_comm', False) and getattr(step, 'n_trunk', 0) > 0 else 0,
                            'how': 'CUDA events around the part of the gradient all-reduce the step waits for, inside the timed steps '
                                   '(U-Net family: the gradients behind the encoder trunk are reduced on the NCCL stream while the trunk\'s backward '
                                   'runs; `overlapped_bytes` of `bytes` are issued before it)'}
    if hasattr(step, 'release'):
        step.release()
    del step, model
    torch.cuda.empty_cache()
    return res


def run_infer_saunet_sharded(ctx, steps, warmup):
    """SURVEY 8e row 2: ONE recording sharded across the ranks for the SAUnet (whose attention mixes the items of a batch): contiguous frame
    ranges on multiples of the reference batch (50 consecutive frames), 37-frame halos of real frames, final NCCL all-gather of [N, 72].
    Strong scaling of a single 30 s clip: value = clip seconds / step time (not multiplied by the number of ranks)."""
    import torch
    from multipitch_architectures_b200.engine import predict_patchwise
    from multipitch_architectures_b200.libdl.data_preprocessing.hcqt import get_plan, C1_HZ
    from multipitch_architectures_b200.parallel import predict_sharded
    from tests import synth as HO
    args, dev = ctx.args, ctx.dev
    model = build_model('train_saunet', 'fp16', dev).eval()
    plan = get_plan(22050, float(C1_HZ / 2 ** ((3 - 1) / (2 * 36))), 512, 36, 6, 5, 1, str(dev))
    clip = torch.from_numpy(HO.synth_clip(4242, seconds=args.seconds)).to(dev)      # the SAME recording on every rank

    def step(i):
        with torch.no_grad():
            hcqt, _ = plan.run_graph(clip)
            return predict_sharded(lambda h, lo, hi: predict_patchwise(model, h, batch=50, lo=lo, hi=hi), hcqt, ctx.world, ctx.rank, multiple=50, gather=True)
    for i in range(warmup):
        out = step(i)
    ms = ctx.timed(step, steps)
    n_frames = int(out.shape[0])
    per_gpu_tf = args.seconds * steps / (ms / 1e3) / ctx.world * FPS * WORKLOADS['train_saunet']['gflop'] / 1e3
    del model
    torch.cuda.empty_cache()
    return {'config': f'SAUnet:L inference of ONE {args.seconds:.0f} s clip ({n_frames} patches) sharded across {ctx.world} GPU(s) on multiples of 50 frames '
                      '(batch-axis attention: reference batches of 50 consecutive frames stay on one rank), HCQT on every rank, NCCL all-gather of the activations',
            'value': args.seconds * steps / (ms / 1e3), 'unit': 'audio-s/s', 'scaling': 'strong', 'n_gpus': ctx.world, 'steps': steps, 'warmup': warmup,
            'ms_per_step': ms / steps, 'dtype': 'fp16', 'roofline_frac_per_gpu': per_gpu_tf / measured_peaks()[0]}


def parity_block(ctx, modes):
    """Each tensor-core mode of the HEADLINE model on the realistic (trained) weights vs the outputs of the UNMODIFIED reference class
    over the whole held-out 30 s clip (tests/golden/realistic_golden.npz), outside every timed region.  The oracle is used here as the
    checker only: its NumPy HCQT of the clip is the input the reference outputs were made from."""
    import numpy as np
    import torch
    from oracle import hcqt_oracle as HQ
    from tests import realistic as R
    from tests import synth
    from multipitch_architectures_b200.engine import CnnStreamEngine
    f, _, _ = HQ.compute_efficient_hcqt(synth.synth_clip(**R.CLIP), **R.HCQT_KW)
    hcqt = torch.from_numpy(np.ascontiguousarray(np.transpose(f, (2, 1, 0)).astype(np.float32))).to(ctx.dev)
    out = {}
    for prec in modes:
        m = build_model('infer_drcnn', prec, ctx.dev).eval()
        with torch.no_grad():
            got = CnnStreamEngine(m, chunk=ctx.args.chunk).predict_hcqt(hcqt).cpu().numpy()
        c = R.compare(got, 'drcnn')
        out[prec] = {'max_abs_vs_reference': c['max_abs'], 'patches': c['frames'], 'threshold_flips': c['flips'], 'tp_fp_fn': list(c['counts']),
                     'tp_fp_fn_reference': list(c['counts_ref']), 'prf': [round(v, 4) for v in c['prf']], 'prf_equal_3dec': c['prf_equal_3dec'],
                     'meets_1e-3': bool(c['max_abs'] <= 1e-3 and c['prf_equal_3dec'])}
        del m
    torch.cuda.empty_cache()
    return out


def dropin_e2e(ctx, precision, steps):
    """The reference's OWN call pattern with only the imports swapped (notebook 02 / exp126a...py:404-436): compute_efficient_hcqt on a
    host array -> np.transpose -> np.pad -> dataset_context(stride 1) -> DataLoader(batch 50) -> model(batch) -> .to('cpu')."""
    import numpy as np
    import torch
    from multipitch_architectures_b200.libdl.data_loaders import dataset_context
    from multipitch_architectures_b200.libdl.data_preprocessing import compute_efficient_hcqt
    from tests import synth
    args = ctx.args
    model = build_model('infer_drcnn', precision, ctx.dev).eval()
    y = synth.synth_clip(1000 * ctx.rank, seconds=args.seconds)

    def once():
        f_hcqt, _, _ = compute_efficient_hcqt(y, **HCQT_KW)
        inputs = np.transpose(f_hcqt, (2, 1, 0))
        targets = np.zeros((inputs.shape[1], 72))
        ic = torch.from_numpy(np.pad(inputs, ((0, 0), (37, 38), (0, 0))))
        tc = torch.from_numpy(np.pad(targets, ((37, 38), (0, 0))))
        gen = torch.utils.data.DataLoader(dataset_context(ic, tc, {'context': 75, 'stride': 1, 'compression': 10}), batch_size=50, shuffle=False)
        pred_tot = np.zeros((0, 72))
        with torch.no_grad():
            for xb, _ in gen:
                yp = model(xb.to(ctx.dev)).to('cpu')
                pred_tot = np.append(pred_tot, torch.squeeze(torch.squeeze(yp, 2), 1).numpy(), axis=0)
        return pred_tot
    once()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        once()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / steps
    del model
    return {'value': args.seconds / dt, 'unit': 'audio-s/s', 'ms_per_step': 1e3 * dt, 'dtype': precision, 'steps': steps,
            'what': "the reference's test loop unmodified (host ndarray in, DataLoader batches of 50, model(batch), .to('cpu')) on this package's "
                    'classes; wall clock, one GPU'}


# ======================================================================================================================= main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=6)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference', 'reference-gpu'])
    ap.add_argument('--seconds', type=float, default=30.0)
    ap.add_argument('--chunk', type=int, default=646)
    ap.add_argument('--cpu-sample', type=int, default=200, help='patches per step of the CPU arm (>= 200: BASELINE.md 3.3)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--preload', type=int, default=6, help='untimed steps run immediately before the timed regions (sustained clocks)')
    ap.add_argument('--e2e-first', action='store_true', help='time the end-to-end loop before the device-resident one (order-effect check)')
    ap.add_argument('--precision', default='auto', choices=['auto', 'fp16', 'bf16', 'fp16x3'],
                    help='inference precision; auto = the fastest mode that is within 1e-3 of the reference on the realistic weight set')
    ap.add_argument('--ring', action='store_true', help='fused schedule with the ring main loop (un-duplicated weight pieces) instead of ready-made tiles')
    ap.add_argument('--plain', action='store_true', help='per-patch conv_tc + separate pool kernels (no fusion / de-duplication)')
    ap.add_argument('--workload', default='all', choices=['all'] + list(WORKLOADS),
                    help='all = headline (infer_drcnn) + short runs of the other BASELINE configs in `workloads`; or one workload alone')
    ap.add_argument('--batch', type=int, default=0, help='training batch per GPU (0 = the workload default)')
    ap.add_argument('--train-precision', default='bf16', choices=['fp32', 'bf16'])
    ap.add_argument('--no-train-graph', action='store_true', help='training: launch every kernel eagerly instead of replaying the captured CUDA graph')
    ap.add_argument('--infer-batch', type=int, default=646, help='patches per forward of the U-Net inference workloads')
    ap.add_argument('--no-extras', action='store_true', help='headline only: skip the `workloads`, `other_modes` and `dropin_e2e` legs')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed step of the headline workload returned (rank 0) as DIR/<name>.npy, float32 or float64, '
                         'at most 64 MB in all; the inputs are seeded, so two builds can be compared output for output')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be >= 1 and --warmup >= 0')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs writes the outputs of the b200 implementation only')

    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    cores = os.cpu_count() or 1
    if args.impl == 'reference':
        return reference_main(args, rank, cores)
    if args.impl == 'reference-gpu':
        return reference_gpu_main(args, cores) if rank == 0 else None

    import torch
    import torch.distributed as dist
    from multipitch_architectures_b200 import _lib
    torch.cuda.set_device(local)
    ctx = Ctx(args, rank, world, local, cores)
    if world > 1:
        dist.init_process_group('nccl', device_id=ctx.dev)
    assert _lib.lib().mpa_device_check() == 0, _lib.last_error()
    headline = 'infer_drcnn' if args.workload == 'all' else args.workload
    spec = WORKLOADS[headline]
    line = {}
    parity = None
    outputs = {} if args.dump_outputs else None
    if spec['kind'] == 'infer':
        precision = args.precision
        if headline == 'infer_drcnn' and not (args.no_extras and precision != 'auto'):
            modes = ['fp16', 'fp16x3', 'bf16']
            parity = parity_block(ctx, modes)
            if world > 1:                                   # every rank must take the same decision
                flag = torch.tensor([1 if parity['fp16']['meets_1e-3'] else 0], device=ctx.dev)
                dist.all_reduce(flag, op=dist.ReduceOp.MIN)
                parity['fp16']['meets_1e-3'] = bool(flag.item())
        if precision == 'auto':
            precision = 'fp16' if (parity is None or parity['fp16']['meets_1e-3']) else 'fp16x3'
        r = run_infer(ctx, headline, precision, args.steps, args.warmup, args.preload, detail=True, e2e_first=args.e2e_first, outputs=outputs)
        metric, unit = 'audio_seconds_per_second', 'audio-s/s'
    else:
        r = run_train(ctx, headline, args.train_precision, args.steps, args.warmup, args.preload, outputs=outputs)
        metric, unit = 'train_patches_per_second', 'patches/s'
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, outputs)
    line = {'metric': metric, 'value': r.pop('value'), 'unit': unit, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': r.pop('ms_per_step'), 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': r.pop('dtype'),
            'data': 'synthetic', 'config': workload_config(headline, args)}
    line.update(r)
    line['run'] = {'preload_steps': args.preload, 'parallelism': (f'{world} ranks, one clip (or one batch) per rank per step' if world > 1 else 'single GPU'),
                   'precision_choice': args.precision}
    if parity is not None:
        line['parity'] = {'mode': line['dtype'], 'weights': 'realistic: DRCNN trained 1,512 steps with loop.fit on labelled synthetic audio (F = 0.95 vs labels)',
                          'reference': 'outputs of the unmodified reference class on the same weights and inputs (tests/golden/realistic_golden.npz)',
                          'tolerance': 1e-3, **parity[line['dtype']], 'all_modes': parity}
    extras = args.workload == 'all' and not args.no_extras
    if extras:
        sub_steps, sub_warm = max(3, min(args.steps, 6)), 3
        # second figures: the other precisions of the headline
        line['other_modes'] = {}
        for prec in ('fp16x3', 'fp16', 'bf16'):
            if prec == line['dtype']:
                continue
            o = run_infer(ctx, 'infer_drcnn', prec, sub_steps, sub_warm, 2, detail=(prec == 'fp16x3'))
            line['other_modes'][prec] = {'value': o['value'], 'unit': unit, 'ms_per_step': o['ms_per_step'], 'e2e': o['e2e']['value'],
                                         'roofline_frac': o['roofline']['frac'], 'executed_tensor_tflops': o['roofline'].get('executed_tensor_tflops'),
                                         'parity': parity[prec] if parity else None}
        line['workloads'] = {}
        for wl in EXTRA_WORKLOADS:
            s = WORKLOADS[wl]
            if s['kind'] == 'infer':
                o = run_infer(ctx, wl, 'fp16', sub_steps, sub_warm, 2)
                u = 'audio-s/s'
            else:
                o = run_train(ctx, wl, args.train_precision, sub_steps, sub_warm, 2)
                u = 'patches/s'
            line['workloads'][wl] = {'config': workload_config(wl, args)['workload'], 'value': o['value'], 'unit': u, 'n_gpus': world, 'steps': sub_steps,
                                     'warmup': sub_warm, 'ms_per_step': o['ms_per_step'], 'dtype': o['dtype'], 'e2e': o['e2e'],
                                     'roofline_frac_per_gpu': o['roofline']['frac'], 'gpu_launches': o['gpu_launches'],
                                     **({'allreduce': o['allreduce'], 'parallelism': o['parallelism']} if 'allreduce' in o else {})}
        line['workloads']['infer_saunet_sharded'] = run_infer_saunet_sharded(ctx, sub_steps, sub_warm)
        if rank == 0:
            line['dropin_e2e'] = dropin_e2e(ctx, line['dtype'], 2)
        if world > 1:
            dist.barrier()
    if rank == 0:
        if not args.no_cpu_baseline:
            if spec['kind'] == 'infer':
                c = cpu_infer_arm(headline, args, cores, 1, 0, args.cpu_sample)
            else:
                c = cpu_train_arm(headline, args, cores, 2, 1)
            line['cpu_baseline'] = {'value': c['value'], 'unit': unit, 'cores': cores, 'kind': c['kind'], 'sample': c['sample']}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
