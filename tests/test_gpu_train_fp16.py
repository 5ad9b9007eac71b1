"""`-m gpu`: fp16 training on the tensor-core tapes with dynamic loss scaling.  Gradients of both model families against the fp32 oracle, the
launches of the fp16 tapes against the bf16 ones, the device-side loss scaler of the fused step (overflow skip, back-off, growth, graph
replay, the drop-in path under torch.amp.GradScaler, two GPUs), its kernels, and a short `fit`."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.test_gpu_autograd_eval import _build, _grad_metrics, _loss, _oracle, _spec, _spy_calls, _zero_dropout
from tests.weights import fill_state_dict, synth_patches, synth_targets

pytestmark = pytest.mark.gpu

S16 = 2.0 ** 16          # torch.amp.GradScaler's initial scale


def _step_cls(name):
    from multipitch_architectures_b200 import training
    from multipitch_architectures_b200.training_unet import UnetTrainStep
    return training.TrainStep if 'cnn' in _spec(name)['cls'] else UnetTrainStep


def _model(name, precision, seed, scheme='torch_default', train=True):
    m = _build(name, precision)
    m.load_state_dict(fill_state_dict(m.state_dict(), seed, scheme=scheme))
    return m.cuda().train(train)


# ---------------------------------------------------------------------------------------------------------------- fidelity
# Gates per (model, mode): (input-gradient cosine, cosine of all parameter gradients) against the fp32 oracle, B = 3, seed 51, the loss
# scaled by 2^16 as a GradScaler would.  Each is stricter than the bf16 gate of the same case (tests/test_gpu_autograd_eval.py: CNN 0.99 /
# 0.9999; U-Net family eval 0.93 / 0.9999, train 0.84 / 0.94).  Measured on one NVIDIA B200 at a 1,000 W power limit (input / parameters):
# CNN:XS 0.99917 / 0.999998 in both modes; unet_s8 eval 0.99516 / 1.000000, train 0.98530 / 0.99634; saunet_s8 eval 0.99417 / 1.000000,
# train 0.98638 / 0.99538.  (An fp32 oracle whose convolutions round to fp16 predicts ~0.995 eval input, ~0.987 / 0.997 train.)
FP16_CASES = [
    ('cnn_xs', 'adversarial', dict(eval=(0.995, 0.99999), train=(0.995, 0.99999))),
    ('unet_s8', 'torch_default', dict(eval=(0.99, 0.99999), train=(0.975, 0.99))),
    ('saunet_s8', 'torch_default', dict(eval=(0.99, 0.99999), train=(0.975, 0.99))),
]


@pytest.mark.parametrize('mode', ['eval', 'train'])
@pytest.mark.parametrize('name,scheme,gates', FP16_CASES, ids=[c[0] for c in FP16_CASES])
def test_fp16_gradients_match_the_oracle(name, scheme, gates, mode):
    from multipitch_architectures_b200 import training, training_unet
    B, seed = 3, 51
    m = _build(name, 'fp16')
    sd = fill_state_dict(m.state_dict(), seed, scheme=scheme)
    m.load_state_dict(sd)
    _zero_dropout(m)
    m = m.cuda().train(mode == 'train')
    x, t = synth_patches(B, seed), synth_targets(B, seed)
    xc = x.cuda().requires_grad_(True)
    if 'cnn' in _spec(name)['cls']:
        assert training._cp8_resident(m, training._exec.cnn_blocks(m), x.shape[3])
    else:
        assert training_unet.cp8_tape_eligible(m, xc)
    loss = _loss(m(xc), t.cuda())
    (loss * S16).backward()
    l_ref, gx_ref, gp_ref = _oracle(name, sd, x, t, mode == 'train')
    gp = {k: p.grad.cpu() / S16 for k, p in m.named_parameters()}
    ex, cx, worst, cp = _grad_metrics(xc.grad.cpu() / S16, gx_ref, gp, gp_ref)
    print(f'{name}/fp16/{mode}: loss {loss.item():.6f} (oracle {l_ref:.6f}); input gradient max|d|/max|ref| {ex:.2e}, cosine {cx:.6f}; '
          f'parameter gradients worst per-tensor deviation {worst:.2e}, cosine {cp:.6f}')
    assert abs(loss.item() - l_ref) < 2e-2 * max(1.0, abs(l_ref))
    min_cx, min_cp = gates[mode]
    assert cx >= min_cx and cp >= min_cp


# ---------------------------------------------------------------------------------------------------------------- paths
LOSS_SCALE_CALLS = ('nonfinite_check_f32',)
AS_BF16 = {'bce_fwd_bwd_scaled_f32': 'bce_fwd_bwd_f32', 'ce_count_fwd_bwd_scaled_f32': 'ce_count_fwd_bwd_f32', 'adamw_scaled_f32': 'adamw_f32'}


@pytest.mark.parametrize('name', ['cnn_xs', 'drcnn_tiny', 'saunet_s8', 'punet_tiny'])
def test_fp16_tapes_launch_what_bf16_launches(name, monkeypatch):
    """Two fused steps (the second one under the pack plan) and a drop-in eval-mode backward: the fp16 model issues the bf16 model's
    entry points in the same order — apart from the loss-scale kernels — and notes the kernel path the bf16 model notes (none on the CP8
    tapes; never the fp32 CUDA-core tape)."""
    from multipitch_architectures_b200 import _lib
    from multipitch_architectures_b200.libdl.nn_models import _exec
    x, t = synth_patches(3, 65).cuda(), synth_targets(3, 65).cuda()
    notes = {}

    def traced(prec):
        m = _model(name, prec, 65)
        step = _step_cls(name)(m)
        monkeypatch.setattr(_exec, 'note_path', lambda model, what: notes.setdefault(prec, []).append(what))
        calls = _spy_calls(monkeypatch)
        n0 = _lib.launch_count()
        for _ in range(2):
            step(x, t)
        m.eval()
        xr = x.clone().requires_grad_(True)
        _loss(m(xr), t).backward()
        torch.cuda.synchronize()
        n = _lib.launch_count() - n0
        monkeypatch.undo()
        return [c[0] for c in calls], n
    bf, n_bf = traced('bf16')
    fp, n_fp = traced('fp16')
    assert fp.count('nonfinite_check_f32') == 2 and 'adamw_scaled_f32' in fp and 'adamw_f32' not in fp
    assert [AS_BF16.get(c, c) for c in fp if c not in LOSS_SCALE_CALLS] == bf
    assert n_fp == n_bf + 2 * 2                      # per step: the overflow check and the scaler update
    assert any(c.startswith('conv_wgrad_tc') or c.startswith('gemm_tc') for c in fp)
    assert notes.get('fp16', []) == notes.get('bf16', []), notes
    assert not any('CUDA-core' in w for w in notes.get('fp16', [])), notes
    if name in ('cnn_xs', 'saunet_s8'):
        assert 'fp16' not in notes, notes


# ---------------------------------------------------------------------------------------------------------------- scaler
def _snapshot(step):
    return [v.clone() for v in (step.flat_p, step.m, step.v)]


def _scaler_state(step):
    sc = step.scaler
    return float(sc.scale.item()), int(sc.growth_tracker.item()), int(sc.applied_steps.item()), int(sc.found_inf.item())


def test_overflow_skips_the_step_and_backs_off():
    from multipitch_architectures_b200.training import TrainStep
    m = _model('cnn_xs', 'fp16', 66)
    step = TrainStep(m, lr=1e-3)
    assert step.loss_scale == S16
    batch = lambda i: (synth_patches(4, 80 + i).cuda(), synth_targets(4, 80 + i).cuda())
    step(*batch(0))
    assert _scaler_state(step) == (S16, 1, 1, 0)
    huge = 2.0 ** 40                                  # gradients of ~1e-3 times 2^40 overflow the fp16 planes
    step.scaler.scale.fill_(huge)
    skipped = 0
    for i in range(1, 40):
        before = _snapshot(step)
        scale = step.loss_scale
        loss = step(*batch(i))
        assert torch.isfinite(loss).all()            # the reported loss is not scaled, and the forward is unaffected
        s, tracker, applied, found = _scaler_state(step)
        if found:
            skipped += 1
            assert all(torch.equal(a, b) for a, b in zip(before, _snapshot(step)))     # p, m, v bit for bit
            assert s == scale / 2 and tracker == 0 and applied == 1
            continue
        # the first step whose gradients fit trains: the counter moves and the parameters change
        assert s == scale and applied == 2 and tracker == 1
        assert not torch.equal(before[0], step.flat_p)
        break
    else:
        pytest.fail('the scale never backed off far enough to train')
    print(f'loss scale 2^40 -> {step.loss_scale:.0f} after {skipped} skipped steps')
    assert skipped >= 1


def test_loss_scale_grows_after_the_interval():
    from multipitch_architectures_b200.training import TrainStep
    step = TrainStep(_model('cnn_xs', 'fp16', 67), lr=1e-3)
    step.scaler.growth_interval = 3
    got = []
    for i in range(6):
        step(synth_patches(4, 90 + i).cuda(), synth_targets(4, 90 + i).cuda())
        got.append(_scaler_state(step)[:3])
    assert got == [(S16, 1, 1), (S16, 2, 2), (2 * S16, 0, 3), (2 * S16, 1, 4), (2 * S16, 2, 5), (4 * S16, 0, 6)], got


def test_graph_replayed_steps_with_a_skip_follow_the_eager_steps():
    """TrainStep(graph=True), dropout on, with an overflow forced at step 4 (a replayed step) and the scale restored at step 5: the skip
    decisions and the whole scaler state match the eager run bit for bit, and so do p / m / v across the skipped step.  Parameters are
    compared across the two runs to a tolerance only: the weight-gradient kernels finish with fp32 atomics, whose order varies."""
    from multipitch_architectures_b200.training import TrainStep
    res = {}
    for graph in (False, True):
        m = _model('cnn_xs', 'fp16', 68)
        assert m.p_dropout > 0
        step = TrainStep(m, lr=1e-6, graph=graph)
        losses, states = [], []
        for i in range(7):
            if i == 3:
                step.scaler.scale.fill_(2.0 ** 40)
            if i == 4:
                step.scaler.scale.fill_(S16)
            before = _snapshot(step)
            losses.append(float(step(synth_patches(4, 100 + i).cuda(), synth_targets(4, 100 + i).cuda()).item()))
            states.append(_scaler_state(step))
            if i == 3:
                assert all(torch.equal(a, b) for a, b in zip(before, _snapshot(step)))
        if graph:
            assert step.replays == 5
        res[graph] = losses, states, step.flat_p.clone()
    (l0, s0, p0), (l1, s1, p1) = res[False], res[True]
    print('eager', l0, s0, '\ngraph', l1, s1)
    assert s0 == s1 and s0[3] == (2.0 ** 39, 0, 3, 1) and s0[-1] == (S16, 3, 6, 0)
    assert all(abs(a - b) <= 2e-4 * max(1.0, abs(a)) for a, b in zip(l0, l1))
    assert len(set(round(v, 4) for v in l1)) == 7                      # fresh dropout masks on every replay
    assert (p0 - p1).abs().max().item() <= 1e-5


def test_fused_fp16_steps_track_grad_scaler_and_adamw():
    """Three fused fp16 steps against the drop-in path of the same model under torch.amp.GradScaler + torch.optim.AdamW.  Tolerance: the
    losses to 2e-4 relative; the parameter updates as tests/test_gpu_training.py bounds them (an element whose gradient is at noise level
    may take a random +-lr step at some step, so the mean and the share of outliers are bounded, not the maximum)."""
    from multipitch_architectures_b200.training import TrainStep
    sd = None
    models = []
    for _ in range(2):
        m = _build('cnn_xs', 'fp16')
        sd = fill_state_dict(m.state_dict(), 69, scheme='torch_default') if sd is None else sd
        m.load_state_dict(sd)
        _zero_dropout(m)
        models.append(m.cuda().train())
    fused, drop = models
    step = TrainStep(fused, lr=1e-3, weight_decay=0.01)
    opt = torch.optim.AdamW(drop.parameters(), lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.01)
    scaler = torch.amp.GradScaler('cuda')
    for it in range(3):
        x, t = synth_patches(4, 110 + it).cuda(), synth_targets(4, 110 + it).cuda()
        l_f = float(step(x, t).item())
        opt.zero_grad()
        loss = F.binary_cross_entropy(drop(x), t)
        scaler.scale(loss).backward()
        scaler.step(opt)
        scaler.update()
        assert abs(l_f - loss.item()) < 2e-4 * max(1.0, abs(loss.item())), (it, l_f, loss.item())
        assert step.loss_scale == scaler.get_scale()
    for (k, p), q in zip(fused.named_parameters(), drop.parameters()):
        d = ((p.detach() - sd[k].cuda()) - (q.detach() - sd[k].cuda())).abs()
        assert d.mean() < 0.02 * 3e-3 and (d > 0.3e-3).float().mean() < 0.02, k


# ---------------------------------------------------------------------------------------------------------------- kernels
def _flag(x, found=7):
    from multipitch_architectures_b200 import _lib
    f = torch.full((1,), found, dtype=torch.int32, device='cuda')
    _lib.call('nonfinite_check_f32', x, _lib.i64(x.numel()), f, _lib.stream_ptr())
    return int(f.item())


@pytest.mark.parametrize('n', [1, 3, 4, 4099, 1_000_003])
def test_nonfinite_check_finds_one_bad_value_anywhere(n):
    base = torch.randn(n + 1, device='cuda') * 1e4
    for x in (base[:n], base[1:]):                   # 16-byte aligned, and not (the element-wise path)
        assert _flag(x.contiguous() if x.data_ptr() % 16 == 0 else x) == 0
        for pos in sorted({0, n // 2, n - 1, max(0, n - 3), n // 4 * 4}):
            if pos >= n:
                continue
            for bad in (float('inf'), float('-inf'), float('nan')):
                y = x.clone() if x.data_ptr() % 16 == 0 else base.clone()[1:]
                y[pos] = bad
                assert _flag(y) == 1, (n, pos, bad, y.data_ptr() % 16)


def _adam_state(n, seed):
    g = torch.Generator().manual_seed(seed)
    mk = lambda s=1.0: (torch.randn(n, generator=g) * s).cuda()
    return mk(), mk(1e-3), mk(1e-3), mk(1e-3).abs() ** 2


@pytest.mark.parametrize('world', [1.0, 0.5])
def test_scaled_adamw_equals_adamw_on_the_unscaled_gradient(world):
    from multipitch_architectures_b200 import _lib
    n, S, k = 100_003, 2.0 ** 14, 5
    p, g, m, v = _adam_state(n, 3)
    g = g * S                                         # the gradient as the scaled loss leaves it
    hp = dict(lr=1e-3, b1=0.9, b2=0.999, eps=1e-8, wd=0.01)
    ref = [t.clone() for t in (p, m, v)]
    _lib.call('adamw_f32', ref[0], g, ref[1], ref[2], _lib.i64(n), hp['lr'], hp['b1'], hp['b2'], hp['eps'], hp['wd'], k, float(world / S),
              _lib.stream_ptr())
    i32 = lambda v: torch.tensor([v], dtype=torch.int32, device='cuda')

    def scaled(found):
        st = [t.clone() for t in (p, m, v)]
        scale, tracker, applied, flag = torch.tensor([S], device='cuda'), i32(7), i32(k - 1), i32(found)
        _lib.call('adamw_scaled_f32', st[0], g, st[1], st[2], _lib.i64(n), hp['lr'], hp['b1'], hp['b2'], hp['eps'], hp['wd'], float(world),
                  flag, scale, tracker, applied, 2.0, 0.5, 2000, _lib.stream_ptr())
        return st, (float(scale.item()), int(tracker.item()), int(applied.item()))
    (p1, m1, v1), state = scaled(0)
    assert torch.equal(m1, ref[1]) and torch.equal(v1, ref[2])
    # the bias corrections are formed on the device from the applied-step counter (powf there, on the host for adamw_f32)
    assert torch.allclose(p1, ref[0], rtol=2e-7, atol=1e-9)
    assert state == (S, 8, k)
    (p2, m2, v2), state = scaled(1)
    assert torch.equal(p2, p) and torch.equal(m2, m) and torch.equal(v2, v)
    assert state == (S / 2, 0, k - 1)


def test_scaled_losses_scale_only_the_gradient():
    from multipitch_architectures_b200 import _lib, ops
    y = torch.rand(3, 1, 1, 72, device='cuda') * 0.98 + 0.01
    t = (torch.rand(3, 1, 1, 72, device='cuda') < 0.1).float()
    S = torch.tensor([S16], device='cuda')
    l0, g0 = ops.bce_fwd_bwd(y, t)
    l1, g1 = ops.bce_fwd_bwd(y, t, loss_scale=S)
    assert torch.equal(l0, l1) and torch.equal(g1, g0 * S16)
    logits = torch.randn(3, 24, device='cuda')
    tt = (torch.rand(3, 1, 1, 72, device='cuda') < 0.05).float()
    out = []
    for scaled in (False, True):
        loss, gl = torch.zeros(1, device='cuda'), torch.empty_like(logits)
        if scaled:
            _lib.call('ce_count_fwd_bwd_scaled_f32', logits, tt, loss, gl, 3, 24, 72, 1.0 / 25.0, 0, S, _lib.stream_ptr())
        else:
            _lib.call('ce_count_fwd_bwd_f32', logits, tt, loss, gl, 3, 24, 72, 1.0 / 25.0, 0, _lib.stream_ptr())
        out.append((loss, gl))
    assert torch.equal(out[1][1], out[0][1] * S16)
    # the items' losses meet in fp32 atomics, whose order varies from call to call
    assert torch.allclose(out[0][0], out[1][0], rtol=1e-6, atol=0.0)


# ---------------------------------------------------------------------------------------------------------------- two GPUs
def _ddp_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ['MASTER_ADDR'], os.environ['MASTER_PORT'] = '127.0.0.1', str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=torch.device('cuda', rank))
    from multipitch_architectures_b200.training import TrainStep
    step = TrainStep(_model('cnn_xs', 'fp16', 70), lr=1e-3)
    dist.broadcast(step.flat_p, src=0)
    log = []
    for i in range(6):
        if i == 2 and rank == 0:
            step.scaler.scale.fill_(2.0 ** 40)        # only rank 0 overflows
        if i == 3:
            step.scaler.scale.fill_(S16)
        before = _snapshot(step)
        step(synth_patches(4, 120 + 10 * i + rank).cuda(), synth_targets(4, 120 + 10 * i + rank).cuda())
        unchanged = all(torch.equal(a, b) for a, b in zip(before, _snapshot(step)))
        log.append((_scaler_state(step)[2:], unchanged))
    flat = step.flat_p.double()
    q.put((rank, log, float(flat.sum().item()), float(flat.abs().max().item())))
    dist.barrier()
    dist.destroy_process_group()


def test_an_overflow_on_one_rank_skips_the_step_on_both():
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    procs = [ctx.Process(target=_ddp_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=300) for _ in range(2))
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    (_, log0, sum0, mx0), (_, log1, sum1, mx1) = res
    print(log0, log1)
    assert log0 == log1                               # (applied steps, found-inf) and the skip, step by step, on both ranks
    assert [e[1] for e in log0] == [False, False, True, False, False, False]
    assert log0[2][0] == (2, 1) and log0[-1][0] == (5, 0)
    assert sum0 == sum1 and mx0 == mx1                # the replicas stay bit-identical


# ---------------------------------------------------------------------------------------------------------------- convergence
def test_fp16_fit_lowers_the_training_loss_as_bf16_does():
    from multipitch_architectures_b200.loop import fit
    from tests.refshapes import build_model
    from tests.test_gpu_ext import _toy_sets
    hist = {}
    for prec in ('bf16', 'fp16'):
        torch.manual_seed(7)
        m = build_model('cnn_xs', precision=prec).cuda()
        h = fit(m, _toy_sets(2, 150, 1, {}), None, batch_size=16, lr=2e-3, max_epochs=4, max_batches_per_epoch=10, seed=5, graph=True,
                scheduler=False, early=False, log=lambda s: None)
        hist[prec] = [r['train_loss'] for r in h]
    print('train loss per epoch', hist)
    for prec, tl in hist.items():
        assert np.isfinite(tl).all() and tl[-1] < tl[0], prec
    assert abs(hist['fp16'][-1] - hist['bf16'][-1]) < 0.1 * hist['bf16'][0]
