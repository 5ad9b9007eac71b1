"""`-m gpu`: training path of the U-Net family (SURVEY 8a N4-N9/N11, configuration 5).  Backward kernels against torch autograd
of the same op; whole-model loss / gradients / BatchNorm running statistics against the REFERENCE goldens
(tests/golden/nn_train_golden.npz: loss.backward() on the unmodified reference modules in train mode); the fused
UnetTrainStep (BCE [+ CE/25] + backward + AdamW kernels) against torch.optim.AdamW driving the oracle."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.refshapes import build_model
from tests.weights import MODEL_SPECS, fill_state_dict, synth_patches, synth_targets

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def train_golden():
    return np.load(os.path.join(ROOT, 'tests', 'golden', 'nn_train_golden.npz'))


def rnd(*shape, seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g) * scale


def _call(name, *a):
    from multipitch_architectures_b200 import _lib
    _lib.call(name, *a, _lib.stream_ptr())


def test_bn_relu_bwd():
    B, C, H, W = 3, 5, 9, 13
    x = rnd(B, C, H, W, seed=1).requires_grad_(True)
    w, b = (1 + 0.2 * rnd(C, seed=2)).requires_grad_(True), (0.1 * rnd(C, seed=3)).requires_grad_(True)
    y = torch.relu(F.batch_norm(x, None, None, w, b, training=True, eps=1e-5))
    g = rnd(B, C, H, W, seed=4)
    y.backward(g)
    from multipitch_architectures_b200 import ops
    xc = x.detach().cuda()
    stats = ops.bn_stats(xc)
    out = ops.bn_apply(xc, stats, w.detach().cuda(), b.detach().cuda(), 1e-5, ops.ACT_RELU, 0.0)
    assert (out.cpu() - y.detach()).abs().max() < 1e-5
    dx, dw, db, scr = torch.empty_like(xc), torch.empty(C).cuda(), torch.empty(C).cuda(), torch.empty(2 * C).cuda()
    _call('bn_relu_bwd_f32', xc, out, g.cuda(), stats, w.detach().cuda(), dx, dw, db, scr, B, C, H * W, 1e-5, 1)
    assert (dx.cpu() - x.grad).abs().max() < 2e-5
    assert (dw.cpu() - w.grad).abs().max() < 1e-4 and (db.cpu() - b.grad).abs().max() < 1e-4


@pytest.mark.parametrize('k,s,shape', [((2, 2), (2, 2), (2, 3, 9, 27)), ((2, 2), (2, 2), (2, 3, 75, 216)), ((2, 5), (1, 2), (3, 4, 3, 9))])
def test_maxpool2d_bwd(k, s, shape):
    x = rnd(*shape, seed=5).requires_grad_(True)
    y = F.max_pool2d(x, k, s)
    g = rnd(*y.shape, seed=6)
    y.backward(g)
    gi = torch.empty(*shape).cuda()
    B, C, H, W = shape
    _call('maxpool2d_bwd_f32', x.detach().cuda(), g.cuda(), gi, B, C, H, W, k[0], k[1], s[0], s[1])
    assert (gi.cpu() - x.grad).abs().max() < 1e-6


@pytest.mark.parametrize('lo,sk', [((2, 3, 4, 13), (2, 5, 9, 27)), ((2, 4, 9, 27), (2, 2, 18, 54)), ((1, 2, 37, 108), (1, 3, 75, 216))])
def test_upsample_concat_bwd(lo, sk):
    from oracle import nn_oracle as NO
    low, skip = rnd(*lo, seed=7).requires_grad_(True), rnd(*sk, seed=8).requires_grad_(True)
    cat = NO.upconcat(low, skip)
    g = rnd(*cat.shape, seed=9)
    cat.backward(g)
    g_skip, g_low = torch.empty(*sk).cuda(), torch.empty(*lo).cuda()
    _call('upsample2x_concat_bwd_f32', g.cuda(), g_skip, 0, g_low, lo[0], lo[1], lo[2], lo[3], sk[1], sk[2], sk[3])
    assert (g_skip.cpu() - skip.grad).abs().max() < 1e-6
    assert (g_low.cpu() - low.grad).abs().max() < 1e-5


def test_attention_and_layernorm_bwd():
    B, S, E, H = 5, 7, 32, 8
    hd = E // H
    qkv = rnd(B * S, 3 * E, seed=10).requires_grad_(True)
    q, k, v = [qkv[:, i * E:(i + 1) * E].reshape(B, S, H, hd).permute(1, 2, 0, 3) for i in range(3)]
    att = torch.softmax((q @ k.transpose(-1, -2)) / hd ** 0.5, dim=-1)
    o = (att @ v).permute(2, 0, 1, 3).reshape(B * S, E)
    g = rnd(B * S, E, seed=11)
    o.backward(g)
    oc, gq = torch.empty(B * S, E).cuda(), torch.empty(B * S, 3 * E).cuda()
    _call('batch_axis_attention_f32', qkv.detach().cuda(), oc, B, S, E, H)
    assert (oc.cpu() - o.detach()).abs().max() < 1e-5
    _call('batch_axis_attention_bwd_f32', qkv.detach().cuda(), g.cuda(), gq, B, S, E, H)
    assert (gq.cpu() - qkv.grad).abs().max() < 1e-5
    from multipitch_architectures_b200 import _lib
    u = rnd(B * S, E, seed=12).requires_grad_(True)
    w, b = (1 + 0.1 * rnd(E, seed=13)).requires_grad_(True), (0.1 * rnd(E, seed=14)).requires_grad_(True)
    F.layer_norm(u, (E,), w, b, 1e-5).backward(g)
    gu, gw, gb = torch.empty(B * S, E).cuda(), torch.empty(E).cuda(), torch.empty(E).cuda()
    _lib.call('layernorm_tok_bwd_f32', u.detach().cuda(), g.cuda(), w.detach().cuda(), gu, gw, gb, _lib.i64(B * S), E, 1e-5, _lib.stream_ptr())
    assert (gu.cpu() - u.grad).abs().max() < 1e-5
    assert (gw.cpu() - w.grad).abs().max() < 1e-4 and (gb.cpu() - b.grad).abs().max() < 1e-4


def test_gemm_modes_colsum_ce():
    A, Bm = rnd(37, 19, seed=15), rnd(19, 70, seed=16)
    C = torch.empty(37, 70).cuda()
    _call('gemm_f32', A.cuda(), Bm.cuda(), C, 37, 70, 19, 0, 0)
    assert (C.cpu() - A @ Bm).abs().max() < 1e-4
    At = rnd(19, 37, seed=17)
    _call('gemm_f32', At.cuda(), Bm.cuda(), C, 37, 70, 19, 1, 1)
    assert (C.cpu() - (A @ Bm + At.T @ Bm)).abs().max() < 1e-4
    s = torch.empty(70).cuda()
    _call('colsum_f32', Bm.cuda(), s, 19, 70)
    assert (s.cpu() - Bm.sum(0)).abs().max() < 1e-5
    logits = rnd(6, 24, seed=18).requires_grad_(True)
    yt = synth_targets(6, 3).reshape(6, 72)
    yt[0, :30] = 1.0                                              # class index clamps at K-1 (the reference would raise)
    cls = yt.sum(-1).long().clamp(max=23)
    loss = F.cross_entropy(logits, cls) / 25.0
    loss.backward()
    ls, gl = torch.zeros(1).cuda(), torch.empty(6, 24).cuda()
    _call('ce_count_fwd_bwd_f32', logits.detach().cuda(), yt.cuda(), ls, gl, 6, 24, 72, 1.0 / 25.0, 0)
    assert abs(ls.item() - loss.item()) < 1e-6 and (gl.cpu() - logits.grad).abs().max() < 1e-7


def _zero_dropout(m):
    m.p_dropout = 0.0
    for mod in m.modules():
        if hasattr(mod, 'p_dropout'):
            mod.p_dropout = 0.0


@pytest.mark.parametrize('name', ['unet_tiny', 'saunet_tiny', 'punet_tiny', 'sausnet_tiny'])
def test_model_loss_grads_and_running_stats_match_reference_golden(train_golden, name):
    tag = f'{name}__train'
    B, seed = [int(v) for v in train_golden[tag + '__meta']]
    m = build_model(name)
    m.load_state_dict(fill_state_dict(m.state_dict(), seed))
    _zero_dropout(m)
    m = m.cuda().train()
    x, t = synth_patches(B, seed).cuda(), synth_targets(B, seed).cuda()
    y = m(x)                                                    # autograd path (training.TrainFunction)
    if isinstance(y, tuple):
        y, n_pred = y
        assert np.abs(n_pred.detach().cpu().numpy() - train_golden[tag + '__n']).max() < 1e-3
        n_target = torch.sum(t, dim=-1, keepdims=True).long().squeeze(3)
        loss = torch.nn.BCELoss(reduction='mean')(y, t) + torch.nn.CrossEntropyLoss(reduction='mean')(n_pred, n_target) / 25.0
    else:
        loss = torch.nn.BCELoss(reduction='mean')(y, t)
    assert np.abs(y.detach().cpu().numpy() - train_golden[tag + '__y']).max() < 1e-3
    loss.backward()
    assert abs(loss.item() - float(train_golden[tag + '__loss'][0])) < 2e-5
    worst = 0.0
    # conv biases in front of a train-mode BatchNorm have a mathematically zero gradient (rounding noise on both sides): every
    # tensor is judged against max(its own scale, 1e-3 of the largest gradient in the model)
    gmax = max(np.abs(train_golden[tag + '__grad__' + k]).max() for k, _ in m.named_parameters())
    for k, p in m.named_parameters():
        g = train_golden[tag + '__grad__' + k]
        d = np.abs(p.grad.cpu().numpy() - g)
        scale = max(np.abs(g).max(), 1e-3 * gmax)
        worst = max(worst, d.max() / scale)
        # fp32 summation-order noise + rare max-pool / ReLU near-tie flips: bound the maximum loosely and the mean tightly
        # (a single max-pool / ReLU near-tie that flips moves a few elements by several per cent: bound the bulk tightly, outliers loosely)
        assert d.max() <= 0.25 * scale and (d.mean() <= 1e-2 * scale or d.size < 64) and (d.size < 1024 or (d > 2e-2 * scale).mean() <= 0.01), \
            (k, d.max() / scale, d.mean() / scale)
    print(f'{tag}: worst relative gradient deviation {worst:.2e}')
    for k, v in m.state_dict().items():
        if 'running_' in k:
            assert np.abs(v.cpu().numpy() - train_golden[tag + '__stat__' + k]).max() < 1e-4, k


@pytest.mark.parametrize('name', ['saunet_tiny', 'punet_tiny'])
def test_fused_train_step_matches_torch_adamw_on_oracle(name):
    from oracle import nn_oracle as NO
    from multipitch_architectures_b200.training_unet import UnetTrainStep
    m = build_model(name)
    sd0 = fill_state_dict(m.state_dict(), 33)
    m.load_state_dict(sd0)
    _zero_dropout(m)
    m = m.cuda().train()
    step = UnetTrainStep(m, lr=1e-3, weight_decay=0.01)
    ref = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and 'running_' not in k else v.clone()) for k, v in sd0.items()}
    params = [v for v in ref.values() if v.requires_grad]
    opt = torch.optim.AdamW(params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.01)
    pe = MODEL_SPECS[name]['kw'].get('pos_encoding')
    for it in range(2):
        x, t = synth_patches(4, 60 + it), synth_targets(4, 60 + it)
        l_gpu = step(x.cuda(), t.cuda()).item()
        opt.zero_grad()
        y = NO.unet_forward(ref, x, train=True, pos_encoding=pe)
        if isinstance(y, tuple):
            y, n_pred = y
            l_ref = NO.bce_mean(y, t) + F.cross_entropy(n_pred, t.sum(-1, keepdim=True).long().squeeze(3)) / 25.0
        else:
            l_ref = NO.bce_mean(y, t)
        l_ref.backward()
        opt.step()
        assert abs(l_gpu - l_ref.item()) < 5e-4 * max(1.0, abs(l_ref.item())), (it, l_gpu, l_ref.item())
    # inference after training sees the updated weights
    m.eval()


def test_train_mode_dropout_is_active_and_deterministic():
    m = build_model('saunet_tiny')
    m.load_state_dict(fill_state_dict(m.state_dict(), 35))
    m = m.cuda().train()
    x = synth_patches(3, 70).cuda()
    with torch.no_grad():
        m._train_calls = 0
        y1 = m(x)
        m._train_calls = 0
        y2 = m(x)
        y3 = m(x)
    assert torch.equal(y1, y2) and not torch.equal(y1, y3)


def _loss_and_grads(name, precision, scheme, seed, B):
    m = build_model(name, precision=precision)
    m.load_state_dict(fill_state_dict(m.state_dict(), seed, scheme=scheme))
    _zero_dropout(m)
    m = m.cuda().train()
    x, t = synth_patches(B, seed).cuda(), synth_targets(B, seed).cuda()
    y = m(x)
    if isinstance(y, tuple):
        y, n_pred = y
        n_target = torch.sum(t, dim=-1, keepdims=True).long().squeeze(3)
        loss = torch.nn.BCELoss(reduction='mean')(y, t) + torch.nn.CrossEntropyLoss(reduction='mean')(n_pred, n_target) / 25.0
    else:
        loss = torch.nn.BCELoss(reduction='mean')(y, t)
    loss.backward()
    return loss.item(), {k: p.grad.cpu().numpy() for k, p in m.named_parameters()}


def _cosines(ga, gb):
    dots = n1 = n2 = 0.0
    worst = (1.0, '')
    gnorm = sum(float((g ** 2).sum()) for g in gb.values()) ** 0.5
    for k, g in gb.items():
        d = ga[k]
        assert np.isfinite(d).all(), k
        dd, gg, dg = float((d * d).sum()), float((g * g).sum()), float((d * g).sum())
        dots += dg; n1 += dd; n2 += gg
        if gg ** 0.5 > 1e-2 * gnorm:                      # tensors that carry a visible share of the gradient
            worst = min(worst, (dg / max(dd ** 0.5 * gg ** 0.5, 1e-30), k))
    return dots / (n1 ** 0.5 * n2 ** 0.5), worst


@pytest.mark.parametrize('name,scheme,min_cos,min_worst', [
    ('cnn_xs', 'adversarial', 0.999, 0.98), ('drcnn_tiny', 'adversarial', 0.999, 0.98),
    ('unet_tiny', 'torch_default', 0.95, 0.80), ('saunet_tiny', 'torch_default', 0.96, 0.80), ('punet_tiny', 'torch_default', 0.90, 0.80),
    ('unet_tiny', 'adversarial', 0.83, 0.60), ('saunet_tiny', 'adversarial', 0.95, 0.80), ('punet_tiny', 'adversarial', 0.87, 0.75),
    ('sausnet_tiny', 'torch_default', 0.90, 0.75)])
def test_bf16_tensor_core_training_tracks_the_fp32_path(name, scheme, min_cos, min_worst):
    """precision='bf16': every stride-1 'same' convolution runs forward / data-gradient / weight-gradient on the tensor cores
    (16-bit operands, fp32 accumulate; layer-level parity <= 4e-3 is in test_gpu_wgrad_tc.py).  Model-level stated bound against the
    fp32 path (itself pinned to the reference's loss.backward()): loss within 2 %; cosine similarity of the whole gradient and of
    every tensor carrying >= 1 % of its norm as parametrised.  CNN family: >= 0.999.  U-Net family: train-mode BatchNorm over a batch
    of 3 amplifies the bf16 rounding of the convolution outputs; the bounds sit just below what the ORACLE gives when its convolutions
    are run with bf16-rounded operands and outputs on the CPU (same seeds: unet 0.969 / 0.875, punet 0.912 / 0.890 for default-init /
    adversarial weights; measured here 0.966 / 0.855 and 0.918 / 0.894), i.e. the deviation is the format's, not the kernels'."""
    B, seed = 3, 41
    l32, g32 = _loss_and_grads(name, 'fp32', scheme, seed, B)
    l16, g16 = _loss_and_grads(name, 'bf16', scheme, seed, B)
    cos, worst = _cosines(g16, g32)
    print(f'{name}/{scheme}: loss bf16 {l16:.5f} fp32 {l32:.5f}; gradient cosine {cos:.5f}; worst tensor {worst[1]} {worst[0]:.4f}')
    assert abs(l16 - l32) < 2e-2 * max(1.0, abs(l32))
    assert cos >= min_cos and worst[0] >= min_worst


def test_sausnet_eval_fp32_matches_reference_and_tensor_core_path_matches_fp32(train_golden):
    """simple_u_net_doubleselfattn_twolayers (SAUSnet): eval output of the fp32 path against the reference's own output; the tcgen05
    path (BatchNorm folded, attention on the bottleneck and on the lowest skip) against the fp32 path on a chunk-aligned variant."""
    tag = 'sausnet_tiny__train'
    B, seed = [int(v) for v in train_golden[tag + '__meta']]
    m = build_model('sausnet_tiny')
    m.load_state_dict(fill_state_dict(m.state_dict(), seed))
    m = m.cuda().eval()
    with torch.no_grad():
        y = m(synth_patches(B, seed).cuda())
    assert np.abs(y.cpu().numpy() - train_golden[tag + '__eval_y']).max() < 1e-3
    x = synth_patches(4, 77).cuda()
    outs = {}
    for prec in ('fp32', 'fp16'):
        m = build_model('sausnet_s8', precision=prec)
        m.load_state_dict(fill_state_dict(m.state_dict(), 78, scheme='torch_default'))
        m = m.cuda().eval()
        with torch.no_grad():
            outs[prec] = m(x)
    assert (outs['fp16'] - outs['fp32']).abs().max().item() < 1e-3


def test_graph_replayed_step_equals_eager_step():
    """UnetTrainStep(graph=True): steps 3.. replay ONE captured forward+backward CUDA graph; with dropout on, every replayed step must be the
    eager step of the same number (dropout offsets come from the device-side step counter).  The learning rate is tiny so that the fp32-atomic
    noise of the weight-gradient kernels is not amplified through the parameters: the loss of step k then depends on the data and the
    dropout masks of step k only (a wrong mask moves it by ~1e-2)."""
    from multipitch_architectures_b200.training_unet import UnetTrainStep
    from tests.refshapes import build_model
    from tests.weights import fill_state_dict, synth_patches, synth_targets
    res = {}
    for mode in (False, True):
        m = build_model('saunet_tiny', precision='bf16')
        m.load_state_dict(fill_state_dict(m.state_dict(), 5, scheme='torch_default'))
        m = m.cuda().train()
        assert m.p_dropout > 0
        step = UnetTrainStep(m, lr=1e-6, graph=mode)
        losses = []
        for i in range(6):
            x, y = synth_patches(5, 50 + i).cuda(), synth_targets(5, 50 + i).cuda()
            losses.append(float(step(x, y).item()))
        res[mode] = (losses, step.flat_p.clone())
        if mode:
            assert step.replays == 4 and step.launches_per_replay > 100
    le, lg = res[False][0], res[True][0]
    print('eager', le, 'graph', lg)
    assert all(abs(a - b) <= 2e-4 * max(1.0, abs(a)) for a, b in zip(le, lg))
    assert len(set(round(v, 4) for v in lg)) == len(lg)                   # every step saw its own data / masks
    assert (res[False][1] - res[True][1]).abs().max().item() < 1e-5       # fp32 atomics (split-K, wgrad flush) are not order-stable


# ---------------------------------------------------------------------------------------------------------------------------------
# full-size SAUnet:L (BASELINE configs[4]): the reference's loss.backward() and a bf16-vs-fp32 training run
def _sample_index(numel, k=256):
    return np.arange(numel) if numel <= k else (np.arange(k, dtype=np.int64) * numel) // k


@pytest.fixture(scope='module')
def saunet_l_golden():
    import os
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'saunet_l_train_golden.npz'))


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_full_size_saunet_l_loss_and_gradients_vs_reference(saunet_l_golden, precision):
    """SAUnet:L [128,80,50,30] sc=4 E=128 mlp=8192 (8.1 M parameters), train mode, batch 4: loss, outputs, BatchNorm running statistics and
    every parameter gradient (norm + a 256-element sample per tensor) against the REFERENCE class's loss.backward()
    (tests/golden/make_golden.py saunet_l_train).  fp32 path: 1e-3 relative; bf16 tensor-core path: its stated looser bound."""
    g = saunet_l_golden
    tag = 'saunet_l__train'
    B, seed = [int(v) for v in g[tag + '__meta']]
    m = build_model('saunet_l', precision=precision)
    m.load_state_dict(fill_state_dict(m.state_dict(), seed, scheme='torch_default'))
    _zero_dropout(m)
    m = m.cuda().train()
    x, t = synth_patches(B, seed).cuda(), synth_targets(B, seed).cuda()
    y = m(x)
    loss = torch.nn.BCELoss(reduction='mean')(y, t)
    loss.backward()
    fp32 = precision == 'fp32'
    assert abs(loss.item() - float(g[tag + '__loss'][0])) < (1e-5 if fp32 else 2e-3)
    assert np.abs(y.detach().cpu().numpy() - g[tag + '__y']).max() < (1e-4 if fp32 else 5e-3)
    dots = n1 = n2 = 0.0
    gnorm_total = sum(float(g[k][0]) ** 2 for k in g.files if '__gnorm__' in k) ** 0.5
    worst = (1.0, '')
    for k, p in m.named_parameters():
        got = p.grad.detach().float().cpu().numpy().reshape(-1)
        ref_norm, ref_s = float(g[tag + '__gnorm__' + k][0]), g[tag + '__gsamp__' + k]
        got_s = got[_sample_index(got.size)]
        assert np.isfinite(got).all(), k
        if fp32 and ref_norm > 1e-3 * gnorm_total:
            assert abs(np.sqrt((got.astype(np.float64) ** 2).sum()) - ref_norm) < 1e-2 * ref_norm, k
            # element-wise: train-mode BatchNorm over a batch of 4 amplifies the fp32 summation-order differences between the two
            # implementations to ~1 % of a tensor's largest gradient entry; the cosine below is the tight check
            assert np.abs(got_s - ref_s).max() < 5e-2 * max(np.abs(ref_s).max(), 1e-12) + 1e-7, k
        dg, dd, gg = float((got_s * ref_s).sum()), float((got_s ** 2).sum()), float((ref_s ** 2).sum())
        dots += dg; n1 += dd; n2 += gg
        if ref_norm > 1e-2 * gnorm_total:
            worst = min(worst, (dg / max(dd ** 0.5 * gg ** 0.5, 1e-30), k))
    cos = dots / (n1 ** 0.5 * n2 ** 0.5)
    print(f'SAUnet:L {precision}: loss {loss.item():.6f} (reference {float(g[tag + "__loss"][0]):.6f}); sampled-gradient cosine {cos:.5f}; worst tensor {worst[1]} {worst[0]:.4f}')
    assert cos > (0.9999 if fp32 else 0.97) and worst[0] > (0.999 if fp32 else 0.80)      # bf16 observed: 0.998 / 0.857
    if fp32:
        for k, v in m.state_dict().items():
            if 'running_' in k:
                assert np.abs(v.cpu().numpy() - g[tag + '__stat__' + k]).max() < 1e-4, k


def test_saunet_l_bf16_training_run_follows_the_fp32_run():
    """60 optimiser steps of the full-size SAUnet:L on the same 6 cycling batches of 25 patches (dropout on, same masks: the Philox offsets
    depend on the step number only), once on the fp32 CUDA-core path and once on the bf16 tensor-core path: the two loss curves must
    stay together (the model memorises the batches: the loss falls by > 25 %; smoothed curves within 6 % of each other on average, no point
    further apart than 25 % of the initial loss, the plateaus within 15 % of each other)."""
    from multipitch_architectures_b200.training_unet import UnetTrainStep
    curves = {}
    data = [(synth_patches(25, 900 + i).cuda(), synth_targets(25, 900 + i).cuda()) for i in range(6)]
    for precision in ('fp32', 'bf16'):
        m = build_model('saunet_l', precision=precision)
        m.load_state_dict(fill_state_dict(m.state_dict(), 3, scheme='torch_default'))
        m = m.cuda().train()
        step = UnetTrainStep(m, lr=1e-3, weight_decay=0.01, graph=(precision == 'bf16'))
        curves[precision] = [float(step(*data[i % 6]).item()) for i in range(60)]
        step.release()
    a, b = np.array(curves['fp32']), np.array(curves['bf16'])
    sm = lambda v: np.convolve(v, np.ones(6) / 6, mode='valid')
    print('fp32 loss', np.round(sm(a)[::9], 4), 'bf16 loss', np.round(sm(b)[::9], 4))
    assert np.isfinite(a).all() and np.isfinite(b).all()
    assert sm(a)[-1] < 0.75 * sm(a)[0] and sm(b)[-1] < 0.75 * sm(b)[0]
    # The steep steps 3-12 at lr 1e-3 are chaotic: two runs of the SAME precision already wander apart there when the summation order of the
    # fp32 atomics changes (observed between repeated bf16 runs: up to 0.03 of 0.285, i.e. 15 % of the local loss), so the point-wise bound
    # only catches gross divergence; the curve as a whole and the plateau are held tightly.
    dev = np.abs(sm(a) - sm(b))
    print('max deviation', dev.max(), 'mean deviation', dev.mean(), 'plateau', a[-12:].mean(), b[-12:].mean())
    assert dev.max() < 0.25 * sm(a).max()
    assert dev.mean() < 0.06 * sm(a).mean()
    # plateau (memorising phase, still falling): observed over repeated runs fp32 0.155-0.162, bf16 0.148-0.168 (the runs are chaotic and the
    # atomics' summation order changes from run to run): within 15 % of each other
    assert abs(a[-12:].mean() - b[-12:].mean()) < 0.15 * a[-12:].mean()
    assert abs(a[0] - b[0]) < 2e-3 * a[0]


@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_fused_attention_half_equals_the_stage_by_stage_path(precision):
    """enc_train.cu (one CTA per bottleneck position; fold / fold-backward in one launch each) against the separate GEMM / attention /
    LayerNorm launches, dropout ON (p = 0.2, same Philox sites): loss and every gradient agree to fp32 summation-order noise."""
    from multipitch_architectures_b200 import training_unet
    from multipitch_architectures_b200.libdl import nn_models as M
    res = {}
    for fused in (True, False):
        m = M.simple_u_net_doubleselfattn(n_chan_input=6, n_chan_layers=[16, 10, 8, 5], n_bins_in=216, n_bins_out=72, scalefac=8, embed_dim=64,
                                          num_heads=8, mlp_dim=128, pos_encoding='sinusoidal', precision=precision)
        m.load_state_dict(fill_state_dict(m.state_dict(), 11, scheme='torch_default'))
        m = m.cuda().train()
        x, t = synth_patches(5, 11).cuda(), synth_targets(5, 11).cuda()
        old = training_unet.ENC_FUSED
        training_unet.ENC_FUSED = fused
        try:
            m._train_calls = 0
            y = m(x)
            loss = torch.nn.BCELoss(reduction='mean')(y, t)
            loss.backward()
        finally:
            training_unet.ENC_FUSED = old
        res[fused] = (loss.item(), y.detach().cpu().numpy(), {k: p.grad.cpu().numpy() for k, p in m.named_parameters()})
    (la, ya, ga), (lb, yb, gb) = res[True], res[False]
    tol = 1e-5 if precision == 'fp32' else 2e-3        # bf16: the MLP GEMMs round their (slightly different) inputs to 16 bits
    assert abs(la - lb) < tol * abs(lb) and np.abs(ya - yb).max() < 10 * tol
    cos, worst = _cosines(ga, gb)
    print(f'fused vs staged ({precision}): gradient cosine {cos:.7f}, worst tensor {worst[1]} {worst[0]:.6f}')
    # bf16: the two attention halves differ by ~1e-6; where that flips a 16-bit rounding of the bottleneck the flip travels through the
    # decoder and the trunk's backward, whose bf16 gradients carry rounding noise of ~25 % of their norm on this tiny-batch model anyway
    # (cosine 0.96 against fp32, tests/test_gpu_unet_cp8.py) — observed 0.99999 without and 0.993 / 0.96 (one tensor) with such flips
    assert cos > (0.99999 if precision == 'fp32' else 0.985) and worst[0] > (0.9999 if precision == 'fp32' else 0.93)
    if precision == 'fp32':
        for k in ga:
            if 'attention' in k:
                assert np.abs(ga[k] - gb[k]).max() < 1e-4 * max(np.abs(gb[k]).max(), 1e-6) + 1e-7, k
