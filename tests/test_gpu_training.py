"""`-m gpu`: training path (SURVEY 8a N2/N11, configuration 2) — backward kernels against torch autograd of the same op,
whole-model loss/gradients against the REFERENCE goldens (loss.backward() on the reference modules), and the fused
TrainStep (BCE + backward + AdamW kernels) against torch.optim.AdamW driving the oracle."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F
import torch.nn.functional as F_

from tests.refshapes import build_model
from tests.weights import fill_state_dict, synth_patches, synth_targets

pytestmark = pytest.mark.gpu


def rnd(*shape, seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g) * scale


@pytest.mark.parametrize('cfg', [
    # B, Cin, Cout, H, W, KH, KW, sh, sw, ph, pw
    (3, 6, 20, 30, 216, 15, 15, 1, 1, 7, 7), (2, 20, 20, 75, 216, 3, 3, 1, 3, 1, 0), (4, 20, 10, 75, 72, 75, 1, 1, 1, 0, 0),
    (4, 10, 1, 1, 72, 1, 1, 1, 1, 0, 0), (2, 8, 8, 20, 50, 15, 15, 1, 1, 7, 7), (2, 40, 40, 12, 40, 15, 15, 1, 1, 7, 7),
])
def test_conv_dgrad_wgrad(cfg):
    import torch.nn as nn
    from multipitch_architectures_b200 import training as TR
    B, Cin, Cout, H, W, KH, KW, sh, sw, ph, pw = cfg
    conv = nn.Conv2d(Cin, Cout, (KH, KW), stride=(sh, sw), padding=(ph, pw))
    x = rnd(B, Cin, H, W, seed=1).requires_grad_(True)
    y = conv(x)
    g = rnd(*y.shape, seed=2)
    y.backward(g)
    convc = nn.Conv2d(Cin, Cout, (KH, KW), stride=(sh, sw), padding=(ph, pw)).cuda()
    convc.load_state_dict(conv.state_dict())
    gi = TR._dgrad(convc, g.cuda(), x.shape).cpu()
    assert (gi - x.grad).abs().max() < 2e-5 * max(1.0, x.grad.abs().max().item())
    gw, gb = torch.empty_like(convc.weight), torch.empty_like(convc.bias)
    TR._wgrad(convc, x.detach().cuda(), g.cuda(), gw, gb)
    assert (gw.cpu() - conv.weight.grad).abs().max() < 1e-4 * max(1.0, conv.weight.grad.abs().max().item())
    assert (gb.cpu() - conv.bias.grad).abs().max() < 1e-4 * max(1.0, conv.bias.grad.abs().max().item())


@pytest.mark.parametrize('k', [3, 13])
def test_pool_act_bwd_and_dropout(k):
    from multipitch_architectures_b200 import training as TR, ops
    y = rnd(2, 5, 75, 40, seed=3).requires_grad_(True)
    a = F.leaky_relu(y, 0.3)
    p = F.max_pool2d(a, (k, 1), (1, 1), (k // 2, 0))
    g = rnd(*p.shape, seed=4)
    p.backward(g)
    got = TR._pool_bwd(a.detach().cuda(), g.cuda(), k, ops.ACT_LRELU, 0.3).cpu()
    assert (got - y.grad).abs().max() < 1e-5      # up to k windows add into one row in arbitrary order
    x = torch.ones(100003).cuda()
    d = TR._dropout(x, 0.2, 7, 3)
    keep = (d != 0).float().mean().item()
    assert abs(keep - 0.8) < 0.01 and abs(d.max().item() - 1.25) < 1e-6
    assert torch.equal(d, TR._dropout(x, 0.2, 7, 3)) and not torch.equal(d, TR._dropout(x, 0.2, 7, 4))


@pytest.mark.parametrize('name', ['cnn_xs', 'drcnn_tiny'])
def test_model_loss_and_grads_match_reference_golden(nn_golden, name):
    tag = f'{name}__eval'
    B, seed, _ = nn_golden[tag + '__meta']
    B, seed = int(B), int(seed)
    m = build_model(name)
    m.load_state_dict(fill_state_dict(m.state_dict(), seed))
    m.p_dropout = 0.0
    m = m.cuda().train()
    x, t = synth_patches(B, seed).cuda(), synth_targets(B, seed).cuda()
    y = m(x)                                                    # autograd path (training.TrainFunction)
    loss = torch.nn.BCELoss(reduction='mean')(y, t)
    loss.backward()
    assert abs(loss.item() - float(nn_golden[tag + '__loss'][0])) < 1e-5
    for k, p in m.named_parameters():
        g = nn_golden[tag + '__grad__' + k]
        d = np.abs(p.grad.cpu().numpy() - g)
        # fp32 summation-order noise of 48600-term signed sums + max-pool near-tie flips (see test_oracle_pinned.py)
        assert d.max() <= 5e-3 * np.abs(g).max() and d.mean() <= 1e-3 * np.abs(g).max(), k


def test_fused_train_step_matches_torch_adamw_on_oracle():
    from oracle import nn_oracle as NO
    from multipitch_architectures_b200.training import TrainStep
    m = build_model('cnn_xs')
    sd0 = fill_state_dict(m.state_dict(), 31)
    m.load_state_dict(sd0)
    m.p_dropout = 0.0
    m = m.cuda().train()
    step = TrainStep(m, lr=1e-3, weight_decay=0.01)
    ref = {k: v.clone().requires_grad_(True) for k, v in sd0.items()}
    opt = torch.optim.AdamW(list(ref.values()), lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.01)
    losses = []
    for it in range(3):
        x, t = synth_patches(4, 40 + it), synth_targets(4, 40 + it)
        l_gpu = step(x.cuda(), t.cuda()).item()
        opt.zero_grad()
        l_ref = NO.bce_mean(NO.cnn_forward(ref, x), t)
        l_ref.backward()
        opt.step()
        losses.append((l_gpu, l_ref.item()))
        assert abs(l_gpu - l_ref.item()) < 2e-4 * max(1.0, abs(l_ref.item())), losses
    for k, p in m.named_parameters():
        # Adam's first steps move every weight by ~lr regardless of gradient scale; compare the UPDATE, not the value
        upd_ref = (ref[k].detach() - sd0[k])
        upd_gpu = (p.detach().cpu() - sd0[k])
        # elements whose gradient is at fp32-noise level at some step get a random +-lr there (sign of m/sqrt(v)), so
        # bound the mean and the share of outliers rather than the maximum
        d = (upd_gpu - upd_ref).abs()
        assert d.mean() < 0.02 * 3e-3 and (d > 0.3e-3).float().mean() < 0.02, k
    # inference after training sees the updated weights (packed-operand cache invalidated)
    m.eval()
    x = synth_patches(2, 50)
    with torch.no_grad():
        y = m(x.cuda()).cpu()
        yr = NO.cnn_forward({k: v.detach() for k, v in ref.items()}, x)
    assert (y - yr).abs().max() < 1e-3


def test_wide_cnn_head_conv4_stays_on_the_fp32_row_kernels(monkeypatch):
    """bf16 CNN whose conv3 and conv4.0 both have more than 10 output channels: conv3 takes the tensor-core GEMMs, conv4.0 (one-row 1x1
    after conv3) the fp32 conv_rows kernels, in the fused step and in the autograd path."""
    from multipitch_architectures_b200 import training as TR
    from multipitch_architectures_b200.libdl import nn_models as M
    calls = []

    def spy(name):
        orig = getattr(TR, name)

        def fn(conv, *args):
            calls.append((name, tuple(conv.weight.shape)))
            return orig(conv, *args)
        return fn
    for name in ('_rows_tc_forward', '_rows_tc_backward'):
        monkeypatch.setattr(TR, name, spy(name))
    m = M.basic_cnn_segm_sigmoid(n_chan_input=6, n_chan_layers=[20, 20, 16, 16], n_bins_in=216, n_bins_out=72, precision='bf16')
    m.load_state_dict(fill_state_dict(m.state_dict(), 3, scheme='torch_default'))
    m = m.cuda().train()
    x, t = synth_patches(3, 5).cuda(), synth_targets(3, 5).cuda()
    torch.nn.BCELoss()(m(x), t).backward()
    TR.TrainStep(m)(x, t)
    conv3 = tuple(m.conv3[0].weight.shape)
    assert calls == [('_rows_tc_forward', conv3), ('_rows_tc_backward', conv3)] * 2, calls


def test_cnn_graph_replayed_step_equals_eager_step():
    """TrainStep(graph=True): steps 3.. replay one captured forward+backward CUDA graph with dropout on; tiny learning rate so that the
    loss of step k depends on the data and the dropout masks of step k only."""
    from multipitch_architectures_b200.training import TrainStep
    from tests.refshapes import build_model
    from tests.weights import fill_state_dict, synth_patches, synth_targets
    res = {}
    for mode in (False, True):
        m = build_model('drcnn_tiny', precision='bf16')
        m.load_state_dict(fill_state_dict(m.state_dict(), 5, scheme='torch_default'))
        m = m.cuda().train()
        assert m.p_dropout > 0
        step = TrainStep(m, lr=1e-6, graph=mode)
        losses = []
        for i in range(6):
            losses.append(float(step(synth_patches(6, 70 + i).cuda(), synth_targets(6, 70 + i).cuda()).item()))
        res[mode] = losses
        if mode:
            assert step.replays == 4 and step.launches_per_replay > 20
    print('eager', res[False], 'graph', res[True])
    assert all(abs(a - b) <= 2e-4 * max(1.0, abs(a)) for a, b in zip(res[False], res[True]))
    assert len(set(round(v, 4) for v in res[True])) == 6


@pytest.mark.parametrize('B,C,F,p,act', [(3, 20, 72, 0.2, 'lrelu'), (2, 5, 216, 0.0, 'lrelu'), (1, 3, 8, 0.5, 'relu'), (2, 7, 36, 0.2, 'none')])
def test_pool13_backward_table_kernel(B, C, F, p, act):
    """backward.cu maxpool13_bwd_table_kernel (T = 75, k = 13: doubling-table first arg-max, shared-memory routing, quad-shared Philox
    draws) against torch autograd of MaxPool2d((13,1), 1, (6,0)) on plateau inputs (ties: the first maximum wins) and against
    dropout -> backward in two kernels (same masks)."""
    from multipitch_architectures_b200 import _lib, ops
    from multipitch_architectures_b200.training import ctypes_u64
    T, seed, off = 75, 0x5EED, 41
    code = {'lrelu': ops.ACT_LRELU, 'relu': ops.ACT_RELU, 'none': ops.ACT_NONE}[act]
    z = (rnd(B, C, T, F, seed=11) * 2).round() / 2 + 0.25     # plateaus: many ties inside a window; no exact zeros (the kernel's lrelu'(0) = 1)
    z.requires_grad_(True)
    a = {'lrelu': lambda v: F_.leaky_relu(v, 0.3), 'relu': F_.relu, 'none': lambda v: v}[act](z)
    g = rnd(B, C, T, F, seed=12)
    gm = torch.empty_like(g).cuda()
    if p > 0:
        _lib.call('dropout_f32', g.cuda(), gm, _lib.i64(g.numel()), float(p), ctypes_u64(seed), ctypes_u64(off), _lib.stream_ptr())
    else:
        gm.copy_(g)
    F_.max_pool2d(a, (13, 1), stride=1, padding=(6, 0)).backward(gm.cpu())
    got = torch.empty_like(gm)
    _lib.call('maxpool_time_bwd_dropout_f32', a.detach().cuda(), g.cuda(), got, B, C, T, F, 13, code, 0.3, float(p), ctypes_u64(seed), ctypes_u64(off),
              None, ctypes_u64(0), _lib.stream_ptr())
    assert (got.cpu() - z.grad).abs().max() <= 1e-6 * max(1.0, z.grad.abs().max().item())
    two = torch.empty_like(gm)
    _lib.call('maxpool_time_bwd_f32', a.detach().cuda(), gm, two, B, C, T, F, 13, code, 0.3, _lib.stream_ptr())
    assert torch.equal(two, got)
    # the generic column kernel (any T) on the same columns, cut to T - 1 rows where the last window differs: compare rows far from the cut
    a74, g74 = a.detach()[:, :, :74].contiguous().cuda(), gm[:, :, :74].contiguous()
    old = torch.empty_like(g74)
    _lib.call('maxpool_time_bwd_f32', a74, g74, old, B, C, 74, F, 13, code, 0.3, _lib.stream_ptr())
    assert torch.equal(old[:, :, :60], two[:, :, :60])


def test_fused_pool_dropout_kernels_equal_the_separate_kernels():
    """MaxPool -> Dropout (-> + residual) in one kernel and its backward with the mask re-drawn on the fly: bit-identical to
    maxpool_time -> dropout -> add and dropout -> maxpool_time_bwd (same Philox convention), through a whole training step."""
    from multipitch_architectures_b200 import training as TR
    from tests.refshapes import build_model
    from tests.weights import fill_state_dict, synth_patches, synth_targets
    res = {}
    for fuse in (True, False):
        TR.FUSE_POOL_DROPOUT = fuse
        try:
            m = build_model('drcnn_tiny')
            m.load_state_dict(fill_state_dict(m.state_dict(), 9, scheme='torch_default'))
            m = m.cuda().train()
            assert m.p_dropout > 0
            x, t = synth_patches(4, 81).cuda(), synth_targets(4, 81).cuda()
            m.dropout_seed, m._train_calls = 1234, 0
            y = m(x)
            loss = torch.nn.BCELoss()(y, t)
            loss.backward()
            res[fuse] = (y.detach().clone(), {k: p.grad.clone() for k, p in m.named_parameters()})
        finally:
            TR.FUSE_POOL_DROPOUT = True
    assert torch.equal(res[True][0], res[False][0])
    for k in res[True][1]:
        a, b = res[True][1][k], res[False][1][k]
        assert (a - b).abs().max().item() <= 1e-6 * max(1.0, b.abs().max().item()), k       # weight gradients meet in fp32 atomics


def _bf16_valued(*shape, seed=0, scale=1.0):
    return (rnd(*shape, seed=seed, scale=scale).bfloat16().float()).cuda()


@pytest.mark.parametrize('B,C,T,F,p', [(1, 5, 75, 216, 0.2), (3, 20, 75, 216, 0.2), (2, 8, 2, 40, 0.5), (2, 11, 1, 8, 0.2), (2, 20, 30, 216, 0.0)])
def test_cp8_pool_dropout_kernels_equal_the_nchw_kernels(B, C, T, F, p):
    """train_cp8.cu: MaxPool(3,1)+Dropout forward / backward and the bias-gradient sum on the 16-bit CP8 planes = the fp32 NCHW kernels
    behind the converters, bit for bit (same Philox element indexing, fp32 sums in the same order, one rounding on the store)."""
    from multipitch_architectures_b200 import _lib, ops
    from multipitch_architectures_b200.training import ctypes_u64
    fmt = ops.FMT_BF16
    seed, off = 0x1234, 77
    a = torch.where(_bf16_valued(B, C, T, F, seed=1) > 0.5, _bf16_valued(B, C, T, F, seed=1), torch.zeros(()).cuda()) - 0.25   # many ties
    a = a.bfloat16().float().contiguous()
    ac = ops.nchw_to_cp8(a, fmt=fmt)
    # forward
    want = torch.empty_like(a)
    if p > 0:
        _lib.call('maxpool_time_dropout_f32', a, None, want, B, C, T, F, 3, float(p), ctypes_u64(seed), ctypes_u64(off), None, ctypes_u64(0),
                  _lib.stream_ptr())
    else:
        want = ops.maxpool_time(a, 3)
    zc = ac.like()
    _lib.call('pool3_dropout_cp8', ac.ptr(), zc.ptr(), B, C, T, F, ac.pitch, ac.pf, ac.pt, fmt, float(p), ctypes_u64(seed), ctypes_u64(off), None,
              ctypes_u64(0), _lib.stream_ptr())
    assert torch.equal(ops.cp8_to_nchw(zc), want.bfloat16().float())
    assert torch.equal(zc.buf[..., :zc.pf, :], torch.zeros_like(zc.buf[..., :zc.pf, :])) and (zc.buf[:, :, 0] == 0).all()     # borders stay zero
    # backward
    g = _bf16_valued(B, C, T, F, seed=2)
    gc = ops.nchw_to_cp8(g, fmt=fmt)
    want = torch.empty_like(a)
    if T > 1:
        _lib.call('maxpool_time_bwd_dropout_f32', a, g, want, B, C, T, F, 3, ops.ACT_LRELU, 0.3, float(p), ctypes_u64(seed), ctypes_u64(off), None,
                  ctypes_u64(0), _lib.stream_ptr())
    else:
        keep = torch.empty_like(g)
        _lib.call('dropout_f32', g, keep, _lib.i64(g.numel()), float(p), ctypes_u64(seed), ctypes_u64(off), _lib.stream_ptr())
        want = keep * torch.where(a >= 0, 1.0, 0.3)
    gac = ac.like()
    _lib.call('pool3_bwd_dropout_cp8', ac.ptr(), gc.ptr(), gac.ptr(), B, C, T, F, ac.pitch, ac.pf, ac.pt, fmt, ops.ACT_LRELU, 0.3, float(p),
              ctypes_u64(seed), ctypes_u64(off), None, ctypes_u64(0), _lib.stream_ptr())
    got = ops.cp8_to_nchw(gac)
    assert torch.equal(got, want.bfloat16().float())
    # bias gradient from the planes
    s = ops.channel_sum_cp8(gac)
    ref = got.double().sum(dim=(0, 2, 3))
    assert s.shape == (C,) and (s.double() - ref).abs().max().item() <= 1e-5 * max(1.0, got.double().abs().sum(dim=(0, 2, 3)).max().item())


@pytest.mark.parametrize('B,C,T,F,gamma', [(3, 6, 75, 216, 0.0), (2, 6, 7, 216, 10.0), (5, 3, 1, 40, 0.0), (1, 8, 9, 256, 0.0)])
def test_layernorm_pixel_kernels_cp8(B, C, T, F, gamma):
    """train_cp8.cu pixel-per-thread LayerNorm([C,F]) -> CP8 planes (+ per-row mean / rstd) and the parameter gradient that reads them:
    against nn.LayerNorm + autograd on the transposed view (basic_cnns.py:371,411) and against the row kernels they replace."""
    from multipitch_architectures_b200 import ops
    fmt = ops.FMT_BF16
    x = rnd(B, C, T, F, seed=3).abs().contiguous()
    w, b = 1 + 0.1 * rnd(C, F, seed=4), 0.1 * rnd(C, F, seed=5)
    xin = torch.log(1 + gamma * x) if gamma > 0 else x
    wt, bt = w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    ref = F_ln(xin, wt, bt)
    xc, wc, bc = x.cuda(), w.cuda(), b.cuda()
    stats = torch.empty(B * T, 2, device='cuda')
    out = ops.layernorm_cf_cp8(xc, wc, bc, 1e-5, ops.CP8(B, C, T, F, fmt=fmt), gamma_log=gamma, stats=stats)
    got = ops.cp8_to_nchw(out).cpu()
    assert (got - ref.detach().bfloat16().float()).abs().max() <= 2 ** -7 * ref.detach().abs().max()          # one bf16 rounding of the same value
    assert (got - ref.detach()).abs().max() <= 2 ** -8 * ref.detach().abs().max() + 1e-6
    assert torch.equal(out.buf[..., :out.pf, :], torch.zeros_like(out.buf[..., :out.pf, :])) and (out.buf[:, :, 0] == 0).all()
    if C < 8:
        assert (out.buf[..., C:] == 0).all()
    mu = xin.transpose(1, 2).reshape(B * T, -1).mean(1)
    var = xin.transpose(1, 2).reshape(B * T, -1).var(1, unbiased=False)
    assert (stats[:, 0].cpu() - mu).abs().max() < 1e-5 and (stats[:, 1].cpu() * torch.sqrt(var + 1e-5) - 1).abs().max() < 1e-5
    # parameter gradients from a 16-bit gradient on the planes
    g = rnd(B, C, T, F, seed=6).bfloat16().float()
    ref.backward(g)
    gcp = ops.nchw_to_cp8(g.cuda(), fmt=fmt)
    gw, gb = torch.empty(C, F, device='cuda'), torch.empty(C, F, device='cuda')
    ops.layernorm_cf_param_grad_cp8(xc, gcp, gw, gb, 1e-5, gamma_log=gamma, stats=stats)
    tol = 2e-5 * max(1.0, wt.grad.abs().max().item())
    assert (gw.cpu() - wt.grad).abs().max() < tol and (gb.cpu() - bt.grad).abs().max() < tol
    if C * F <= 1408:                                                                                          # the row kernel's limit
        gw0, gb0 = torch.empty_like(gw), torch.empty_like(gb)
        ops.layernorm_cf_param_grad_cp8(xc, gcp, gw0, gb0, 1e-5, gamma_log=gamma)                              # row kernel (no saved statistics)
        assert (gw0 - gw).abs().max() < tol and (gb0 - gb).abs().max() < tol


def F_ln(x, w, b):
    C, Fb = w.shape
    return F.layer_norm(x.transpose(1, 2), [C, Fb], w, b, 1e-5).transpose(1, 2)


@pytest.mark.parametrize('name,p', [('cnn_xs', None), ('dcnn_tiny', None), ('dcnn_tiny', 0.0)])
def test_cp8_resident_training_step_equals_the_converter_path(name, p):
    """bf16 CNN training with activations / gradients resident in CP8 between the convolutions (no nchw<->CP8 converters, pools on the
    planes) against the same step through the converters and the fp32 NCHW pool kernels: same outputs bit for bit; gradients up to
    the order of the fp32 atomics, block bias gradients up to the 16-bit rounding of the summed gradient."""
    from multipitch_architectures_b200 import training as TR
    res = {}
    for resident in (True, False, 'pixel_ln'):
        TR.CP8_RESIDENT = bool(resident)
        TR.LN_PIXEL = resident == 'pixel_ln'      # the row LayerNorm kernels sum in the order of the fp32 NCHW path: bit-for-bit comparison
        try:
            m = build_model(name, precision='bf16')
            m.load_state_dict(fill_state_dict(m.state_dict(), 9, scheme='torch_default'))
            if p is not None:
                m.p_dropout = p
            m = m.cuda().train()
            x, t = synth_patches(5, 83).cuda(), synth_targets(5, 83).cuda()
            m.dropout_seed, m._train_calls = 4321, 0
            n0 = TR._lib.launch_count()
            y = m(x)
            loss = torch.nn.BCELoss()(y, t)
            loss.backward()
            res[resident] = (y.detach().clone(), {k: q.grad.clone() for k, q in m.named_parameters()}, TR._lib.launch_count() - n0)
        finally:
            TR.CP8_RESIDENT = TR.LN_PIXEL = True
    assert torch.equal(res[True][0], res[False][0])
    assert res[True][2] < res[False][2]                        # fewer launches: the converters are gone
    # default path (pixel-per-thread LayerNorm, another fp32 summation order: single 16-bit roundings of the normalised input flip)
    assert (res['pixel_ln'][0] - res[True][0]).abs().max().item() < 2e-3
    gn = sum(float((g.double() ** 2).sum()) for g in res[True][1].values()) ** 0.5
    for k in res[True][1]:
        # flipped roundings move single arg-max routings of the pools: compare the tensors as a whole
        a, b = res['pixel_ln'][1][k].double(), res[True][1][k].double()
        assert float((a - b).norm()) <= 0.1 * float(b.norm()) + 1e-3 * gn, (k, float((a - b).norm()), float(b.norm()), gn)
    n_blocks = 1 if name == 'cnn_xs' else 3
    block_bias = {'conv1.0.bias'} | {f'prefilt_list.{i}.0.bias' for i in range(n_blocks - 1)}
    for k in res[True][1]:
        a, b = res[True][1][k], res[False][1][k]
        tol = 2e-2 if k in block_bias else 1e-5
        assert (a - b).abs().max().item() <= tol * max(1e-6, b.abs().max().item()), (k, (a - b).abs().max().item(), b.abs().max().item())


@pytest.mark.parametrize('B,C,T,F', [(2, 5, 75, 72), (1, 3, 75, 216), (2, 2, 9, 8), (1, 2, 30, 40)])
def test_pool13_bwd_with_dropout_equals_dropout_then_pool_bwd(B, C, T, F):
    """k = 13 backward with the dropout mask re-drawn on the fly == dropout_kernel followed by the plain backward == torch autograd of
    max_pool2d on the masked gradient (plateaus in the input: the first maximum of a window must win)."""
    from multipitch_architectures_b200 import training as TR, ops
    a = torch.where(rnd(B, C, T, F, seed=5) > 0.3, rnd(B, C, T, F, seed=5), torch.zeros(())) - 0.2        # plateaus: ties inside the windows
    g = rnd(B, C, T, F, seed=6)
    ac, gc = a.cuda().contiguous(), g.cuda().contiguous()
    fused = TR._pool_bwd_dropout(ac, gc, 13, ops.ACT_LRELU, 0.3, 0.25, 99, 5)
    gm = TR._dropout(gc, 0.25, 99, 5)
    assert torch.equal(fused, TR._pool_bwd(ac, gm, 13, ops.ACT_LRELU, 0.3))
    # torch reference: `a` is the pool input (post-activation); the activation derivative is applied from its sign
    ar = a.clone().requires_grad_(True)
    torch.nn.functional.max_pool2d(ar, (13, 1), (1, 1), (6, 0)).backward(gm.cpu())
    want = ar.grad * torch.where(a >= 0, 1.0, 0.3)
    assert (fused.cpu() - want).abs().max() < 1e-5
