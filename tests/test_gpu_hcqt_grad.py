"""`-m gpu`: autograd from the pitch activations to the raw audio.  The three adjoint kernels against the inner-product identity, the HCQT
gradient against torch.autograd of the float64 restatement of HCQTPlan.run (tests/hcqt_ref.py, pinned to the oracle by
tests/test_hcqt_grad_host.py), ops.gather_patches against torch.autograd of log1p(gamma * unfold), determinism, the unchanged inference
calls, and engine.audio_vjp against a plain autograd composition (and, for an fp32 DRCNN, against float64 CPU autograd of the restatement
followed by oracle/nn_oracle.py)."""
import ctypes
import functools

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import hcqt_oracle as Q
from tests import hcqt_ref as R
from tests.weights import MODEL_SPECS, fill_state_dict

pytestmark = pytest.mark.gpu

TUNE = 50


@functools.lru_cache(maxsize=2)
def plan(efficient):
    return R.make_plan(efficient, 'cuda')


def _tun():
    return torch.tensor([TUNE], dtype=torch.int32, device='cuda')


def _dot(a, b):
    return float((a.double() * b.double()).sum())


# ---------------------------------------------------------------------------------------------------------------- adjoint identities
@pytest.mark.parametrize('factor,n', [(2, 4001), (2, 4000), (4, 1001), (4, 1000), (8, 999), (8, 100)])
def test_decimate_adjoint_identity(factor, n):
    """<D x, w> = <x, D^T w> for the 2:1 chain step and the one-shot 2^c:1 early down-sampling (gain sqrt(D)); n = 100 at D = 8 is shorter
    than the 255-tap filter, so most taps fall outside the signal."""
    from multipitch_architectures_b200 import _lib
    from multipitch_architectures_b200.libdl.data_preprocessing import _filterbank as FB
    g = torch.Generator(device='cuda').manual_seed(n)
    taps = torch.from_numpy(FB.kaiser_fast_half_taps(factor)).cuda()
    gain = ctypes.c_double(float(np.sqrt(factor)))
    x = torch.randn(n, device='cuda', generator=g)
    w = torch.randn(-(-n // factor), device='cuda', generator=g)
    dx = torch.empty_like(w)
    _lib.call('decimate_gain_f32', x, dx, taps, taps.numel(), factor, gain, _lib.i64(n), _lib.stream_ptr())
    dtw = torch.empty_like(x)
    _lib.call('decimate_adjoint_f32', w, dtw, taps, taps.numel(), factor, gain, _lib.i64(n), 0, _lib.stream_ptr())
    lhs, rhs = _dot(dx, w), _dot(x, dtw)
    rel = abs(lhs - rhs) / (float(dx.double().norm() * w.double().norm()) + float(x.double().norm() * dtw.double().norm()))
    print(f'decimate D={factor} n={n}: <Dx,w> = {lhs:.6f}, <x,D^T w> = {rhs:.6f}, rel {rel:.1e}')
    assert rel < 1e-6
    # accumulate flag: adds to what the buffer holds; same bits twice
    acc = torch.full_like(x, 0.25)
    _lib.call('decimate_adjoint_f32', w, acc, taps, taps.numel(), factor, gain, _lib.i64(n), 1, _lib.stream_ptr())
    assert torch.allclose(acc, dtw + 0.25, rtol=0, atol=1e-6)
    again = torch.empty_like(x)
    _lib.call('decimate_adjoint_f32', w, again, taps, taps.numel(), factor, gain, _lib.i64(n), 0, _lib.stream_ptr())
    assert torch.equal(again, dtw)


@pytest.mark.parametrize('stride', [1, 3])
def test_gather_patches_adjoint_identity(stride):
    from multipitch_architectures_b200 import _lib
    C, NT, Fq, T, n = 3, 200, 40, 75, 20
    i0 = (NT - T) // stride - n + 1                          # the last patch ends at (or just before) the last frame
    g = torch.Generator(device='cuda').manual_seed(stride)
    x = torch.randn(C, NT, Fq, device='cuda', generator=g)
    w = torch.randn(n, C, T, Fq, device='cuda', generator=g)
    gx = torch.empty(n, C, T, Fq, device='cuda')
    _lib.call('gather_patches_f32', x, gx, C, NT, Fq, i0, n, T, stride, 0.0, _lib.stream_ptr())
    gtw = torch.full_like(x, 7.0)                            # every element is written: rows no patch covers come out 0
    _lib.call('gather_patches_bwd_f32', w, None, gtw, C, NT, Fq, i0, n, T, stride, 0.0, _lib.stream_ptr())
    lhs, rhs = _dot(gx, w), _dot(x, gtw)
    rel = abs(lhs - rhs) / float(gx.double().norm() * w.double().norm())
    print(f'gather_patches stride {stride}: rel {rel:.1e}')
    assert rel < 1e-6
    assert (gtw[:, :i0 * stride] == 0).all() and (gtw[:, (i0 + n - 1) * stride + T:] == 0).all()


# ---------------------------------------------------------------------------------------------------------------- HCQT gradient
# Tolerance: the GPU backward recomputes the forward's fp32 spectrum and runs the transposed contraction and the second FFT in fp32 (the
# decimators and the overlap-add in float64); the forward itself meets the oracle to 2e-4 of its largest magnitude.  Relative to the
# largest gradient element 1e-3 leaves margin for the fp32 FFTs of up to 2048 points and the 1/|C| factor of rows with small responses.
GRAD_TOL = 1e-3
CLIPS = [(True, 400), (True, 44100), (True, 661500), (False, 1500), (False, 44100), (False, 661500)]


@pytest.mark.parametrize('efficient,n', CLIPS, ids=[f'{"efficient" if e else "per_harmonic"}-{n}' for e, n in CLIPS])
def test_hcqt_gradient_matches_float64_autograd(efficient, n):
    p = plan(efficient)
    y = torch.from_numpy(Q.synth_clip(31, seconds=n / 22050)[:n].copy()).cuda()
    if n < 22050:
        y = torch.randn(n, generator=torch.Generator().manual_seed(n)).cuda()
    yg = y.clone().requires_grad_(True)
    out, tun = p.run(yg, _tun())
    assert out.grad_fn is not None and not tun.requires_grad
    g = torch.randn(out.shape, generator=torch.Generator().manual_seed(7)).cuda()
    out.backward(g)
    y64 = y.double().requires_grad_(True)
    ref = R.hcqt(p, y64, TUNE)
    ferr = float((out.double() - ref).abs().max() / ref.abs().max())
    ref.backward(g.double())
    gr = y64.grad
    err = float((yg.grad.double() - gr).abs().max() / gr.abs().max())
    print(f'efficient={efficient} n={n}: forward {ferr:.1e}, gradient max|d| / max|ref| = {err:.2e}')
    assert ferr < 2e-4
    assert torch.isfinite(yg.grad).all() and err < GRAD_TOL


@pytest.mark.parametrize('efficient', [True, False])
def test_hcqt_gradient_silence_and_determinism(efficient):
    p = plan(efficient)
    y = torch.zeros(30000, device='cuda', requires_grad=True)
    out, _ = p.run(y, _tun())
    out.backward(torch.ones_like(out))
    assert torch.isfinite(y.grad).all() and (y.grad == 0).all()
    x = torch.from_numpy(Q.synth_clip(5, seconds=3.0)).cuda()
    grads = []
    for _ in range(2):
        xg = x.clone().requires_grad_(True)
        out, _ = p.run(xg)                                  # tuning estimated on the device, held constant
        out.backward(torch.linspace(-1, 1, out.numel(), device='cuda').view_as(out))
        grads.append(xg.grad)
    assert torch.equal(grads[0], grads[1])


def test_hcqt_without_grad_is_unchanged():
    from multipitch_architectures_b200 import _lib
    for efficient in (True, False):
        p = plan(efficient)
        y = torch.from_numpy(Q.synth_clip(8, seconds=2.0)).cuda()
        n0 = _lib.launch_count()
        out, tun = p.run(y)
        n_launch = _lib.launch_count() - n0
        # tuning estimate (2) + one launch per decimated signal + the filterbank (one launch, or one per level beyond 16 levels)
        n_dec = len([s for s in p.signals if s != (0, 0)])
        assert n_launch == 2 + n_dec + (1 if len(p.levels) <= 16 else len(p.levels))
        assert out.grad_fn is None and not out.requires_grad
        with torch.no_grad():
            out2, _ = p.run(y.clone().requires_grad_(True))
        assert out2.grad_fn is None and torch.equal(out, out2)
        out3, tun3 = p.run(y.clone().requires_grad_(True))
        assert out3.grad_fn is not None and torch.equal(out, out3) and torch.equal(tun, tun3)
        graph_out, _ = p.run_graph(y.clone().requires_grad_(True))
        assert graph_out.grad_fn is None and torch.equal(graph_out, out)


# ---------------------------------------------------------------------------------------------------------------- gather_patches
@pytest.mark.parametrize('stride,i0,n', [(1, 0, 30), (1, 95, 30), (3, 0, 12), (3, 29, 12)])
def test_gather_patches_backward_matches_autograd(stride, i0, n):
    from multipitch_architectures_b200 import ops
    C, NT, Fq, T = 6, 200, 216, 75
    assert (i0 + n - 1) * stride + T <= NT
    gen = torch.Generator().manual_seed(i0 + 10 * stride)
    x = torch.rand(C, NT, Fq, generator=gen) * 0.2
    g = torch.randn(n, C, T, Fq, generator=gen)
    xr = x.double().requires_grad_(True)
    ref = torch.stack([torch.log1p(10.0 * xr[:, (i0 + b) * stride:(i0 + b) * stride + T]) for b in range(n)])
    ref.backward(g.double())
    xc = x.cuda().requires_grad_(True)
    out = ops.gather_patches(xc, i0, n, T, stride, 10.0)
    assert out.grad_fn is not None
    assert torch.equal(out.detach(), ops.gather_patches(x.cuda(), i0, n, T, stride, 10.0))
    assert float((out.detach().double().cpu() - ref.detach()).abs().max()) < 1e-6
    out.backward(g.cuda())
    err = float((xc.grad.double().cpu() - xr.grad).abs().max() / xr.grad.abs().max())
    print(f'gather_patches backward stride {stride} i0 {i0}: {err:.1e}')
    assert err < 1e-5
    xc2 = x.cuda().requires_grad_(True)
    ops.gather_patches(xc2, i0, n, T, stride, 10.0).backward(g.cuda())
    assert torch.equal(xc.grad, xc2.grad)


# ---------------------------------------------------------------------------------------------------------------- end to end
LOCAL = {'saunet_small': dict(cls='simple_u_net_doubleselfattn', kw=dict(n_chan_input=6, n_chan_layers=[16, 10, 8, 5], n_bins_in=216, n_bins_out=72,
                                                                          scalefac=16, embed_dim=32, num_heads=8, mlp_dim=64,
                                                                          pos_encoding='sinusoidal'))}


def _model(name, precision, seed=3):
    from multipitch_architectures_b200.libdl import nn_models as M
    spec = LOCAL.get(name) or MODEL_SPECS[name]
    m = getattr(M, spec['cls'])(**spec['kw'], precision=precision)
    sd = fill_state_dict(m.state_dict(), seed, scheme='adversarial' if 'cnn' in spec['cls'] else 'torch_default')
    m.load_state_dict(sd)
    return m.cuda().eval(), sd


def _composition_vjp(model, y, p, g_act, batch, tun):
    """plan.run -> zero padding -> gather_patches -> model, one autograd graph over the whole clip, batched as predict_patchwise."""
    from multipitch_architectures_b200 import ops
    yg = y.clone().requires_grad_(True)
    h, _ = p.run(yg, tun)
    C, N, Fq = h.shape
    padded = F.pad(h, (0, 0, 37, 38))
    loss = 0.0
    for i0 in range(0, N, batch):
        n = min(batch, N - i0)
        out = model(ops.gather_patches(padded, i0, n, 75, 1, 10.0))
        out = out[0] if isinstance(out, tuple) else out
        loss = loss + (out.reshape(n, -1) * g_act[i0:i0 + n]).sum()
    loss.backward()
    return yg.grad


def _cos(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float(a @ b / (a.norm() * b.norm()))


@pytest.mark.parametrize('name,precision', [('drcnn_tiny', 'fp32'), ('drcnn_tiny', 'bf16'), ('saunet_small', 'fp32'), ('punet_tiny', 'fp32')])
def test_audio_vjp_matches_autograd_composition(name, precision):
    from multipitch_architectures_b200 import engine
    p = plan(True)
    m, _ = _model(name, precision)
    y = torch.from_numpy(Q.synth_clip(41, seconds=2.0)).cuda()
    N = p.n_frames(y.numel())
    g_act = torch.randn(N, 72, generator=torch.Generator().manual_seed(2)).cuda()
    got = engine.audio_vjp(m, y, p, g_act, batch=50, tuning_idx=_tun())
    assert got.shape == y.shape and torch.isfinite(got).all() and got.abs().max() > 0
    assert all(q.grad is None for q in m.parameters())
    ref = _composition_vjp(m, y, p, g_act, 50, _tun())
    err, cos = float((got - ref).abs().max() / ref.abs().max()), _cos(got, ref)
    print(f'audio_vjp {name}/{precision}: max|d| / max|ref| = {err:.1e}, cosine {cos:.8f}')
    # the same kernels on the same batches: only the order of the per-batch sums into the padded HCQT differs
    if precision == 'fp32':
        assert err < 1e-4
    else:
        assert cos > 0.999
    # a sub-range on the same batch boundaries: rows of g_act outside lo..hi do not matter
    g2 = g_act.clone()
    g2[:50] = 0
    part = engine.audio_vjp(m, y, p, g_act, lo=50, batch=50, tuning_idx=_tun())
    full = engine.audio_vjp(m, y, p, g2, batch=50, tuning_idx=_tun())
    assert float((part - full).abs().max()) <= 1e-5 * float(full.abs().max())


def test_audio_vjp_drcnn_fp32_matches_float64_oracle():
    from multipitch_architectures_b200 import engine
    from oracle import nn_oracle as NO
    p = plan(True)
    m, sd = _model('drcnn_tiny', 'fp32')
    y = torch.from_numpy(Q.synth_clip(43, seconds=2.0)).cuda()
    N = p.n_frames(y.numel())
    g_act = torch.randn(N, 72, generator=torch.Generator().manual_seed(4)).cuda()
    got = engine.audio_vjp(m, y, p, g_act, batch=50, tuning_idx=_tun()).cpu()
    sd64 = {k: v.double() if v.is_floating_point() else v for k, v in sd.items()}
    y64 = y.cpu().double().requires_grad_(True)
    h = F.pad(R.hcqt(p, y64, TUNE), (0, 0, 37, 38))
    X = torch.log1p(10.0 * h.unfold(1, 75, 1)[:, :N].permute(1, 0, 3, 2))    # [N, C, 75, F]
    out = NO.cnn_forward(sd64, X, residual=True).reshape(N, 72)
    (out * g_act.cpu().double()).sum().backward()
    err = float((got.double() - y64.grad).abs().max() / y64.grad.abs().max())
    cos = _cos(got, y64.grad)
    print(f'audio_vjp drcnn_tiny fp32 vs float64 oracle composition: max|d| / max|ref| = {err:.2e}, cosine {cos:.8f}')
    # the fp32 HCQT gradient (gated at 1e-3 of its largest element above) seen through the adversarial-gain random DRCNN weights; measured
    # on a B200: 1.0e-3, cosine 0.9999997
    assert err < 3e-3 and cos > 0.99999


def test_predict_patchwise_unchanged():
    from multipitch_architectures_b200 import _lib, engine
    m, _ = _model('drcnn_tiny', 'fp32')
    h = torch.rand(6, 120, 216, generator=torch.Generator().manual_seed(9)).cuda() * 0.1
    got = engine.predict_patchwise(m, h, batch=50)
    padded = torch.zeros(6, 120 + 75, 216, device='cuda')
    padded[:, 37:157] = h
    outs = []
    for i0 in range(0, 120, 50):
        n = min(50, 120 - i0)
        x = torch.empty(n, 6, 75, 216, device='cuda')
        _lib.call('gather_patches_f32', padded, x, 6, 195, 216, i0, n, 75, 1, 10.0, _lib.stream_ptr())
        with torch.no_grad():
            outs.append(m(x).reshape(n, -1))
    assert torch.equal(got, torch.cat(outs))
