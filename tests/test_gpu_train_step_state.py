"""`-m gpu`: what a fused training step keeps between its calls (training.StepState: pooled planes, pack plan, side stream) belongs to that
step alone — it goes when the step goes, a later step never sees it, and a stage that raises leaves the step usable."""
import gc

import pytest
import torch

from tests.refshapes import build_model
from tests.weights import fill_state_dict, synth_patches, synth_targets

pytestmark = pytest.mark.gpu

BATCH = {'cnn_xs': 16, 'saunet_tiny': 8}


def _model(name, seed):
    m = build_model(name, precision='bf16')
    m.load_state_dict(fill_state_dict(m.state_dict(), seed, scheme='torch_default'))
    return m.cuda().train()


def _step(name, model, **kw):
    from multipitch_architectures_b200.training import TrainStep
    from multipitch_architectures_b200.training_unet import UnetTrainStep
    return (TrainStep if name == 'cnn_xs' else UnetTrainStep)(model, **kw)


def _batches(name, n, first=0):
    return [(synth_patches(BATCH[name], 70 + i).cuda(), synth_targets(BATCH[name], 70 + i).cuda()) for i in range(first, first + n)]


@pytest.mark.parametrize('graph', [False, True])
@pytest.mark.parametrize('name', ['cnn_xs', 'saunet_tiny'])
def test_dropped_step_frees_its_pooled_planes(name, graph):
    """Three steps (the third one captured and replayed with graph=True) pool tens of MB of planes; dropping the step without release()
    gives all of it back."""
    data = _batches(name, 3)
    warm = _step(name, _model(name, 1), graph=graph)     # process-wide caches (zero rows, positional encodings) exist before the count
    for x, t in data:
        warm(x, t)
    del warm
    gc.collect()
    step = _step(name, _model(name, 2), graph=graph)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    for x, t in data:
        step(x, t)
    torch.cuda.synchronize()
    assert torch.cuda.memory_allocated() - base > 8 << 20
    del step
    gc.collect()
    torch.cuda.synchronize()
    assert torch.cuda.memory_allocated() <= base


@pytest.mark.parametrize('a,b', [('cnn_xs', 'saunet_tiny'), ('saunet_tiny', 'cnn_xs')])
def test_dropped_step_leaves_nothing_to_the_next_one(a, b):
    """A graph-replayed run on model B, a step on model A dropped without release(), then the run on a fresh copy of B: the last run is the
    first one (losses and parameters to the tolerances of the graph-vs-eager tests) and its pack plan recorded the same jobs."""
    data = _batches(b, 6)

    def run_b():
        step = _step(b, _model(b, 5), lr=1e-6, graph=True)
        return step, [float(step(x, t).item()) for x, t in data]
    ref, ref_losses = run_b()
    ref_p, ref_jobs = ref.flat_p.clone(), len(ref._state.plan.jobs)
    ref.release()
    del ref
    other = _step(a, _model(a, 6), lr=1e-6, graph=True)
    for x, t in _batches(a, 3, first=10):
        other(x, t)
    del other
    gc.collect()
    step, losses = run_b()
    print('reference', ref_losses, 'after a dropped step', losses)
    assert all(abs(u - v) <= 2e-4 * max(1.0, abs(u)) for u, v in zip(ref_losses, losses))
    assert (step.flat_p - ref_p).abs().max().item() < 1e-5
    assert len(step._state.plan.jobs) == ref_jobs > 0


def _cp8_entries(v):
    from multipitch_architectures_b200 import ops
    if isinstance(v, ops.CP8):
        yield v
    elif isinstance(v, dict):
        for u in v.values():
            yield from _cp8_entries(u)
    elif isinstance(v, (list, tuple)):
        for u in v:
            yield from _cp8_entries(u)


@pytest.mark.parametrize('name', ['cnn_xs', 'saunet_tiny'])
def test_pooled_planes_keep_the_zero_gap_condition(name):
    """mpa_conv_wgrad_tc sums over every pixel of the padded rows, so its results are right only when the gap columns of its planes are
    zero and everything it reads is finite.  After three bf16 training steps with dropout on, every pooled CP8 buffer with pad rows holds
    zeros in the pad rows and gap columns of its real channels, and no NaN or Inf anywhere."""
    model = _model(name, 4)
    assert model.p_dropout > 0
    step = _step(name, model)
    for x, t in _batches(name, 3):
        step(x, t)
    torch.cuda.synchronize()
    seen = 0
    for key, a in step._state.pool.items():
        for v in _cp8_entries(a):
            if v.pt < 1:
                continue
            seen += 1
            assert bool(torch.isfinite(v.buf).all()), f'{key}: non-finite values'
            pl = v.buf[:v.B, v.chunk0:v.chunk0 + v.NC].float()
            real = torch.zeros(pl.shape[2:4], dtype=torch.bool, device=pl.device)
            real[v.pt:v.pt + v.T, v.pf:v.pf + v.F] = True
            for k in range(v.NC):
                nl = min(8, v.C - 8 * k)
                gap = pl[:, k][:, ~real][..., :nl]
                bad = int((gap != 0).sum())
                assert bad == 0, f'{key}: {bad} non-zero values in the pad rows / gap columns of chunk {k}'
    print(f'{name}: {seen} pooled CP8 buffers checked')
    assert seen > 0


@pytest.mark.parametrize('name,stage', [('cnn_xs', 'channel_sum_cp8'), ('saunet_tiny', 'gemm_tc_chunks')])
def test_stage_that_raises_leaves_the_step_usable(name, stage, monkeypatch):
    """A Python stage raises once after weight gradients were forked onto the side stream: the exception reaches the caller, no step state
    is left active, the side stream is joined and its kept tensors let go, and the next call of the same step trains normally."""
    from multipitch_architectures_b200 import ops, training
    step = _step(name, _model(name, 3), lr=1e-6)
    st, orig, seen = step._state, getattr(ops, stage), {}

    def failing(*args, **kw):
        if not seen and st.dirty:
            seen['keep'] = len(st.keep)
            raise RuntimeError('injected stage failure')
        return orig(*args, **kw)
    monkeypatch.setattr(ops, stage, failing)
    (x, t), = _batches(name, 1)
    with pytest.raises(RuntimeError, match='injected stage failure'):
        step(x, t)
    assert seen and (name == 'cnn_xs' or seen['keep'] > 0)          # the U-Net's encoder MLP keeps its gradient for the side stream
    assert training._active is None
    assert st.keep == [] and not st.dirty
    loss = step(x, t)
    assert torch.isfinite(loss).all()
