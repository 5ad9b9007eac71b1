"""The training loop of the reference's experiment scripts (exp126a_musicnet_cnn_basic.py:240-373) on top of this package's pieces:
`dataset_context` objects resident in HBM (patch cut + augmentation in one kernel per batch), the fused `TrainStep` / `UnetTrainStep`
(forward + loss + backward replayed from a CUDA graph, NCCL all-reduce, fused AdamW), validation, ReduceLROnPlateau, early stopping and
checkpointing of the best model.  Everything here is host control flow; the arithmetic is in the kernels.

Semantics kept from the reference: one shuffled permutation over ALL (file, patch) pairs per epoch (ConcatDataset + DataLoader(shuffle)),
batches that straddle files, an optional cap on batches per epoch, the validation pass in TRAIN mode (the scripts never call
model.eval() before it: dropout and BatchNorm batch statistics stay active, exp126a...py:333-345), scheduler.step(val_loss) and
early stopping / checkpointing on the validation loss."""
import numpy as np
import torch

from . import ops
from .libdl.metrics import early_stopping
from .libdl.nn_models.basic_cnns import basic_cnn_segm_sigmoid, deep_cnn_segm_sigmoid


class ReduceLROnPlateau:
    """torch.optim.lr_scheduler.ReduceLROnPlateau(mode='min', threshold_mode='rel') for an object with an `lr` attribute (the fused
    train steps read `lr` on every call)."""

    def __init__(self, step, factor=0.5, patience=5, threshold=1e-4, cooldown=0, min_lr=1e-6, eps=1e-8):
        self.step_obj, self.factor, self.patience, self.threshold = step, factor, patience, threshold
        self.cooldown, self.min_lr, self.eps = cooldown, min_lr, eps
        self.best, self.num_bad_epochs, self.cooldown_counter = float('inf'), 0, 0

    def step(self, metric):
        metric = float(metric)
        if metric < self.best * (1.0 - self.threshold):
            self.best, self.num_bad_epochs = metric, 0
        else:
            self.num_bad_epochs += 1
        if self.cooldown_counter > 0:
            self.cooldown_counter -= 1
            self.num_bad_epochs = 0
        if self.num_bad_epochs > self.patience:
            new_lr = max(self.step_obj.lr * self.factor, self.min_lr)
            if self.step_obj.lr - new_lr > self.eps:
                self.step_obj.lr = new_lr
            self.cooldown_counter, self.num_bad_epochs = self.cooldown, 0
        return self.step_obj.lr


class PatchSampler:
    """Batches over the concatenation of several dataset_context objects: (dataset id, patch index) pairs in one shuffled permutation
    per epoch, cut into batches of `batch_size` (the last one may be short), each gathered into ONE [n,C,T,F] tensor."""

    def __init__(self, datasets, batch_size, shuffle=True, seed=0, max_batches=None, rank=0, world=1):
        """Data-parallel runs: every rank draws the SAME permutation (same seed) and keeps the items rank, rank+world, ... of it, so the
        ranks see disjoint patches and together cover the epoch (torch's DistributedSampler scheme); all ranks run the same number of
        batches (the tail is padded by wrapping around), which the per-step gradient all-reduce needs."""
        self.datasets, self.batch_size, self.shuffle, self.max_batches = list(datasets), int(batch_size), shuffle, max_batches
        self.rank, self.world = int(rank), int(world)
        self.rng = np.random.default_rng(seed)
        self.lengths = np.array([len(d) for d in self.datasets], dtype=np.int64)
        self.offsets = np.concatenate([[0], np.cumsum(self.lengths)])

    def _per_rank(self):
        return int(-(-int(self.offsets[-1]) // self.world))

    def __len__(self):
        n = int(-(-self._per_rank() // self.batch_size))
        return n if self.max_batches is None else min(n, int(self.max_batches))

    def epoch(self):
        total = int(self.offsets[-1])
        order = self.rng.permutation(total) if self.shuffle else np.arange(total)
        if self.world > 1:
            padded = np.concatenate([order, order[:self._per_rank() * self.world - total]])
            order = padded[self.rank::self.world]
        for k in range(len(self)):
            yield self.gather(order[k * self.batch_size:(k + 1) * self.batch_size])

    def gather(self, flat):
        ds_id = np.searchsorted(self.offsets, flat, side='right') - 1
        d0 = self.datasets[0]
        C, _, F = d0.inputs.shape
        dev, n = d0.inputs.device, len(flat)
        X = torch.empty(n, C, d0.context, F, dtype=torch.float32, device=dev)
        y = torch.empty(n, 1, 1, d0.targets.shape[1], dtype=torch.float32, device=dev)
        pos = 0
        for d in np.unique(ds_id):                      # items of one file are cut (and augmented) by one launch, written in place
            sel = np.flatnonzero(ds_id == d)
            idx = flat[sel] - self.offsets[d]
            k = len(sel)
            self.datasets[d].gather(idx, out=(X[pos:pos + k], y[pos:pos + k]))
            pos += k
        return X, y


def _train_mode_loss(model, step, x, t):
    """Forward in train mode + BCE (+ CE/25) WITHOUT a parameter update: the reference's validation pass."""
    with torch.no_grad():
        if isinstance(model, (basic_cnn_segm_sigmoid, deep_cnn_segm_sigmoid)):
            from .training import cnn_train_forward
            step.val_calls = getattr(step, 'val_calls', 0) + 1
            y = cnn_train_forward(model, x, {}, step.seed ^ 0x5A5A, step.val_calls)[0]
            return ops.bce_fwd_bwd(y.d, t.contiguous())[0]
        out = model(x)
        y, n_pred = out if isinstance(out, tuple) else (out, None)
        t = t.contiguous()
        loss = ops.bce_fwd_bwd(y, t)[0]
        if n_pred is not None:                            # PUnet: + CrossEntropy(n_pred, number of active pitches) / 25
            from ._lib import call, stream_ptr
            B, K = n_pred.shape[0], n_pred.shape[1]
            call('ce_count_fwd_bwd_f32', n_pred.contiguous(), t, loss, torch.empty_like(n_pred), B, K, t.numel() // B, float(step.ce_scale), 1,
                 stream_ptr())
        return loss


def fit(model, train_sets, val_sets=None, batch_size=25, val_batch_size=50, lr=1e-3, weight_decay=0.01, max_epochs=100,
        max_batches_per_epoch=None, scheduler=None, early=None, seed=0, save_path=None, graph=True, log=print):
    """Train `model` (CUDA, .train() mode is set here) on CUDA-resident dataset_context objects.  scheduler / early: dicts of
    ReduceLROnPlateau / early_stopping keyword arguments (None = the scripts' defaults; False = off).  -> history (list of dicts)."""
    from .training import TrainStep
    from .training_unet import UnetTrainStep
    model.train()
    cnn = isinstance(model, (basic_cnn_segm_sigmoid, deep_cnn_segm_sigmoid))
    step = (TrainStep if cnn else UnetTrainStep)(model, lr=lr, weight_decay=weight_decay, graph=graph)
    import torch.distributed as dist
    world, rank = (dist.get_world_size(), dist.get_rank()) if (dist.is_available() and dist.is_initialized()) else (1, 0)
    sampler = PatchSampler(train_sets, batch_size, shuffle=True, seed=seed, max_batches=max_batches_per_epoch, rank=rank, world=world)
    vsampler = PatchSampler(val_sets, val_batch_size, shuffle=False) if val_sets else None       # every rank validates on the whole set
    sched = None if scheduler is False or vsampler is None else ReduceLROnPlateau(step, **(scheduler or {}))
    es = None if early is False or vsampler is None else early_stopping(**dict(dict(mode='min', min_delta=1e-5, patience=12, percentage=False),
                                                                                **(early or {})))
    if world > 1:
        dist.broadcast(step.flat_p, src=0)              # replicas start from rank 0's parameters

    def across_ranks(v):
        """Mean over the ranks: scheduler and early-stopping decisions must be identical everywhere (a rank that stopped alone would
        leave the others waiting in the gradient all-reduce)."""
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=step.flat_p.device)
        dist.all_reduce(t)
        return float(t.item()) / world
    history = []
    full = None
    for epoch in range(max_epochs):
        acc, n_batches = torch.zeros((), device=next(model.parameters()).device), 0
        for X, y in sampler.epoch():
            if full is None:
                full = X.shape[0]
            if step.use_graph and X.shape[0] != full:
                continue                                  # a short last batch does not fit the captured graph: skipped (drop_last)
            acc += step(X, y).reshape(())
            n_batches += 1
        rec = {'epoch': epoch, 'train_loss': across_ranks(float(acc.item()) / max(1, n_batches)), 'lr': step.lr}
        if vsampler is not None:
            vacc, n_val = torch.zeros_like(acc), 0
            for X, y in vsampler.epoch():
                vacc += _train_mode_loss(model, step, X, y).reshape(())
                n_val += 1
            rec['val_loss'] = across_ranks(float(vacc.item()) / max(1, n_val))
            if sched is not None:
                sched.step(rec['val_loss'])
        history.append(rec)
        if rank == 0:
            log('Epoch #%d finished. Train Loss: %.4f%s with lr: %.5f' % (epoch, rec['train_loss'],
                                                                          (', Val Loss: %.4f' % rec['val_loss']) if 'val_loss' in rec else '', rec['lr']))
        if es is not None:
            if save_path and rank == 0 and (epoch == 0 or es.curr_is_better(rec['val_loss'])):
                torch.save(model.state_dict(), save_path)
            if es.step(rec['val_loss']):
                break
    if save_path and es is None and rank == 0:
        torch.save(model.state_dict(), save_path)
    return history
