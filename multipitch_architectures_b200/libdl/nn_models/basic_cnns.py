"""CNN / DCNN / DRCNN multi-pitch networks with the reference's constructor signature and state_dict layout
(/root/reference/libdl/nn_models/basic_cnns.py:133-195, 342-423), executed by libmpa CUDA kernels.

The torch.nn layer objects below are parameter holders only (they give the drop-in key names
`conv1.0.weight`, `prefilt_list.2.0.bias`, ... and the reference's default initialisation); `forward` runs
the kernel sequence in _exec.py.  `precision`: 'fp32' (exact CUDA-core path) or 'bf16' (tcgen05 tensor-core
path for the 15x15 stacks, fp32 accumulate)."""
import torch
import torch.nn as nn

from . import _exec


class _Stage(nn.Module):
    """Placeholder keeping the reference's nn.Sequential indices (activation / pool / dropout slots own no
    parameters; their arithmetic is fused into the CUDA epilogues)."""

    def __init__(self, what):
        super().__init__()
        self.what = what

    def extra_repr(self):
        return self.what

    def forward(self, x):  # pragma: no cover
        raise RuntimeError('stages are executed by libmpa kernels, not called')


def _prefilt(cin, cout, a, p):
    return nn.Sequential(nn.Conv2d(cin, cout, (15, 15), stride=(1, 1), padding=(7, 7)),
                         _Stage(f'LeakyReLU({a})'), _Stage('MaxPool(3,1)/s1/p(1,0)'), _Stage(f'Dropout({p})'))


def _head(model, c0, n_ch, n_bins_in, n_bins_out, a, p):
    last_kernel_size = n_bins_in // 3 + 1 - n_bins_out
    model.conv2 = nn.Sequential(nn.Conv2d(c0, n_ch[1], (3, 3), stride=(1, 3), padding=(1, 0)),
                                _Stage(f'LeakyReLU({a})'), _Stage('MaxPool(13,1)/s1/p(6,0)'), _Stage(f'Dropout({p})'))
    model.conv3 = nn.Sequential(nn.Conv2d(n_ch[1], n_ch[2], (75, 1)), _Stage(f'LeakyReLU({a})'), _Stage(f'Dropout({p})'))
    model.conv4 = nn.Sequential(nn.Conv2d(n_ch[2], n_ch[3], (1, 1)), _Stage(f'LeakyReLU({a})'), _Stage(f'Dropout({p})'),
                                nn.Conv2d(n_ch[3], 1, (1, last_kernel_size)), _Stage('Sigmoid'))


class _MpaModel(nn.Module):
    # eval mode + autograd recording: True records the eval tape (dropout off, BatchNorm frozen at its running statistics) even when the
    # input needs no gradient — fine-tuning with frozen statistics; False (default) keeps that forward on the inference path, no grad_fn
    eval_backward = False

    def _init_common(self, n_chan_input, n_bins_in, a_lrelu, p_dropout, precision):
        if precision is None:
            precision = _exec.DEFAULT_PRECISION          # the reference's constructors take no such keyword: package-level default
        if precision not in _exec.PRECISIONS:
            raise ValueError(f'precision must be one of {_exec.PRECISIONS}')
        self.n_chan_input, self.n_bins_in = n_chan_input, n_bins_in
        self.a_lrelu, self.p_dropout, self.precision = a_lrelu, p_dropout, precision
        self._cache = _exec.ParamCache()



def _dispatch(model, x):
    """Autograd recording -> the training tape (in eval mode only when a graph is asked for: x requires grad, or model.eval_backward; then
    with dropout off); train mode under no_grad -> the training forward with its tape discarded (dropout stays active exactly as in the
    reference, whose validation pass runs in train mode: exp126a...py:333-345); eval -> inference path."""
    if torch.is_grad_enabled() and (model.training or x.requires_grad or model.eval_backward):
        from ...training import cnn_train_forward, forward_train
        return forward_train(cnn_train_forward, model, x)
    if model.training and model.p_dropout > 0:
        from ...training import cnn_train_forward
        model._train_calls = getattr(model, '_train_calls', 0) + 1
        return cnn_train_forward(model, x, {}, getattr(model, 'dropout_seed', 0x5EED), model._train_calls)[0].d
    return _exec.cnn_forward(model, x)


class basic_cnn_segm_sigmoid(_MpaModel):
    """CNN (paper: CNN:XS..L).  Args as the reference: n_chan_input, n_chan_layers, n_bins_in, n_bins_out,
    a_lrelu, p_dropout."""

    def __init__(self, n_chan_input=6, n_chan_layers=[20, 20, 10, 1], n_bins_in=216, n_bins_out=12, a_lrelu=0.3,
                 p_dropout=0.2, precision=None):
        super().__init__()
        self._init_common(n_chan_input, n_bins_in, a_lrelu, p_dropout, precision)
        n_ch = n_chan_layers
        self.layernorm = nn.LayerNorm(normalized_shape=[n_chan_input, n_bins_in])
        self.conv1 = _prefilt(n_chan_input, n_ch[0], a_lrelu, p_dropout)
        _head(self, n_ch[0], n_ch, n_bins_in, n_bins_out, a_lrelu, p_dropout)

    def forward(self, x):
        x = _exec._check_input(x, self.n_chan_input, self.n_bins_in)
        return _dispatch(self, x)


class deep_cnn_segm_sigmoid(_MpaModel):
    """DCNN / DRCNN: n_prefilt_layers 15x15 blocks, optional residual connections."""

    def __init__(self, n_chan_input=6, n_chan_layers=[20, 20, 10, 1], n_prefilt_layers=1, residual=False, n_bins_in=216,
                 n_bins_out=12, a_lrelu=0.3, p_dropout=0.2, precision=None):
        super().__init__()
        self._init_common(n_chan_input, n_bins_in, a_lrelu, p_dropout, precision)
        n_ch = n_chan_layers
        self.layernorm = nn.LayerNorm(normalized_shape=[n_chan_input, n_bins_in])
        self.conv1 = _prefilt(n_chan_input, n_ch[0], a_lrelu, p_dropout)
        self.n_prefilt_layers = n_prefilt_layers
        self.prefilt_list = nn.ModuleList(_prefilt(n_ch[0], n_ch[0], a_lrelu, p_dropout) for _ in range(1, n_prefilt_layers))
        self.residual = residual
        _head(self, n_ch[0], n_ch, n_bins_in, n_bins_out, a_lrelu, p_dropout)

    def forward(self, x):
        x = _exec._check_input(x, self.n_chan_input, self.n_bins_in)
        return _dispatch(self, x)
