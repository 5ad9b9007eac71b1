"""Unet / SAUnet / SAUSnet / PUnet / BLUnet multi-pitch networks with the reference's constructor signatures and
state_dict layout (/root/reference/libdl/nn_models/unet_cnns.py:30-159, 220-243, 333-407, 496-575, 670-754, 1000-1101,
2251-2335), executed by libmpa CUDA kernels (see _exec.py).  torch.nn layers are parameter holders only."""
import ctypes

import torch
import torch.nn as nn

from ... import _lib, ops
from . import _exec
from .basic_cnns import _MpaModel, _Stage, _head


class double_conv(nn.Module):
    """(Conv k x k -> BatchNorm2d -> ReLU -> Dropout(convdrop)) x 2; index layout 0,1,(2,3),4,5,(6,7) as in the
    reference's default branch (convdrop=0, alt_order=False, unet_cnns.py:49-59)."""

    def __init__(self, in_channels, out_channels, mid_channels=None, kernel_size=(3, 3), padding=(1, 1), convdrop=0,
                 residual=False, alt_order=False):
        super().__init__()
        if alt_order:
            raise NotImplementedError('alt_order=True (ELU/BN pre-activation variant) is not used by any experiment')
        if residual:
            raise NotImplementedError('residual double_conv is not used by the BASELINE configurations')
        if not mid_channels:
            mid_channels = out_channels
        self.residual, self.out_channels = residual, out_channels
        layers = [nn.Conv2d(in_channels, mid_channels, kernel_size=kernel_size, padding=padding), nn.BatchNorm2d(mid_channels),
                  _Stage('ReLU')]
        if convdrop is not None:
            layers.append(_Stage(f'Dropout({convdrop})'))
        layers += [nn.Conv2d(mid_channels, out_channels, kernel_size=kernel_size, padding=padding), nn.BatchNorm2d(out_channels),
                   _Stage('ReLU')]
        if convdrop is not None:
            layers.append(_Stage(f'Dropout({convdrop})'))
        self.double_conv = nn.Sequential(*layers)
        if convdrop is None:
            raise NotImplementedError('convdrop=None changes the Sequential indices; the experiments use convdrop=0')


class transformer_enc_layer(nn.Module):
    """Parameter holder of the bottleneck encoder layer (unet_cnns.py:107-159).  The sinusoidal table is a plain
    attribute in the reference (not in the state_dict); here it is rebuilt on the input's device."""

    def __init__(self, embed_dim=32, num_heads=8, mlp_dim=512, p_dropout=0.2, pos_encoding=None):
        super().__init__()
        if pos_encoding not in (None, 'sinusoidal'):
            raise NotImplementedError("pos_encoding='learnable' is not used by any experiment")
        self.embed_dim, self.num_heads, self.mlp_dim, self.pos_encoding = embed_dim, num_heads, mlp_dim, pos_encoding
        self.p_dropout = p_dropout
        self.q_linear = nn.Linear(embed_dim, embed_dim, bias=False)
        self.v_linear = nn.Linear(embed_dim, embed_dim, bias=False)
        self.k_linear = nn.Linear(embed_dim, embed_dim, bias=False)
        self.attn = nn.MultiheadAttention(embed_dim=embed_dim, num_heads=num_heads)
        self.o_linear = nn.Linear(embed_dim, embed_dim, bias=False)
        self.mlp = nn.Sequential(nn.Linear(embed_dim, mlp_dim), _Stage('ReLU'), nn.Linear(mlp_dim, embed_dim))
        self.layernorm1 = nn.LayerNorm(normalized_shape=[embed_dim])
        self.layernorm2 = nn.LayerNorm(normalized_shape=[embed_dim])
        self._cache = _exec.ParamCache()

    def run(self, x, fmt=None):
        """fmt None: the fused fp32 sequence (mpa_encoder_layer_f32).  fmt = ops.FMT_F16 / FMT_BF16 (tensor-core models): the same
        stages as separate calls with the MLP's two Linear layers — > 95 % of the layer's FLOPs — on tcgen05 (mpa_gemm_tc_f16)."""
        B, E, Th, Fw = x.shape
        S = Th * Fw
        at = self.attn

        def fold():
            Wi, bi = at.in_proj_weight, at.in_proj_bias
            wq = Wi[:E] @ self.q_linear.weight
            wk = Wi[E:2 * E] @ self.k_linear.weight
            wv = Wi[2 * E:] @ self.v_linear.weight
            w_qkv = torch.cat([wq, wk, wv], 0).contiguous()
            w_proj = (self.o_linear.weight @ at.out_proj.weight).contiguous()
            b_proj = (self.o_linear.weight @ at.out_proj.bias).contiguous()
            return w_qkv, bi.contiguous(), w_proj, b_proj
        w_qkv, b_qkv, w_proj, b_proj = self._cache.get(
            'fold', [at.in_proj_weight, at.in_proj_bias, self.q_linear.weight, self.k_linear.weight, self.v_linear.weight,
                     self.o_linear.weight, at.out_proj.weight, at.out_proj.bias], fold)
        pe = None
        if self.pos_encoding == 'sinusoidal':
            pe = self._cache.get(f'pe{S}', [self.layernorm1.weight], lambda: _exec.sinusoidal_pe(S, E, x.device).contiguous())
        if fmt is not None:
            return self._run_tc(x, fmt, pe, w_qkv, b_qkv, w_proj, b_proj)
        ws_bytes = _lib.lib().mpa_encoder_layer_workspace(B, E, S, self.mlp_dim)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
        out = torch.empty_like(x)
        _lib.call('encoder_layer_f32', x, out, B, E, Th, Fw, self.num_heads, self.mlp_dim, pe, w_qkv, b_qkv, w_proj, b_proj,
                  self.layernorm1.weight, self.layernorm1.bias, self.mlp[0].weight, self.mlp[0].bias, self.mlp[2].weight,
                  self.mlp[2].bias, self.layernorm2.weight, self.layernorm2.bias, float(self.layernorm1.eps), ws,
                  _lib.usize(ws_bytes), _lib.stream_ptr())
        return out


def _enc_run_tc(self, x, fmt, pe, w_qkv, b_qkv, w_proj, b_proj):
    B, E, Th, Fw = x.shape
    S, M, dev = Th * Fw, B * Th * Fw, x.device
    f32 = lambda *shape: torch.empty(*shape, dtype=torch.float32, device=dev)
    sp = _lib.stream_ptr
    h1, h1c = f32(M, E), None
    if B <= 64 and E % 16 == 0 and 64 <= E <= 128 and 2 * E + 128 <= (3 * E + 127) // 128 * 128:
        # the attention half in ONE launch: gather + PE, folded q/k/v and out-projection on tcgen05, batch-axis softmax, residual, LayerNorm1
        wqc = self._cache.get(f'wqkvc{fmt}', [self.attn.in_proj_weight, self.q_linear.weight, self.k_linear.weight, self.v_linear.weight],
                              lambda: ops.gemm_tc_chunks(w_qkv, 128, fmt))
        wpc = self._cache.get(f'wprojc{fmt}', [self.o_linear.weight, self.attn.out_proj.weight], lambda: ops.gemm_tc_chunks(w_proj, 128, fmt))
        h1c = torch.empty(_lib.lib().mpa_gemm_tc_chunked_bytes(M, E, 256), dtype=torch.uint8, device=dev)
        _lib.call('enc_attn_block_tc', x, pe, wqc, b_qkv, wpc, b_proj, self.layernorm1.weight, self.layernorm1.bias, h1, h1c, B, E, S,
                  self.num_heads, float(self.layernorm1.eps), fmt, sp())
    else:
        tok = f32(M, E)
        _lib.call('enc_gather_f32', x, pe, tok, B, E, S, sp())
        qkv = f32(M, 3 * E)
        _lib.call('gemm_nt_f32', tok, w_qkv, b_qkv, qkv, M, 3 * E, E, 0, sp())
        att = f32(M, E)
        _lib.call('batch_axis_attention_f32', qkv, att, B, S, E, self.num_heads, sp())
        proj = f32(M, E)
        _lib.call('gemm_nt_f32', att, w_proj, b_proj, proj, M, E, E, 0, sp())
        _lib.call('add_layernorm_tok_f32', tok, proj, self.layernorm1.weight, self.layernorm1.bias, h1, None, _lib.i64(M), E, S,
                  float(self.layernorm1.eps), sp())
    W1, W2 = self.mlp[0].weight, self.mlp[2].weight
    w1c = self._cache.get(f'w1c{fmt}', [W1], lambda: ops.gemm_tc_chunks(W1, 128, fmt))
    w2c = self._cache.get(f'w2c{fmt}', [W2], lambda: ops.gemm_tc_chunks(W2, 128, fmt))
    # hidden activation [M, mlp_dim]: written by the first product's epilogue as the 16-bit X operand of the second one (no fp32 copy,
    # no converter pass: at 646 patches the fp32 tensor alone was 1.1 GB per layer)
    Dm = self.mlp_dim
    Mp, Np8 = (M + 255) // 256 * 256, (Dm + 127) // 128 * 16
    if h1c is None:
        h1c = ops.gemm_tc_chunks(h1, 256, fmt)
    hid_feat = torch.empty(Np8 * Mp * 16, dtype=torch.uint8, device=dev)
    ops.gemm_tc_ex(h1c, w1c, self.mlp[0].bias, M, Dm, E, True, fmt, y_feat=hid_feat, y_feat_rows=Mp)
    out = torch.empty_like(x)
    if E <= 128:
        # residual + LayerNorm2 in the second product's epilogue, written straight to NCHW: the layer is 3 launches (attention half, MLP
        # product 1, MLP product 2).  Few token tiles (the reference batch of 50: 11 tiles): the product is split over K, the slices meet
        # in atomics on `mo`, and the slice that arrives last finishes the tile's LayerNorm from L2.
        ops.gemm_tc_ex(hid_feat, w2c, self.mlp[2].bias, M, E, Dm, False, fmt, y=f32(M, E),
                       ln=(h1, self.layernorm2.weight, self.layernorm2.bias, self.layernorm2.eps, out, S))
        return out
    mo = ops.gemm_tc_ex(hid_feat, w2c, self.mlp[2].bias, M, E, Dm, False, fmt, y=f32(M, E))
    _lib.call('add_layernorm_tok_f32', h1, mo, self.layernorm2.weight, self.layernorm2.bias, None, out, _lib.i64(M), E, S,
              float(self.layernorm2.eps), sp())
    return out


transformer_enc_layer._run_tc = _enc_run_tc


class blstm_temporal_enc_layer(nn.Module):
    """BLSTM over the time axis of a U-Net level (unet_cnns.py:220-243): the (channel, bin) plane of every frame is one
    input vector; `num_layers` stacked bidirectional nn.LSTM layers (parameter holder: `blstm`), zero initial state."""

    def __init__(self, embed_dim=32, hidden_size=512, num_layers=1, batch_first=True, bidirectional=True):
        super().__init__()
        self.embed_dim, self.hidden_size, self.num_layers = embed_dim, hidden_size, num_layers
        self.blstm = nn.LSTM(input_size=embed_dim, hidden_size=hidden_size, num_layers=num_layers, batch_first=True, bidirectional=True)
        self._cache = _exec.ParamCache()

    def run(self, x):
        B, C, T, F = x.shape
        H, I = self.hidden_size, C * F
        if I != self.embed_dim:
            raise RuntimeError(f'input.size(-1) must be equal to input_size. Expected {self.embed_dim}, got {I}')
        c_out = self.embed_dim // F                      # embed_dim_scaled of the reference's .view
        if 2 * H != c_out * F:
            raise RuntimeError(f'shape [-1, {c_out}, {F}, {T}] is invalid for the BLSTM output of {2 * H} features per frame')
        sp, dev = _lib.stream_ptr, x.device
        seq = torch.empty(B, T, I, dtype=torch.float32, device=dev)
        _lib.call('lstm_seq_from_nchw_f32', x, seq, B, C, T, F, sp())
        ws_bytes = _lib.lib().mpa_lstm_layer_workspace(B, T, H, 2)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        for l in range(self.num_layers):
            names = [f'{p}_l{l}{sfx}' for p in ('weight_ih', 'weight_hh', 'bias_ih', 'bias_hh') for sfx in ('', '_reverse')]
            params = [getattr(self.blstm, n) for n in names]
            w_ih, w_hh, b_ih, b_hh = self._cache.get(f'l{l}', params, lambda: tuple(
                torch.stack([params[2 * i].detach().float(), params[2 * i + 1].detach().float()]).contiguous() for i in range(4)))
            out = torch.empty(B, T, 2 * H, dtype=torch.float32, device=dev)
            _lib.call('lstm_layer_f32', seq, w_ih, w_hh, b_ih, b_hh, out, B, T, seq.shape[2], H, 2, ws, _lib.usize(ws_bytes), sp())
            seq = out
        y = torch.empty(B, c_out, T, F, dtype=torch.float32, device=dev)
        _lib.call('lstm_seq_to_nchw_f32', seq, y, B, c_out, T, F, sp())
        return y


def _down(cin, cout, k, **kw):
    return nn.Sequential(_Stage('MaxPool(2,2)'), double_conv(cin, cout, mid_channels=cout, kernel_size=(k, k), padding=(k // 2, k // 2), **kw))


class _UnetBase(_MpaModel):
    def _build_trunk(self, n_in, n_ch, sc, **kw):
        self.inc = double_conv(n_in, 64 // sc, mid_channels=64 // sc, kernel_size=(15, 15), padding=(7, 7),
                               **{k: v for k, v in kw.items() if k != 'residual'})
        self.down1 = _down(64 // sc, 128 // sc, 15, **kw)
        self.down2 = _down(128 // sc, 256 // sc, 9, **kw)
        self.down3 = _down(256 // sc, 512 // sc, 5, **kw)
        self.down4 = _down(512 // sc, 1024 // (sc * 2), 3, **kw)

    def _build_up(self, n_ch, sc, **kw):
        self.upconcat = _Stage('bilinear x2 (align_corners) + pad + concat')
        self.upconv1 = double_conv(1024 // sc, 512 // (sc * 2), mid_channels=1024 // (sc * 2), kernel_size=(3, 3), padding=(1, 1), **kw)
        self.upconv2 = double_conv(512 // sc, 256 // (sc * 2), mid_channels=512 // (sc * 2), kernel_size=(5, 5), padding=(2, 2), **kw)
        self.upconv3 = double_conv(256 // sc, 128 // (sc * 2), mid_channels=256 // (sc * 2), kernel_size=(9, 9), padding=(4, 4), **kw)
        self.upconv4 = double_conv(128 // sc, n_ch[0], mid_channels=128 // (sc * 2), kernel_size=(15, 15), padding=(7, 7), **kw)

    def _bn_train(self):
        return self.training

    def _eval_tape(self, x):
        """Eval mode, autograd recording, and a graph asked for: x requires grad (saliency), or `eval_backward` is set (fine-tuning with
        frozen BatchNorm statistics).  Anything else in eval mode — the reference's `model.eval(); model(batch)` test loop included — takes
        the inference path and returns a tensor without grad_fn."""
        return not self.training and torch.is_grad_enabled() and (x.requires_grad or self.eval_backward)

    def predict_frames(self, plane, i0, n):
        """Eval-mode forward of the n stride-1 patches starting at frames i0.. of a recording whose LayerNorm'ed (+ log-compressed) frames
        sit in the 16-bit frame-major `plane` [rows][pitch][8] (mpa_layernorm_frames; engine.predict_patchwise builds it once per
        recording).  The first convolution gathers its 75-row windows straight from the plane: no patch is materialised.  Same result as
        forward() on the materialised patches (same kernels, same operand values)."""
        y, x5 = _exec.unet_forward_tc(self, None, frames=(plane, int(i0), int(n)))
        return self._finish(y, x5 if hasattr(self, 'convP') else None)

    def _finish(self, y, x5):
        return y

    def _run(self, x):
        x = _exec._check_input(x, self.n_chan_input, self.n_bins_in)
        if x.shape[2] < 75:
            raise ValueError('U-Net models need at least 75 frames of context')
        if self.training:
            # train mode (BatchNorm batch statistics, dropout): the tape-driven training path, with or without autograd recording
            from ...training import forward_train
            from ...training_unet import unet_train_forward
            if torch.is_grad_enabled():
                out = forward_train(unet_train_forward, self, x)
                return out if isinstance(out, tuple) else (out, None)
            self._train_calls = getattr(self, '_train_calls', 0) + 1
            y, n_pred, _ = unet_train_forward(self, x, {}, getattr(self, 'dropout_seed', 0x5EED), self._train_calls)
            return y.d, (n_pred.d if n_pred is not None else None)
        if self._eval_tape(x):
            # eval mode with a graph asked for: the training tape with dropout off and BatchNorm frozen at its running statistics
            from ...training import forward_train
            from ...training_unet import unet_train_forward
            out = forward_train(unet_train_forward, self, x)
            return out if isinstance(out, tuple) else (out, None)
        train = self._bn_train()
        if _exec.unet_tc_eligible(self, x):
            y, x5c = _exec.unet_forward_tc(self, x)
            return y, (x5c if hasattr(self, 'convP') else None)          # PUnet: the bottleneck stays in its CP8 planes for convP
        x1, x2, x3, x4, x5 = _exec.unet_trunk_f32(self, x, train)
        x5 = self._bottleneck(x5)
        x4 = self._skip4(x4)                  # (SAUSnet: attention on the lowest skip, after x5 was taken from the original x4)
        u = _exec.unet_up_f32(self, x5, (x1, x2, x3, x4), train)
        return _exec.head_f32(self._cache, self, u, self.a_lrelu), x5

    def _bottleneck(self, x5):
        return x5

    def _skip4(self, x4):
        return x4


class simple_u_net_largekernels(_UnetBase):
    def __init__(self, n_chan_input=6, n_chan_layers=[64, 30, 20, 10], n_bins_in=216, n_bins_out=12, a_lrelu=0.3, p_dropout=0.2,
                 scalefac=16, precision=None):
        super().__init__()
        self._init_common(n_chan_input, n_bins_in, a_lrelu, p_dropout, precision)
        self.layernorm = nn.LayerNorm(normalized_shape=[n_chan_input, n_bins_in])
        self._build_trunk(n_chan_input, n_chan_layers, scalefac)
        self._build_up(n_chan_layers, scalefac)
        _head(self, n_chan_layers[0], n_chan_layers, n_bins_in, n_bins_out, a_lrelu, p_dropout)

    def forward(self, x):
        return self._run(x)[0]


class simple_u_net_doubleselfattn(_UnetBase):
    def __init__(self, n_chan_input=6, n_chan_layers=[64, 30, 20, 10], n_bins_in=216, n_bins_out=12, a_lrelu=0.3, p_dropout=0.2,
                 convdrop=0, residual=False, alt_order=False, scalefac=16, embed_dim=4 * 8, num_heads=8, mlp_dim=512,
                 pos_encoding=None, precision=None):
        super().__init__()
        self._init_common(n_chan_input, n_bins_in, a_lrelu, p_dropout, precision)
        kw = dict(convdrop=convdrop, residual=residual, alt_order=alt_order)
        self.layernorm = nn.LayerNorm(normalized_shape=[n_chan_input, n_bins_in])
        self._build_trunk(n_chan_input, n_chan_layers, scalefac, **kw)
        self.attention1 = transformer_enc_layer(embed_dim=embed_dim, num_heads=num_heads, mlp_dim=mlp_dim, pos_encoding=pos_encoding)
        self.attention2 = transformer_enc_layer(embed_dim=embed_dim, num_heads=num_heads, mlp_dim=mlp_dim)
        self._build_up(n_chan_layers, scalefac, **kw)
        _head(self, n_chan_layers[0], n_chan_layers, n_bins_in, n_bins_out, a_lrelu, p_dropout)

    def _bottleneck(self, x5):
        return self.attention2.run(self.attention1.run(x5))

    def forward(self, x):
        return self._run(x)[0]


class simple_u_net_doubleselfattn_twolayers(_UnetBase):
    """SAUSnet (unet_cnns.py:670-754): two encoder layers at the bottleneck AND two on the lowest skip connection x4.  The reference
    hands its own p_dropout to the encoder layers here (the SAUnet above leaves them at their default 0.2)."""

    def __init__(self, n_chan_input=6, n_chan_layers=[64, 30, 20, 10], n_bins_in=216, n_bins_out=12, a_lrelu=0.3, p_dropout=0.2,
                 convdrop=0, residual=False, scalefac=16, embed_dim=4 * 8, num_heads=8, mlp_dim=512, pos_encoding=None, precision=None):
        super().__init__()
        self._init_common(n_chan_input, n_bins_in, a_lrelu, p_dropout, precision)
        kw = dict(convdrop=convdrop, residual=residual)
        self.layernorm = nn.LayerNorm(normalized_shape=[n_chan_input, n_bins_in])
        self._build_trunk(n_chan_input, n_chan_layers, scalefac, **kw)
        enc = dict(embed_dim=embed_dim, num_heads=num_heads, mlp_dim=mlp_dim, p_dropout=p_dropout)
        self.attention1 = transformer_enc_layer(pos_encoding=pos_encoding, **enc)
        self.attention2 = transformer_enc_layer(**enc)
        self.attention3 = transformer_enc_layer(pos_encoding=pos_encoding, **enc)
        self.attention4 = transformer_enc_layer(**enc)
        self._build_up(n_chan_layers, scalefac, **kw)
        _head(self, n_chan_layers[0], n_chan_layers, n_bins_in, n_bins_out, a_lrelu, p_dropout)

    def _bottleneck(self, x5):
        return self.attention2.run(self.attention1.run(x5))

    def _skip4(self, x4):
        return self.attention4.run(self.attention3.run(x4))

    def forward(self, x):
        return self._run(x)[0]


class simple_u_net_polyphony_classif_softmax(_UnetBase):
    def __init__(self, n_chan_input=6, n_chan_layers=[64, 30, 20, 10], n_bins_in=216, n_bins_out=12, a_lrelu=0.3, p_dropout=0.2,
                 scalefac=16, num_polyphony_steps=24, precision=None):
        super().__init__()
        self._init_common(n_chan_input, n_bins_in, a_lrelu, p_dropout, precision)
        sc = scalefac
        self.layernorm = nn.LayerNorm(normalized_shape=[n_chan_input, n_bins_in])
        self._build_trunk(n_chan_input, n_chan_layers, sc)
        self._build_up(n_chan_layers, sc)
        _head(self, n_chan_layers[0], n_chan_layers, n_bins_in, n_bins_out, a_lrelu, p_dropout)
        self.convP = nn.Sequential(nn.Conv2d(1024 // (sc * 2), 1024 // (sc * 4), (2, 5)), _Stage(f'LeakyReLU({a_lrelu})'),
                                   _Stage('MaxPool(2,5)/s(1,2)'), _Stage(f'Dropout({p_dropout})'),
                                   nn.Conv2d(1024 // (sc * 4), num_polyphony_steps, (2, 3)))

    def forward(self, x):
        y, x5 = self._run(x)
        if self.training or self._eval_tape(x):
            return y, x5                     # the training tape evaluates convP itself (x5 slot = n_pred)
        return self._finish(y, x5)

    def _finish(self, y, x5):
        if isinstance(x5, ops.CP8):
            p = _exec.conv_even_valid_tc(self._cache, 'convP.0', self.convP[0], x5, ops.ACT_LRELU, self.a_lrelu)
        else:
            p = _exec.conv_f32(self._cache, 'convP.0', self.convP[0], x5, ops.ACT_LRELU, self.a_lrelu)
        p = ops.maxpool2d(p, (2, 5), (1, 2))
        c4 = self.convP[4]
        if tuple(p.shape[2:]) == tuple(c4.kernel_size):
            # the (2,3) VALID convolution covers its whole input: one GEMM row per item
            n_pred = torch.empty(p.shape[0], c4.weight.shape[0], 1, 1, dtype=torch.float32, device=p.device)
            w = self._cache.get('convP.4:flat', [c4.weight], lambda: c4.weight.detach().reshape(c4.weight.shape[0], -1).contiguous())
            _lib.call('gemm_nt_f32', p, w, c4.bias, n_pred, p.shape[0], w.shape[0], w.shape[1], 0, _lib.stream_ptr())
        else:
            n_pred = _exec.conv_f32(self._cache, 'convP.4', c4, p)
        return y, n_pred


class u_net_blstm_varlayers(_UnetBase):
    """BLUnet (unet_cnns.py:1000-1101; experiments exp186b/d/e): the large-kernel U-Net with `lstm_number` stacked BLSTM layers over
    time at the bottleneck (lstm_depth 1) and, for lstm_depth > 1, on the skip connections from the bottom up."""

    def __init__(self, n_chan_input=6, n_chan_layers=[64, 30, 20, 10], n_bins_in=216, n_bins_out=12, a_lrelu=0.3, p_dropout=0.2,
                 scalefac=8, embed_dim=4 * 16, hidden_size=512, lstm_depth=0, lstm_number=2, precision=None):
        super().__init__()
        self._init_common(n_chan_input, n_bins_in, a_lrelu, p_dropout, precision)
        self.lstm_depth, self.lstm_number = lstm_depth, lstm_number
        self.layernorm = nn.LayerNorm(normalized_shape=[n_chan_input, n_bins_in])
        self._build_trunk(n_chan_input, n_chan_layers, scalefac)
        for depth, name in enumerate(('lstm5', 'lstm4', 'lstm3', 'lstm2', 'lstm1')):
            if lstm_depth > depth:
                setattr(self, name, blstm_temporal_enc_layer(embed_dim=embed_dim, hidden_size=hidden_size, num_layers=lstm_number))
        self._build_up(n_chan_layers, scalefac)
        _head(self, n_chan_layers[0], n_chan_layers, n_bins_in, n_bins_out, a_lrelu, p_dropout)

    def _bottleneck(self, x5):
        return self.lstm5.run(x5) if self.lstm_depth > 0 else x5

    def _skip4(self, x4):
        return self.lstm4.run(x4) if self.lstm_depth > 1 else x4

    def forward(self, x):
        if self.lstm_depth > 2:
            raise NotImplementedError('BLSTM layers on the upper skip connections (lstm_depth > 2) are not used by any experiment')
        return self._run(x)[0]
