"""Training path of the U-Net family (simple_u_net_largekernels / _doubleselfattn / _polyphony_classif_softmax):
train-mode forward (BatchNorm batch statistics, dropout, batch-axis attention) with saved activations and the
hand-written backward of every stage — all libmpa kernels (fp32), sequenced by the reverse-mode tape of training.py (UnetTape adds
the stages only this family has).

Reference loop being replaced (experiments/Exp2_SectionIV-C/RETRAIN4_exp180d_..._doubleselfattn_moresamples.py, same
shape as exp126a...py:315-329; PUnet: RETRAIN4_exp195f..._rerun1.py:337-350):
    y_pred[, n_pred] = model(X); loss = BCELoss(y_pred, y) [+ CrossEntropyLoss(n_pred, sum(y).long())/25]
    optimizer.zero_grad(); loss.backward(); optimizer.step()

Semantics kept from the reference modules (unet_cnns.py:30-159):
  * double_conv = (Conv -> BatchNorm2d(train: batch mean / biased variance, running stats updated) -> ReLU -> Dropout(0)) x 2
  * MaxPool2d(2) floor mode, gradient to the first maximum; bilinear x2 (align_corners) + pad + concat
  * transformer_enc_layer: q/k/v Linear -> nn.MultiheadAttention over the BATCH axis -> o Linear -> add&LN -> MLP -> add&LN,
    dropout after the positional encoding, the attention branch and the MLP branch (p = 0.2, the layer's own default)
The q/k/v (and o/out_proj) Linear pairs are evaluated as ONE folded matrix each (W_in.W_q, W_o.W_out); the tape
back-propagates through the fold to the reference's separate parameters."""
import torch

from . import _lib, ops
from ._lib import call, stream_ptr
from .libdl.nn_models import _exec
from .training import (FusedTrainStep, Node, Tape, TcConv, ctypes_u64, note_fp32_tape, tape_fmt, _act_bwd, _add, _s3_split_eligible, _split_buf,
                       _step_args, _tc_s3_eligible)

SITES_PER_STEP = 256      # dropout sites reserved per step of the U-Net tape: offset = step * 256 + site


class UnetTape(Tape):
    """The U-Net family's stages: BatchNorm, double_conv, max-pool / up-sampling / concat (fp32 NCHW and on the CP8 planes), the encoder
    layer and the BLSTM."""

    def bn_relu(self, name, bn, y):
        """BatchNorm2d in training mode (batch statistics) + ReLU; running statistics updated as nn.BatchNorm2d does.  frozen_bn: eval mode
        (the running statistics normalise and stay untouched; the convolution's own backward sums its bias gradient from dx)."""
        B, C, H, W = y.d.shape
        if self.frozen_bn:
            stats = ops.bn_frozen_stats(bn)
            out = Node(ops.bn_apply(y.d, stats, bn.weight, bn.bias, bn.eps, ops.ACT_RELU, 0.0))

            def bwd_frozen():
                dx = torch.empty_like(y.d)
                scratch = torch.empty(2 * C, dtype=torch.float32, device=y.d.device)
                call('bn_relu_bwd_frozen_f32', y.d, out.d, out.g, stats, bn.weight, dx, self.grads[name + '.weight'], self.grads[name + '.bias'],
                     None, scratch, B, C, H * W, float(bn.eps), 1, stream_ptr())
                y.acc(dx)
            self.push(bwd_frozen)
            return out
        stats = ops.bn_stats(y.d)
        if bn.track_running_stats:
            n = B * H * W
            m = bn.momentum if bn.momentum is not None else 0.1
            bn.running_mean.mul_(1 - m).add_(stats[:C], alpha=m)
            bn.running_var.mul_(1 - m).add_(stats[C:] * (n / max(n - 1, 1)), alpha=m)
            bn.num_batches_tracked += 1
        out = Node(ops.bn_apply(y.d, stats, bn.weight, bn.bias, bn.eps, ops.ACT_RELU, 0.0))

        def bwd():
            dx = torch.empty_like(y.d)
            scratch = torch.empty(2 * C, dtype=torch.float32, device=y.d.device)
            call('bn_relu_bwd_f32', y.d, out.d, out.g, stats, bn.weight, dx, self.grads[name + '.weight'], self.grads[name + '.bias'],
                 scratch, B, C, H * W, float(bn.eps), 1, stream_ptr())
            y.acc(dx)
        self.push(bwd)
        return out

    def double_conv(self, name, dc, x, need_dx=True):
        seq = dc.double_conv
        y = self.bn_relu(name + '.double_conv.1', seq[1], self.conv(name + '.double_conv.0', seq[0], x, need_dx=need_dx))
        return self.bn_relu(name + '.double_conv.5', seq[5], self.conv(name + '.double_conv.4', seq[4], y))

    def maxpool2d(self, x, k, s):
        out = Node(ops.maxpool2d(x.d, k, s))

        def bwd():
            B, C, H, W = x.d.shape
            gi = torch.empty_like(x.d)
            call('maxpool2d_bwd_f32', x.d, out.g, gi, B, C, H, W, k[0], k[1], s[0], s[1], stream_ptr())
            x.acc(gi)
        self.push(bwd)
        return out

    def upconcat(self, low, skip):
        out = Node(ops.upsample2x_concat(low.d, skip.d))

        def bwd():
            B, Cl, Hl, Wl = low.d.shape
            _, Cs, Hs, Ws = skip.d.shape
            g_skip, g_low = torch.empty_like(skip.d), torch.empty_like(low.d)
            call('upsample2x_concat_bwd_f32', out.g, g_skip, 0, g_low, B, Cl, Hl, Wl, Cs, Hs, Ws, stream_ptr())
            skip.acc(g_skip)
            low.acc(g_low)
        self.push(bwd)
        return out

    # ---------------------------------------------------------------------------------------------- CP8-resident stages (bf16 / fp16)
    # Nodes whose .d / .g are ops.CP8 planes: between two tensor-core convolutions nothing leaves the 16-bit planes (train_unet_cp8.cu).
    # Every such node has ONE consumer, except the skip connections (max-pool + concat), whose two gradients meet in maxpool_cp8's backward.
    def conv_cp8(self, name, conv, x, need_dx=True):
        """Conv2d (+ bias) on the planes -> the raw (pre-BatchNorm) output; the bias gradient is left to the BatchNorm backward."""
        out = Node(TcConv.forward_cp8(name, conv, x.d, ops.ACT_NONE, 0.0))

        def bwd():
            gx = TcConv.backward_cp8(name, conv, x.d, out.g, self.grads[name + '.weight'], None, need_dx)
            if need_dx:
                x.g = gx
        self.push(bwd)
        return out

    def bn_relu_cp8(self, name, bn, y, dst, conv_bias_name, split=0, conv_bias=None):
        """BatchNorm2d (train mode, running statistics updated) + ReLU on the planes, written into `dst` (a buffer or a channel view of a
        concat buffer; split = s: phase-split planes, the hand-over to the head's stride-(1, s) convolution and back).  frozen_bn: eval mode,
        normalised with the running statistics, which stay untouched."""
        frozen = self.frozen_bn
        stats = ops.bn_frozen_stats(bn) if frozen else ops.bn_stats_cp8(y.d, bn, pivot=conv_bias)
        out = Node(ops.bn_relu_apply_cp8(y.d, stats, bn, dst, split))

        def bwd():
            yc = y.d
            dy = TcConv._buf(name + ':dy', yc.B, yc.C, yc.T, yc.F, yc.buf.device, yc.fmt)
            bwd_fn = ops.bn_relu_bwd_frozen_cp8 if frozen else ops.bn_relu_bwd_cp8
            y.g = bwd_fn(out.g, yc, stats, bn, dy, self.grads[name + '.weight'], self.grads[name + '.bias'], self.grads[conv_bias_name], split)
        self.push(bwd)
        return out

    def double_conv_cp8(self, name, dc, x, dst=None, need_dx=True, split=0):
        seq = dc.double_conv
        n0, n1, n4, n5 = (f'{name}.double_conv.{i}' for i in (0, 1, 4, 5))
        xc = x.d
        mid = TcConv._buf(n1 + ':a', xc.B, seq[0].weight.shape[0], xc.T, xc.F, xc.buf.device, xc.fmt)
        a1 = self.bn_relu_cp8(n1, seq[1], self.conv_cp8(n0, seq[0], x, need_dx), mid, n0 + '.bias', conv_bias=seq[0].bias)
        if dst is None:
            dst = TcConv._buf(n5 + ':a', xc.B, seq[4].weight.shape[0], xc.T, xc.F, xc.buf.device, xc.fmt)
        return self.bn_relu_cp8(n5, seq[5], self.conv_cp8(n4, seq[4], a1), dst, n4 + '.bias', split, conv_bias=seq[4].bias)

    def maxpool_cp8(self, tag, x):
        xc = x.d
        out = Node(ops.maxpool2x2_cp8(xc, TcConv._buf(tag + ':pool', xc.B, xc.C, xc.T // 2, xc.F // 2, xc.buf.device, xc.fmt)))

        def bwd():
            # x.g: the gradient the skip connection already delivered (decoder side runs first in the backward), or None
            x.g = ops.maxpool2x2_bwd_cp8(xc, out.g, x.g, TcConv._buf(tag + ':gpool', xc.B, xc.C, xc.T, xc.F, xc.buf.device, xc.fmt))
        self.push(bwd)
        return out

    def upcat_cp8(self, tag, low, skip, cat, c_skip):
        """`skip` already sits in channels [0, c_skip) of `cat`; the bilinear x2 up-sampling of `low` fills the rest."""
        lc = low.d
        ops.upsample2x_cp8(lc, cat.channels(c_skip, lc.C))
        out = Node(cat)

        def bwd():
            g = out.g
            skip.g = g.channels(0, c_skip)
            low.g = ops.upsample2x_bwd_cp8(g.channels(c_skip, lc.C), TcConv._buf(tag + ':glow', lc.B, lc.C, lc.T, lc.F, lc.buf.device, lc.fmt))
        self.push(bwd)
        return out

    def cp8_to_f32(self, tag, x):
        """planes -> fp32 NCHW node (the encoder layers and the 72-bin head stay fp32)."""
        xc = x.d
        out = Node(ops.cp8_to_nchw(xc))

        def bwd():
            x.g = ops.nchw_to_cp8(out.g, out=TcConv._buf(tag + ':g16', xc.B, xc.C, xc.T, xc.F, xc.buf.device, xc.fmt), fmt=xc.fmt)
        self.push(bwd)
        return out

    def f32_to_cp8(self, tag, x, fmt):
        B, C, T, F = x.d.shape
        out = Node(ops.nchw_to_cp8(x.d, out=TcConv._buf(tag + ':x16', B, C, T, F, x.d.device, fmt), fmt=fmt))

        def bwd():
            x.acc(ops.cp8_to_nchw(out.g))
        self.push(bwd)
        return out

    # ---------------------------------------------------------------------------------------------- encoder layer
    def _enc_attn_fused(self, name, layer, x, p_drop, pe, gemm, colsum):
        """Attention half of the layer in one launch per direction (enc_train.cu): gather + PE + dropout + folded q/k/v + batch-axis attention
        + folded out-projection + dropout + residual + LayerNorm1, one CTA per bottleneck position; the parameter folds and their chain rule
        are one launch each.  Only the weight gradients (reductions over all B*S tokens) remain GEMM launches."""
        B, E, Th, Fw = x.d.shape
        S, H, dev = Th * Fw, layer.num_heads, x.d.device
        M = B * S
        at = layer.attn
        G = self.grads
        f32 = lambda *shape: torch.empty(*shape, dtype=torch.float32, device=dev)
        params = (at.in_proj_weight, layer.q_linear.weight, layer.k_linear.weight, layer.v_linear.weight, layer.o_linear.weight, at.out_proj.weight,
                  at.out_proj.bias)
        w_qkv, w_qkvT, w_proj, w_projT, b_proj = f32(3 * E, E), f32(E, 3 * E), f32(E, E), f32(E, E), f32(E)
        call('enc_fold_f32', *params, w_qkv, w_qkvT, w_proj, w_projT, b_proj, E, stream_ptr())
        site_tok = site_att = 0
        if p_drop > 0.0:
            if pe is not None:
                self.site += 1
                site_tok = self.site
            self.site += 1
            site_att = self.site
        sd, sm = _step_args()
        t, qkv, att, u1, h1 = f32(M, E), f32(M, 3 * E), f32(M, E), f32(M, E), f32(M, E)
        call('enc_attn_train_fwd_f32', x.d, pe, w_qkvT, at.in_proj_bias, w_projT, b_proj, layer.layernorm1.weight, layer.layernorm1.bias,
             float(layer.layernorm1.eps), t, qkv, att, u1, h1, B, E, S, H, float(p_drop), ctypes_u64(self.seed), ctypes_u64(site_tok),
             ctypes_u64(site_att), sd, sm, stream_ptr())
        h1 = Node(h1)

        def bwd():
            g_p, g_qkv, g_x = f32(M, E), f32(M, 3 * E), f32(B, E, Th, Fw)
            sd_b, sm_b = _step_args()
            call('enc_attn_train_bwd_f32', h1.g, u1, qkv, w_qkv, w_proj, layer.layernorm1.weight, float(layer.layernorm1.eps), g_p, g_qkv, g_x,
                 G[name + '.layernorm1.weight'], G[name + '.layernorm1.bias'], B, E, S, H, int(pe is not None), float(p_drop),
                 ctypes_u64(self.seed), ctypes_u64(site_tok), ctypes_u64(site_att), sd_b, sm_b, stream_ptr())
            x.acc(g_x)

            def weight_grads():                                     # reductions over all tokens: off the data-gradient chain
                dWp = gemm(g_p, att, E, E, M, 1)                    # [E,E] = g_p^T att
                dbp = colsum(g_p, M, E)
                dWf = gemm(g_qkv, t, 3 * E, E, M, 1)                # [3E,E] = g_qkv^T t
                colsum(g_qkv, M, 3 * E, out=G[name + '.attn.in_proj_bias'])
                call('enc_fold_bwd_f32', dWf, dWp, dbp, *params, G[name + '.attn.in_proj_weight'], G[name + '.q_linear.weight'],
                     G[name + '.k_linear.weight'], G[name + '.v_linear.weight'], G[name + '.o_linear.weight'], G[name + '.attn.out_proj.weight'],
                     G[name + '.attn.out_proj.bias'], E, stream_ptr())
            TcConv.wgrad_async(weight_grads, keep=(g_p, g_qkv, att, t))
        self.push(bwd)
        return h1

    def encoder_layer(self, name, layer, x, p_drop):
        """transformer_enc_layer.forward (unet_cnns.py:148-159) on [B,E,Th,Fw]; tokens are rows (b*S+s) of [B*S, E]."""
        B, E, Th, Fw = x.d.shape
        S, H, dev = Th * Fw, layer.num_heads, x.d.device
        M = B * S
        at = layer.attn
        Wi, bi = at.in_proj_weight, at.in_proj_bias
        Wq, Wk, Wv, Wo, Wout, bout = (layer.q_linear.weight, layer.k_linear.weight, layer.v_linear.weight, layer.o_linear.weight,
                                      at.out_proj.weight, at.out_proj.bias)
        f32 = lambda *shape: torch.empty(*shape, dtype=torch.float32, device=dev)

        def gemm(A, Bm, Mm, Nn, Kk, mode, out=None, accumulate=0):
            out = f32(Mm, Nn) if out is None else out
            call('gemm_f32', A, Bm, out, Mm, Nn, Kk, mode, accumulate, stream_ptr())
            return out

        def gemm_nt(A, W, bias, Mm, Nn, Kk, relu=0):
            out = f32(Mm, Nn)
            call('gemm_nt_f32', A, W, bias, out, Mm, Nn, Kk, relu, stream_ptr())
            return out

        def colsum(A, Mm, Nn, out=None):
            out = f32(Nn) if out is None else out
            call('colsum_f32', A, out, Mm, Nn, stream_ptr())
            return out
        G = self.grads
        pe = _exec.sinusoidal_pe(S, E, dev).contiguous() if layer.pos_encoding == 'sinusoidal' else None
        W1, b1, W2, b2 = layer.mlp[0].weight, layer.mlp[0].bias, layer.mlp[2].weight, layer.mlp[2].bias
        Dm = W1.shape[0]
        if ENC_FUSED and _lib.lib().mpa_enc_train_supported(B, E, H):
            h1 = self._enc_attn_fused(name, layer, x, p_drop, pe, gemm, colsum)
        else:
            # folded projections (one-off E x E products of parameters)
            w_qkv = f32(3 * E, E)
            for i, Wx in enumerate((Wq, Wk, Wv)):
                gemm(Wi[i * E:(i + 1) * E], Wx, E, E, E, 0, out=w_qkv[i * E:(i + 1) * E])
            w_proj = gemm(Wo, Wout, E, E, E, 0)
            b_proj = gemm(Wo, bout, E, 1, E, 0).reshape(E)

            # Closures are pushed in forward order (the tape runs them in reverse); they only dereference nodes when they run.
            tok0 = f32(M, E)
            call('enc_gather_f32', x.d, pe, tok0, B, E, S, stream_ptr())
            tok = Node(tok0)
            self.push(lambda: x.acc(self._tok_to_nchw(tok.g, B, E, S, Th, Fw)))
            t = self.dropout(tok, p_drop) if pe is not None else tok

            # -- attention branch: qkv -> batch-axis attention -> folded out_proj . o_linear
            qkv = Node(gemm_nt(t.d, w_qkv, bi, M, 3 * E, E))
            att = f32(M, E)
            call('batch_axis_attention_f32', qkv.d, att, B, S, E, H, stream_ptr())
            att = Node(att)
            proj = Node(gemm_nt(att.d, w_proj, b_proj, M, E, E))

            def bwd_attn():
                g_p = proj.g
                dWp = gemm(g_p, att.d, E, E, M, 1)                      # [E,E] = g_p^T att
                dbp = colsum(g_p, M, E)
                # w_proj = Wo @ Wout, b_proj = Wo @ bout
                call('gemm_nt_f32', dWp, Wout, None, G[name + '.o_linear.weight'], E, E, E, 0, stream_ptr())          # dWp @ Wout^T
                gemm(dbp, bout, E, E, 1, 0, out=G[name + '.o_linear.weight'], accumulate=1)                           # + dbp bout^T
                gemm(Wo, dWp, E, E, E, 1, out=G[name + '.attn.out_proj.weight'])                                       # Wo^T dWp
                gemm(Wo, dbp, E, 1, E, 1, out=G[name + '.attn.out_proj.bias'])                                         # Wo^T dbp
                g_att = gemm(g_p, w_proj, M, E, E, 0)
                g_qkv = f32(M, 3 * E)
                call('batch_axis_attention_bwd_f32', qkv.d, g_att, g_qkv, B, S, E, H, stream_ptr())
                dWf = gemm(g_qkv, t.d, 3 * E, E, M, 1)                  # [3E,E]
                colsum(g_qkv, M, 3 * E, out=G[name + '.attn.in_proj_bias'])
                gWi = G[name + '.attn.in_proj_weight']
                for i, (Wx, nm) in enumerate(((Wq, 'q'), (Wk, 'k'), (Wv, 'v'))):
                    blk = dWf[i * E:(i + 1) * E]
                    call('gemm_nt_f32', blk, Wx, None, gWi[i * E:(i + 1) * E], E, E, E, 0, stream_ptr())            # dWf_i @ Wx^T
                    gemm(Wi[i * E:(i + 1) * E], blk, E, E, E, 1, out=G[f'{name}.{nm}_linear.weight'])                 # Wi_i^T dWf_i
                t.acc(gemm(g_qkv, w_qkv, M, E, 3 * E, 0))
            self.push(bwd_attn)
            d1 = self.dropout(proj, p_drop)

            # -- add & LayerNorm 1
            u1 = _add(t.d, d1.d)
            h1 = f32(M, E)
            call('add_layernorm_tok_f32', t.d, d1.d, layer.layernorm1.weight, layer.layernorm1.bias, h1, None, _lib.i64(M), E, S,
                 float(layer.layernorm1.eps), stream_ptr())
            h1 = Node(h1)

            def bwd_ln1():
                g_u1 = f32(M, E)
                call('layernorm_tok_bwd_f32', u1, h1.g, layer.layernorm1.weight, g_u1, G[name + '.layernorm1.weight'],
                     G[name + '.layernorm1.bias'], _lib.i64(M), E, float(layer.layernorm1.eps), stream_ptr())
                t.acc(g_u1)
                d1.acc(g_u1)
            self.push(bwd_ln1)

        # -- MLP
        fm = tape_fmt(self.model)
        tc_mlp = fm is not None
        if tc_mlp:
            # Both Linear layers and the four products of their backward on the tensor cores (16-bit operands, fp32 accumulate).  The hidden
            # activation [M, mlp_dim] and its gradient exist ONLY as 16-bit operand-layout copies written by the GEMM epilogues
            # (token-chunked for the weight-gradient products, feature-chunked for the next layer): no fp32 round trip, no converter pass,
            # ReLU backward and the bias gradient inside the epilogue (mpa_gemm_tc_ex_f16).
            Mp, KCt, rows_t, Np8 = (M + 255) // 256 * 256, (M + 63) // 64 * 8, (Dm + 255) // 256 * 256, (Dm + 127) // 128 * 16
            hid_tok = TcConv._raw(name + ':hid_tok', KCt * rows_t * 16, True, dev)
            hid_feat = TcConv._raw(name + ':hid_feat', Np8 * Mp * 16, False, dev)
            ops.gemm_tc_ex(ops.gemm_tc_chunks(h1.d, 256, fm), ops.gemm_tc_chunks(W1, 128, fm), b1, M, Dm, E, True, fm, y_tok=hid_tok,
                           y_tok_rows=rows_t, y_tok_chunks=KCt, y_feat=hid_feat, y_feat_rows=Mp)
            m2 = Node(ops.gemm_tc_ex(hid_feat, ops.gemm_tc_chunks(W2, 128, fm), b2, M, E, Dm, False, fm, y=f32(M, E)))
        else:
            hid = Node(gemm_nt(h1.d, W1, b1, M, Dm, E, relu=1))
            m2 = Node(gemm_nt(hid.d, W2, b2, M, E, Dm))

        def bwd_mlp_tc():
            g_m2 = m2.g

            def dw2():                                              # dW2 [E, Dm] = g_m2^T hid, d b2: off the data-gradient chain
                ops.gemm_tc_ex(ops.gemm_tc_chunks(g_m2, 256, fm, True), hid_tok, None, E, Dm, M, False, fm, y=G[name + '.mlp.2.weight'],
                               w_rows=rows_t)
                colsum(g_m2, M, E, out=G[name + '.mlp.2.bias'])
            TcConv.wgrad_async(dw2, keep=(g_m2,))
            # g_hid = (g_m2 W2) * [hid > 0] -> both operand layouts, bias gradient = its column sums
            ghid_tok = TcConv._raw(name + ':ghid_tok', KCt * rows_t * 16, True, dev)
            ghid_feat = TcConv._raw(name + ':ghid_feat', Np8 * Mp * 16, False, dev)
            gb1 = G[name + '.mlp.0.bias']
            gb1.zero_()
            ops.gemm_tc_ex(ops.gemm_tc_chunks(g_m2, 256, fm), ops.gemm_tc_chunks(W2, 128, fm, True), None, M, Dm, E, False, fm, y_tok=ghid_tok,
                           y_tok_rows=rows_t, y_tok_chunks=KCt, y_feat=ghid_feat, y_feat_rows=Mp, mask_tok=hid_tok, colsum=gb1)
            # dW1 [Dm, E] = g_hid^T h1;  g_h1 [M, E] = g_hid W1
            TcConv.wgrad_async(lambda: ops.gemm_tc_ex(ghid_tok, ops.gemm_tc_chunks(h1.d, 128, fm, True), None, Dm, E, M, False, fm,
                                                      y=G[name + '.mlp.0.weight'], x_rows=rows_t), keep=(h1.d,))
            h1.acc(ops.gemm_tc_ex(ghid_feat, ops.gemm_tc_chunks(W1, 128, fm, True), None, M, E, Dm, False, fm, y=f32(M, E)))

        def bwd_mlp():
            if tc_mlp:
                return bwd_mlp_tc()
            g_m2 = m2.g
            gemm(g_m2, hid.d, E, Dm, M, 1, out=G[name + '.mlp.2.weight'])
            colsum(g_m2, M, E, out=G[name + '.mlp.2.bias'])
            g_hid = _act_bwd(hid.d, gemm(g_m2, W2, M, Dm, E, 0), ops.ACT_RELU)
            gemm(g_hid, h1.d, Dm, E, M, 1, out=G[name + '.mlp.0.weight'])
            colsum(g_hid, M, Dm, out=G[name + '.mlp.0.bias'])
            h1.acc(gemm(g_hid, W1, M, E, Dm, 0))
        self.push(bwd_mlp)
        d2 = self.dropout(m2, p_drop)

        # -- add & LayerNorm 2, back to NCHW
        u2 = _add(h1.d, d2.d)
        out = f32(B, E, Th, Fw)
        call('add_layernorm_tok_f32', h1.d, d2.d, layer.layernorm2.weight, layer.layernorm2.bias, None, out, _lib.i64(M), E, S,
             float(layer.layernorm2.eps), stream_ptr())
        out = Node(out)

        def bwd_ln2():
            g_tok = f32(M, E)
            call('nchw_tokens_f32', out.g, g_tok, B, E, S, 1, stream_ptr())
            g_u2 = f32(M, E)
            call('layernorm_tok_bwd_f32', u2, g_tok, layer.layernorm2.weight, g_u2, G[name + '.layernorm2.weight'],
                 G[name + '.layernorm2.bias'], _lib.i64(M), E, float(layer.layernorm2.eps), stream_ptr())
            h1.acc(g_u2)
            d2.acc(g_u2)
        self.push(bwd_ln2)
        return out

    # ---------------------------------------------------------------------------------------------- BLSTM (BLUnet bottleneck)
    def blstm(self, name, layer, x):
        """blstm_temporal_enc_layer.forward (unet_cnns.py:233-243) on [B,C,T,F] with the backward through time of every stacked
        bidirectional layer (mpa_lstm_layer_train_f32 / mpa_lstm_layer_bwd_f32)."""
        B, C, T, F = x.d.shape
        H, I0, dev = layer.hidden_size, C * F, x.d.device
        if I0 != layer.embed_dim or 2 * H != (layer.embed_dim // F) * F:
            raise RuntimeError(f'BLSTM of input size {layer.embed_dim} / hidden {H} does not fit a [{C},{F}] plane per frame')
        c_out = layer.embed_dim // F
        f32 = lambda *shape: torch.empty(*shape, dtype=torch.float32, device=dev)
        seq = f32(B, T, I0)
        call('lstm_seq_from_nchw_f32', x.d, seq, B, C, T, F, stream_ptr())
        saved = []
        ws = f32(2 * B * H)
        for l in range(layer.num_layers):
            stk = lambda p: torch.stack([getattr(layer.blstm, f'{p}_l{l}').detach(), getattr(layer.blstm, f'{p}_l{l}_reverse').detach()]).contiguous()
            w_ih, w_hh, b_ih, b_hh = stk('weight_ih'), stk('weight_hh'), stk('bias_ih'), stk('bias_hh')
            I = seq.shape[2]
            out, gates, c_all = f32(B, T, 2 * H), f32(2, B * T, 4 * H), f32(2, B, T, H)
            call('lstm_layer_train_f32', seq, w_ih, w_hh, b_ih, b_hh, out, gates, c_all, B, T, I, H, 2, ws, _lib.usize(ws.numel() * 4), stream_ptr())
            saved.append((seq, w_ih, w_hh, gates, c_all, out, I))
            seq = out
        y = f32(B, c_out, T, F)
        call('lstm_seq_to_nchw_f32', seq, y, B, c_out, T, F, stream_ptr())
        res = Node(y)
        G = self.grads

        def bwd():
            g = f32(B, T, 2 * H)
            call('lstm_seq_from_nchw_f32', res.g, g, B, c_out, T, F, stream_ptr())
            wsb_bytes = _lib.lib().mpa_lstm_layer_bwd_workspace(B, T, H, 2)
            wsb = torch.empty(wsb_bytes, dtype=torch.uint8, device=dev)
            for l in range(layer.num_layers - 1, -1, -1):
                xin, w_ih, w_hh, gates, c_all, out, I = saved[l]
                g_x, g_wih, g_whh, g_b = f32(B, T, I), f32(2, 4 * H, I), f32(2, 4 * H, H), f32(2, 4 * H)
                call('lstm_layer_bwd_f32', xin, w_ih, w_hh, gates, c_all, out, g, g_x, g_wih, g_whh, g_b, B, T, I, H, 2, wsb, _lib.usize(wsb_bytes),
                     stream_ptr())
                for d, sfx in enumerate(('', '_reverse')):
                    G[f'{name}.blstm.weight_ih_l{l}{sfx}'].copy_(g_wih[d])
                    G[f'{name}.blstm.weight_hh_l{l}{sfx}'].copy_(g_whh[d])
                    G[f'{name}.blstm.bias_ih_l{l}{sfx}'].copy_(g_b[d])
                    G[f'{name}.blstm.bias_hh_l{l}{sfx}'].copy_(g_b[d])
                g = g_x
            gx = f32(B, C, T, F)
            call('lstm_seq_to_nchw_f32', g, gx, B, C, T, F, stream_ptr())
            x.acc(gx)
        self.push(bwd)
        return res

    @staticmethod
    def _tok_to_nchw(g_tok, B, E, S, Th, Fw):
        out = torch.empty(B, E, Th, Fw, dtype=torch.float32, device=g_tok.device)
        call('nchw_tokens_f32', g_tok, out, B, E, S, 0, stream_ptr())
        return out


ENC_FUSED = True           # test knob: False = the attention half of an encoder layer as separate GEMM / attention / LayerNorm launches
CP8_TAPE = True            # test knob: False = the fp32 NCHW tape with converters around every tensor-core convolution


def cp8_tape_eligible(model, x):
    """bf16 / fp16 U-Net / SAUnet whose every double_conv convolution runs on the tensor cores with whole channel chunks: the training step keeps
    activations and gradients on the CP8 planes between the convolutions."""
    if not CP8_TAPE or tape_fmt(model) is None:
        return False
    if hasattr(model, 'convP') or hasattr(model, 'attention3') or getattr(model, 'lstm_depth', 0) > 0:
        return False
    T, F = x.shape[2], x.shape[3]
    geo = _exec.level_geometry(T, F)
    blocks = [(model.inc, 0)] + [(getattr(model, f'down{i}')[1], i) for i in (1, 2, 3, 4)] + \
             [(getattr(model, f'upconv{i + 1}'), lv) for i, lv in enumerate((3, 2, 1, 0))]
    for dc, lv in blocks:
        Tl, Fl, _ = geo[lv]
        for conv in (dc.double_conv[0], dc.double_conv[4]):
            if not (TcConv.eligible(model, conv, Fl) and Tl >= 2 and conv.weight.shape[0] % 8 == 0):
                return False
    return geo[4][0] >= 1 and _tc_s3_eligible(model, model.conv2[0], F) and model.conv2[0].weight.shape[1] % 8 == 0


def _unet_train_forward_cp8(model, x, grads, seed, step, need_input_grad=False, frozen_bn=False):
    """The CP8-resident tape: LayerNorm -> planes -> [conv -> BN stats -> BN+ReLU]* with max-pool / up-sampling / concat on the planes ->
    (encoder layers in fp32 tokens) -> head conv2 on the planes -> fp32 72-bin head."""
    p = model.p_dropout if model.training else 0.0
    fmt = tape_fmt(model)
    tp = UnetTape(grads, seed, step, SITES_PER_STEP, model, need_input_grad, frozen_bn)
    B, C, T, F = x.shape
    dev = x.device
    geo = _exec.level_geometry(T, F)
    c = [model.inc.double_conv[4].weight.shape[0]] + [getattr(model, f'down{i}')[1].double_conv[4].weight.shape[0] for i in (1, 2, 3, 4)]
    up_out = [getattr(model, f'upconv{i}').double_conv[4].weight.shape[0] for i in (1, 2, 3, 4)]
    buf = lambda tag, lv, ch: TcConv._buf(tag, B, ch, geo[lv][0], geo[lv][1], dev, fmt)
    z = tp.layernorm_cf_cp8(model.layernorm, x, TcConv._buf('inc.in:x16', B, C, T, F, dev, fmt)) if C <= 8 else \
        tp.f32_to_cp8('inc.in', tp.layernorm_cf(model.layernorm, x), fmt)
    cat = {3: buf('cat3', 3, c[3] + c[4]), 2: buf('cat2', 2, c[2] + up_out[0]), 1: buf('cat1', 1, c[1] + up_out[1]),
           0: buf('cat0', 0, c[0] + up_out[2])}
    xs = [tp.double_conv_cp8('inc', model.inc, z, cat[0].channels(0, c[0]))]
    for lv in (1, 2, 3, 4):
        dst = cat[lv].channels(0, c[lv]) if lv < 4 else None
        xs.append(tp.double_conv_cp8(f'down{lv}.1', getattr(model, f'down{lv}')[1], tp.maxpool_cp8(f'down{lv}', xs[-1]), dst))
    x5 = xs[4]
    tp.trunk_mark = len(tp.ops)
    if hasattr(model, 'attention1'):
        t5 = tp.cp8_to_f32('x5', x5)
        for nm in ('attention1', 'attention2'):
            layer = getattr(model, nm)
            t5 = tp.encoder_layer(nm, layer, t5, layer.p_dropout if model.training else 0.0)
        x5 = tp.f32_to_cp8('x5a', t5, fmt)
    u = x5
    split = 3 if _s3_split_eligible(model, model.conv2[0], F) else 0
    for i, lv in enumerate((3, 2, 1, 0)):
        last = lv == 0 and split
        dst = _split_buf('upconv4:as', B, up_out[3], T, F, 3, dev, fmt) if last else None       # hand-over to conv2 in phase-split planes
        u = tp.double_conv_cp8(f'upconv{i + 1}', getattr(model, f'upconv{i + 1}'), tp.upcat_cp8(f'up{i + 1}', u, xs[lv], cat[lv], c[lv]), dst,
                               split=split if last else 0)
    return tp.head(u, p, split), None, tp


def unet_train_forward(model, x, grads, seed=0, step=0, need_input_grad=False, frozen_bn=False):
    """-> (y_pred [B,1,T-74,72], n_pred or None, tape).  Train mode: BatchNorm batch statistics, dropout when p > 0.  Eval mode: dropout
    off (encoder layers and convP included); frozen_bn: BatchNorm normalises with its running statistics and leaves them as they are.
    need_input_grad: the tape also leaves the gradient wrt x in tape.input_grad."""
    if cp8_tape_eligible(model, x):
        return _unet_train_forward_cp8(model, x, grads, seed, step, need_input_grad, frozen_bn)
    if not model.training:
        note_fp32_tape(model)
    a, p = model.a_lrelu, (model.p_dropout if model.training else 0.0)
    tp = UnetTape(grads, seed, step, SITES_PER_STEP, model, need_input_grad, frozen_bn)
    z = tp.layernorm_cf(model.layernorm, x)
    x1 = tp.double_conv('inc', model.inc, z)       # (the gradient wrt z feeds the LayerNorm parameter gradients)
    xs = [x1]
    for lv in (1, 2, 3, 4):
        xs.append(tp.double_conv(f'down{lv}.1', getattr(model, f'down{lv}')[1], tp.maxpool2d(xs[-1], (2, 2), (2, 2))))
    x5 = xs[4]
    tp.trunk_mark = len(tp.ops)
    if getattr(model, 'lstm_depth', 0) > 0:             # BLUnet: BLSTM over time at the bottleneck (and on the lowest skip for depth 2)
        x5 = tp.blstm('lstm5', model.lstm5, x5)
    if getattr(model, 'lstm_depth', 0) > 1:
        xs[3] = tp.blstm('lstm4', model.lstm4, xs[3])
    if hasattr(model, 'attention1'):
        for nm in ('attention1', 'attention2'):
            layer = getattr(model, nm)
            x5 = tp.encoder_layer(nm, layer, x5, layer.p_dropout if model.training else 0.0)
    if hasattr(model, 'attention3'):                    # SAUSnet: the lowest skip passes two encoder layers (after x5 was taken from it)
        for nm in ('attention3', 'attention4'):
            layer = getattr(model, nm)
            xs[3] = tp.encoder_layer(nm, layer, xs[3], layer.p_dropout if model.training else 0.0)
    u = x5
    for i, lv in enumerate((3, 2, 1, 0)):
        u = tp.double_conv(f'upconv{i + 1}', getattr(model, f'upconv{i + 1}'), tp.upconcat(u, xs[lv]))
    y = tp.head(u, p)
    n_pred = None
    if hasattr(model, 'convP'):
        q = tp.conv('convP.0', model.convP[0], x5, ops.ACT_LRELU, a)
        q = tp.dropout(tp.maxpool2d(q, (2, 5), (1, 2)), p)
        n_pred = tp.conv('convP.4', model.convP[4], q)
    return y, n_pred, tp


class UnetTrainStep(FusedTrainStep):
    """Fused training step of a U-Net-family model (FusedTrainStep): forward, BCE (+ CE/25 for the PUnet), backward, ONE gradient
    all-reduce, fused AdamW.  graph=True replays ~3,500 kernel launches of the SAUnet:L (more host launch time than GPU time) from one graph."""
    sites_per_step = SITES_PER_STEP
    build = staticmethod(unet_train_forward)

    def __init__(self, model, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.01, seed=0x5EED, process_group=None, ce_scale=1.0 / 25.0,
                 graph=False, overlap_comm=True):
        super().__init__(model, lr, betas, eps, weight_decay, seed, process_group, graph)
        self.ce_scale = ce_scale
        # Data-parallel runs overlap the gradient all-reduce with the backward: the parameters of the encoder trunk (layernorm, inc, down1-4)
        # are a PREFIX of the flat buffer; everything behind it (attention, decoder, head: ~3/4 of the SAUnet:L's bytes) is final once the
        # backward has reached the bottleneck, and is reduced on NCCL's stream while the trunk's backward still runs.
        self.overlap_comm = bool(overlap_comm)
        seen_other = False
        for name, p in model.named_parameters():
            trunk = name.startswith(('layernorm.', 'inc.', 'down'))
            if trunk and seen_other:
                self.n_trunk = 0                       # not a prefix (unknown model layout): one flat all-reduce after the backward
                break
            if trunk:
                self.n_trunk += p.numel()
            else:
                seen_other = True
