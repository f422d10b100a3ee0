"""Training step of the drop-in encoder: forward with saved activations + hand-written backward.

What ``torch.autograd`` does for the reference module under fairseq's ``train_step``
(examples/speech_recognition/tasks/speech_recognition.py:234-263 -> criterions/ctc_multi_loss.py:20-46 ->
``optimizer.backward``) is done here by ONE ``torch.autograd.Function`` whose forward and backward are chains of
the sm_100a kernels (no PyTorch arithmetic on activations; torch only owns memory, the parameter tensors and a
few [C]-sized views / permutes of weight gradients):

* forward = the reference's training-mode forward (conv_transformer.py:195-276): Conv2d -> ReLU ->
  BatchNorm2d with BATCH statistics over the padded batch (+ running-stat update) -> dropout(max(p, .1));
  fc3 + ReLU + positions -> dropout(p); per layer LN -> qkv -> attention with probability dropout ->
  out_proj -> dropout -> residual; LN -> fc1 -> ReLU -> activation dropout -> fc2 -> dropout -> residual
  (fairseq/modules/transformer_layer.py:87-139); CTC compression; final LN.  In ``eval()`` with grad enabled
  the same chain runs with running statistics and no dropout (deterministic: what the gradient-parity tests
  compare with the reference).
* backward: for every linear layer dX = dY W (tcgen05 GEMM on a transposed weight copy), dW = dY^T X (split-K
  tcgen05 GEMM over token-contiguous operand copies), db = column sums; flash-style attention backward on
  tcgen05 (scores recomputed, no L x L buffer); LayerNorm / BatchNorm / ReLU / dropout backward as streaming
  kernels (dropout masks are regenerated from (seed, site, position)); conv2 as im2col GEMMs, conv1 (K = 9)
  as a reduction kernel; CTC compression backward (W is constant: d x[t] = W[t, seg(t)] d out[seg(t)]).

Operand precision: bf16 GEMM operands / fp16 conv-front-end activations, fp32 accumulation, fp32 residual
stream and fp32 parameter gradients in the reference's parameter layout (so fairseq's optimizers, gradient
clipping and the legacy DDP all-reduce see exactly what they expect).
"""
import torch

from . import ops

_SITE_CONV1, _SITE_CONV2, _SITE_EMB = 1, 2, 3


def _layer_sites(li):
    base = 16 + 8 * li
    return dict(att=base, out=base + 1, act=base + 2, ffn=base + 3)


def prepare_train_weights(enc):
    """bf16 / fp16 operand copies of the master parameters for one training step (re-derived whenever a
    parameter's version counter changes, i.e. after every optimizer step)."""
    params = list(enc.parameters())
    key = tuple((p._version, p.data_ptr()) for p in params)
    if getattr(enc, "_train_prep_key", None) == key:
        return enc._train_prep
    with torch.no_grad():
        C = enc.conv_channels
        dev = params[0].device
        W = {}
        W["w1"] = enc.convolutions[0].weight.detach().reshape(C, 9).float().contiguous()
        W["b1"] = enc.convolutions[0].bias.detach().float().contiguous()
        w2 = enc.convolutions[1].weight.detach().float()
        W["w2"] = ops.prep_conv2_weight(w2)  # [9][Cout][Cin] fp16
        W["b2"] = enc.convolutions[1].bias.detach().float().contiguous()
        # conv2 dgrad as a GEMM: dcol[pix, (tap, ci)] = sum_co dz2[pix, co] W2[co, ci, tap]
        W["w2d"] = ops.cast_bf16(w2.permute(2, 3, 1, 0).reshape(9 * C, C).contiguous())
        W["w3"] = ops.prep_fc3_weight(enc.fc3.weight.detach().float(), C, enc.feat_out)  # [D, F2*C] fp16
        W["b3"] = enc.fc3.bias.detach().float().contiguous()
        # bf16 operand copies + transposed copies of every nn.Linear weight: ONE batched launch per 48 matrices
        # into buffers that persist across steps (~130 cat / cast / transpose launches per step before)
        bufs = getattr(enc, "_train_bufs", None)
        if bufs is None or bufs["device"] != dev:
            bufs = enc._train_bufs = dict(device=dev)
        jobs = []

        def buf(name, rows, cols, zero_pad=False):
            t = bufs.get(name)
            if t is None:
                pitch = (cols + 7) // 8 * 8
                t = (torch.zeros if zero_pad else torch.empty)(rows, pitch, dtype=torch.bfloat16, device=dev)
                bufs[name] = t
            return t[:, :cols]

        def linear_weight(name, blocks, want_copy=True, zero_pad=False):
            """blocks: row blocks [n_i, k] of one logical weight [sum n_i, k] -> (copy [N, k], transposed [k, N])."""
            N, K = sum(w.shape[0] for w in blocks), blocks[0].shape[1]
            cp = buf(name, N, K) if want_copy else None
            tr = buf(name + "T", K, N, zero_pad)
            r = 0
            for w in blocks:
                w = w.detach()
                n = w.shape[0]
                jobs.append((w if w.stride(1) == 1 else w.contiguous(), cp[r:r + n] if cp is not None else None,
                             tr[:, r:r + n]))
                r += n
            return cp, tr
        _, W["w3T"] = linear_weight("w3", [W["w3"]], want_copy=False)  # [F2*C, D] bf16 from the fp16 fc3 operand
        layers = []
        for li, lyr in enumerate(enc.layers):
            sa = lyr.self_attn
            if hasattr(sa, "in_proj_weight"):
                qkv_blocks, bqkv = [sa.in_proj_weight], sa.in_proj_bias.detach().float().contiguous()
            else:
                qkv_blocks = [sa.q_proj.weight, sa.k_proj.weight, sa.v_proj.weight]
                bqkv = torch.cat([sa.q_proj.bias, sa.k_proj.bias, sa.v_proj.bias], 0).detach().float()
            d = dict(bqkv=bqkv, bo=sa.out_proj.bias.detach().float().contiguous(),
                     b1=lyr.fc1.bias.detach().float().contiguous(), b2=lyr.fc2.bias.detach().float().contiguous(),
                     g1=lyr.self_attn_layer_norm.weight.detach().float().contiguous(),
                     be1=lyr.self_attn_layer_norm.bias.detach().float().contiguous(),
                     g2=lyr.final_layer_norm.weight.detach().float().contiguous(),
                     be2=lyr.final_layer_norm.bias.detach().float().contiguous(),
                     eps1=lyr.self_attn_layer_norm.eps, eps2=lyr.final_layer_norm.eps)
            d["wqkv"], d["wqkvT"] = linear_weight("l%d.wqkv" % li, qkv_blocks)
            d["wo"], d["woT"] = linear_weight("l%d.wo" % li, [sa.out_proj.weight])
            d["w1"], d["w1T"] = linear_weight("l%d.w1" % li, [lyr.fc1.weight])
            d["w2"], d["w2T"] = linear_weight("l%d.w2" % li, [lyr.fc2.weight])
            layers.append(d)
        W["layers"] = layers
        W["gf"] = enc.layer_norm.weight.detach().float().contiguous()
        W["bf"] = enc.layer_norm.bias.detach().float().contiguous()
        if enc.ctc_compress_out:
            # wcT: [D, V] view of a [D, ceil8(V)] buffer whose pad columns stay zero (the dgrad GEMM contracts
            # over the padded V)
            W["wc"], W["wcT"] = linear_weight("wc", [enc.ctc_fc.weight], zero_pad=True)
            W["bc"] = enc.ctc_fc.bias.detach().float().contiguous()
        ops.prep_batch(jobs)
    enc._train_prep, enc._train_prep_key = W, key
    return W


def flat_parameters(enc):
    """The parameters the Function differentiates, in a fixed order (matches ``_assemble_grads``)."""
    ps = [enc.convolutions[0].weight, enc.convolutions[0].bias, enc.bn[0].weight, enc.bn[0].bias,
          enc.convolutions[1].weight, enc.convolutions[1].bias, enc.bn[1].weight, enc.bn[1].bias,
          enc.fc3.weight, enc.fc3.bias]
    for lyr in enc.layers:
        sa = lyr.self_attn
        if hasattr(sa, "in_proj_weight"):
            ps += [sa.in_proj_weight, sa.in_proj_bias]
        else:
            ps += [sa.q_proj.weight, sa.q_proj.bias, sa.k_proj.weight, sa.k_proj.bias, sa.v_proj.weight,
                   sa.v_proj.bias]
        ps += [sa.out_proj.weight, sa.out_proj.bias, lyr.self_attn_layer_norm.weight, lyr.self_attn_layer_norm.bias,
               lyr.fc1.weight, lyr.fc1.bias, lyr.fc2.weight, lyr.fc2.bias, lyr.final_layer_norm.weight,
               lyr.final_layer_norm.bias]
    ps += [enc.layer_norm.weight, enc.layer_norm.bias]
    if enc.ctc_compress_out:
        ps += [enc.ctc_fc.weight, enc.ctc_fc.bias]
    return ps


def _bn_state(enc, i, y_relu, train):
    """(mean, rstd, scale, shift) of BatchNorm i for this step: batch statistics (+ running-stat update,
    nn.BatchNorm2d momentum 0.1) in training, running statistics in eval."""
    bn = enc.bn[i]
    if train:
        m, r, sc, sh = ops.bn_batch_stats(y_relu, bn.weight.detach().float(), bn.bias.detach().float(), bn.eps,
                                          bn.momentum if bn.momentum is not None else 0.1, bn.running_mean,
                                          bn.running_var)
        bn.num_batches_tracked += 1
        return m, r, sc, sh
    sc, sh = ops.prep_bn_affine(bn.weight.detach().float(), bn.bias.detach().float(), bn.running_mean.float(),
                                bn.running_var.float(), bn.eps)
    mean = bn.running_mean.float().contiguous()
    rstd = (bn.running_var.float() + bn.eps).rsqrt().contiguous()  # [C]: parameter-sized, not activations
    return mean, rstd, sc, sh


def pretranspose(S):
    """Token-contiguous (transposed) bf16 copies of the activations the weight-gradient GEMMs read, for the saved
    state ``S`` of one training forward: one batched launch (+ conv2's im2col).  Idempotent."""
    if S is None or S.get("pretransposed"):
        return
    S["pretransposed"] = True
    x_in = S["x_in"]
    dev = x_in.device
    jobs = []

    def tjob(t):
        out = ops.transposed_buffer(t.shape[0], t.shape[1], dev)
        jobs.append((t, None, out))
        return out
    y2 = S["y2"]
    S["y2T"] = tjob(y2.view(y2.shape[0] * y2.shape[1], -1))
    ops.prep_batch(jobs)
    S["colT"] = ops.conv2_im2col_t(S["y1"])


class EncoderTrainFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, enc, src_tokens, len_host, seed, *params):
        dev = src_tokens.device
        train = enc.training
        ctx.set_materialize_grads(False)  # an unused output (ctc_out or the tap) must arrive as None, not zeros
        W = prepare_train_weights(enc)
        B, T, Fd = src_tokens.shape
        C, D, H = enc.conv_channels, enc.embed_dim, enc.heads
        p = enc.dropout if train else 0.0
        p_conv = max(enc.dropout, 0.1) if train else 0.0  # conv_transformer.py:214
        p_att = enc.attention_dropout if train else 0.0
        p_act = enc.activation_dropout if train else 0.0
        x_in = src_tokens.float().contiguous()
        sub = [((n + 1) // 2 + 1) // 2 for n in len_host]
        L = ((T + 1) // 2 + 1) // 2
        lengths = torch.tensor(sub, dtype=torch.int32, device=dev)
        ones = torch.ones(C, dtype=torch.float32, device=dev)
        zeros = torch.zeros(C, dtype=torch.float32, device=dev)
        S = dict(B=B, T=T, Fd=Fd, L=L, train=train, seed=seed, p=p, p_conv=p_conv, p_att=p_att, p_act=p_act,
                 x_in=x_in, lengths=lengths)

        # ---- conv front end: ReLU(conv) kept (BatchNorm / ReLU backward need it), BN + dropout as its own pass
        y1r = ops.conv1_relu_bn(x_in, W["w1"], W["b1"], ones, zeros)
        bn1 = _bn_state(enc, 0, y1r, train)
        y1 = ops.bn_apply(y1r, bn1[2], bn1[3], p_conv, seed, _SITE_CONV1)
        y2r = ops.conv2_relu_bn(y1, W["w2"], W["b2"], ones, zeros)
        bn2 = _bn_state(enc, 1, y2r, train)
        y2 = ops.bn_apply(y2r, bn2[2], bn2[3], p_conv, seed, _SITE_CONV2)
        assert y2.shape[1] == L
        S.update(y1r=y1r, y1=y1, y2r=y2r, y2=y2, bn1=bn1[:2], bn2=bn2[:2])
        h3 = ops.linear(y2.view(B * L, -1), W["w3"], W["b3"], relu=True, out_dtype=torch.float32)
        S["h3b"] = ops.cast_bf16(h3)  # ReLU mask for the backward ((b, t) row order)
        table = enc._positions(L + 1, dev) if enc.embed_positions is not None else None
        x0, _, _ = ops.embed_remap_stats(h3, L, B, table, lengths if table is not None else None)
        lay0 = W["layers"][0] if W["layers"] else None
        # embedding dropout (conv_transformer.py:232) fused with the first layer's LayerNorm
        if lay0 is not None:
            x, ln = ops.dropout_add_ln(x0, None, lay0["g1"], lay0["be1"], lay0["eps1"], p, seed, _SITE_EMB)
        else:
            x, ln = ops.dropout_add_ln(x0, None, None, None, 1e-5, p, seed, _SITE_EMB)
        mask = ops.lengths_to_mask(lengths, L)[0] if min(sub) < L else None
        ctc_mask, x_ctc, states = mask, None, []
        cur_L, cur_len, cur_host = L, lengths, sub
        saved = []
        n_layers = len(W["layers"])
        for li, Wl in enumerate(W["layers"]):
            torch.empty(1).uniform_()  # LayerDrop draw of the reference (:241): keep its CPU RNG stream
            sites = _layer_sites(li)
            M = cur_L * B
            qkv = ops.linear(ln, Wl["wqkv"], Wl["bqkv"])
            att, lse = ops.attention_train_fwd(qkv, cur_len, cur_L, B, H, enc.log_penalty, p_att, seed, sites["att"])
            a = ops.linear(att, Wl["wo"], Wl["bo"], out_dtype=torch.float32)
            x1, ln2 = ops.dropout_add_ln(a, x, Wl["g2"], Wl["be2"], Wl["eps2"], p, seed, sites["out"])
            f = ops.linear(ln2, Wl["w1"], Wl["b1"], relu=True)
            ops.dropout_(f, p_act, seed, sites["act"])
            o = ops.linear(f, Wl["w2"], Wl["b2"], out_dtype=torch.float32)
            ctc_here = enc.ctc_compress_out and enc.ctc_layer == li + 1
            last = li + 1 == n_layers
            rec = dict(x=x, ln1=ln, qkv=qkv, att=att, lse=lse, x1=x1, ln2=ln2, f=f, L=cur_L, lengths=cur_len,
                       sites=sites, ctc=None)
            if ctc_here or last:
                x2, _ = ops.dropout_add_ln(o, x1, None, None, 1e-5, p, seed, sites["ffn"])
                ln = None
            else:
                nxt = W["layers"][li + 1]
                x2, ln = ops.dropout_add_ln(o, x1, nxt["g1"], nxt["be1"], nxt["eps1"], p, seed, sites["ffn"])
            if ctc_here:
                # conv_transformer.py:278-291: logits WITH grad, argmax / segments / weights without
                xb = ops.cast_bf16(x2)
                V = enc.ctc_fc.out_features
                logits = ops.linear(xb, W["wc"], W["bc"], out_dtype=torch.float32)  # [M, V] view, pitch ceil8(V)
                x_ctc = logits.view(cur_L, B, V)
                hooked = x_ctc  # forward hooks (d hooked / d logits = identity): their output is what is returned
                for hook in enc.ctc_fc._forward_hooks.values():  # test / bench logit injection (SURVEY F9)
                    r = hook(enc.ctc_fc, (x2.view(cur_L, B, D),), hooked)
                    hooked = hooked if r is None else r
                if enc.ctc_logit_bump is not None:  # the inference path's built-in injection, same semantics
                    bl, bm = enc.ctc_logit_bump
                    bl = bl(cur_L, B) if callable(bl) else bl
                    bump = torch.full((cur_L, B, 1), float(bm), dtype=hooked.dtype, device=dev)
                    if hooked is x_ctc:  # our own fresh buffer: in place (no 771 MB copy, rows stay 16-byte aligned)
                        hooked.scatter_add_(2, bl.long().unsqueeze(-1), bump)
                    else:
                        hooked = hooked.scatter_add(2, bl.long().unsqueeze(-1), bump)
                lg = hooked.reshape(M, V) if hooked.stride(-1) == 1 else hooked.contiguous().view(M, V)
                want_prob = enc.ctc_compress_strategy != "avg"
                labels, prob = ops.ctc_argmax(lg, cur_len, cur_L, B, V, want_prob)
                seg_id, seg_start, weight, new_len, max_new = ops.ctc_segment(
                    labels, prob, cur_len, enc.ctc_compress_strategy, cur_L, B)
                xc = ops.ctc_compress(x2, seg_id, seg_start, weight, cur_len, new_len, max_new, cur_L, B)
                new_host = new_len.cpu().tolist()  # the step's one shape synchronisation
                L2 = max(new_host)
                rec["ctc"] = dict(xb=xb, seg_id=seg_id, weight=weight, L2=L2, V=V)
                ctc_ret, ctc_tap = hooked, x2  # (x2: the projection's input, handed out as a gradient tap)
                x2 = xc[: L2 * B]
                cur_L, cur_len, cur_host = L2, new_len, new_host
                mask = ops.lengths_to_mask(cur_len, cur_L)[0] if min(cur_host) < cur_L else None
                if not last:
                    nxt = W["layers"][li + 1]
                    _, ln = ops.dropout_add_ln(x2, None, nxt["g1"], nxt["be1"], nxt["eps1"], want_x=False)
            saved.append(rec)
            states.append(x2.view(cur_L, B, D))
            x = x2
        xf = ops.layernorm(x, W["gf"], W["bf"], out_dtype=torch.float32, eps=enc.layer_norm.eps)
        S.update(layers=saved, x_last=x, L_out=cur_L)
        # The weight-gradient GEMMs contract over tokens and want token-contiguous operands; the activation halves
        # of those operands depend on the forward only.  `pretranspose(S)` makes them in one batched launch; it is
        # called by whoever runs first in the backward (criterion.CtcProjLossFn: before the decoder's backward,
        # which is bound by the host's launch rate and leaves the GPU idle) -- inside this node's backward they
        # sit on the GPU-bound critical path (44 launches, ~1.3 ms per cfg4 step).
        mode = getattr(enc, "pretranspose_activations", True)
        mode = "bwd" if mode is True else ("off" if not mode else mode)
        enc._train_pending = S if mode == "bwd" else None
        if mode == "fwd":
            pretranspose(S)
        ctx.S, ctx.enc = S, enc
        if getattr(enc, "keep_train_state", False):  # tests: the activation patterns of this forward
            enc.last_train_state = S
        ctx.n_params = len(params)
        out = xf.view(cur_L, B, D)
        states[-1] = out
        ctx.has_ctc = x_ctc is not None
        extras = dict(mask=mask, ctc_mask=ctc_mask, states=states, out_len=cur_host)
        enc._train_extras = extras
        # the intermediate states (x2 after each layer but the last, compressed after the CTC layer) come last:
        # a loss on one of them (the CTC-multitask recipe without --ctc-compress-out projects encoder_states[k-1])
        # sends its gradient back into this node.  They are the saved activations the backward reads.
        if x_ctc is None:
            return (out,) + tuple(states[:-1])
        # third output: the CTC projection's INPUT.  A criterion that computes the projection's backward itself
        # (criterion.CtcProjLossFn: early in the backward, while the decoder's backward keeps the host busy)
        # sends d loss / d x back through it; with any other criterion the gradient arrives through ctc_ret
        return (out, ctc_ret, ctc_tap) + tuple(states[:-1])

    @staticmethod
    def backward(ctx, d_out, *d_rest):
        d_ctc, d_tap = (d_rest[0], d_rest[1]) if ctx.has_ctc else (None, None)
        d_states = d_rest[2:] if ctx.has_ctc else d_rest
        S, enc = ctx.S, ctx.enc
        if getattr(enc, "_train_pending", None) is S:  # no criterion node did it earlier: one batched launch here
            enc._train_pending = None
            pretranspose(S)
        elif not S.get("pretransposed") and getattr(enc, "pretranspose_activations", True):
            pretranspose(S)
        W = prepare_train_weights(enc)
        B, L, D, H, C = S["B"], S["L"], enc.embed_dim, enc.heads, enc.conv_channels
        seed, p, p_act, p_att, p_conv = S["seed"], S["p"], S["p_act"], S["p_att"], S["p_conv"]
        # every reduction whose result is only read when the backward returns (bias gradients, split-K slices of
        # the weight gradients, LayerNorm parameter gradients: ~120 per step) is queued and launched as ONE batch
        with ops.deferred_reductions():
            G = {}
            M_out = S["L_out"] * B
            if d_out is None:
                dx = torch.zeros(M_out, D, dtype=torch.float32, device=S["x_in"].device)
            else:
                dy = d_out.reshape(M_out, D).float().contiguous()
                dx, G["gf"], G["bf"] = ops.ln_bwd(dy, S["x_last"], W["gf"], eps=enc.layer_norm.eps)
            for li in range(len(S["layers"]) - 1, -1, -1):
                R, Wl = S["layers"][li], W["layers"][li]
                cur_L, cur_len, sites = R["L"], R["lengths"], R["sites"]
                M = cur_L * B
                g = {}
                d_state = d_states[li] if li < len(d_states) else None
                if d_state is not None:
                    # dx is d loss / d (this layer's output): the state's own gradient joins it here, on the
                    # compressed rows for the CTC layer (before ctc_compress_bwd)
                    dx += d_state.reshape(dx.shape)
                if R["ctc"] is not None:
                    ct = R["ctc"]
                    # dx holds the L2*B compressed rows; a frame's segment id is < its utterance's new length <= L2
                    dx = ops.ctc_compress_bwd(dx, ct["seg_id"], ct["weight"], cur_L, B)
                    if d_tap is not None:
                        dx += d_tap.reshape(M, D)
                    if d_ctc is not None:
                        V = ct["V"]
                        Vp = (V + 7) // 8 * 8
                        gc = d_ctc.reshape(M, V)
                        if gc.dtype != torch.float32 or gc.stride(-1) != 1:
                            gc = gc.float().contiguous()
                        gb, gT, G["bc"] = ops.grad_prep(gc, n_pad=Vp)
                        G["wc"] = ops.linear_wgrad(gT, ops.transpose_bf16(ct["xb"]))
                        wcT = W["wcT"]
                        wcT_full = wcT if Vp == V else torch.as_strided(wcT, (D, Vp), (wcT.stride(0), 1))
                        dx = ops.linear(gb, wcT_full, None, residual=dx, out_dtype=torch.float32)
                # ---- feed-forward block (transformer_layer.py:124-136).  The weight gradients read the saved
                # activations in their natural [tokens, features] layout (both operands MN-major in the tensor
                # cores), not token-contiguous transposed copies: measured (cfg4, r02x) backward 20.7 -> 20.05 ms
                g2, _, g["b2"] = ops.grad_prep(dx, p=p, seed=seed, site=sites["ffn"], dp_cols=D, want_gT=False)
                g["w2"] = ops.linear_wgrad_nt(g2, R["f"])
                df = ops.linear(g2, Wl["w2T"])
                dh, _, g["b1"] = ops.grad_prep(df, act=R["f"], act_scale=1.0 / (1.0 - p_act) if p_act > 0 else 1.0,
                                               want_gT=False)
                g["w1"] = ops.linear_wgrad_nt(dh, R["ln2"])
                dln2 = ops.linear(dh, Wl["w1T"], out_dtype=torch.float32)
                dx, g["g2"], g["be2"] = ops.ln_bwd(dln2, R["x1"], Wl["g2"], dx=dx, eps=Wl["eps2"])
                # ---- self-attention block (:104-122)
                g1, _, g["bo"] = ops.grad_prep(dx, p=p, seed=seed, site=sites["out"], dp_cols=D, want_gT=False)
                g["wo"] = ops.linear_wgrad_nt(g1, R["att"])
                dO = ops.linear(g1, Wl["woT"])
                dqkv = ops.attention_train_bwd(R["qkv"], R["att"], dO, R["lse"], cur_len, cur_L, B, H, enc.log_penalty,
                                               p_att, seed, sites["att"])
                _, _, g["bqkv"] = ops.grad_prep(dqkv, want_gb=False, want_gT=False)
                g["wqkv"] = ops.linear_wgrad_nt(dqkv, R["ln1"])
                dln1 = ops.linear(dqkv, Wl["wqkvT"], out_dtype=torch.float32)
                dx, g["g1"], g["be1"] = ops.ln_bwd(dln1, R["x"], Wl["g1"], dx=dx, eps=Wl["eps1"])
                G[li] = g
            # ---- embedding dropout, positions (constant), fc3 + ReLU (conv_transformer.py:225-232)
            F2C = S["y2"].shape[2] * C
            dh3, dh3T, G["b3"] = ops.grad_prep(dx, act=S["h3b"], remap=(L, B), p=p, seed=seed, site=_SITE_EMB, dp_cols=D)
            y2T = S["y2T"] if "y2T" in S else ops.transpose_bf16(S["y2"].view(B * L, F2C))
            dW3p = ops.linear_wgrad(dh3T, y2T)  # [D, F2*C] (f, c) order
            dy2 = ops.linear(dh3, W["w3T"])  # [B*L, F2*C] bf16 == [B, T2, F2, C]
            # ---- conv2 block
            bn = enc.bn[1]
            dz2, G["bn1_b"], G["bn1_w"] = ops.bn_relu_bwd(dy2.view(S["y2"].shape), S["y2r"], bn.weight.detach().float(),
                                                          S["bn2"][0], S["bn2"][1], S["train"], p_conv, seed, _SITE_CONV2)
            P2 = dz2.numel() // C
            _, dz2T, G["cb2"] = ops.grad_prep(dz2.view(P2, C), want_gb=False)
            dW2p = ops.linear_wgrad(dz2T, S["colT"] if "colT" in S else ops.conv2_im2col_t(S["y1"]))  # [Cout, (tap, ci)]
            dcol = ops.linear(dz2.view(P2, C), W["w2d"])
            T1, F1 = S["y1"].shape[1], S["y1"].shape[2]
            dy1 = ops.conv2_col2im(dcol, B, T1, F1, C)
            # ---- conv1 block
            bn = enc.bn[0]
            dz1, G["bn0_b"], G["bn0_w"] = ops.bn_relu_bwd(dy1, S["y1r"], bn.weight.detach().float(), S["bn1"][0],
                                                          S["bn1"][1], S["train"], p_conv, seed, _SITE_CONV1)
            dW1, G["cb1"] = ops.conv1_wgrad(dz1, S["x_in"])
            G["cw1"] = dW1.reshape(C, 1, 3, 3)
        G["w3"] = dW3p.view(D, enc.feat_out, C).permute(0, 2, 1).reshape(D, C * enc.feat_out)
        G["cw2"] = dW2p.view(C, 3, 3, C).permute(0, 3, 1, 2).contiguous()
        ctx.S = None  # release the saved activations
        grads = _assemble_grads(enc, G, d_ctc is not None)
        # fp16 training (`--fp16`: model.half(), fp32 master copy in fairseq's FP16Optimizer): autograd wants
        # every gradient in its parameter's dtype
        grads = [g if g is None or g.dtype == p.dtype else g.to(p.dtype) for g, p in zip(grads, flat_parameters(enc))]
        return (None, None, None, None) + tuple(grads)


def _assemble_grads(enc, G, have_ctc):
    D = enc.embed_dim
    out = [G["cw1"], G["cb1"], G["bn0_w"], G["bn0_b"], G["cw2"], G["cb2"], G["bn1_w"], G["bn1_b"], G["w3"], G["b3"]]
    for li, lyr in enumerate(enc.layers):
        g = G[li]
        if hasattr(lyr.self_attn, "in_proj_weight"):
            out += [g["wqkv"], g["bqkv"]]
        else:
            for k in range(3):
                out += [g["wqkv"][k * D:(k + 1) * D], g["bqkv"][k * D:(k + 1) * D]]
        out += [g["wo"], g["bo"], g["g1"], g["be1"], g["w1"], g["b1"], g["w2"], g["b2"], g["g2"], g["be2"]]
    out += [G.get("gf"), G.get("bf")]
    if enc.ctc_compress_out:
        out += [G.get("wc"), G.get("bc")] if have_ctc else [None, None]
    return out


def forward_train(enc, src_tokens, src_lengths, return_all_hiddens):
    """The encoder's forward when gradients are required: returns the reference's output tuple, with
    ``encoder_out``, ``ctc_out`` and (``return_all_hiddens``) every entry of ``encoder_states`` attached to the
    autograd graph: a loss on an intermediate state (CTC multitask without --ctc-compress-out) trains the layers
    below it.  The intermediate states are the saved activations the backward reads: consumers must not modify
    them in place (fairseq does not; autograd refuses it in fp32, where they are views the node created)."""
    from .encoder import CTCAwareEncoderOut, EncoderOut  # (resolved late: the plugin swaps in fairseq's types)
    from . import encoder as _e
    if enc.training and enc.encoder_layerdrop > 0:
        raise NotImplementedError("fbkst_b200: LayerDrop is not supported in training (--encoder-layerdrop 0)")
    if enc.layernorm_embedding is not None:
        raise NotImplementedError("fbkst_b200: layernorm_embedding is not supported in training")
    if enc.embed_positions is not None and enc.embed_positions.learned:
        raise NotImplementedError("fbkst_b200: learned positional embeddings are inference-only (no reference "
                                  "architecture enables --encoder-learned-pos)")
    len_host = src_lengths.tolist()
    # one 63-bit seed per step from torch's CPU generator (fairseq re-seeds it per update: trainer.py:655-661)
    seed = int(torch.empty((), dtype=torch.int64).random_().item()) if enc.training else 0
    params = flat_parameters(enc)
    res = EncoderTrainFn.apply(enc, src_tokens, len_host, seed, *params)
    ex = enc._train_extras
    enc._train_extras = None
    n_head = len(res) - (len(ex["states"]) - 1)
    res, mid = res[:n_head], list(res[n_head:])
    tap = res[2] if len(res) > 2 else None
    res = res[:2]
    out = res[0]
    odt = enc.layer_norm.weight.dtype
    if odt != torch.float32:  # model.half(): hand fp16 activations to the fp16 decoder (differentiable casts)
        res = tuple(r.to(odt) for r in res)
        out = res[0]
    if tap is not None and getattr(enc, "ctc_grad_tap", True):
        # read by criterion.ctc_loss_train (same tensor object, i.e. as long as nobody transforms ctc_out on the
        # way to the criterion): (projection input with grad_fn, encoder)
        res[1]._fbkst_tap = (tap, enc)
    states = None
    if return_all_hiddens:
        if odt != torch.float32:
            mid = [s.to(odt) for s in mid]
        for s in mid:  # read by criterion.CtcProjection: whose pending activation transposes its backward starts
            s._fbkst_encoder = enc
        states = mid + [out]
    out_lengths = torch.tensor(ex["out_len"], dtype=src_lengths.dtype, device=src_tokens.device)
    if enc.ctc_compress_out:
        return _e.CTCAwareEncoderOut(out, ex["mask"], None, states, src_tokens, out_lengths,
                                     res[1] if len(res) > 1 else None, ex["ctc_mask"])
    return _e.EncoderOut(out, ex["mask"], None, states, src_tokens, out_lengths)
