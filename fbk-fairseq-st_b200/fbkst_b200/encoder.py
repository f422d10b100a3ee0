"""Drop-in ``ConvolutionalTransformerEncoder`` whose forward runs on the sm_100a kernels.

Mirrors the reference module interface
(examples/speech_recognition/models/conv_transformer.py:124-345):

  * ``__init__(args, dictionary, audio_features=40)`` reading the same ``args`` fields;
  * ``forward(src_tokens, src_lengths, cls_input=None, return_all_hiddens=False, **ignored)``
    returning ``EncoderOut`` / ``CTCAwareEncoderOut`` with the reference's field order;
  * ``reorder_encoder_out``, ``forward_non_torchscript``, ``output_batch_first``;
  * the same parameter names and shapes, so reference checkpoints load with ``strict=True``
    (both self-attention layouts of SURVEY F6).

``torch.nn`` modules are used only as parameter containers (state_dict layout); none of their
``forward`` methods run.  There is no CPU / PyTorch fallback: without the CUDA library and a B200
the forward raises.  Round 1 implements inference (``eval()``); the training backward is not
implemented and ``forward`` raises in training mode instead of silently degrading.
"""
import math
from typing import Dict, List, NamedTuple, Optional

import torch
import torch.nn as nn
from torch import Tensor

from . import ops

try:  # plug into fairseq when it is importable (train.py / generate.py --user-dir)
    from fairseq.models import FairseqEncoder as _Base  # type: ignore
    _HAVE_FAIRSEQ = True
except Exception:  # standalone (tests, bench, the GPU box)
    _HAVE_FAIRSEQ = False

    class _Base(nn.Module):
        def __init__(self, dictionary):
            super().__init__()
            self.dictionary = dictionary

        def max_positions(self):
            return 1e6


class _PinnedPool:
    """Pinned int32 staging vectors, one per in-flight use.  A vector goes back to the pool only when
    its user is done with it: ``give(t)`` after the host has read a D2H result, ``give(t, event)`` for
    an H2D source (it is handed out again only once ``event`` -- recorded after the copy -- has
    completed).  The host can run any number of launches ahead of the GPU without a staging vector
    being rewritten under a copy that has not executed yet (ADVICE r01: the fixed 8-slot rings could)."""

    def __init__(self):
        self._free = {}

    def take(self, n):
        lst = self._free.setdefault(n, [])
        for i, (t, ev) in enumerate(lst):
            if ev is None or ev.query():
                lst.pop(i)
                return t
        return torch.empty(n, dtype=torch.int32).pin_memory()

    def give(self, t, event=None):
        self._free.setdefault(t.numel(), []).append((t, event))


class EncoderOut(NamedTuple):
    """fairseq/models/fairseq_encoder.py:11-21"""
    encoder_out: Tensor  # T x B x C
    encoder_padding_mask: Optional[Tensor]  # B x T
    encoder_embedding: Optional[Tensor]
    encoder_states: Optional[List[Tensor]]
    src_tokens: Optional[Tensor]
    src_lengths: Optional[Tensor]


class CTCAwareEncoderOut(NamedTuple):
    """conv_transformer.py:28-32"""
    encoder_out: Tensor
    encoder_padding_mask: Optional[Tensor]
    encoder_embedding: Optional[Tensor]
    encoder_states: Optional[List[Tensor]]
    src_tokens: Optional[Tensor]
    src_lengths: Optional[Tensor]
    ctc_out: Tensor  # T x B x V
    ctc_padding_mask: Optional[Tensor]


# ---------------------------------------------------------------- parameter containers + init
def _conv2d(cin, cout, k, dropout):
    """conv_transformer.py:348-354"""
    m = nn.Conv2d(cin, cout, kernel_size=k, padding=k // 2, stride=2)
    std = math.sqrt((4 * (1.0 - dropout)) / (m.kernel_size[0] * cin))
    nn.init.normal_(m.weight, mean=0, std=std)
    nn.init.constant_(m.bias, 0)
    return m


def _linear(i, o):
    """conv_transformer.py:371-375"""
    m = nn.Linear(i, o)
    nn.init.xavier_uniform_(m.weight)
    nn.init.constant_(m.bias, 0.0)
    return m


class _LocalAttentionParams(nn.Module):
    """Parameter layout of modules/local_attention.py:33-47 (fused in-projection)."""

    def __init__(self, D):
        super().__init__()
        self.in_proj_weight = nn.Parameter(torch.empty(3 * D, D))
        self.in_proj_bias = nn.Parameter(torch.zeros(3 * D))
        self.out_proj = nn.Linear(D, D)
        nn.init.xavier_uniform_(self.in_proj_weight)
        nn.init.xavier_uniform_(self.out_proj.weight)
        nn.init.constant_(self.out_proj.bias, 0.0)

    def qkv(self):
        return self.in_proj_weight, self.in_proj_bias


class _MultiheadAttentionParams(nn.Module):
    """Parameter layout of fairseq/modules/multihead_attention.py:61-65 (separate q/k/v)."""

    def __init__(self, D):
        super().__init__()
        self.k_proj, self.v_proj, self.q_proj = nn.Linear(D, D), nn.Linear(D, D), nn.Linear(D, D)
        self.out_proj = nn.Linear(D, D)
        for m in (self.k_proj, self.v_proj, self.q_proj):  # multihead_attention.py:88-94
            nn.init.xavier_uniform_(m.weight, gain=1 / math.sqrt(2))
        nn.init.xavier_uniform_(self.out_proj.weight)
        nn.init.constant_(self.out_proj.bias, 0.0)

    def qkv(self):
        w = torch.cat([self.q_proj.weight, self.k_proj.weight, self.v_proj.weight], 0)
        b = torch.cat([self.q_proj.bias, self.k_proj.bias, self.v_proj.bias], 0)
        return w, b


class _EncoderLayerParams(nn.Module):
    """fairseq/modules/transformer_layer.py:32-57 + modules/conv_transformer_layer.py:9-19."""

    def __init__(self, D, Dff, log_penalty):
        super().__init__()
        self.self_attn = _LocalAttentionParams(D) if log_penalty else _MultiheadAttentionParams(D)
        self.self_attn_layer_norm = nn.LayerNorm(D)
        self.fc1 = nn.Linear(D, Dff)
        self.fc2 = nn.Linear(Dff, D)
        self.final_layer_norm = nn.LayerNorm(D)


class _SinusoidalParams(nn.Module):
    """Keeps the reference's only persistent buffer (``_float_tensor``)."""

    def __init__(self):
        super().__init__()
        self.register_buffer("_float_tensor", torch.zeros(1))


class _PositionalParams(nn.Module):
    """``PositionalEmbeddingAudio`` (modules/positional_embedding_audio.py:13-19) as a parameter container:
    sinusoidal (one persistent buffer) or, with ``--encoder-learned-pos``, an ``nn.Embedding`` with
    ``padding_idx = 0`` exactly like ``LearnedPositionalEmbedding(num_embeddings, dim, 0)`` (same state_dict key
    ``embed_positions.embeddings.weight``, same default initialisation).  Both are read the same way by the
    kernel: row t + 1 for frame t < length, the padding row 0 beyond (fairseq/utils.py:192-202)."""

    def __init__(self, learned=False, num_embeddings=0, dim=0):
        super().__init__()
        self.learned = learned
        self.embeddings = nn.Embedding(num_embeddings, dim, padding_idx=0) if learned else _SinusoidalParams()


class CtcProjection(nn.Linear):
    """``ctc_fc`` (conv_transformer.py:190): an ``nn.Linear`` whose forward is the tcgen05 GEMM,
    so forward hooks registered on it behave as on the reference module.  Input L x B x D fp32,
    output L x B x V logits in FP32 like the reference's (fp32 accumulators written unrounded; rows
    padded to a multiple of 8 columns in memory): the CTC argmax, the pooling probabilities and the
    CTC loss all see un-rounded logits, so near-ties between the top two labels are not turned into
    exact ties by a bf16 store (ADVICE r01).  ``logits_dtype = torch.bfloat16`` is an opt-in that halves
    the 2 x L*B*V*4 bytes this costs, for callers that accept bf16-rounded logits."""
    logits_dtype = torch.float32
    precision = "bf16"  # set by the encoder's ``precision``: "fp32" runs the split-TF32 GEMM on fp32 operands

    def forward(self, x):  # noqa: D401
        L, B, D = x.shape
        if self.precision == "fp32":
            self._bf16_operand = None
            w, b = self._prepared_f32()
            return ops.linear_f32(x.reshape(L * B, D).contiguous(), w, b).view(L, B, -1)
        w, b = self._prepared()
        pre = getattr(self, "_bf16_operand", None)  # (data_ptr of x, bf16(x)) left by the fc2 epilogue
        self._bf16_operand = None
        if pre is not None and pre[0] == x.data_ptr() and pre[1].shape == (L * B, D):
            a = pre[1]
        else:
            a = ops.cast_bf16(x.reshape(L * B, D))
        return ops.linear(a, w, b, out_dtype=self.logits_dtype).view(L, B, -1)

    def project_argmax(self, x2d, xb, lengths, L, B, want_prob, bump):
        """Fused path (no forward hooks to honour): logits + frame arg-max from one GEMM (ops.linear_argmax)."""
        w, b = self._prepared()
        a = xb if xb is not None else ops.cast_bf16(x2d)
        return ops.linear_argmax(a, w, b, lengths, L, B, want_prob=want_prob, bump=bump)

    def _prepared(self):
        key = (self.weight._version, self.bias._version, self.weight.data_ptr())
        if getattr(self, "_prep_key", None) != key:
            self._prep = (ops.cast_bf16(self.weight.detach()), self.bias.detach().float().contiguous())
            self._prep_key = key
        return self._prep

    def _prepared_f32(self):
        key = (self.weight._version, self.bias._version, self.weight.data_ptr())
        if getattr(self, "_prep32_key", None) != key:
            self._prep32 = (self.weight.detach().float().contiguous(), self.bias.detach().float().contiguous())
            self._prep32_key = key
        return self._prep32


PRECISIONS = ("bf16", "fp32")


def make_encoder_class(base):
    """The encoder class on top of ``base`` (fairseq's ``FairseqEncoder`` inside fairseq, a small
    ``nn.Module`` shim standalone).  ``fairseq_model.py:247`` asserts ``isinstance(encoder,
    FairseqEncoder)``, so the plugin instantiates this with the real base class."""

    class ConvolutionalTransformerEncoder(base):
        def __init__(self, args, dictionary, audio_features=40):
            super().__init__(dictionary)
            convs = eval(args.encoder_convolutions) if args.encoder_convolutions is not None \
                else ((512, 3),) * 2
            if len(convs) != 2:
                raise NotImplementedError("fbkst_b200: exactly two subsampling convolutions are supported")
            self.dropout = args.dropout
            # training-mode dropout sites (local_attention.py:136; fairseq/modules/transformer_layer.py:43-46)
            self.attention_dropout = float(getattr(args, "attention_dropout", 0.0) or 0.0)
            self.activation_dropout = float(getattr(args, "activation_dropout", 0) or 0)
            if self.activation_dropout == 0:
                self.activation_dropout = float(getattr(args, "relu_dropout", 0) or 0)
            if getattr(args, "activation_fn", "relu") != "relu":
                raise NotImplementedError("fbkst_b200: only activation_fn=relu is supported")
            if getattr(args, "attn_2d", False):
                raise NotImplementedError(
                    "fbkst_b200: ConvAttention2D is outside the accelerated path; pass --no-attn-2d")
            penalty = getattr(args, "distance_penalty", False)
            if penalty is True:
                penalty = "log"
            if penalty not in (False, None, "log"):
                raise NotImplementedError("fbkst_b200: distance penalty %r is not supported (the "
                                          "reference's 'gauss' penalty crashes on construction)" % penalty)
            self.log_penalty = penalty == "log"
            if not getattr(args, "encoder_normalize_before", True):
                raise NotImplementedError("fbkst_b200: only pre-LayerNorm encoders (all reference archs)")

            self.convolutions = nn.ModuleList()
            cin = 1
            for spec in convs:
                cout, k = spec[0], spec[1]
                if k != 3 or (len(spec) > 2 and spec[2] != 3):
                    raise NotImplementedError("fbkst_b200: only 3x3 convolutions are supported")
                self.convolutions.append(_conv2d(cin, cout, k, self.dropout))
                cin = cout
            self.conv_channels = cin
            if convs[0][0] != convs[1][0] or cin not in (64, 128):
                raise NotImplementedError("fbkst_b200: conv channels must be equal and 64 or 128")
            self.bn = nn.ModuleList([nn.BatchNorm2d(cin) for _ in range(2)])

            D = args.encoder_embed_dim
            self.embed_dim = D
            self.heads = args.encoder_attention_heads
            if D != 64 * self.heads:
                raise NotImplementedError("fbkst_b200: head_dim must be 64 (all reference archs)")
            flat = audio_features
            for _ in range(2):
                flat = math.ceil(flat / 2)
            self.feat_out = flat
            self.fc3 = _linear(flat * cin, D)
            self.embed_positions = None if getattr(args, "no_token_positional_embeddings", False) \
                else _PositionalParams(bool(getattr(args, "encoder_learned_pos", False)),
                                       int(getattr(args, "max_source_positions", 0) or 0), D)
            self.encoder_layerdrop = getattr(args, "encoder_layerdrop", 0.0)
            self.layers = nn.ModuleList(
                [_EncoderLayerParams(D, args.encoder_ffn_embed_dim, self.log_penalty)
                 for _ in range(args.encoder_layers)])
            self.num_layers = len(self.layers)
            self.layer_norm = nn.LayerNorm(D)
            self.layernorm_embedding = nn.LayerNorm(D) if getattr(args, "layernorm_embedding", False) \
                else None
            self.ctc_compress_out = getattr(args, "ctc_compress_out", False)
            if self.ctc_compress_out:
                self.ctc_fc = CtcProjection(D, len(dictionary))
                # conv_transformer.py:191 asserts the criterion; the plugin's device-side variant qualifies too
                assert str(args.criterion).startswith("ctc_multi_loss")
                self.ctc_layer = args.ctc_encoder_layer
                self.ctc_compress_strategy = args.ctc_compress_strategy
                if self.ctc_compress_strategy not in ("avg", "weighted", "softmax"):
                    raise ValueError("unknown --ctc-compress-strategy %r" % self.ctc_compress_strategy)
            self._prep = None
            self._prep_key = None
            self._prep32 = None
            self._prep32_key = None
            self._precision = "bf16"
            self._pos_table = None
            self._ws = None
            self._ws_key = None
            # opt-in: replay one captured CUDA graph per input shape instead of ~90 launches
            self.use_cuda_graph = False
            self.max_graphs = 16  # cached graphs (each pins its activations: ~1.2 GB at 96 k frames, d512)
            self._graphs = {}
            # graphs (and the activations they own) are per lane: EncoderPipeline keeps one forward in
            # flight per lane/stream and sets this before every launch
            self.graph_lane = 0
            # benchmark / test logit injection without a forward hook (keeps the fused ctc_fc + arg-max epilogue):
            # (labels [L, B] int32 device tensor, margin) -> logits[t, b, labels[t, b]] += margin   (SURVEY F9)
            self.ctc_logit_bump = None
            self._pins = _PinnedPool()  # pinned staging vectors for lengths (H2D sources, D2H results)

        @property
        def precision(self):
            """Operand precision of the inference forward: ``"bf16"`` (default; bf16 / fp16 tensor-core operands,
            fp32 accumulation) or ``"fp32"`` (split-TF32 tensor-core operands, about 21 significant bits, fp32
            softmax and LayerNorm: within 1e-3 of an fp32 reference).  Training runs in bf16 only."""
            return self._precision

        @precision.setter
        def precision(self, value):
            if value not in PRECISIONS:
                raise ValueError("fbkst_b200: precision must be one of %s, got %r" % (PRECISIONS, value))
            self._precision = value
            if self.ctc_compress_out:
                self.ctc_fc.precision = value

        # ------------------------------------------------------------------ derived operand formats
        def _params_key(self):
            return tuple((p._version, p.data_ptr()) for p in list(self.parameters()) + list(self.buffers()))

        def _prepared_active(self):
            return self._prepared_f32() if self._precision == "fp32" else self._prepared()

        def _prepared_f32(self):
            """Operands of the fp32 path: plain fp32 (the kernels split them), no LayerNorm folding (the fold
            feeds an uncentred operand); the conv and fc3 weights permuted to the channels-last patch order."""
            key = self._params_key()
            if self._prep32_key == key:
                return self._prep32
            f32 = lambda t: t.detach().float().contiguous()
            with torch.no_grad():
                P = {}
                C = self.conv_channels
                P["w1"] = f32(self.convolutions[0].weight.reshape(C, 9))
                P["b1"] = f32(self.convolutions[0].bias)
                P["w2"] = ops.prep_conv2_weight_f32(self.convolutions[1].weight)
                P["b2"] = f32(self.convolutions[1].bias)
                for i in range(2):
                    bn = self.bn[i]
                    P["bn%d" % i] = ops.prep_bn_affine(f32(bn.weight), f32(bn.bias), f32(bn.running_mean),
                                                       f32(bn.running_var), bn.eps)
                P["w3"] = ops.prep_fc3_weight_f32(self.fc3.weight, C, self.feat_out)
                P["b3"] = f32(self.fc3.bias)
                D = self.embed_dim
                layers = []
                for lyr in self.layers:
                    w, b = lyr.self_attn.qkv()
                    w, b = w.detach().float().clone(), b.detach().float().clone()
                    w[:D] *= 64 ** -0.5  # head_dim ** -0.5 on the q rows (exact: 2^-3), local_attention.py:98
                    b[:D] *= 64 ** -0.5
                    ln1, ln2 = lyr.self_attn_layer_norm, lyr.final_layer_norm
                    layers.append(dict(
                        ln1=(f32(ln1.weight), f32(ln1.bias)), eps1=ln1.eps, wqkv=w.contiguous(), bqkv=b.contiguous(),
                        wo=f32(lyr.self_attn.out_proj.weight), bo=f32(lyr.self_attn.out_proj.bias),
                        ln2=(f32(ln2.weight), f32(ln2.bias)), eps2=ln2.eps,
                        w1=f32(lyr.fc1.weight), b1=f32(lyr.fc1.bias), w2=f32(lyr.fc2.weight), b2=f32(lyr.fc2.bias)))
                P["layers"] = layers
                P["lnf"] = (f32(self.layer_norm.weight), f32(self.layer_norm.bias))
                if self.layernorm_embedding is not None:
                    P["lne"] = (f32(self.layernorm_embedding.weight), f32(self.layernorm_embedding.bias))
            self._prep32, self._prep32_key = P, key
            return P

        def _prepared(self):
            params = list(self.parameters()) + list(self.buffers())
            key = tuple((p._version, p.data_ptr()) for p in params)
            if self._prep_key == key:
                return self._prep
            with torch.no_grad():
                P = {}
                C = self.conv_channels
                P["w1"] = self.convolutions[0].weight.detach().reshape(C, 9).float().contiguous()
                P["b1"] = self.convolutions[0].bias.detach().float().contiguous()
                P["w2"] = ops.prep_conv2_weight(self.convolutions[1].weight.detach().float())
                P["b2"] = self.convolutions[1].bias.detach().float().contiguous()
                for i in range(2):
                    bn = self.bn[i]
                    P["bn%d" % i] = ops.prep_bn_affine(bn.weight.detach().float(), bn.bias.detach().float(),
                                                       bn.running_mean.float(), bn.running_var.float(),
                                                       bn.eps)
                P["w3"] = ops.prep_fc3_weight(self.fc3.weight.detach().float(), C, self.feat_out)
                P["b3"] = self.fc3.bias.detach().float().contiguous()
                D = self.embed_dim
                # head_dim ** -0.5 folded into the q rows of the in-projection (exact: 2^-3)
                qscale = torch.ones(3 * D, device=self.fc3.weight.device)
                qscale[:D] = 64 ** -0.5
                layers = []
                for lyr in self.layers:
                    # the two LayerNorms of the block are folded into the GEMMs they feed
                    # (ops.fold_layernorm; transformer_layer.py:108-110 and :126-131)
                    w, b = lyr.self_attn.qkv()
                    wqkv, cqkv = ops.fold_layernorm(w, b, lyr.self_attn_layer_norm.weight,
                                                    lyr.self_attn_layer_norm.bias, row_scale=qscale)
                    w1, c1 = ops.fold_layernorm(lyr.fc1.weight, lyr.fc1.bias, lyr.final_layer_norm.weight,
                                                lyr.final_layer_norm.bias)
                    layers.append(dict(
                        wqkv=wqkv, bqkv=cqkv, eps1=lyr.self_attn_layer_norm.eps,
                        wo=ops.cast_bf16(lyr.self_attn.out_proj.weight.detach().float()),
                        bo=lyr.self_attn.out_proj.bias.detach().float().contiguous(),
                        w1=w1, b1=c1, eps2=lyr.final_layer_norm.eps,
                        w2=ops.cast_bf16(lyr.fc2.weight.detach().float()),
                        b2=lyr.fc2.bias.detach().float().contiguous()))
                P["layers"] = layers
                P["lnf"] = (self.layer_norm.weight.detach().float().contiguous(),
                            self.layer_norm.bias.detach().float().contiguous())
                if self.layernorm_embedding is not None:
                    P["lne"] = (self.layernorm_embedding.weight.detach().float().contiguous(),
                                self.layernorm_embedding.bias.detach().float().contiguous())
            self._prep, self._prep_key = P, key
            return P

        def _positions(self, rows, device):
            if self.embed_positions.learned:  # --encoder-learned-pos: the embedding matrix IS the table
                w = self.embed_positions.embeddings.weight
                if w.shape[0] < rows:
                    raise ValueError("fbkst_b200: %d positions needed but --max-source-positions is %d"
                                     % (rows, w.shape[0]))
                return w.detach().float().contiguous()
            t = self._pos_table
            if t is None or t.shape[0] < rows or t.device != device:
                t = ops.sinusoidal_table(max(rows, 1024), self.embed_dim, device)
                self._pos_table = t
            return t

        # ------------------------------------------------------------------------------- forward
        def forward(self, src_tokens, src_lengths, cls_input: Optional[Tensor] = None,
                    return_all_hiddens: bool = False, **unused):
            if not src_tokens.is_cuda:
                raise RuntimeError("fbkst_b200: src_tokens must be a CUDA tensor (no CPU fallback)")
            # Training semantics (BatchNorm batch statistics, dropout) whenever the module is in train();
            # the differentiable chain also serves eval() with gradients enabled (running statistics, no
            # dropout) when a parameter or the input features require a gradient (attribution with a frozen
            # model).  Both run fbkst_b200.train: hand-written forward + backward kernels, no PyTorch
            # arithmetic.  Everything else is the inference path.
            if self.training or (torch.is_grad_enabled() and (
                    src_tokens.requires_grad or any(p.requires_grad for p in self.parameters()))):
                if self._precision != "bf16":
                    raise NotImplementedError(
                        "fbkst_b200: precision=%r is inference only (eval() under torch.no_grad()); training and "
                        "the backward run with precision='bf16'" % self._precision)
                from .train import forward_train
                return forward_train(self, src_tokens, src_lengths, return_all_hiddens)
            with torch.no_grad():
                return self._forward(src_tokens, src_lengths, return_all_hiddens)

        def _forward(self, src_tokens, src_lengths, return_all_hiddens):
            return self._finish(self._launch(src_tokens, src_lengths, return_all_hiddens))

        # The forward is split where its single host synchronisation sits: ``_launch`` enqueues every
        # kernel (and, after CTC compression, an async copy of the new lengths into pinned memory),
        # ``_finish`` waits for that copy and cuts the worst-case buffers to the exact output shape.
        # ``forward`` runs both back to back; ``EncoderPipeline`` puts the next batch's ``_launch``
        # between them so the GPU never waits for the host.
        def launch(self, src_tokens, src_lengths):
            """Asynchronous half of ``forward`` (inference, no hidden states): returns a handle for
            ``finish``.  Buffers owned by a CUDA graph (``ctc_out``) stay valid until the next launch
            with the same input shape on the same ``graph_lane``."""
            if self.training:
                raise RuntimeError("fbkst_b200: launch/finish is the inference API (call eval())")
            if not src_tokens.is_cuda:
                raise RuntimeError("fbkst_b200: src_tokens must be a CUDA tensor (no CPU fallback)")
            with torch.no_grad():
                return self._launch(src_tokens, src_lengths, False)

        def finish(self, handle):
            """Blocking half of ``forward``: the reference's output tuple for a ``launch`` handle."""
            with torch.no_grad():
                return self._finish(handle)

        def _launch(self, src_tokens, src_lengths, return_all_hiddens):
            dev = src_tokens.device
            B, T, Fd = src_tokens.shape
            x_in = src_tokens if src_tokens.dtype == torch.float32 else src_tokens.float()
            x_in = x_in.contiguous()
            L = ((T + 1) // 2 + 1) // 2
            # Lengths drive all shape logic.  Host lengths: used directly.  DEVICE lengths (fairseq's
            # utils.move_to_cuda puts them there): subsampled on the device and read back together
            # with the compressed lengths by the forward's single deferred host sync (``_finish``) --
            # no blocking .cpu() at the top of the forward.  Only ``return_all_hiddens`` (exact
            # per-layer shapes, which synchronises anyway) still needs them on the host up front.
            len_dev = None
            if src_lengths.is_cuda and not return_all_hiddens:
                len_dev = ops.subsample_lengths(src_lengths.contiguous(), 2)
                len_host = None
            else:
                len_host = src_lengths.tolist() if not src_lengths.is_cuda else src_lengths.cpu().tolist()
                len_host = [((n + 1) // 2 + 1) // 2 for n in len_host]  # ceil(ceil(n/2)/2), :213
            for _ in range(self.num_layers):
                torch.empty(1).uniform_()  # LayerDrop draws: keep the CPU RNG stream of the reference
            compress = self.ctc_compress_out and 0 < self.ctc_layer <= self.num_layers
            if self.use_cuda_graph and not return_all_hiddens:
                r = self._replay(x_in, len_host, len_dev, B, T, Fd, L)
            else:
                lengths = len_dev if len_dev is not None else \
                    torch.tensor(len_host, dtype=torch.int32).to(dev, non_blocking=True)
                r = self._run_body(self._prepared_active(), x_in, lengths, len_host, L, B, return_all_hiddens,
                                   self._workspace(L * B, dev) if compress and not return_all_hiddens else None)
            x, limit, new_len, states = r["x"], r["limit"], r["new_len"], r["states"]
            mask_in = r["mask"]
            if self.use_cuda_graph and not return_all_hiddens:
                mask_in = mask_in.clone()  # do not hand out a buffer the next replay overwrites
            # :298-299: the mask is None when nothing is padded (decided in _finish for device lengths)
            mask = None if len_host is None or min(len_host) >= L else mask_in
            ctc_mask = mask
            if return_all_hiddens and compress:
                len_host, L = r["len_host"], r["L"]
                mask = r["mask2"] if min(len_host) < L else None
            xf = ops.layernorm(x, *self._prepared_active()["lnf"], out_dtype=torch.float32, rows_limit=limit)
            deferred = limit is not None or len_host is None
            h = dict(xf=xf, mask=mask, ctc_mask=ctc_mask, mask_in=mask_in, states=states, len_host=len_host,
                     L=L, B=B, x_ctc=r["x_ctc"], src_tokens=src_tokens, len_dtype=src_lengths.dtype, dev=dev,
                     return_all_hiddens=return_all_hiddens, deferred=deferred, compressed=limit is not None)
            if deferred:
                pin = h["pin"] = self._pins.take(2 * B)  # [subsampled input lengths | compressed lengths]
                if len_host is None:
                    pin[:B].copy_(r["lengths_in"], non_blocking=True)
                if limit is not None:
                    h["mask_full"] = ops.lengths_to_mask(new_len, L)[0]
                    pin[B:].copy_(new_len, non_blocking=True)
                h["ev"] = torch.cuda.Event()
                h["ev"].record()
            return h

        def _finish(self, h):
            xf, mask, ctc_mask, states, L, B = h["xf"], h["mask"], h["ctc_mask"], h["states"], h["L"], h["B"]
            len_host = h["len_host"]
            D, dev = self.embed_dim, h["dev"]
            if h["deferred"]:
                h["ev"].synchronize()  # the single host sync of the forward
                vals = h["pin"].tolist()
                self._pins.give(h.pop("pin"))
                if len_host is None:  # device lengths: the None-when-unpadded decision is made here
                    len_host = vals[:B]
                    mask = ctc_mask = h["mask_in"] if min(len_host) < L else None
                if h["compressed"]:
                    len_host = vals[B:]
                    L2 = max(len_host)
                    xf = xf[: L2 * B]
                    mask = None if min(len_host) >= L2 else h["mask_full"][:, :L2].contiguous()
                    L = L2
            h["out_len_host"] = len_host
            xf = xf.view(L, B, D)
            # `model.half()` (generate.py --fp16, fairseq_cli/generate.py:84-87): the decoder's weights are fp16,
            # so the encoder hands over fp16 like the reference module would (a cast of the final result)
            odt = self.layer_norm.weight.dtype
            if odt != torch.float32:
                xf = xf.to(odt)
            if h["return_all_hiddens"]:
                states[-1] = xf
            out_lengths = torch.tensor(len_host, dtype=h["len_dtype"]).to(dev, non_blocking=True)
            if self.ctc_compress_out:
                return CTCAwareEncoderOut(xf, mask, None, states, h["src_tokens"], out_lengths, h["x_ctc"],
                                          ctc_mask)
            return EncoderOut(xf, mask, None, states, h["src_tokens"], out_lengths)

        def _body(self, P, x_in, lengths, len_host, L, B, want_states, ws):
            """Everything between the input batch and the final LayerNorm.  Shape-static when
            ``want_states`` is False (no host synchronisation, every launch sized for the worst case
            with device-side row limits after CTC compression), so it can be captured in a CUDA graph.
            ``lengths``: subsampled lengths, int32 on the device; ``len_host``: the same on the host
            (only needed when ``want_states``)."""
            dev = x_in.device
            D, H = self.embed_dim, self.heads
            y = ops.conv1_relu_bn(x_in, P["w1"], P["b1"], *P["bn0"])
            y = ops.conv2_relu_bn(y, P["w2"], P["b2"], *P["bn1"])  # [B, T2, F2, C]
            assert y.shape[1] == L
            a = y.view(B * L, -1)
            # fc3 + ReLU on the CTA-pair GEMM in the conv layout's (b, t) row order; the transpose to
            # time-major rows, the positions and the first layer's LayerNorm statistics are one
            # row-per-warp pass (:225-229)
            h3 = ops.linear(a, P["w3"], P["b3"], relu=True, out_dtype=torch.float32)
            table = self._positions(L + 1, dev) if self.embed_positions is not None else None
            x, xb, st = ops.embed_remap_stats(h3, L, B, table, lengths if table is not None else None)
            if self.layernorm_embedding is not None:
                x = ops.layernorm(x, *P["lne"], out_dtype=torch.float32)
                xb, st = ops.row_stats_cast(x)
            mask = ops.lengths_to_mask(lengths, L)[0]
            r = dict(mask=mask, mask2=None, x_ctc=None, len_host=len_host, L=L, lengths_in=lengths,
                     tables=table if self.embed_positions is not None else None)
            states = [] if want_states else None
            # After CTC compression the number of valid rows is known only on the device.  Unless the
            # caller wants every hidden state (exact shapes per layer), the remaining layers are
            # launched for the worst case with a device-side row limit and persistent, finite
            # workspaces; the single host sync of the forward is the final read of the new lengths.
            limit, new_len = None, None
            # Folded LayerNorm: every x travels with its bf16 copy and per-row slice statistics, written
            # by the epilogue that produced x (out_proj / fc2) or by row_stats_cast (fc3 output,
            # compressed rows); QKV / fc1 apply 1/sigma in their epilogues.  No LayerNorm launches
            # inside the layer stack.
            n_layers = len(P["layers"])
            for li, W in enumerate(P["layers"]):
                ctc_here = self.ctc_compress_out and self.ctc_layer == li + 1
                need_ln = li + 1 < n_layers or ctc_here  # the last x only feeds the final LayerNorm
                if limit is None:
                    qkv = ops.linear_ln(xb, W["wqkv"], W["bqkv"], stats_in=st, ln_eps=W["eps1"])
                    att = ops.attention(qkv, lengths, L, B, H, self.log_penalty)
                    x, xb, st = ops.linear_ln(att, W["wo"], W["bo"], residual=x, out_dtype=torch.float32,
                                              ln_out=True)
                    f = ops.linear_ln(xb, W["w1"], W["b1"], relu=True, stats_in=st, ln_eps=W["eps2"])
                    if need_ln:
                        x, xb, st = ops.linear_ln(f, W["w2"], W["b2"], residual=x, out_dtype=torch.float32,
                                                  ln_out=True)
                    else:
                        x = ops.linear(f, W["w2"], W["b2"], residual=x, out_dtype=torch.float32)
                else:
                    lo = (ws["h"], ws["st"])
                    qkv = ops.linear_ln(xb, W["wqkv"], W["bqkv"], stats_in=st, ln_eps=W["eps1"],
                                        out=ws["qkv"], rows_limit=limit)
                    att = ops.attention(qkv, lengths, L, B, H, self.log_penalty, out=ws["att"],
                                        q_limit=limit[0])  # rows t >= max new length are never read
                    x1, xb, st = ops.linear_ln(att, W["wo"], W["bo"], residual=x, out_dtype=torch.float32,
                                               out=ws["x1"], ln_out=lo, rows_limit=limit)
                    f = ops.linear_ln(xb, W["w1"], W["b1"], relu=True, stats_in=st, ln_eps=W["eps2"],
                                      out=ws["f"], rows_limit=limit)
                    if need_ln:
                        x, xb, st = ops.linear_ln(f, W["w2"], W["b2"], residual=x1, out_dtype=torch.float32,
                                                  out=ws["x0"], ln_out=lo, rows_limit=limit)
                    else:
                        x = ops.linear(f, W["w2"], W["b2"], residual=x1, out_dtype=torch.float32,
                                       out=ws["x0"], rows_limit=limit)
                if ctc_here:
                    self.ctc_fc._bf16_operand = (x.data_ptr(), xb)  # bf16(x) is already there
                    if want_states:
                        r["x_ctc"], x, lengths, len_host, L = self._ctc_compress(x, lengths, L, B)
                        r["mask2"] = ops.lengths_to_mask(lengths, L)[0]
                        r["len_host"], r["L"] = len_host, L
                        if li + 1 < n_layers:
                            xb, st = ops.row_stats_cast(x)
                    else:
                        r["x_ctc"], x, lengths, max_new = self._ctc_compress(x, lengths, L, B, out=ws["x0"])
                        new_len = lengths
                        limit = (max_new, B)
                        if li + 1 < n_layers:
                            xb, st = ops.row_stats_cast(x, out=(ws["h"], ws["st"]), rows_limit=limit)
                if want_states:
                    states.append(x.view(L, B, D))
            r.update(x=x, limit=limit, new_len=new_len, states=states)
            return r

        def _run_body(self, *args):
            return (self._body_f32 if self._precision == "fp32" else self._body)(*args)

        def _body_f32(self, P, x_in, lengths, len_host, L, B, want_states, ws):
            """``_body`` with fp32 activations and split-TF32 operands (``precision = "fp32"``): the same
            shapes, row limits and outputs, explicit LayerNorms in fp32, no bf16 copies."""
            dev = x_in.device
            D, H = self.embed_dim, self.heads
            f32 = torch.float32
            y = ops.conv1_relu_bn_f32(x_in, P["w1"], P["b1"], *P["bn0"])
            y = ops.conv2_relu_bn_f32(y, P["w2"], P["b2"], *P["bn1"])  # [B, T2, F2, C]
            assert y.shape[1] == L
            h3 = ops.linear_f32(y.view(B * L, -1), P["w3"], P["b3"], relu=True)  # (b, t) rows, :227
            table = self._positions(L + 1, dev) if self.embed_positions is not None else None
            x = ops.embed_remap_stats(h3, L, B, table, lengths if table is not None else None)[0]
            if self.layernorm_embedding is not None:
                x = ops.layernorm(x, *P["lne"], out_dtype=f32)
            mask = ops.lengths_to_mask(lengths, L)[0]
            r = dict(mask=mask, mask2=None, x_ctc=None, len_host=len_host, L=L, lengths_in=lengths,
                     tables=table)
            states = [] if want_states else None
            limit, new_len = None, None
            for li, W in enumerate(P["layers"]):
                ctc_here = self.ctc_compress_out and self.ctc_layer == li + 1
                if limit is None:  # transformer_layer.py:105-135 (pre-LayerNorm)
                    h = ops.layernorm(x, *W["ln1"], out_dtype=f32, eps=W["eps1"])
                    qkv = ops.linear_f32(h, W["wqkv"], W["bqkv"])
                    att = ops.attention_f32(qkv, lengths, L, B, H, self.log_penalty)
                    x = ops.linear_f32(att, W["wo"], W["bo"], residual=x)
                    h = ops.layernorm(x, *W["ln2"], out_dtype=f32, eps=W["eps2"])
                    f = ops.linear_f32(h, W["w1"], W["b1"], relu=True)
                    x = ops.linear_f32(f, W["w2"], W["b2"], residual=x)
                else:
                    h = ops.layernorm(x, *W["ln1"], out_dtype=f32, eps=W["eps1"], out=ws["h"], rows_limit=limit)
                    qkv = ops.linear_f32(h, W["wqkv"], W["bqkv"], out=ws["qkv"], rows_limit=limit)
                    att = ops.attention_f32(qkv, lengths, L, B, H, self.log_penalty, out=ws["att"],
                                            q_limit=limit[0])
                    x1 = ops.linear_f32(att, W["wo"], W["bo"], residual=x, out=ws["x1"], rows_limit=limit)
                    h = ops.layernorm(x1, *W["ln2"], out_dtype=f32, eps=W["eps2"], out=ws["h"], rows_limit=limit)
                    f = ops.linear_f32(h, W["w1"], W["b1"], relu=True, out=ws["f"], rows_limit=limit)
                    x = ops.linear_f32(f, W["w2"], W["b2"], residual=x1, out=ws["x0"], rows_limit=limit)
                if ctc_here:
                    if want_states:
                        r["x_ctc"], x, lengths, len_host, L = self._ctc_compress(x, lengths, L, B)
                        r["mask2"] = ops.lengths_to_mask(lengths, L)[0]
                        r["len_host"], r["L"] = len_host, L
                    else:
                        r["x_ctc"], x, lengths, max_new = self._ctc_compress(x, lengths, L, B, out=ws["x0"])
                        new_len = lengths
                        limit = (max_new, B)
                if want_states:
                    states.append(x.view(L, B, D))
            r.update(x=x, limit=limit, new_len=new_len, states=states)
            return r

        # ------------------------------------------------------------------------- CUDA graphs
        def _graph_key(self, B, T, Fd, dev):
            hooks = tuple(sorted(self.ctc_fc._forward_hooks)) if self.ctc_compress_out else ()
            bump = None if self.ctc_logit_bump is None else (id(self.ctc_logit_bump[0]), self.ctc_logit_bump[1])
            prep_key = self._prep32_key if self._precision == "fp32" else self._prep_key
            return (B, T, Fd, str(dev), self._precision, prep_key, hooks, bump, self.graph_lane)

        def _replay(self, x_in, len_host, len_dev, B, T, Fd, L):
            """Graph mode (``use_cuda_graph``): the ~90 launches of ``_body`` for one input shape are
            captured once and replayed with one ``cudaGraphLaunch``; the batch is copied into the
            graph's static input buffer (device-to-device) and the subsampled lengths into its static
            length vector.  ``ctc_out`` then aliases a buffer owned by the graph: it is valid until
            the next forward with the same input shape."""
            dev = x_in.device
            P = self._prepared_active()
            key = self._graph_key(B, T, Fd, dev)
            G = self._graphs.get(key)
            if G is None:
                if len(self._graphs) >= self.max_graphs:  # bounded: every graph pins its activations
                    self._graphs.pop(next(iter(self._graphs)))
                G = self._capture(P, B, T, Fd, L, dev)
                self._graphs[key] = G
            if len_dev is not None:
                G["lengths"].copy_(len_dev, non_blocking=True)
            else:
                # pinned staging vector from the pool: handed out again only after the event recorded
                # behind the H2D copy has completed (the host may run many launches ahead of the GPU)
                pin = self._pins.take(B)
                pin.copy_(torch.tensor(len_host, dtype=torch.int32))
                G["lengths"].copy_(pin, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record()
                self._pins.give(pin, ev)
            if x_in.data_ptr() != G["x"].data_ptr():  # the caller may have produced x in place (static_input)
                G["x"].copy_(x_in, non_blocking=True)
            G["graph"].replay()
            ops._count(G["launches"])
            return G["out"]

        def static_input(self, B, T, Fd, dev):
            """Graph mode: the captured graph's input buffer [B,T,F] fp32 for this shape on the current
            ``graph_lane`` (None before the first forward of that shape).  A producer that writes the
            batch straight into it (e.g. ``ops.cmvn(raw, lengths, out=buf)``) and passes it to
            ``launch`` / ``forward`` saves the device-to-device copy of the replay."""
            if not self.use_cuda_graph:
                return None
            G = self._graphs.get(self._graph_key(B, T, Fd, dev))
            return None if G is None else G["x"]

        def _capture(self, P, B, T, Fd, L, dev):
            compress = self.ctc_compress_out and 0 < self.ctc_layer <= self.num_layers
            G = dict(x=torch.zeros(B, T, Fd, dtype=torch.float32, device=dev),
                     lengths=torch.full((B,), L, dtype=torch.int32, device=dev),
                     P=P,
                     ws=self._make_workspace(L * B, dev) if compress else None)
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):  # warm-up outside capture: lazy one-time initialisation
                self._run_body(P, G["x"], G["lengths"], None, L, B, False, G["ws"])
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            graph = torch.cuda.CUDAGraph()
            n0 = ops.LAUNCHES
            with torch.cuda.graph(graph):
                G["out"] = self._run_body(P, G["x"], G["lengths"], None, L, B, False, G["ws"])
            G["launches"] = ops.LAUNCHES - n0
            G["graph"] = graph
            return G

        def _make_workspace(self, M, dev):
            """Zero-initialised buffers for the layers after compression (rows beyond the device-side
            limit are never written, so they must hold finite values: 0 * NaN would poison the P.V
            product of a partially valid key tile)."""
            D, Dff = self.embed_dim, self.layers[0].fc1.out_features
            z = lambda n, dt: torch.zeros(M, n, dtype=dt, device=dev)
            if self._precision == "fp32":
                f32 = torch.float32
                return dict(h=z(D, f32), qkv=z(3 * D, f32), att=z(D, f32), f=z(Dff, f32), x0=z(D, f32), x1=z(D, f32))
            return dict(h=z(D, torch.bfloat16), qkv=z(3 * D, torch.bfloat16), att=z(D, torch.bfloat16),
                        f=z(Dff, torch.bfloat16), x0=z(D, torch.float32), x1=z(D, torch.float32),
                        st=torch.zeros(M, (D + 127) // 128, 2, dtype=torch.float32, device=dev))

        def _workspace(self, M, dev):
            """The eager path keeps one workspace per lane (for the last shape seen on it)."""
            key = (M, str(dev), self._precision)
            if self._ws is None:
                self._ws = {}
            got = self._ws.get(self.graph_lane)
            if got is None or got[0] != key:
                got = self._ws[self.graph_lane] = (key, self._make_workspace(M, dev))
            return got[1]

        def _ctc_compress(self, x, lengths, L, B, out=None):
            """conv_transformer.py:278-291 on device.  With ``out`` (workspace mode) nothing is read
            back: returns (logits, out, new_len, max_new) as device tensors.  Otherwise one D2H copy
            (the new lengths) gives the exact output shape."""
            D = self.embed_dim
            want_prob = self.ctc_compress_strategy != "avg"
            bump = None
            if self.ctc_logit_bump is not None:
                bl, bm = self.ctc_logit_bump
                if callable(bl):  # per-shape label plans (ragged streams): fn(L, B) -> [L, B] int32
                    bl = bl(L, B)
                if tuple(bl.shape) != (L, B) or bl.dtype != torch.int32 or not bl.is_contiguous():
                    raise ValueError("fbkst_b200: ctc_logit_bump labels must be a contiguous [L, B] int32 tensor")
                bump = (bl.view(L * B), float(bm))
            # fused epilogue: measured 269 us against 217 (GEMM) + 116 (arg-max pass) at cfg2 for `avg`; with the
            # sum of exponentials (weighted / softmax) the 8 epilogue warps become the bottleneck (342 us against
            # 217 + 127: a tie), so those strategies keep the separate pass (scripts/bench_ctc_fc.py)
            fused = (not self.ctc_fc._forward_hooks and not self.ctc_fc._forward_pre_hooks
                     and self.ctc_fc.logits_dtype == torch.float32 and not want_prob and self._precision == "bf16")
            if fused:
                # ctc_fc on tcgen05 with the arg-max (+ sum exp) folded into its epilogue: the logits are written
                # once and never re-read (conv_transformer.py:279 + :282-284)
                pre = getattr(self.ctc_fc, "_bf16_operand", None)
                self.ctc_fc._bf16_operand = None
                xb = pre[1] if pre is not None and pre[0] == x.data_ptr() else None
                lg, labels, prob, _ = self.ctc_fc.project_argmax(x, xb, lengths, L, B, want_prob, bump)
                V = lg.shape[1]
                logits = lg.view(L, B, V)
            else:
                logits = self.ctc_fc(x.view(L, B, D))  # module call: forward hooks apply
                V = logits.shape[-1]
                if bump is not None:  # test / benchmark logit injection on the unfused path (in place)
                    logits.scatter_add_(2, bump[0].view(L, B, 1).long(),
                                        torch.full((L, B, 1), bump[1], dtype=logits.dtype, device=logits.device))
                try:
                    lg = logits.view(L * B, V)
                except RuntimeError:
                    lg = logits.contiguous().view(L * B, V)
                if lg.stride(-1) != 1:
                    lg = lg.contiguous()
                labels, prob = ops.ctc_argmax(lg, lengths, L, B, V, want_prob)
            seg_id, seg_start, weight, new_len, max_new = ops.ctc_segment(
                labels, prob, lengths, self.ctc_compress_strategy, L, B)
            res = ops.ctc_compress(x, seg_id, seg_start, weight, lengths, new_len, max_new, L, B, out=out)
            if out is not None:
                return logits, res, new_len, max_new
            new_host = new_len.cpu().tolist()  # host sync: exact shapes for encoder_states
            L2 = max(new_host)
            return logits, res[: L2 * B], new_len, new_host, L2

        # ----------------------------------------------------------------- reference interface
        @property
        def output_batch_first(self):
            return False

        @torch.jit.unused
        def forward_non_torchscript(self, net_input: Dict[str, Tensor]):
            encoder_input = {k: v for k, v in net_input.items()
                             if k not in ("prev_output_tokens", "transcript_prev_output_tokens")}
            return self.forward(**encoder_input)

        def reorder_encoder_out(self, encoder_out, new_order):
            """conv_transformer.py:315-345: index_select batch dim by ``new_order`` (beam search).
            Same values as the reference; the tensors returned additionally remember which columns
            of the ORIGINAL encoder output they hold (``cross_attention.reorder_tagged``), so
            ``CrossAttention`` projects K/V once per utterance instead of once per hypothesis, and a
            chain of reorders is one gather from the original.  With ``lazy_beam_reorder = True``
            (opt-in; every consumer must be a ``CrossAttention``) nothing is gathered at all: the
            un-replicated tensors travel with the row vector."""
            from .cross_attention import reorder_tagged
            lazy = getattr(self, "lazy_beam_reorder", False)
            memo = {}
            if encoder_out.encoder_out is not None:
                encoder_out = encoder_out._replace(
                    encoder_out=reorder_tagged(encoder_out.encoder_out, 1, new_order, lazy, memo))
            if encoder_out.encoder_padding_mask is not None:
                encoder_out = encoder_out._replace(
                    encoder_padding_mask=reorder_tagged(encoder_out.encoder_padding_mask, 0, new_order,
                                                        lazy, memo))
            if encoder_out.encoder_embedding is not None:
                encoder_out = encoder_out._replace(
                    encoder_embedding=encoder_out.encoder_embedding.index_select(0, new_order))
            if encoder_out.encoder_states is not None:
                for idx, state in enumerate(encoder_out.encoder_states):
                    encoder_out.encoder_states[idx] = state.index_select(1, new_order)
            return encoder_out

    return ConvolutionalTransformerEncoder


ConvolutionalTransformerEncoder = make_encoder_class(_Base)
