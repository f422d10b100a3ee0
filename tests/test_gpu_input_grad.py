"""Gradients of the encoder with respect to its input features (saliency / attribution, input-gradient losses)
and the selective backward: the training node computes only the gradients autograd asks for.

* ``ops.conv1_dgrad`` against torch.autograd of ``F.conv2d(stride=2, padding=1)`` in fp64, on the same bf16
  upstream gradient and fp32 weights;
* ``src_tokens.grad`` of a frozen model in eval() against the fp32 oracle's input gradient: with our ReLU
  patterns (what remains is bf16 rounding) and as it is (cosine);
* the requested gradients are bitwise those of the full backward whatever else is frozen, in eval() and in
  train() (batch-statistics BatchNorm, dropout); frozen parameters keep ``.grad is None``;
* the skipped work is not launched (profiler trace + call counts of the weight-gradient GEMMs)."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from helpers import build_encoder, rel_err  # noqa: E402
from oracle import encoder_oracle as O  # noqa: E402  (checker only)
from fbkst_b200 import ops  # noqa: E402

TINY = dict(embed_dim=128, ffn_dim=256, heads=2, layers=3, conv_channels=64, feat_dim=40, vocab=64,
            distance_penalty="log", ctc_layer=2, ctc_strategy="weighted")


# ---------------------------------------------------------------------------------------------- the kernel
def _dgrad_fp64(dz1, w1, T, Fd):
    B, T1, F1, C = dz1.shape
    x = torch.zeros(B, 1, T, Fd, dtype=torch.float64, requires_grad=True)
    z = F.conv2d(x, w1.double().view(C, 1, 3, 3), stride=2, padding=1)
    assert z.shape == (B, C, T1, F1)
    z.backward(dz1.double().permute(0, 3, 1, 2))
    return x.grad[:, 0]


KERNEL_CASES = [(C, Fd, T) for C in (64, 128) for Fd in (40, 41, 80) for T in (1, 2, 3, 5, 257, 1500)]


@pytest.mark.parametrize("C,Fd,T", KERNEL_CASES)
def test_conv1_dgrad_vs_fp64(C, Fd, T):
    i = KERNEL_CASES.index((C, Fd, T))
    B = 1 + i % 5
    g = torch.Generator().manual_seed(1000 + i)
    T1, F1 = (T + 1) // 2, (Fd + 1) // 2
    dz1 = torch.randn(B, T1, F1, C, generator=g).bfloat16()
    w1 = torch.randn(C, 9, generator=g) * 0.3
    ref = _dgrad_fp64(dz1, w1, T, Fd)
    a = ops.conv1_dgrad(dz1.cuda(), w1.cuda(), T, Fd)
    b = ops.conv1_dgrad(dz1.cuda(), w1.cuda(), T, Fd)
    torch.cuda.synchronize()
    assert a.shape == (B, T, Fd) and a.dtype == torch.float32
    assert torch.equal(a, b)  # fixed summation order
    err = ((a.double().cpu() - ref).abs().max() / ref.abs().max()).item()
    assert err <= 1e-5, err


def test_conv1_dgrad_rejects_mismatched_shapes():
    dz1 = torch.zeros(1, 3, 20, 64, dtype=torch.bfloat16, device="cuda")
    w1 = torch.zeros(64, 9, device="cuda")
    with pytest.raises(ValueError):
        ops.conv1_dgrad(dz1, w1, 7, 40)  # T1 of 7 frames is 4
    with pytest.raises(ValueError):
        ops.conv1_dgrad(dz1, w1[:, :8].contiguous(), 6, 40)


# ------------------------------------------------------------------------------ end to end against the oracle
def _upstream(ref, lens_in, seed):
    """Random upstream gradients, zero at padded output rows (what a decoder / F.ctc_loss produce)."""
    g = torch.Generator().manual_seed(seed)
    r_out = torch.randn(ref["encoder_out"].shape, generator=g)
    for b, n in enumerate(ref["src_lengths"].tolist()):
        r_out[n:, b] = 0
    r_ctc = None
    if ref["ctc_out"] is not None:
        r_ctc = torch.randn(ref["ctc_out"].shape, generator=g) * 0.05
        for b, n in enumerate([((n + 1) // 2 + 1) // 2 for n in lens_in]):
            r_ctc[n:, b] = 0
    return r_out, r_ctc


def _oracle_input_grad(sd, cfg, x, lens, hook, r_out, r_ctc, relu_masks=None):
    xl = x.clone().requires_grad_(True)
    ref = O.encoder_forward(sd, cfg, xl, lens, ctc_logits_hook=hook, relu_masks=relu_masks)
    if r_out is None:
        return ref, None
    loss = (ref["encoder_out"] * r_out).sum()
    if r_ctc is not None:
        loss = loss + (ref["ctc_out"] * r_ctc).sum()
    loss.backward()
    return ref, xl.grad


def _input_grad_case(cfg, lens_in, seed, feat=40):
    sd = O.init_state_dict(cfg, seed=seed)
    x, lens = O.synthetic_batch(lens_in, feat, seed=seed + 100)
    T = max(lens_in)
    L = ((T + 1) // 2 + 1) // 2
    B = len(lens_in)
    hook = labels = None
    if cfg.get("ctc_layer", 0) > 0:
        labels = O.synthetic_ctc_bump(L, B, cfg["vocab"], seed=seed + 7)
        hook = O.bump_hook(labels, 30.0)
    ref, _ = _oracle_input_grad(sd, cfg, x, lens, hook, None, None)
    r_out, r_ctc = _upstream(ref, lens_in, seed + 1)
    ref, gx = _oracle_input_grad(sd, cfg, x, lens, hook, r_out, r_ctc)

    enc = build_encoder(cfg, sd)  # eval(), every parameter frozen
    enc.keep_train_state = True
    if hook is not None:
        dev_hook = O.bump_hook(labels.cuda(), 30.0)
        enc.ctc_fc.register_forward_hook(lambda m, i, o: dev_hook(o))
    xd = x.cuda().requires_grad_(True)
    out = enc(xd, lens.cuda())
    assert out.encoder_out.requires_grad
    assert out.src_lengths.cpu().tolist() == ref["src_lengths"].tolist()
    loss = (out.encoder_out * r_out.cuda()).sum()
    if r_ctc is not None:
        loss = loss + (out.ctc_out * r_ctc.cuda()).sum()
    loss.backward()
    assert all(p.grad is None for p in enc.parameters())
    dx = xd.grad
    assert dx is not None and dx.shape == x.shape and dx.dtype == torch.float32
    assert torch.isfinite(dx).all()

    # the oracle with our activation patterns: what remains is rounding
    S = enc.last_train_state
    masks = {"conv0": (S["y1r"] > 0).permute(0, 3, 1, 2).cpu(), "conv1": (S["y2r"] > 0).permute(0, 3, 1, 2).cpu(),
             "fc3": (S["h3b"] > 0).view(B, L, -1).transpose(0, 1).cpu()}
    for li, R in enumerate(S["layers"]):
        masks["layers.%d.fc1" % li] = (R["f"] > 0).view(R["L"], B, -1).cpu()
    _, gx_m = _oracle_input_grad(sd, cfg, x, lens, hook, r_out, r_ctc, relu_masks=masks)
    a, r0, r1 = dx.double().cpu().flatten(), gx.double().flatten(), gx_m.double().flatten()
    worst = ((a - r1).abs().max() / r1.abs().max()).item()
    cos = (torch.dot(a, r0) / (a.norm() * r0.norm())).item()
    assert worst <= 1e-2, worst
    assert cos >= 0.998, cos
    # padded frames next to valid ones receive gradient through the unmasked convolutions (as in the reference)
    short = min(range(B), key=lambda b: lens_in[b])
    if lens_in[short] < T:
        assert dx[short, lens_in[short]].abs().max() > 0
    return worst, cos


def test_input_grad_tiny_weighted():
    _input_grad_case(TINY, [97, 64, 30], seed=3)


@pytest.mark.parametrize("ctc_layer,strategy", [(0, "avg"), (2, "avg"), (2, "weighted")])
def test_input_grad_big2_shape(ctc_layer, strategy):
    cfg = dict(embed_dim=512, ffn_dim=2048, heads=8, layers=3, conv_channels=64, feat_dim=40, vocab=1005,
               distance_penalty="log", ctc_layer=ctc_layer, ctc_strategy=strategy)
    _input_grad_case(cfg, [601, 598, 411, 203], seed=7)


# ------------------------------------------------------------------------ the selective backward's numbers
def _front_names(n):
    return n.startswith(("convolutions.", "bn.", "fc3."))


def _layer_of(n):
    return int(n.split(".")[1]) if n.startswith("layers.") else None


FREEZE = {
    "nothing": lambda n: False,
    "front": _front_names,
    "front_layers_0_1": lambda n: _front_names(n) or _layer_of(n) in (0, 1),
    "all_but_ctc_fc": lambda n: not n.startswith("ctc_fc."),
    "all": lambda n: True,
}


def _step(cfg, sd, x, lens, labels, frozen, want_x, train, seed=0):
    """One forward + backward; -> (parameter gradients by name or None, input gradient or None)."""
    enc = build_encoder(cfg, sd)
    if train:
        enc.train()
    enc.ctc_logit_bump = (labels, 30.0)
    for n, p in enc.named_parameters():
        p.requires_grad_(not frozen(n))
    xd = x.clone().requires_grad_(want_x)
    torch.manual_seed(seed)  # the step's dropout seed and the LayerDrop draws
    out = enc(xd, lens, return_all_hiddens=True)
    g = torch.Generator().manual_seed(77)
    r = torch.randn(out.encoder_out.shape, generator=g).cuda()
    rc = torch.randn(out.ctc_out.shape, generator=g).cuda() * 0.05
    loss = (out.encoder_out * r).sum() + (out.ctc_out * rc).sum()
    loss.backward()
    grads = {n: (p.grad.clone() if p.grad is not None else None) for n, p in enc.named_parameters()}
    return grads, (xd.grad.clone() if want_x else None)


def _selective_setup(dropout=0.0):
    cfg = dict(TINY, dropout=dropout)
    sd = O.init_state_dict(cfg, seed=31)
    lens_in = [160, 131, 97, 160]
    x, lens = O.synthetic_batch(lens_in, 40, seed=32)
    labels = O.synthetic_ctc_bump(40, len(lens_in), cfg["vocab"], seed=33).to(torch.int32).cuda().contiguous()
    return cfg, sd, x.cuda(), lens.cuda(), labels


@pytest.mark.parametrize("train", [False, True], ids=["eval", "train"])
def test_selective_backward_is_bitwise(train):
    cfg, sd, x, lens, labels = _selective_setup(dropout=0.1 if train else 0.0)
    full, _ = _step(cfg, sd, x, lens, labels, FREEZE["nothing"], False, train)
    assert all(g is not None for g in full.values())
    x_alone = None
    for name, frozen in FREEZE.items():
        for want_x in (False, True):
            if name == "all" and not want_x:
                continue  # nothing requires a gradient: no backward
            grads, gx = _step(cfg, sd, x, lens, labels, frozen, want_x, train)
            for n, gr in grads.items():
                if frozen(n):
                    assert gr is None, (name, n)
                else:
                    assert gr is not None and torch.equal(gr, full[n]), (name, want_x, n)
            if want_x:
                assert gx is not None and torch.isfinite(gx).all() and gx.abs().max() > 0
                if x_alone is None:
                    x_alone = gx
                assert torch.equal(gx, x_alone), (name, "input gradient")


def test_frozen_front_skips_its_work(monkeypatch):
    """Front end and layers 0..1 frozen, no input gradient: the conv-stack backward and the fc3 / conv2
    weight-gradient GEMMs do not run, and only the trainable layer's four weight-gradient GEMMs do."""
    cfg = dict(TINY, ctc_layer=0)
    sd = O.init_state_dict(cfg, seed=41)
    x, lens = O.synthetic_batch([160, 131, 97], 40, seed=42)
    enc = build_encoder(cfg, sd)
    for n, p in enc.named_parameters():
        p.requires_grad_(not (_front_names(n) or _layer_of(n) in (0, 1)))
    calls = {"tn": 0, "nt": 0}
    tn, nt = ops.linear_wgrad, ops.linear_wgrad_nt

    def spy_tn(*a, **k):
        calls["tn"] += 1
        return tn(*a, **k)

    def spy_nt(*a, **k):
        calls["nt"] += 1
        return nt(*a, **k)
    monkeypatch.setattr(ops, "linear_wgrad", spy_tn)
    monkeypatch.setattr(ops, "linear_wgrad_nt", spy_nt)
    out = enc(x.cuda(), lens.cuda())
    r = torch.randn(out.encoder_out.shape, generator=torch.Generator().manual_seed(43)).cuda()
    loss = (out.encoder_out * r).sum()
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        loss.backward()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert any("ln_bwd" in n for n in names), "no backward kernel in the trace"
    for bad in ("conv1_wgrad", "conv1_dgrad", "col2im", "im2col_t", "bn_bwd"):
        assert not any(bad in n for n in names), bad
    assert calls == {"tn": 0, "nt": 4}, calls  # fc3 / conv2 (TN) none; layer 2: fc2, fc1, out_proj, qkv
    assert enc.layers[2].fc1.weight.grad is not None and enc.fc3.weight.grad is None


def test_intermediate_state_loss_reaches_the_input():
    """CTC multitask without compression: a loss on encoder_states[k-1] alone trains the input gradient."""
    cfg = dict(TINY, ctc_layer=0)
    sd = O.init_state_dict(cfg, seed=51)
    x, lens = O.synthetic_batch([120, 99, 64], 40, seed=52)
    gxs = []
    for trainable in (False, True):
        enc = build_encoder(cfg, sd)
        for p in enc.parameters():
            p.requires_grad_(trainable)
        xd = x.cuda().requires_grad_(True)
        out = enc(xd, lens.cuda(), return_all_hiddens=True)
        st = out.encoder_states[1]
        r = torch.randn(st.shape, generator=torch.Generator().manual_seed(53)).cuda()
        (st * r).sum().backward()
        assert xd.grad is not None and torch.isfinite(xd.grad).all() and xd.grad.abs().max() > 0
        if trainable:
            assert enc.layers[2].fc1.weight.grad is None or enc.layers[2].fc1.weight.grad.abs().max() == 0
            assert enc.layers[0].fc1.weight.grad.abs().max() > 0
        gxs.append(xd.grad)
    assert torch.equal(gxs[0], gxs[1])


def test_input_grad_half_precision():
    """model.half() with fp16 features: the input gradient comes back fp16, within fp16 rounding of the fp32
    run on the same (fp16-representable) parameters and features."""
    cfg = dict(TINY, ctc_layer=0)
    sd = {k: (v.half().float() if v.is_floating_point() else v) for k, v in O.init_state_dict(cfg, seed=61).items()}
    x, lens = O.synthetic_batch([150, 111, 64], 40, seed=62)
    x = x.half()
    res = []
    for half in (False, True):
        enc = build_encoder(cfg, sd)
        if half:
            enc = enc.half()
        xd = (x if half else x.float()).cuda().requires_grad_(True)
        out = enc(xd, lens.cuda())
        r = torch.randn(out.encoder_out.shape, generator=torch.Generator().manual_seed(63)).half().cuda()
        (out.encoder_out * r.to(out.encoder_out.dtype)).sum().backward()
        assert xd.grad.dtype == xd.dtype
        res.append(xd.grad)
    g32, g16 = res
    assert rel_err(g16.float(), g32) <= 1e-3


def test_fp32_precision_refuses_input_grad():
    sd = O.init_state_dict(TINY, seed=71)
    x, lens = O.synthetic_batch([64, 50], 40, seed=72)
    enc = build_encoder(TINY, sd)
    enc.precision = "fp32"
    with pytest.raises(NotImplementedError):
        enc(x.cuda().requires_grad_(True), lens.cuda())
    with torch.no_grad():  # the inference path is unchanged
        enc(x.cuda(), lens.cuda())
