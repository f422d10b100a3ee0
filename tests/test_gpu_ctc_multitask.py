"""The CTC-multitask recipe WITHOUT --ctc-compress-out in training: ctc_multi_loss projects an intermediate encoder
state (``encoder_states[ctc_encoder_layer - 1]``) with the criterion's own ``fc_out`` and takes the CTC loss on
it, so the gradient of that state must reach the layers below it and the front end.

* the encoder's differentiable ``encoder_states`` against torch.autograd of the CPU oracle (the comparisons of
  tests/test_gpu_train.py: cosine >= 0.99 against the fp32 oracle, 2e-2 of max against the oracle run with our
  ReLU patterns), without and with CTC compression;
* ``criterion.CtcProjection`` + ``ctc_loss_train`` against an fp64 reference on the same bf16-rounded operands;
  its two backward routes (inside the loss node, its own node) against each other; fp16 (model.half());
  the validation forward;
* with the reference package present: fairseq's training call path, ``ctc_multi_loss`` against
  ``ctc_multi_loss_b200`` (skipped otherwise, as tests/test_gpu_dropin.py)."""
import argparse
import os
import warnings

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from helpers import build_encoder, rel_err  # noqa: E402
from oracle import encoder_oracle as O  # noqa: E402  (checker only)
from oracle import ref_loader as R  # noqa: E402

TOL = 2e-2
COS_MIN = 0.99


def _sub(n):
    return ((n + 1) // 2 + 1) // 2


def _zero_padded(r, lengths):
    for b, n in enumerate(lengths):
        r[n:, b] = 0
    return r


def _oracle_grads(sd, cfg, x, lens, hook, upstream, relu_masks=None):
    """torch.autograd of the oracle for loss = sum over (output, R) pairs of <output, R>; ``upstream(ref)`` ->
    {key: R} with key "out", "ctc" or a state index."""
    leaf = {}
    for k, v in sd.items():
        v = v.clone()
        if v.is_floating_point() and "running" not in k and "_float_tensor" not in k:
            v.requires_grad_(True)
        leaf[k] = v
    ref = O.encoder_forward(leaf, cfg, x, lens, return_all_hiddens=True, ctc_logits_hook=hook,
                            relu_masks=relu_masks)
    rs = upstream(ref)
    loss = 0.0
    for key, r in rs.items():
        loss = loss + (_ref_output(ref, key) * r).sum()
    loss.backward()
    return ref, {k: v.grad for k, v in leaf.items() if v.requires_grad}, rs


def _ref_output(ref, key):
    return ref["encoder_out"] if key == "out" else ref["ctc_out"] if key == "ctc" else ref["encoder_states"][key]


def _our_output(out, key):
    return out.encoder_out if key == "out" else out.ctc_out if key == "ctc" else out.encoder_states[key]


def _masks(enc, B, L, C=64):
    S = enc.last_train_state
    m = {"conv0": (S["y1r"] > 0).permute(0, 3, 1, 2).cpu(), "conv1": (S["y2r"] > 0).permute(0, 3, 1, 2).cpu(),
         "fc3": (S["h3b"] > 0).view(B, L, -1).transpose(0, 1).cpu()}
    for li, Rl in enumerate(S["layers"]):
        m["layers.%d.fc1" % li] = (Rl["f"] > 0).view(Rl["L"], B, -1).cpu()
    return m


def _compare_grads(enc, grads, grads_m):
    worst, cosines = {}, {}
    for name, p in enc.named_parameters():
        assert p.grad is not None, name
        assert torch.isfinite(p.grad).all(), name
        a, r0, r1 = p.grad.double().cpu().flatten(), grads[name].double().flatten(), grads_m[name].double().flatten()
        scale = r1.abs().max()
        if name.endswith("k_proj.bias") or scale < 1e-7:  # exactly zero in exact arithmetic (test_gpu_train.py)
            qb = dict(enc.named_parameters()).get(name.replace("k_proj", "q_proj"))
            ref_scale = qb.grad.abs().max().item() if qb is not None and name.endswith("k_proj.bias") else 1.0
            assert a.abs().max() < 0.05 * ref_scale, (name, a.abs().max().item(), ref_scale)
            continue
        worst[name] = ((a - r1).abs().max() / scale).item()
        cosines[name] = (torch.dot(a, r0) / (a.norm() * r0.norm()).clamp_min(1e-30)).item()
    bad = {k: round(v, 4) for k, v in worst.items() if v >= TOL}
    assert not bad, bad
    lowcos = {k: round(v, 4) for k, v in cosines.items() if v < COS_MIN}
    assert not lowcos, lowcos
    return worst, cosines


def run_state_case(cfg, lens_in, seed, state_ids, feat=40):
    """loss = <encoder_out, R> + sum_i <encoder_states[i], R_i> (+ <ctc_out, R_ctc> with compression), every R zeroed
    at padded rows; every parameter gradient against the oracle's."""
    sd = O.init_state_dict(cfg, seed=seed)
    x, lens = O.synthetic_batch(lens_in, feat, seed=seed + 100)
    B, L = len(lens_in), _sub(max(lens_in))
    sub = [_sub(n) for n in lens_in]
    k = cfg.get("ctc_layer", 0)
    hook = None
    if k > 0:
        labels = O.synthetic_ctc_bump(L, B, cfg["vocab"], seed=seed + 7)
        hook = O.bump_hook(labels, 30.0)
    g = torch.Generator().manual_seed(seed + 1)

    def upstream(ref):
        new_len = ref["src_lengths"].tolist()
        rs = {"out": _zero_padded(torch.randn(ref["encoder_out"].shape, generator=g), new_len)}
        for i in state_ids:  # a state before the CTC layer has the subsampled lengths, from it on the compressed
            st = ref["encoder_states"][i]
            rs[i] = _zero_padded(torch.randn(st.shape, generator=g), sub if k == 0 or i < k - 1 else new_len)
        if ref["ctc_out"] is not None:
            rs["ctc"] = _zero_padded(torch.randn(ref["ctc_out"].shape, generator=g) * 0.05, sub)
        return rs

    ref, grads, rs = _oracle_grads(sd, cfg, x, lens, hook, upstream)
    enc = build_encoder(cfg, sd)  # eval(): running statistics, no dropout
    enc.keep_train_state = True
    if hook is not None:
        dev_hook = O.bump_hook(labels.cuda(), 30.0)
        enc.ctc_fc.register_forward_hook(lambda m, i, o: dev_hook(o))
    for p in enc.parameters():
        p.requires_grad_(True)
    out = enc(x.cuda(), lens.cuda(), return_all_hiddens=True)
    new_len = ref["src_lengths"].tolist()
    assert out.src_lengths.cpu().tolist() == new_len
    assert len(out.encoder_states) == cfg["layers"]
    for i in state_ids:
        st = out.encoder_states[i]
        assert st.requires_grad and st.dtype == torch.float32, i
        lim = sub if k == 0 or i < k - 1 else new_len
        for b, n in enumerate(lim):
            assert rel_err(st.detach()[:n, b], ref["encoder_states"][i].detach()[:n, b]) < TOL, (i, b)
    loss = 0.0
    for key, r in rs.items():
        loss = loss + (_our_output(out, key) * r.cuda()).sum()
    loss.backward()

    ref_m, grads_m, _ = _oracle_grads(sd, cfg, x, lens, hook, lambda r: rs, relu_masks=_masks(enc, B, L))
    assert ref_m["src_lengths"].tolist() == new_len
    return _compare_grads(enc, grads, grads_m)


def test_state_gradient_log_penalty_no_compression():
    """CTC at layer 2 of 3 without compression (log-penalty layout): layers 1..2 and the front end get the
    state's gradient.  (A detached state would train layers <= k with the encoder_out term only.)"""
    cfg = dict(embed_dim=128, ffn_dim=256, heads=2, layers=3, conv_channels=64, feat_dim=40, vocab=64,
               distance_penalty="log", ctc_layer=0, ctc_strategy="avg")
    run_state_case(cfg, [97, 64, 30], seed=31, state_ids=[1])


def test_state_gradient_mha_layout_no_compression():
    """The MHA layout of tests/test_gpu_train.py::test_gradients_mha_layout_no_compression (same model, batch and
    encoder_out gradient) with a loss on the state of layer 1: only layer 0 and the front end see the state's
    gradient, the last layer's gradients are those of that test."""
    cfg = dict(embed_dim=256, ffn_dim=512, heads=4, layers=2, conv_channels=64, feat_dim=40, vocab=50,
               distance_penalty=None, ctc_layer=0, ctc_strategy="avg")
    run_state_case(cfg, [201, 160, 77, 40], seed=5, state_ids=[0])


def test_state_gradients_around_the_compression():
    """With compression at layer 2 of 4: upstream gradients on the state before the CTC layer, on the CTC layer's
    own (compressed) output and on one after it -- the latter two pass through ctc_compress_bwd."""
    cfg = dict(embed_dim=128, ffn_dim=256, heads=2, layers=4, conv_channels=64, feat_dim=40, vocab=61,
               distance_penalty="log", ctc_layer=2, ctc_strategy="weighted")
    run_state_case(cfg, [160, 131, 97, 64], seed=35, state_ids=[0, 1, 2])


# ------------------------------------------------------------------------------------------------------------
# criterion.CtcProjection

def _ctc_problem(T, B, V, seed):
    """Ragged input lengths, targets with repeated labels, utterance 2 infeasible (more labels + repeats than
    frames: zero_infinity)."""
    g = torch.Generator().manual_seed(seed)
    il = torch.tensor([T, T - 7, 9, T - 20][:B])
    U = 12
    tg = torch.randint(1, V, (B, U), generator=g)
    tg[0, 3] = tg[0, 2]  # repeated labels need a blank between them
    tg[1, 5] = tg[1, 4] = tg[1, 3]
    tl = torch.tensor([12, 10, 12, 6][:B])
    for b in range(B):
        tg[b, tl[b]:] = 0
    mask = torch.arange(T).unsqueeze(1) >= il.unsqueeze(0)  # T x B, True = padding
    return il, tg, tl, mask


def _projection(D, V, seed, dtype=torch.float32):
    torch.manual_seed(seed)
    lin = torch.nn.Linear(D, V)
    with torch.no_grad():
        lin.bias.normal_(0, 0.5)
    return lin.to(device="cuda", dtype=dtype)


def test_projection_and_loss_against_fp64():
    from fbkst_b200 import criterion as C
    T, B, D, V, blank = 57, 4, 256, 1005, 0
    il, tg, tl, mask = _ctc_problem(T, B, V, seed=41)
    lin = _projection(D, V, seed=42)
    proj = C.CtcProjection(lin)
    assert proj.weight is lin.weight and proj.bias is lin.bias
    g = torch.Generator().manual_seed(43)
    x = (torch.randn(T, B, D, generator=g) * 2.0).cuda().requires_grad_(True)
    logits = proj(x)
    assert logits.dtype == torch.float32 and tuple(logits.shape) == (T, B, V)
    assert logits._fbkst_tap[0] is x and logits._fbkst_tap[1] is proj
    loss, totals, il_dev = C.ctc_loss_train(logits, mask.cuda(), tg.cuda(), tl.cuda(), blank)
    assert type(loss.grad_fn).__name__.startswith("CtcProjLossFn")
    assert il_dev.cpu().tolist() == il.tolist()
    loss.backward()

    xr = x.detach().cpu().bfloat16().double().requires_grad_(True)
    wr = lin.weight.detach().cpu().bfloat16().double().requires_grad_(True)
    br = lin.bias.detach().cpu().double().requires_grad_(True)
    lr = F.linear(xr, wr, br)
    nll = F.ctc_loss(lr.log_softmax(-1), tg, il, tl, blank=blank, reduction="none", zero_infinity=True)
    assert nll[2].item() == 0.0 and nll[0].item() > 0  # utterance 2 is infeasible
    ref_loss = nll.sum()
    ref_loss.backward()
    assert (logits.detach().double().cpu() - lr.detach()).abs().max() <= 1e-4 * lr.detach().abs().max()
    assert abs(loss.item() - ref_loss.item()) <= 1e-4 * abs(ref_loss.item())
    for name, a, r in (("weight", lin.weight.grad, wr.grad), ("bias", lin.bias.grad, br.grad), ("x", x.grad, xr.grad)):
        assert a is not None and a.dtype == torch.float32, name
        err = (a.double().cpu() - r).abs().max() / r.abs().max()
        assert err <= TOL, (name, err.item())
    assert x.grad[:, 2].abs().max() == 0  # the infeasible utterance contributes nothing
    for b in range(B):  # nor do padded frames
        if il[b] < T:
            assert x.grad[il[b]:, b].abs().max().item() == 0, b


def _multitask_step(enc, proj, x, lens, k, r_out, problem, drop_tap):
    from fbkst_b200 import criterion as C
    il, tg, tl, mask = problem
    out = enc(x, lens, return_all_hiddens=True)
    logits = proj(out.encoder_states[k - 1])
    assert type(logits.grad_fn).__name__ == "_CtcProjectionFnBackward"
    if drop_tap:  # anything between the projection and the loss that makes a new tensor drops the tap
        logits = logits.view_as(logits)
        assert not hasattr(logits, "_fbkst_tap")
    loss_ctc, totals, _ = C.ctc_loss_train(logits, mask.cuda(), tg.cuda(), tl.cuda(), 0)
    name = type(loss_ctc.grad_fn).__name__
    assert name.startswith("CtcLossFn" if drop_tap else "CtcProjLossFn"), name
    loss = (out.encoder_out * r_out).sum() + 0.5 * loss_ctc
    loss.backward()
    return out, loss, totals


def test_tap_route_matches_the_module_backward_route():
    """The loss-node backward (tap) and the module's own backward give the same gradient for every encoder
    parameter and both projection parameters (as test_ctc_projection_backward_in_the_criterion_node for the
    encoder's ctc_fc)."""
    from fbkst_b200 import criterion as C
    cfg = dict(embed_dim=128, ffn_dim=256, heads=2, layers=3, conv_channels=64, feat_dim=40, vocab=61,
               distance_penalty="log", ctc_layer=0, ctc_strategy="avg")
    sd = O.init_state_dict(cfg, seed=51)
    lens_in = [160, 131, 97, 160]
    x, lens = O.synthetic_batch(lens_in, 40, seed=52)
    L, B, V, k = 40, len(lens_in), 61, 2
    sub = torch.tensor([_sub(n) for n in lens_in])
    _, tg, tl, _ = _ctc_problem(L, B, V, seed=53)
    problem = (sub, tg, tl, torch.arange(L).unsqueeze(1) >= sub.unsqueeze(0))
    r = torch.randn(L, B, cfg["embed_dim"], generator=torch.Generator().manual_seed(54)).cuda()
    grads, losses = [], []
    for drop_tap in (False, True):
        enc = build_encoder(cfg, sd)
        for p in enc.parameters():
            p.requires_grad_(True)
        proj = C.CtcProjection(_projection(cfg["embed_dim"], V, seed=55))
        _, loss, _ = _multitask_step(enc, proj, x.cuda(), lens.cuda(), k, r, problem, drop_tap)
        losses.append(loss.item())
        gd = {n: p.grad.clone() for n, p in enc.named_parameters()}
        gd["proj.weight"], gd["proj.bias"] = proj.weight.grad.clone(), proj.bias.grad.clone()
        grads.append(gd)
    assert abs(losses[0] - losses[1]) <= 1e-6 * abs(losses[1])
    for n in grads[0]:
        a, b = grads[0][n], grads[1][n]
        assert (a - b).abs().max() <= 2e-3 * b.abs().max().clamp_min(1e-6), n
    assert grads[0]["proj.weight"].abs().max() > 0
    assert grads[0]["layers.0.fc1.weight"].abs().max() > 0


def test_half_model_states_and_projection():
    """model.half() (fairseq --fp16): states come back fp16, gradients arrive in the fp16 parameters of the
    encoder and of the projection, the loss is finite."""
    from fbkst_b200 import criterion as C
    cfg = dict(embed_dim=128, ffn_dim=256, heads=2, layers=3, conv_channels=64, feat_dim=40, vocab=61,
               distance_penalty="log", ctc_layer=0, ctc_strategy="avg")
    sd = O.init_state_dict(cfg, seed=61)
    lens_in = [160, 131, 97, 160]
    x, lens = O.synthetic_batch(lens_in, 40, seed=62)
    L, B, V, k = 40, len(lens_in), 61, 2
    sub = torch.tensor([_sub(n) for n in lens_in])
    _, tg, tl, _ = _ctc_problem(L, B, V, seed=63)
    problem = (sub, tg, tl, torch.arange(L).unsqueeze(1) >= sub.unsqueeze(0))
    enc = build_encoder(cfg, sd).half()
    for p in enc.parameters():
        p.requires_grad_(True)
    proj = C.CtcProjection(_projection(cfg["embed_dim"], V, seed=64, dtype=torch.float16))
    r = torch.randn(L, B, cfg["embed_dim"], generator=torch.Generator().manual_seed(65)).cuda().half()
    out, loss, _ = _multitask_step(enc, proj, x.cuda().half(), lens.cuda(), k, r, problem, drop_tap=False)
    assert all(s.dtype == torch.float16 for s in out.encoder_states)
    assert torch.isfinite(loss).item()
    for n, p in list(enc.named_parameters()) + [("proj.weight", proj.weight), ("proj.bias", proj.bias)]:
        assert p.grad is not None and p.grad.dtype == torch.float16, n
        assert torch.isfinite(p.grad).all(), n
    assert enc.layers[0].fc1.weight.grad.abs().max() > 0 and proj.weight.grad.abs().max() > 0


def test_validation_forward_matches_the_training_forward():
    from fbkst_b200 import criterion as C
    T, B, D, V = 33, 3, 128, 61
    proj = C.CtcProjection(_projection(D, V, seed=71))
    x = torch.randn(T, B, D, generator=torch.Generator().manual_seed(72)).cuda()
    with torch.no_grad():
        a = proj(x)
    assert a.grad_fn is None and not hasattr(a, "_fbkst_tap")
    b = proj(x.requires_grad_(True))
    assert b.requires_grad and torch.equal(a, b.detach())
    # the operand copies follow the parameters (an optimizer step changes their version counter)
    with torch.no_grad():
        proj.weight.mul_(0.5)
        c = proj(x)
        proj.bias.zero_()
        d = proj(x)
    assert not torch.equal(a, c) and not torch.equal(c, d)
    ref = F.linear(x.detach().bfloat16().double(), proj.weight.detach().bfloat16().double())
    assert (d.double() - ref).abs().max() <= 1e-4 * ref.abs().max()


# ------------------------------------------------------------------------------------------------------------
# fairseq's training call path (needs the reference package, as tests/test_gpu_dropin.py)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PLUGIN = os.path.join(ROOT, "fbk-fairseq-st_b200", "fbkst_b200", "plugin")


class _CritTask:
    def build_criterion(self, args):
        from fairseq import criterions
        return criterions.build_criterion(args, self)


def _args(arch, extra=()):
    from fairseq import options
    parser = options.get_training_parser()
    return options.parse_args_and_arch(parser, [
        "/tmp/nodata", "--user-dir", PLUGIN, "--arch", arch,
        "--task", "speech_translation_with_transcription", "--criterion", "ctc_multi_loss",
        "--underlying-criterion", "label_smoothed_cross_entropy", "--ctc-encoder-layer", "2",
        "--no-attn-2d", "--distance-penalty", "log", "--input-feat-per-channel", "40", "--encoder-layers", "3",
        "--decoder-layers", "2", "--max-tokens", "1000", "--skip-normalization"] + list(extra))


@pytest.mark.skipif(not R.available(), reason="reference package (baseline/_ref) not present")
def test_train_step_through_the_criterion_without_compression():
    """tests/test_gpu_dropin.py::test_train_step_through_the_criterion without --ctc-compress-out: the criterion
    projects encoder_states[1] with its own fc_out (a CtcProjection in ctc_multi_loss_b200).  Loss, UER counts
    and every parameter's gradient (model and criterion) against the reference's, cosine >= 0.99."""
    warnings.simplefilter("ignore")
    R.load()
    from fairseq import criterions, utils
    utils.import_user_module(argparse.Namespace(user_dir=PLUGIN))
    from fairseq.models import MODEL_REGISTRY
    from fbkst_b200 import criterion as C
    import bench
    task = _CritTask()
    task.source_dictionary = R.make_dictionary(120)
    task.target_dictionary = R.make_dictionary(90)
    extra = ["--label-smoothing", "0.1"]
    a_ref = _args("conv_transformer_big2", extra)
    a_our = _args("conv_transformer_big2_b200", extra)
    a_our.criterion = "ctc_multi_loss_b200"
    torch.manual_seed(7)
    ref = MODEL_REGISTRY["conv_transformer"].build_model(a_ref, task)
    ours = MODEL_REGISTRY["conv_transformer_b200"].build_model(a_our, task)
    ours.load_state_dict(ref.state_dict(), strict=True)
    ref, ours = ref.cuda().eval(), ours.cuda().eval()
    crit_ref = criterions.build_criterion(a_ref, task).cuda()
    crit_our = criterions.build_criterion(a_our, task).cuda()
    assert type(crit_our).__name__ == "B200CTCMultiLoss"
    crit_our.load_state_dict(crit_ref.state_dict(), strict=True)  # same keys: the projection keeps its parameters
    _, _, p_ref = C.find_ctc_projection(crit_ref)
    _, _, p_our = C.find_ctc_projection(crit_our)
    assert isinstance(p_our, C.CtcProjection) and isinstance(p_ref, torch.nn.Linear)
    lens_in = [801, 640, 523, 402]
    B, L = len(lens_in), (max(lens_in) + 3) // 4
    plan = bench.label_plan(L, B, len(task.source_dictionary), seed=23).cuda()
    handles = [p.register_forward_hook(lambda mod, i, o: o.scatter_add(
        -1, plan[: o.shape[0]].unsqueeze(-1), torch.full_like(o[..., :1], 30.0))) for p in (p_ref, p_our)]
    g = torch.Generator().manual_seed(1)
    s = O.synthetic_batch(lens_in, 40, seed=9)
    U, U1 = 11, 9
    tgt = torch.randint(4, 89, (B, U), generator=g)
    tgt[:, -1] = task.target_dictionary.eos()
    prev = torch.cat([torch.full((B, 1), task.target_dictionary.eos()), tgt[:, :-1]], 1)
    tr = torch.randint(4, 118, (B, U1), generator=g)
    trl = torch.tensor([9, 8, 7, 5])
    for b in range(B):
        tr[b, trl[b]:] = task.source_dictionary.pad()
    sample = utils.move_to_cuda(dict(
        net_input=dict(src_tokens=s[0], src_lengths=torch.tensor(lens_in, dtype=torch.long), prev_output_tokens=prev),
        target=tgt, transcript_target=tr, transcript_target_lengths=trl, ntokens=int(B * U), nsentences=B))
    try:
        with R.grad_shims():
            loss_ref, ss_ref, log_ref = crit_ref(ref, sample)
            loss_ref.backward()
        loss_our, ss_our, log_our = crit_our(ours, sample)
        loss_our.backward()
        assert ss_ref == ss_our
        assert abs(log_our["ctc_loss"] - log_ref["ctc_loss"]) <= 2e-2 * abs(log_ref["ctc_loss"])
        assert abs(loss_our.item() - loss_ref.item()) <= 2e-2 * abs(loss_ref.item())
        assert log_our["ctc_errors"] == log_ref["ctc_errors"] and log_our["ctc_total"] == log_ref["ctc_total"]
        low = {}
        for tag, mine, theirs in (("model", ours, ref), ("criterion", crit_our, crit_ref)):
            pr = dict(theirs.named_parameters())
            for name, p in mine.named_parameters():
                gr = pr[name].grad
                if gr is None or p.grad is None:
                    assert gr is None and p.grad is None, (tag, name)
                    continue
                a, r = p.grad.double().flatten(), gr.double().flatten()
                if r.abs().max() < 1e-9 or name.endswith("k_proj.bias"):
                    continue
                c = (torch.dot(a, r) / (a.norm() * r.norm()).clamp_min(1e-30)).item()
                if c < 0.99:
                    low[(tag, name)] = round(c, 4)
        assert not low, low
        assert ours.encoder.layers[0].fc1.weight.grad.abs().max() > 0
    finally:
        for h in handles:
            h.remove()
