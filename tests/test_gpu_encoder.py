"""End-to-end parity of the drop-in encoder against golden outputs of the LIVE reference
(tests/golden/*.pt, made by oracle/make_golden.py) and against the CPU oracle at larger sizes.
bf16 path: encoder outputs within 2e-2 (relative to max |ref|); lengths / masks bit-exact."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

from helpers import build_encoder, parity_report, rel_err  # noqa: E402
from oracle import encoder_oracle as O  # noqa: E402  (checker only)
from oracle.golden import load as load_golden  # noqa: E402

TOL = 2e-2


def check_against(out, ref, lens_in, tol=TOL):
    assert out.src_lengths.cpu().tolist() == ref["src_lengths"].tolist()
    if ref["encoder_padding_mask"] is None:
        assert out.encoder_padding_mask is None
    else:
        assert torch.equal(out.encoder_padding_mask.cpu(), ref["encoder_padding_mask"])
    assert out.encoder_out.shape == ref["encoder_out"].shape
    nl = ref["src_lengths"].tolist()
    rep = parity_report(out.encoder_out, ref["encoder_out"], nl)  # valid positions
    assert rep["max_rel"] < tol, rep
    assert rep["elementwise"] < tol, rep  # |a-b| <= tol*|ref| + tol*rms(ref) for every element
    for b, n in enumerate(nl):  # compressed padding rows are exact zeros before the final LayerNorm;
        # after it they are LN(0) = beta on both sides: compare them exactly as "finite and equal rows"
        assert torch.isfinite(out.encoder_out[n:, b]).all()
    assert torch.isfinite(out.encoder_out).all()
    return rep["max_rel"]


@pytest.mark.parametrize("name", ["enc_tiny_log.pt", "enc_tiny_nopen.pt"])
def test_encoder_golden(golden_dir, name):
    fx = load_golden(os.path.join(golden_dir, name))
    cfg = fx["cfg"]
    for strategy, ref in fx["outputs"].items():
        enc = build_encoder(dict(cfg, ctc_strategy=strategy), fx["state_dict"])
        if "bump_labels" in fx:
            hook = O.bump_hook(fx["bump_labels"], fx["bump_margin"])
            enc.ctc_fc.register_forward_hook(lambda m, i, o: hook(o))
        out = enc(fx["src_tokens"].cuda(), fx["src_lengths"].cuda(), return_all_hiddens=True)
        check_against(out, ref, fx["src_lengths"])
        assert len(out.encoder_states) == len(ref["encoder_states"])
        for a, r in zip(out.encoder_states, ref["encoder_states"]):
            assert a.shape == r.shape
        if cfg.get("ctc_layer", 0) > 0:
            assert out.ctc_out.shape == ref["ctc_out"].shape
            n0 = int(fx["src_lengths"][0] + 3) // 4
            assert torch.equal(out.ctc_padding_mask.cpu(), ref["ctc_padding_mask"])


def test_state_dict_layout_matches_reference(golden_dir):
    """Reference checkpoints load strict=True and our keys/shapes equal the reference's."""
    for name in ["enc_tiny_log.pt", "enc_tiny_nopen.pt"]:
        fx = load_golden(os.path.join(golden_dir, name))
        enc = build_encoder(fx["cfg"], fx["state_dict"])
        ours = enc.state_dict()
        assert set(ours.keys()) == set(fx["state_dict"].keys())
        for k, v in fx["state_dict"].items():
            assert tuple(ours[k].shape) == tuple(v.shape), k


def test_encoder_cfg1_vs_oracle():
    """BASELINE configs[0]: 6L d256 h4 ffn768, avg@4, batch 8 x 1000 x 40 (no penalty)."""
    cfg = dict(embed_dim=256, ffn_dim=768, heads=4, layers=6, conv_channels=64, feat_dim=40,
               vocab=105, distance_penalty=None, ctc_layer=4, ctc_strategy="avg")
    sd = O.init_state_dict(cfg, seed=0)
    x, lens = O.synthetic_batch([1000, 950, 900, 800, 700, 600, 500, 400], 40, seed=1234)
    labels = O.synthetic_ctc_bump(250, 8, 105, seed=7)
    hook = O.bump_hook(labels, 30.0)
    ref = O.encoder_forward(sd, cfg, x, lens, ctc_logits_hook=hook)
    enc = build_encoder(cfg, sd)
    enc.ctc_fc.register_forward_hook(lambda m, i, o: hook(o))
    out = enc(x.cuda(), lens.cuda())
    check_against(out, ref, lens)


@pytest.mark.parametrize("strategy", ["avg", "weighted", "softmax"])
def test_encoder_big2_ragged_vs_oracle(strategy):
    """EACL'21 model shape (d512 h8 ffn2048, log penalty) at reduced depth/batch, ragged batch with
    odd conv lengths (SURVEY F5), all three strategies."""
    cfg = dict(embed_dim=512, ffn_dim=2048, heads=8, layers=3, conv_channels=64, feat_dim=40,
               vocab=1005, distance_penalty="log", ctc_layer=2, ctc_strategy=strategy)
    sd = O.init_state_dict(cfg, seed=1)
    x, lens = O.synthetic_batch([601, 598, 411, 203], 40, seed=77)
    labels = O.synthetic_ctc_bump(151, 4, 1005, seed=9)
    hook = O.bump_hook(labels, 30.0)
    ref = O.encoder_forward(sd, cfg, x, lens, ctc_logits_hook=hook)
    enc = build_encoder(cfg, sd)
    enc.ctc_fc.register_forward_hook(lambda m, i, o: hook(o))
    out = enc(x.cuda(), lens.cuda())
    check_against(out, ref, lens)


def test_reorder_and_non_torchscript(golden_dir):
    fx = load_golden(os.path.join(golden_dir, "enc_tiny_log.pt"))
    enc = build_encoder(fx["cfg"], fx["state_dict"])
    net_input = dict(src_tokens=fx["src_tokens"].cuda(), src_lengths=fx["src_lengths"].cuda(),
                     prev_output_tokens=torch.zeros(3, 5), transcript_prev_output_tokens=None)
    out = enc.forward_non_torchscript(net_input)
    order = torch.tensor([2, 0, 0, 1], device="cuda")
    re = enc.reorder_encoder_out(out, order)
    assert re.encoder_out.shape[1] == 4
    assert torch.equal(re.encoder_out[:, 0], out.encoder_out[:, 2])
    assert enc.output_batch_first is False


@pytest.mark.parametrize("graph,lanes", [(False, 1), (True, 1), (True, 2), (True, 3)])
def test_pipeline_matches_direct_calls(golden_dir, graph, lanes):
    """The host-buffer serving loop (copy-in / compute lanes / copy-out streams, asynchronous
    launch + deferred finish) returns exactly what direct calls return."""
    from fbkst_b200 import ops
    from fbkst_b200.pipeline import EncoderPipeline
    fx = load_golden(os.path.join(golden_dir, "enc_tiny_log.pt"))
    enc = build_encoder(fx["cfg"], fx["state_dict"])
    batches = []
    for i, lens in enumerate([[61, 47, 30], [90, 90], [33, 20, 20, 7], [61, 47, 30], [61, 40, 33],
                              [61, 61, 61], [90, 12], [90, 90], [33, 31, 20, 9]]):
        x, l = O.synthetic_batch(lens, 40, seed=50 + i)
        batches.append(((x * 2 + 1).pin_memory(), l))
    direct = []
    for x, l in batches:
        xn = ops.cmvn(x.cuda(), l.to(torch.int32).cuda())
        o = enc(xn, l)
        direct.append((o.encoder_out.cpu(), o.src_lengths.cpu()))
    enc.use_cuda_graph = graph
    pipe = EncoderPipeline(enc, lanes=lanes)
    assert pipe.lanes == lanes
    got = [(h.clone(), l.clone()) for h, l in pipe.run(iter(batches))]
    got += [(h.clone(), l.clone()) for h, l in pipe.run(iter(batches))]  # second pass: cached graphs
    assert len(got) == 2 * len(direct)
    for (a, la), (b, lb) in zip(got, direct + direct):
        assert torch.equal(la, lb)
        assert torch.equal(a, b)
    # device-resident batches through the same lanes
    resident = [(ops.cmvn(x.cuda(), l.to(torch.int32).cuda()), l) for x, l in batches]
    pipe_dev = EncoderPipeline(enc, normalize=False, lanes=lanes)
    outs = [(o.encoder_out.clone(), o.src_lengths.clone()) for o in pipe_dev.run_device(iter(resident))]
    torch.cuda.synchronize()
    assert len(outs) == len(direct)
    for (a, la), (b, lb) in zip(outs, direct):
        assert torch.equal(la.cpu(), lb)
        assert torch.equal(a.cpu(), b)


def test_cuda_graph_mode_is_bit_identical():
    """use_cuda_graph replays the same kernels: outputs equal the eager path bit for bit, across
    batches of one shape with different lengths/content and across a second shape."""
    cfg = dict(embed_dim=256, ffn_dim=512, heads=4, layers=4, conv_channels=64, feat_dim=40,
               vocab=205, distance_penalty="log", ctc_layer=2, ctc_strategy="weighted")
    sd = O.init_state_dict(cfg, seed=3)
    enc = build_encoder(cfg, sd)
    labels = O.synthetic_ctc_bump(80, 4, 205, seed=5).cuda()

    def bump(m, i, o):  # device-resident plan (capturable); the second shape is left as it is
        if tuple(o.shape[:2]) != tuple(labels.shape):
            return o
        return o.scatter_add(2, labels.unsqueeze(-1), torch.full_like(o[..., :1], 30.0))
    enc.ctc_fc.register_forward_hook(bump)
    batches = [O.synthetic_batch(l, 40, seed=s) for s, l in
               enumerate([[320, 301, 222, 95], [320, 320, 320, 320], [317, 200, 100, 64], [200, 111]])]
    eager = []
    for x, l in batches:
        o = enc(x.cuda(), l.cuda())
        eager.append((o.encoder_out.clone(), o.src_lengths.clone(),
                      None if o.encoder_padding_mask is None else o.encoder_padding_mask.clone(),
                      o.ctc_out.float().clone()))
    enc.use_cuda_graph = True
    for rep in range(2):  # second round replays the cached graphs
        for (x, l), (eo, sl, pm, co) in zip(batches, eager):
            o = enc(x.cuda(), l.cuda())
            assert torch.equal(o.src_lengths, sl)
            assert torch.equal(o.encoder_out, eo)
            assert (o.encoder_padding_mask is None) == (pm is None)
            if pm is not None:
                assert torch.equal(o.encoder_padding_mask, pm)
            n = int(l[0] + 3) // 4
            assert torch.equal(o.ctc_out.float()[:n], co[:n])
    assert len(enc._graphs) == 3  # T = 320, 317, 200


@pytest.mark.parametrize("strategy", ["weighted", "softmax"])
def test_encoder_cfg3_long_ragged_vs_oracle(strategy):
    """BASELINE configs[2] shape: big2 model, ragged 200-3000 frame utterances (L up to 750, several
    query tiles and key tiles per utterance, partially valid last tiles), weighted / softmax pooling."""
    cfg = dict(embed_dim=512, ffn_dim=2048, heads=8, layers=2, conv_channels=64, feat_dim=40,
               vocab=505, distance_penalty="log", ctc_layer=1, ctc_strategy=strategy)
    sd = O.init_state_dict(cfg, seed=2)
    lens_in = [3000, 2177, 1203, 640, 201]
    x, lens = O.synthetic_batch(lens_in, 40, seed=31)
    labels = O.synthetic_ctc_bump(750, len(lens_in), 505, seed=11)
    hook = O.bump_hook(labels, 30.0)
    ref = O.encoder_forward(sd, cfg, x, lens, ctc_logits_hook=hook)
    enc = build_encoder(cfg, sd)
    enc.ctc_fc.register_forward_hook(lambda m, i, o: hook(o))
    out = enc(x.cuda(), lens.cuda())
    check_against(out, ref, lens)


def test_encoder_cfg5_shape_vs_oracle():
    """BASELINE configs[4] shape: 80-dim fbank, d1024 h16 ffn4096, 128 conv channels
    (conv_transformer_giant), long utterances (T up to 5000 -> L = 1250), compression at layer 2."""
    cfg = dict(embed_dim=1024, ffn_dim=4096, heads=16, layers=2, conv_channels=128, feat_dim=80,
               vocab=305, distance_penalty="log", ctc_layer=2, ctc_strategy="avg")
    sd = O.init_state_dict(cfg, seed=4)
    lens_in = [5000, 3333]
    x, lens = O.synthetic_batch(lens_in, 80, seed=41)
    labels = O.synthetic_ctc_bump(1250, 2, 305, seed=13)
    hook = O.bump_hook(labels, 30.0)
    ref = O.encoder_forward(sd, cfg, x, lens, ctc_logits_hook=hook)
    enc = build_encoder(cfg, sd)
    enc.ctc_fc.register_forward_hook(lambda m, i, o: hook(o))
    out = enc(x.cuda(), lens.cuda())
    check_against(out, ref, lens)


@pytest.mark.parametrize("ctc_layer", [1, 2, 3])
def test_encoder_cfg5_compression_sweep_vs_oracle(ctc_layer):
    """BASELINE configs[4] sweeps the compression layer (4 / 8 / 12 of 12): here first / middle / last of a
    3-layer d1024 h16 C128 F80 encoder -- compressing before any layer has run, between layers, and after
    the last one (nothing but the final LayerNorm sees the compressed rows)."""
    cfg = dict(embed_dim=1024, ffn_dim=4096, heads=16, layers=3, conv_channels=128, feat_dim=80,
               vocab=305, distance_penalty="log", ctc_layer=ctc_layer, ctc_strategy="avg")
    sd = O.init_state_dict(cfg, seed=6)
    lens_in = [1210, 1000, 517]
    x, lens = O.synthetic_batch(lens_in, 80, seed=43)
    labels = O.synthetic_ctc_bump(303, 3, 305, seed=17)
    hook = O.bump_hook(labels, 30.0)
    ref = O.encoder_forward(sd, cfg, x, lens, ctc_logits_hook=hook)
    enc = build_encoder(cfg, sd)
    dev_hook = O.bump_hook(labels.cuda(), 30.0)  # device-resident plan: capturable in a CUDA graph
    enc.ctc_fc.register_forward_hook(lambda m, i, o: dev_hook(o))
    out = enc(x.cuda(), lens.cuda())
    check_against(out, ref, lens)
    enc.use_cuda_graph = True  # the graph path (worst-case grids + device-side row limits) as well
    out_g = enc(x.cuda(), lens.cuda())
    assert torch.equal(out_g.src_lengths, out.src_lengths)
    assert torch.equal(out_g.encoder_out, out.encoder_out)


def test_encoder_full_size_properties():
    """BASELINE configs[1] at FULL size (64 x 1500 x 40, 11 layers, V=8005) through size-independent
    properties: (1) determinism: two runs are bit-identical; (2) batch-slot permutation: permuting
    the utterances permutes the outputs (same padded extent on both sides, SURVEY F5) up to bf16
    rounding, and the integer outputs (compressed lengths) exactly;
    (3) compressed lengths equal the number of label changes of the injected plan; (4) padding rows
    of the compressed output are exactly 0 and everything is finite."""
    import bench
    cfgb = bench.CONFIGS["cfg2"]
    model = cfgb["model"]
    torch.manual_seed(0)
    from fbkst_b200.config import build_encoder as build
    enc = build(model, None, device="cpu")
    bench.randomise_norm_stats(enc, 1)
    enc = enc.cuda().eval()
    B, T, L = 64, 1500, 375
    g = torch.Generator().manual_seed(5)
    lens_in = torch.randint(700, T + 1, (B,), generator=g).sort(descending=True).values
    lens_in[0] = T
    x, lens = bench.make_batch(lens_in.tolist(), 40, 99)
    plan = bench.label_plan(L, B, model["vocab"], seed=7).cuda()
    state = dict(plan=plan)

    def bump(m, i, o):
        return o.scatter_add(2, state["plan"].unsqueeze(-1), torch.full_like(o[..., :1], 30.0))
    enc.ctc_fc.register_forward_hook(bump)
    from fbkst_b200 import ops
    xn = ops.cmvn(x.cuda(), lens.to(torch.int32).cuda())  # as the bench: CMVN, then the encoder
    o1 = enc(xn, lens.cuda())
    o2 = enc(xn, lens.cuda())
    assert torch.equal(o1.encoder_out, o2.encoder_out) and torch.equal(o1.src_lengths, o2.src_lengths)
    assert torch.isfinite(o1.encoder_out).all()
    sub = [((n + 1) // 2 + 1) // 2 for n in lens.tolist()]
    pl = plan.cpu()
    for b in range(B):
        n = sub[b]
        changes = 1 + int((pl[1:n, b] != pl[: n - 1, b]).sum())
        assert int(o1.src_lengths[b]) == changes, b
        assert bool(o1.encoder_padding_mask[b, changes:].all()) and not bool(o1.encoder_padding_mask[b, :changes].any())
    perm = torch.randperm(B, generator=g)
    state["plan"] = plan[:, perm.cuda()]
    o3 = enc(xn[perm.cuda()].contiguous(), lens[perm].cuda())
    assert torch.equal(o3.src_lengths.cpu(), o1.src_lengths.cpu()[perm])
    L2 = o1.encoder_out.shape[0]
    for k in range(0, B, 5):
        b = int(perm[k])
        n = int(o1.src_lengths[b])
        # not bit for bit: the key tiles of an utterance are split between the two softmax groups
        # by their position in the CTA's tile stream, which moves with the batch slot
        assert rel_err(o3.encoder_out[:n, k], o1.encoder_out[:n, b]) < 5e-3, (k, b)


def test_learned_positional_embeddings():
    """--encoder-learned-pos (positional_embedding_audio.py:13-17): the embedding matrix is read like the
    sinusoidal table (row t+1 inside the utterance, padding row 0 beyond).  Checked against the oracle with the
    positional term swapped for the same lookup."""
    import torch.nn.functional as F
    cfg = dict(embed_dim=128, ffn_dim=256, heads=2, layers=2, conv_channels=64, feat_dim=40, vocab=64,
               distance_penalty="log", ctc_layer=0, ctc_strategy="avg", learned_pos=True, max_source_positions=64)
    sd = O.init_state_dict(cfg, seed=21)
    del sd["embed_positions.embeddings._float_tensor"]
    g = torch.Generator().manual_seed(3)
    W = torch.randn(64, 128, generator=g) * 0.3
    W[0] = 0  # padding_idx row
    sd["embed_positions.embeddings.weight"] = W
    enc = build_encoder(cfg, sd)
    assert "embed_positions.embeddings.weight" in enc.state_dict()
    x, lens = O.synthetic_batch([120, 99, 64], 40, seed=5)
    out = enc(x.cuda(), lens.cuda())
    # oracle with the learned lookup in place of the sinusoidal one
    orig = O.positional_embedding
    try:
        def learned(lengths, dim):
            t = torch.arange(int(lengths.max())).unsqueeze(0)
            pos = torch.where(t < lengths.unsqueeze(1), t + 1, torch.zeros_like(t))
            return F.embedding(pos, W)
        O.positional_embedding = learned
        ref = O.encoder_forward({k: v for k, v in sd.items() if "embed_positions" not in k}, cfg, x, lens)
    finally:
        O.positional_embedding = orig
    check_against(out, ref, lens)


@pytest.mark.parametrize("lens_in", [[5, 3, 1], [1], [9, 9], [130, 2]])
def test_tiny_and_degenerate_batches(lens_in):
    """Edge cases of the shape logic: utterances of 1-9 frames (L = 1-3 after the two stride-2 convs, single
    partly filled tiles everywhere), B = 1, and a batch that mixes a 130-frame utterance with a 2-frame one."""
    cfg = dict(embed_dim=128, ffn_dim=256, heads=2, layers=2, conv_channels=64, feat_dim=40, vocab=64,
               distance_penalty="log", ctc_layer=1, ctc_strategy="weighted")
    sd = O.init_state_dict(cfg, seed=31)
    x, lens = O.synthetic_batch(lens_in, 40, seed=7)
    L = ((max(lens_in) + 1) // 2 + 1) // 2
    labels = O.synthetic_ctc_bump(L, len(lens_in), 64, seed=3)
    hook = O.bump_hook(labels, 30.0)
    ref = O.encoder_forward(sd, cfg, x, lens, ctc_logits_hook=hook)
    enc = build_encoder(cfg, sd)
    dev_hook = O.bump_hook(labels.cuda(), 30.0)
    enc.ctc_fc.register_forward_hook(lambda m, i, o: dev_hook(o))
    out = enc(x.cuda(), lens.cuda())
    check_against(out, ref, lens)
    enc.use_cuda_graph = True
    out_g = enc(x.cuda(), lens)
    assert torch.equal(out_g.encoder_out, out.encoder_out)
    # and the differentiable chain on the same degenerate shapes
    for p in enc.parameters():
        p.requires_grad_(True)
    enc.use_cuda_graph = False
    o2 = enc(x.cuda(), lens.cuda(), return_all_hiddens=True)
    assert o2.src_lengths.cpu().tolist() == ref["src_lengths"].tolist()
    (o2.encoder_out.float().pow(2).sum() + o2.ctc_out.float().pow(2).sum() * 1e-3).backward()
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in enc.parameters())


def test_sustained_ragged_inference_stays_finite_and_identical():
    """Regression (round 2): after CTC compression the remaining layers run on worst-case grids with a
    device-side row limit in a PERSISTENT workspace; the rows between that limit and the end of the last
    256-row GEMM tile are read-modify-written by every residual epilogue.  They used to survive from one
    forward to the next, grew ~1.4x per forward and reached inf after ~70 forwards of a ragged batch, after
    which attention read them as V rows of partially valid key tiles (0 * inf = NaN).  fbkst_ctc_compress
    now zeroes them with the other padding rows: 150 forwards of the same ragged batch stay finite and
    bit-identical to the first one, launch by launch and under graph replay."""
    cfg = dict(embed_dim=256, ffn_dim=768, heads=4, layers=6, conv_channels=64, feat_dim=40,
               vocab=105, distance_penalty=None, ctc_layer=4, ctc_strategy="avg")
    sd = O.init_state_dict(cfg, seed=0)
    x, lens = O.synthetic_batch([1000, 950, 900, 800, 700, 600, 500, 400], 40, seed=1234)
    labels = O.synthetic_ctc_bump(250, 8, 105, seed=7)
    for graph in (False, True):
        enc = build_encoder(cfg, sd)
        enc.ctc_logit_bump = (labels.to(torch.int32).cuda().contiguous(), 30.0)  # (capturable, unlike a hook)
        enc.use_cuda_graph = graph
        xd = x.cuda()
        first = enc(xd, lens)
        torch.cuda.synchronize()
        first_out, first_len = first.encoder_out.clone(), first.src_lengths.clone()
        assert torch.isfinite(first_out).all()
        for _ in range(150):
            out = enc(xd, lens)
        torch.cuda.synchronize()
        assert torch.equal(out.src_lengths, first_len)
        assert torch.isfinite(out.encoder_out).all(), "graph=%s" % graph
        assert torch.equal(out.encoder_out, first_out), "graph=%s" % graph
        if not graph:  # the workspace itself stays bounded (it reached 1e10 before the fix)
            for name, t in enc._ws[0][1].items():
                assert torch.isfinite(t.float()).all(), name
                assert float(t.float().abs().max()) < 1e4, name
