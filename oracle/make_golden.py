"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/*.npz by running the UNMODIFIED reference.

Run where the reference tree is available (oracle/ref_import.py; SDETR_REFERENCE_ROOT points at it):
  python oracle/make_golden.py [fixture ...]      (fixture names: FIXTURES below; default all)
The reference ships no tests / golden vectors (SURVEY.md section 4); these fixtures are outputs of the
reference's own Python modules (imported via oracle/ref_import.py) on small seeded inputs, and are what
pins the oracle (tests/test_oracle_golden.py) and, through it, the CUDA kernels.

Fixtures
  msda_core_{a,b}.npz   multi_scale_deformable_attn_pytorch (ms_deform_attn.py:159-212) forward and its
                        autograd gradients (the contract of _C.ms_deform_attn_forward/backward).
  msda_module.npz       MultiScaleDeformableAttention.forward (ms_deform_attn.py:286-377) incl. state_dict.
  encoder_tiny_{even,ragged}.npz
                        SalienceTransformer.forward lines 106-183 (filter + encoder) of a tiny model:
                        inputs, encoder-half state_dict, the kwargs the filter hands to the encoder, and
                        the encoder memory.  "even": both images full size (tie-free selection);
                        "ragged": second image smaller (padded tokens -> ties, see SURVEY.md 8(a) notes).
  dropin_*.npz, decoder_*.npz
                        the drop-in and decoder-half tests at C = 256: see make_dropin_* / make_decoder_* below.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_import  # noqa: E402
from oracle import oracle as orc  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def np_(t):
    return t.detach().cpu().numpy()


def make_msda_core(name, b, shapes, m, d, nq, p, seed):
    ref = ref_import.load()
    g = torch.Generator().manual_seed(seed)
    shapes_t = torch.tensor(shapes, dtype=torch.int64)
    nv = int(shapes_t.prod(1).sum())
    lsi = torch.cat([shapes_t.new_zeros(1), shapes_t.prod(1).cumsum(0)[:-1]])
    L = len(shapes)
    value = torch.randn(b, nv, m, d, generator=g, requires_grad=True)
    loc = (torch.rand(b, nq, m, L, p, 2, generator=g) * 1.2 - 0.1).requires_grad_(True)
    attn = torch.randn(b, nq, m, L * p, generator=g).softmax(-1).view(b, nq, m, L, p).requires_grad_(True)
    out = ref.msda.multi_scale_deformable_attn_pytorch(value, shapes_t, loc, attn)
    gout = torch.randn(out.shape, generator=g)
    gv, gl, ga = torch.autograd.grad(out, (value, loc, attn), gout)
    np.savez_compressed(os.path.join(OUT, name), value=np_(value), shapes=np_(shapes_t), lsi=np_(lsi),
                        loc=np_(loc), attn=np_(attn), out=np_(out), grad_out=np_(gout), grad_value=np_(gv),
                        grad_loc=np_(gl), grad_attn=np_(ga))


def make_msda_module(seed=3):
    ref = ref_import.load()
    torch.manual_seed(seed)
    mod = ref.msda.MultiScaleDeformableAttention(64, 4, 2, 4).eval()
    with torch.no_grad():  # non-trivial offsets / weights (init has zero weight matrices)
        mod.sampling_offsets.weight.normal_(0, 0.05)
        mod.attention_weights.weight.normal_(0, 0.5)
    shapes = [(9, 12), (5, 6), (3, 3), (2, 2)]
    shapes_t = torch.tensor(shapes)
    nv = int(shapes_t.prod(1).sum())
    lsi = torch.cat([shapes_t.new_zeros(1), shapes_t.prod(1).cumsum(0)[:-1]])
    b, nq = 2, 37
    query = torch.randn(b, nq, 64)
    refp = torch.rand(b, nq, 4, 2)
    value = torch.randn(b, nv, 64)
    mask = torch.rand(b, nv) < 0.15
    with torch.no_grad():
        out = mod(query, refp, value, shapes_t, lsi, mask)
    sd = {"sd." + k: np_(v) for k, v in mod.state_dict().items()}
    np.savez_compressed(os.path.join(OUT, "msda_module.npz"), query=np_(query), ref=np_(refp), value=np_(value),
                        shapes=np_(shapes_t), lsi=np_(lsi), mask=np_(mask), out=np_(out), **sd)


class _Stop(Exception):
    pass


TINY = dict(embed_dim=64, d_ffn=128, n_heads=2, n_levels=4, n_points=4, num_layers=3, num_classes=11,
            level_filter_ratio=(0.4, 0.8, 1.0, 1.0), layer_filter_ratio=(1.0, 0.6, 0.3), topk_sa=20,
            max_num_embedding=40, num_proposals=30)


def make_encoder_tiny(name, image_sizes, padded, seed):
    tr = ref_import.build_transformer(seed=seed, **TINY)
    with torch.no_grad():
        for layer in tr.encoder.layers:  # exercise learned offsets/weights, not only the init ring
            layer.self_attn.sampling_offsets.weight.normal_(0, 0.05)
            layer.self_attn.attention_weights.weight.normal_(0, 0.5)
    feats, masks, pos = orc.synthetic_inputs(image_sizes, padded, TINY["embed_dim"], seed=seed)
    captured = {}
    enc_fwd = tr.encoder.forward
    layer_out = []
    hooks = [l.register_forward_hook(lambda m, i, o: layer_out.append(o.detach().clone())) for l in tr.encoder.layers]

    def spy(**kw):
        captured.update(kw)
        captured["memory"] = enc_fwd(**kw)
        raise _Stop()

    tr.encoder.forward = spy
    try:
        with torch.no_grad():
            tr(feats, masks, pos, None, None, None)
    except _Stop:
        pass
    for h in hooks:
        h.remove()
    sd = {"sd." + k: np_(v) for k, v in tr.state_dict().items()
          if not (k.startswith("decoder") or k.startswith("tgt_embed") or k.startswith("encoder_bbox_head"))}
    arrs = {f"feat{i}": np_(f) for i, f in enumerate(feats)}
    arrs.update({f"mask{i}": np_(m) for i, m in enumerate(masks)})
    arrs.update({f"pos{i}": np_(p) for i, p in enumerate(pos)})
    arrs.update({f"layer_out{i}": np_(o) for i, o in enumerate(layer_out)})
    np.savez_compressed(
        os.path.join(OUT, name),
        memory=np_(captured["memory"]),
        foreground_score=np_(captured["foreground_score"]),
        focus_token_nums=np_(captured["focus_token_nums"]),
        selected_inds=np_(captured["foreground_inds"][0]),
        layer_num_query=np.array([x.shape[1] for x in captured["foreground_inds"]]),
        valid_ratios=np_(captured["valid_ratios"]),
        spatial_shapes=np_(captured["spatial_shapes"]),
        level_start_index=np_(captured["level_start_index"]),
        cfg_keys=np.array(sorted(TINY.keys())),
        **arrs, **sd)


def make_encoder_tiny_grads(name, image_sizes, padded, seed):
    """Gradients of the reference's own autograd through lines 106-183 for the tiny model of ``make_encoder_tiny`` (same
    seed -> same weights and inputs): d loss / d parameter for every parameter the loss reaches and d loss / d feats,
    loss = memory.square().mean().  Pins the training path (MSDA backward kernel inside torch autograd)."""
    tr = ref_import.build_transformer(seed=seed, **TINY).train()  # dropout = 0.0: train() only enables grad paths
    with torch.no_grad():
        for layer in tr.encoder.layers:
            layer.self_attn.sampling_offsets.weight.normal_(0, 0.05)
            layer.self_attn.attention_weights.weight.normal_(0, 0.5)
    feats, masks, pos = orc.synthetic_inputs(image_sizes, padded, TINY["embed_dim"], seed=seed)
    feats = [f.requires_grad_(True) for f in feats]
    captured = {}
    enc_fwd = tr.encoder.forward

    def spy(**kw):
        captured["memory"] = enc_fwd(**kw)
        raise _Stop()

    tr.encoder.forward = spy
    try:
        tr(feats, masks, pos, None, None, None)
    except _Stop:
        pass
    loss = captured["memory"].square().mean()
    loss.backward()
    out = {"loss": np_(loss)}
    for n, p in tr.named_parameters():
        if p.grad is not None:
            out["grad." + n] = np_(p.grad)
    for i, f in enumerate(feats):
        out[f"grad_feat{i}"] = np_(f.grad)
    np.savez_compressed(os.path.join(OUT, name), **out)


C256 = dict(embed_dim=256, d_ffn=256, n_heads=8, n_levels=4, n_points=4, num_layers=2, num_classes=11,
            level_filter_ratio=(0.4, 0.8, 1.0, 1.0), layer_filter_ratio=(1.0, 0.5), topk_sa=64,
            max_num_embedding=80, num_proposals=30)
C256_IMAGES, C256_PADDED, C256_SEED, C256_ROWS = [(384, 512), (384, 512)], (384, 512), 11, 256


def encoder_half_keys(state_dict):
    return {k: tuple(v.shape) for k, v in state_dict.items()
            if not (k.startswith("decoder") or k.startswith("tgt_embed") or k.startswith("encoder_bbox_head")
                    or k.endswith("_filter_ratio"))}


def make_encoder_c256(name="encoder_c256.npz"):
    """Reference width (C = 256, 8 heads of 32) at 4080 tokens per image: exercises the paths that are specialised for
    the real model (fused pre-attention, persistent tensor-core GEMM).  Weights come from
    oracle.deterministic_state_dict (regenerated by the tests), inputs from oracle.synthetic_inputs; the fixture holds
    the reference's outputs: selection, scores, and the encoder memory at C256_ROWS sampled tokens per image plus
    per-token channel means of all tokens."""
    import json
    tr = ref_import.build_transformer(seed=0, **C256)
    shapes = encoder_half_keys(tr.state_dict())
    missing = tr.load_state_dict(orc.deterministic_state_dict(shapes, C256_SEED), strict=False)
    assert not [k for k in missing.unexpected_keys]
    feats, masks, pos = orc.synthetic_inputs(C256_IMAGES, C256_PADDED, C256["embed_dim"], seed=C256_SEED)
    captured = {}
    enc_fwd = tr.encoder.forward

    def spy(**kw):
        captured.update(kw)
        captured["memory"] = enc_fwd(**kw)
        raise _Stop()

    tr.encoder.forward = spy
    try:
        with torch.no_grad():
            tr(feats, masks, pos, None, None, None)
    except _Stop:
        pass
    mem = captured["memory"]
    nv = mem.shape[1]
    rows = torch.stack([torch.randperm(nv, generator=torch.Generator().manual_seed(100 + i))[:C256_ROWS] for i in range(mem.shape[0])])
    np.savez_compressed(
        os.path.join(OUT, name),
        shapes_json=np.array(json.dumps({k: list(v) for k, v in shapes.items()})),
        memory_rows_index=np_(rows),
        memory_rows=np_(torch.gather(mem, 1, rows[..., None].expand(-1, -1, mem.shape[2]))),
        memory_row_mean=np_(mem.mean(-1)), memory_row_absmax=np_(mem.abs().amax(-1)),
        foreground_score=np_(captured["foreground_score"]),
        focus_token_nums=np_(captured["focus_token_nums"]),
        selected_inds=np_(captured["foreground_inds"][0]),
        layer_num_query=np.array([x.shape[1] for x in captured["foreground_inds"]]))


def make_salience_criterion(name="salience_criterion.npz"):
    """SalienceCriterion (models/detectors/salience_detr.py:13-116) + sigmoid_focal_loss (models/bricks/losses.py:4-12).
    The detector module cannot be imported here (pycocotools / accelerate are missing), so the two definitions are compiled
    from the reference's own source files, unmodified, without the modules' import lines; loss, its gradient w.r.t. the
    score maps, and the target maps on seeded boxes."""
    import ast
    from typing import Tuple  # noqa: F401
    from torch import nn
    from torch.nn import functional as F
    from torchvision.ops import boxes as box_ops
    ns = {"torch": torch, "nn": nn, "F": F, "box_ops": box_ops, "Tuple": Tuple}
    for path, kind, ident in ((os.path.join(ref_import.REFERENCE_ROOT, "models/bricks/losses.py"), ast.FunctionDef, "sigmoid_focal_loss"),
                              (os.path.join(ref_import.REFERENCE_ROOT, "models/detectors/salience_detr.py"), ast.ClassDef, "SalienceCriterion")):
        node = [n for n in ast.parse(open(path).read()).body if isinstance(n, kind) and n.name == ident][0]
        exec(compile(ast.Module(body=[node], type_ignores=[]), path, "exec"), ns)
    crit = ns["SalienceCriterion"]()
    g = torch.Generator().manual_seed(0)
    shapes = [(50, 84), (25, 42), (13, 21), (7, 11)]
    fg = [torch.randn(2, 1, h, w, generator=g).requires_grad_(True) for h, w in shapes]

    def boxes(n):
        return torch.cat([torch.rand(n, 2, generator=g) * 0.6 + 0.2, torch.rand(n, 2, generator=g) * 0.5 + 0.02], -1)

    targets = [{"boxes": boxes(7)}, {"boxes": boxes(3)}]
    image_sizes = [(400, 672), (380, 600)]
    strides = [(400 / h, 672 / w) for h, w in shapes]
    loss = crit(fg, targets, strides, image_sizes)["loss_salience"]
    loss.backward()
    mt = []
    for lvl, (shape, st) in enumerate(zip(shapes, strides)):
        cx, cy = crit.get_pixel_coordinate(shape, st, "cpu")
        mt.append(torch.stack([crit.get_mask_single_level(cx, cy, box_ops._box_cxcywh_to_xyxy(t["boxes"]) *
                                                          torch.tensor([iw, ih, iw, ih]), lvl)
                               for t, (ih, iw) in zip(targets, image_sizes)]))
    np.savez_compressed(os.path.join(OUT, name), loss=np_(loss), boxes0=np_(targets[0]["boxes"]), boxes1=np_(targets[1]["boxes"]),
                        image_sizes=np.array(image_sizes), shapes=np.array(shapes), strides=np.array(strides, dtype=np.float64),
                        mask_targets=np_(torch.cat(mt, 1)), **{f"fg{i}": np_(f) for i, f in enumerate(fg)},
                        **{f"grad{i}": np_(f.grad) for i, f in enumerate(fg)})


# ---- fixtures of the drop-in and decoder-half tests (tests/test_dropin_reference.py, tests/test_decoder_half.py) -----------
# Outputs larger than a few KiB are stored at SAMPLE positions (oracle.sample_index, seeded) with their absolute maximum.
SAMPLE = 512


def _store_sampled(arrs, name, t, seed):
    arrs[name + "_sample"] = np_(orc.sampled(t, SAMPLE, seed))
    arrs[name + "_absmax"] = np.float32(t.abs().max().item())


def _load_deterministic(model, seed, skip=("level_filter_ratio", "layer_filter_ratio")):
    """Load oracle.deterministic_state_dict into a reference model -> (shapes_json, aliases_json) to store with the fixture."""
    import json
    sd0 = model.state_dict()
    shapes = {k: list(v.shape) for k, v in sd0.items() if not k.endswith(skip)}
    gen = orc.deterministic_state_dict(shapes, seed)
    res = model.load_state_dict(gen, strict=False)
    assert not res.unexpected_keys and set(res.missing_keys) <= {k for k in sd0 if k.endswith(skip)}
    eff = model.state_dict()
    aliases = {}
    for k in shapes:  # keys sharing one tensor: the value it ended up holding comes from one of them
        if not torch.equal(eff[k], gen[k]):
            src = [j for j in shapes if j != k and eff[j].data_ptr() == eff[k].data_ptr() and torch.equal(eff[k], gen[j])]
            assert src, k
            aliases[k] = src[0]
    assert all(torch.equal(v, eff[k]) for k, v in orc.golden_state_dict(json.dumps(shapes), seed, json.dumps(aliases)).items())
    return json.dumps(shapes), json.dumps(aliases)


def make_dropin_msda_operator(name="dropin_msda_operator.npz", seed=21):
    """MultiScaleDeformableAttention(256, 4 levels, 8 heads, 4 points) forward and the gradients w.r.t. query, value,
    sampling_offsets.weight and value_proj.weight, on its pure-PyTorch path (ms_deform_attn.py:159-212,311-377)."""
    ref = ref_import.load()
    mod = ref.msda.MultiScaleDeformableAttention(256, 4, 8, 4)
    shapes_json, aliases_json = _load_deterministic(mod, seed)
    shapes = torch.tensor([(30, 40), (15, 20), (8, 10), (4, 5)])
    lsi = torch.cat([shapes.new_zeros(1), shapes.prod(1).cumsum(0)[:-1]])
    nv, b, nq = int(shapes.prod(1).sum()), 2, 333
    g = torch.Generator().manual_seed(1)
    query = torch.randn(b, nq, 256, generator=g).requires_grad_(True)
    refp = torch.rand(b, nq, 4, 2, generator=g)
    value = torch.randn(b, nv, 256, generator=g).requires_grad_(True)
    mask = torch.rand(b, nv, generator=g) < 0.1
    gout = torch.randn(b, nq, 256, generator=g)
    out = mod(query, refp, value, shapes, lsi, mask)
    grads = torch.autograd.grad(out, [query, value, mod.sampling_offsets.weight, mod.value_proj.weight], gout)
    arrs = dict(shapes_json=np.array(shapes_json), aliases_json=np.array(aliases_json), seed=np.int64(seed))
    for i, (n, t) in enumerate(zip(("out", "grad_query", "grad_value", "grad_sampling_offsets_weight", "grad_value_proj_weight"),
                                   (out,) + tuple(grads))):
        _store_sampled(arrs, n, t, i)
    np.savez_compressed(os.path.join(OUT, name), **arrs)


DROPIN = dict(embed_dim=256, d_ffn=512, n_heads=8, n_levels=4, n_points=4, num_layers=3, num_classes=17,
              level_filter_ratio=(0.4, 0.8, 1.0, 1.0), layer_filter_ratio=(1.0, 0.7, 0.4), topk_sa=100,
              max_num_embedding=100, num_proposals=50)


def make_dropin_encoder(name, image_sizes, seed=4, input_seed=9):
    """SalienceTransformer.forward lines 106-183 at C = 256 with a 3-layer encoder: what its salience filter hands to the
    encoder (the selection, scores and token budgets) and the encoder memory."""
    import json
    tr = ref_import.build_transformer(seed=0, **DROPIN)
    shapes_json, aliases_json = _load_deterministic(tr, seed)
    feats, masks, pos = orc.synthetic_inputs(image_sizes, (480, 640), DROPIN["embed_dim"], seed=input_seed)
    mem, kw = ref_import.run_encoder_half(tr, feats, masks, pos)
    arrs = dict(shapes_json=np.array(shapes_json), aliases_json=np.array(aliases_json), seed=np.int64(seed),
                geo_json=np.array(json.dumps(DROPIN)), encoder_kwargs=np.array(sorted(kw)),
                valid_ratios=np_(kw["valid_ratios"]), foreground_score=np_(kw["foreground_score"]),
                focus_token_nums=np_(kw["focus_token_nums"]), selected_inds=np_(kw["foreground_inds"][0]).astype(np.int16),
                layer_num_query=np.array([x.shape[1] for x in kw["foreground_inds"]]))
    _store_sampled(arrs, "memory", mem, 0)
    np.savez_compressed(os.path.join(OUT, name), **arrs)


DECODER = dict(embed_dim=256, d_ffn=512, n_heads=8, num_layers=2, num_classes=17, level_filter_ratio=(0.4, 0.8, 1.0, 1.0),
               layer_filter_ratio=(1.0, 0.5), topk_sa=100, max_num_embedding=100, num_proposals=300, dec_layers=3)


def _decoder_reference(neck=None, seed=2):
    ref = ref_import.load()
    st, c = ref.st, DECODER["embed_dim"]
    relu = torch.nn.ReLU(inplace=True)
    enc = st.SalienceTransformerEncoder(st.SalienceTransformerEncoderLayer(c, DECODER["d_ffn"], 0.0, DECODER["n_heads"], relu, 4, 4,
                                                                           topk_sa=DECODER["topk_sa"]),
                                        DECODER["num_layers"], max_num_embedding=DECODER["max_num_embedding"])
    dec = st.SalienceTransformerDecoder(st.SalienceTransformerDecoderLayer(c, DECODER["d_ffn"], DECODER["n_heads"], 0.0, relu, 4, 4),
                                        DECODER["dec_layers"], DECODER["num_classes"])
    tr = st.SalienceTransformer(enc, None, dec, DECODER["num_classes"], 4, DECODER["num_proposals"],
                                DECODER["level_filter_ratio"], DECODER["layer_filter_ratio"])
    shapes_json, aliases_json = _load_deterministic(tr, seed)
    tr.neck = neck
    return tr.eval(), shapes_json, aliases_json


def make_decoder_half(name, image_sizes, seed=2, input_seed=13):
    """The whole SalienceTransformer.forward (filter, encoder, two-stage selection, decoder; :97-239) and the decoder alone
    (:498-674) on the proposals of that forward with value = the flattened input features, with and without 20 denoising
    queries behind an attention mask."""
    import json
    tr, shapes_json, aliases_json = _decoder_reference(seed=seed)
    feats, masks, pos = orc.synthetic_inputs(image_sizes, (480, 640), DECODER["embed_dim"], seed=input_seed)
    cap = {}
    dec_fwd = tr.decoder.forward

    def spy(**kw):
        cap.update(kw)
        return dec_fwd(**kw)

    tr.decoder.forward = spy
    with torch.no_grad():
        want = tr(feats, masks, pos, None, None, None)
    del tr.decoder.forward
    arrs = dict(shapes_json=np.array(shapes_json), aliases_json=np.array(aliases_json), seed=np.int64(seed),
                geo_json=np.array(json.dumps(DECODER)), decoder_kwargs=np.array(sorted(cap)),
                valid_ratios=np_(cap["valid_ratios"]), reference_points=np_(cap["reference_points"]),
                enc_outputs_coord=np_(want[3]))
    for i, (n, t) in enumerate(zip(("outputs_classes", "outputs_coords", "enc_outputs_class"), want[:3])):
        _store_sampled(arrs, n, t, i)
    _store_sampled(arrs, "salience", torch.cat([s.flatten(1) for s in want[4]], 1), 3)
    # the decoder alone
    kw = dict(cap, value=orc.flatten_levels(feats))
    b, nq = kw["query"].shape[:2]
    g = torch.Generator().manual_seed(4)
    dn_q = torch.randn(b, 20, DECODER["embed_dim"], generator=g)
    dn_b = torch.rand(b, 20, 4, generator=g) * 0.5 + 0.25
    mask = torch.zeros(nq + 20, nq + 20, dtype=torch.bool)
    mask[20:, :20] = True
    kw_dn = dict(kw, query=torch.cat([dn_q, kw["query"]], 1), reference_points=torch.cat([dn_b, kw["reference_points"]], 1),
                 attn_mask=mask)
    with torch.no_grad():
        for tag, k in (("dec", kw), ("dec_dn", kw_dn)):
            cls, box = tr.decoder(**k)
            _store_sampled(arrs, tag + "_classes", cls, 4)
            _store_sampled(arrs, tag + "_coords", box, 5)
    np.savez_compressed(os.path.join(OUT, name), **arrs)


NMS_CASES = (([(60, 80), (30, 40), (15, 20), (8, 10)], 1200), ([(100, 168), (50, 84), (25, 42), (13, 21)], 3600),
             ([(20, 20), (10, 10)], 450))


def make_nms_topk(name="decoder_nms_topk.npz"):
    """SalienceTransformer.nms_on_topk_index (:249-295, torchvision batched_nms) on seeded distinct scores, three geometries."""
    tr, _, _ = _decoder_reference()
    tr.two_stage_num_proposals = 900
    g = torch.Generator().manual_seed(0)
    arrs = {}
    for i, (shapes, k) in enumerate(NMS_CASES):
        st = torch.tensor(shapes)
        lsi = torch.cat([st.new_zeros(1), st.prod(1).cumsum(0)[:-1]])
        scores = torch.rand(2, int(st.prod(1).sum()), generator=g)
        topk_scores, topk_index = torch.topk(scores, k, dim=1)
        arrs[f"kept{i}"] = np_(tr.nms_on_topk_index(topk_scores, topk_index, st, lsi, iou_threshold=0.3)).astype(np.int16)
        arrs[f"shapes{i}"], arrs[f"k{i}"] = np.array(shapes), np.int64(k)
    np.savez_compressed(os.path.join(OUT, name), **arrs)


def make_decoder_neck(name="decoder_neck.npz", seed=2, input_seed=13):
    """SalienceTransformer.forward with a neck (oracle.TopDownNeck) between encoder and decoder (:185-192): the memory that
    leaves the neck, as the decoder's `value` input."""
    import json
    tr, shapes_json, aliases_json = _decoder_reference(neck=orc.TopDownNeck(DECODER["embed_dim"], 4), seed=seed)
    feats, masks, pos = orc.synthetic_inputs([(480, 640), (480, 640)], (480, 640), DECODER["embed_dim"], seed=input_seed)
    cap = {}

    def spy(**kw):
        cap["value"] = kw["value"]
        raise _Stop()

    tr.decoder.forward = spy
    try:
        with torch.no_grad():
            tr(feats, masks, pos, None, None, None)
    except _Stop:
        pass
    arrs = dict(shapes_json=np.array(shapes_json), aliases_json=np.array(aliases_json), seed=np.int64(seed),
                geo_json=np.array(json.dumps(DECODER)))
    _store_sampled(arrs, "value", cap["value"], 0)
    np.savez_compressed(os.path.join(OUT, name), **arrs)


FIXTURES = {
    "msda_core": lambda: (make_msda_core("msda_core_a.npz", b=2, shapes=[(10, 12), (5, 6), (3, 3), (2, 2)], m=4, d=32, nq=40,
                                         p=4, seed=1),
                          make_msda_core("msda_core_b.npz", b=1, shapes=[(7, 5), (4, 3)], m=2, d=16, nq=23, p=2, seed=2)),
    "msda_module": make_msda_module,
    "encoder_tiny": lambda: (make_encoder_tiny("encoder_tiny_even.npz", [(96, 128), (96, 128)], (96, 128), seed=5),
                             make_encoder_tiny("encoder_tiny_ragged.npz", [(96, 128), (72, 90)], (96, 128), seed=6)),
    "encoder_c256": make_encoder_c256,
    "encoder_tiny_grads": lambda: make_encoder_tiny_grads("encoder_tiny_even_grads.npz", [(96, 128), (96, 128)], (96, 128),
                                                          seed=5),
    "salience_criterion": make_salience_criterion,
    "dropin": lambda: (make_dropin_msda_operator(),
                       make_dropin_encoder("dropin_encoder_even.npz", [(480, 640), (480, 640)]),
                       make_dropin_encoder("dropin_encoder_ragged.npz", [(480, 640), (400, 500)])),
    "decoder": lambda: (make_decoder_half("decoder_half_even.npz", [(480, 640), (480, 640)]),
                        make_decoder_half("decoder_half_ragged.npz", [(480, 640), (400, 500)]),
                        make_nms_topk(), make_decoder_neck()),
}


def main():
    """python oracle/make_golden.py [fixture ...]  (default: all of FIXTURES)"""
    os.makedirs(OUT, exist_ok=True)
    for name in sys.argv[1:] or FIXTURES:
        FIXTURES[name]()
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)) // 1024, "KiB")
    print("torch", torch.__version__)


if __name__ == "__main__":
    main()
