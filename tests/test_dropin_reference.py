"""Drop-in tests against outputs of the UNMODIFIED reference (row (b) of SURVEY.md section 8).

The fixtures (tests/golden/dropin_*.npz, made by ``oracle/make_golden.py dropin``) hold what the reference's own modules
computed on its pure-PyTorch path, with weights regenerated from a seed (``oracle.golden_state_dict``) and seeded inputs.
Three levels of "drops in unchanged":

1. operator: the reference's ``MultiScaleDeformableAttention`` arithmetic (the oracle restatement, pinned by
   tests/test_oracle_golden.py) calling this package's ``_C.ms_deform_attn_forward/backward`` exactly as the reference's
   autograd Function does (models/bricks/ms_deform_attn.py:35-84,361-372), forward and backward;
2. module: this package's ``SalienceTransformerEncoder`` / ``SalienceTransformerEncoderLayer`` built as a reference config
   would (configs/salience_detr/salience_detr_resnet50_800_1333.py:44-62), loaded with the reference encoder's state_dict
   and called with the keyword arguments the reference's salience filter hands to its encoder (:106-183);
3. transformer: this package's ``SalienceTransformer.forward_encoder`` with the reference's ``state_dict``.
"""
import json
import os

import numpy as np
import pytest
import torch
from torch.autograd.function import once_differentiable

from oracle import oracle as orc

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

GEO = dict(embed_dim=256, d_ffn=512, n_heads=8, n_levels=4, n_points=4, num_layers=3, num_classes=17,
           level_filter_ratio=(0.4, 0.8, 1.0, 1.0), layer_filter_ratio=(1.0, 0.7, 0.4), topk_sa=100,
           max_num_embedding=100, num_proposals=50)


@pytest.fixture(scope="module")
def pkg():
    import salience_detr_b200 as p
    p.cabi.lib()
    return p


@pytest.fixture(autouse=True)
def _fp32_matmul(pkg):
    prev, mode = torch.backends.cuda.matmul.allow_tf32, pkg.gemm.MODE
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32 = prev
    pkg.gemm.MODE = mode


def _golden(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


def _weights(z):
    return orc.golden_state_dict(str(z["shapes_json"]), int(z["seed"]), str(z["aliases_json"]))


def _check_sampled(z, name, got, tol, seed, relative=False):
    want = torch.from_numpy(z[name + "_sample"])
    scale = max(1.0, float(z[name + "_absmax"])) if relative else 1.0
    assert abs(got.abs().max().item() - float(z[name + "_absmax"])) < tol * scale, name
    err = (orc.sampled(got, want.numel(), seed) - want).abs().max().item()
    assert err < tol * scale, (name, err)


def _inputs(ragged=False):
    sizes = [(480, 640), (400, 500)] if ragged else [(480, 640), (480, 640)]
    feats, masks, pos = orc.synthetic_inputs(sizes, (480, 640), GEO["embed_dim"], seed=9)
    return [f.to(DEV) for f in feats], [m.to(DEV) for m in masks], [p.to(DEV) for p in pos]


class _ReferenceFunction(torch.autograd.Function):
    """The reference's MultiScaleDeformableAttnFunction calls into ``_C`` (ms_deform_attn.py:35-84); ``_C`` is this
    package's."""

    @staticmethod
    def forward(ctx, value, shapes, lsi, loc, attn, im2col_step, C):
        ctx.im2col_step, ctx.C = im2col_step, C
        out = C.ms_deform_attn_forward(value, shapes, lsi, loc, attn, ctx.im2col_step)
        ctx.save_for_backward(value, shapes, lsi, loc, attn)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        value, shapes, lsi, loc, attn = ctx.saved_tensors
        gv, gl, ga = ctx.C.ms_deform_attn_backward(value, shapes, lsi, loc, attn, grad_output.contiguous(), ctx.im2col_step)
        return gv, None, None, gl, ga, None, None


def test_operator_C_dropin_forward_backward(pkg):
    """The reference module's arithmetic with `_C.ms_deform_attn_forward/backward` of THIS package (ms_deform_attn.py:361-370)
    against the reference module on its pure-PyTorch path."""
    z = _golden("dropin_msda_operator.npz")
    sd = {k: v.to(DEV) for k, v in _weights(z).items()}
    for k in ("sampling_offsets.weight", "value_proj.weight"):
        sd[k].requires_grad_(True)
    shapes = torch.tensor([(30, 40), (15, 20), (8, 10), (4, 5)], device=DEV)
    lsi = torch.cat([shapes.new_zeros(1), shapes.prod(1).cumsum(0)[:-1]])
    nv, b, nq = int(shapes.prod(1).sum()), 2, 333
    g = torch.Generator().manual_seed(1)
    query = torch.randn(b, nq, 256, generator=g).to(DEV).requires_grad_(True)
    refp = torch.rand(b, nq, 4, 2, generator=g).to(DEV)
    value = torch.randn(b, nv, 256, generator=g).to(DEV).requires_grad_(True)
    mask = (torch.rand(b, nv, generator=g) < 0.1).to(DEV)
    gout = torch.randn(b, nq, 256, generator=g).to(DEV)

    def core(v, s, l, loc, w):
        return _ReferenceFunction.apply(v.contiguous(), s, l, loc.contiguous(), w.contiguous(), 64, pkg._C)

    n0 = pkg.cabi.launch_count()
    out = orc.msda_module(sd, "", query, refp, value, shapes, lsi, mask, 8, 4, 4, core=core)
    grads = torch.autograd.grad(out, [query, value, sd["sampling_offsets.weight"], sd["value_proj.weight"]], gout)
    assert pkg.cabi.launch_count() >= n0 + 2  # our forward and backward kernels really ran
    _check_sampled(z, "out", out.detach(), 1e-4, 0)
    for i, (n, t) in enumerate(zip(("grad_query", "grad_value", "grad_sampling_offsets_weight", "grad_value_proj_weight"),
                                   grads)):
        _check_sampled(z, n, t, 1e-3, i + 1, relative=True)


def _encoder_golden(ragged):
    z = _golden("dropin_encoder_ragged.npz" if ragged else "dropin_encoder_even.npz")
    assert json.loads(str(z["geo_json"])) == {k: list(v) if isinstance(v, tuple) else v for k, v in GEO.items()}
    return z, {k: v.to(DEV) for k, v in _weights(z).items()}


def _reference_encoder_kwargs(z, feats, masks, pos, level_embeds):
    """What the reference's filter hands to its encoder (salience_transformer.py:171-183): the selection, scores and budgets
    from the fixture, the token layouts of the inputs."""
    from salience_detr_b200 import flatten_levels
    shapes = torch.tensor([list(m.shape[-2:]) for m in masks], device=DEV)
    inds = torch.from_numpy(z["selected_inds"].astype(np.int64)).to(DEV)
    kw = dict(query=flatten_levels(feats),
              query_pos=flatten_levels([p + e.view(1, -1, 1, 1) for p, e in zip(pos, level_embeds)]),
              query_key_padding_mask=flatten_levels(masks), spatial_shapes=shapes,
              level_start_index=torch.cat([shapes.new_zeros(1), shapes.prod(1).cumsum(0)[:-1]]),
              valid_ratios=torch.from_numpy(z["valid_ratios"]).to(DEV),
              foreground_score=torch.from_numpy(z["foreground_score"]).to(DEV),
              focus_token_nums=torch.from_numpy(z["focus_token_nums"]).to(DEV),
              foreground_inds=[inds[:, :int(n)] for n in z["layer_num_query"]], multi_level_masks=masks)
    assert sorted(kw) == z["encoder_kwargs"].tolist()
    return kw


@pytest.mark.parametrize("ragged", [False, True])
@pytest.mark.parametrize("mode", ["fp32", "auto"])
def test_reference_transformer_with_our_encoder(pkg, ragged, mode):
    """This package's encoder classes, built and loaded as a reference config does, on the reference filter's selection:
    both sides process identical tokens, so the memory agrees with the reference's within 1e-3."""
    z, sd = _encoder_golden(ragged)
    feats, masks, pos = _inputs(ragged)
    layer = pkg.SalienceTransformerEncoderLayer(GEO["embed_dim"], GEO["d_ffn"], 0.0, GEO["n_heads"],
                                                torch.nn.ReLU(inplace=True), GEO["n_levels"], GEO["n_points"],
                                                topk_sa=GEO["topk_sa"])
    enc = pkg.SalienceTransformerEncoder(layer, GEO["num_layers"], max_num_embedding=GEO["max_num_embedding"]).to(DEV)
    enc_sd = {k[len("encoder."):]: v for k, v in sd.items() if k.startswith("encoder.")}
    res = enc.load_state_dict(enc_sd, strict=False)  # same parameter names as the reference encoder;
    assert not res.missing_keys and set(res.unexpected_keys) == {"enhance_mcsp.weight", "enhance_mcsp.bias"}  # (:79 alias)
    head = torch.nn.Linear(GEO["embed_dim"], GEO["num_classes"]).to(DEV)  # the reference transformer's encoder_class_head,
    head.load_state_dict({"weight": sd["encoder_class_head.weight"], "bias": sd["encoder_class_head.bias"]})
    enc.enhance_mcsp = head                                               # injected into the encoder by its constructor (:79)
    kw = _reference_encoder_kwargs(z, feats, masks, pos, sd["level_embeds"])
    pkg.gemm.MODE = mode
    n0 = pkg.cabi.launch_count()
    with torch.no_grad():
        got = enc(**kw)
    assert pkg.cabi.launch_count() > n0 + 10
    _check_sampled(z, "memory", got, 1e-3, 0)


@pytest.mark.parametrize("ragged", [False, True])
def test_our_transformer_with_reference_state_dict(pkg, ragged):
    """This package's SalienceTransformer (fused filter + encoder) loaded with the reference's state_dict."""
    z, sd = _encoder_golden(ragged)
    feats, masks, pos = _inputs(ragged)
    layer = pkg.SalienceTransformerEncoderLayer(GEO["embed_dim"], GEO["d_ffn"], 0.0, GEO["n_heads"],
                                                torch.nn.ReLU(inplace=True), GEO["n_levels"], GEO["n_points"],
                                                topk_sa=GEO["topk_sa"])
    enc = pkg.SalienceTransformerEncoder(layer, GEO["num_layers"], max_num_embedding=GEO["max_num_embedding"])
    ours = pkg.SalienceTransformer(enc, None, None, GEO["num_classes"], GEO["n_levels"], GEO["num_proposals"],
                                   GEO["level_filter_ratio"], GEO["layer_filter_ratio"]).to(DEV).eval()
    res = ours.load_state_dict(sd, strict=False)
    assert set(res.missing_keys) <= {"level_filter_ratio", "layer_filter_ratio"}  # buffers of the config, not weights
    assert all(k.startswith(("decoder.", "tgt_embed.", "encoder_bbox_head.")) for k in res.unexpected_keys)
    kw = _reference_encoder_kwargs(z, feats, masks, pos, ours.level_embeds)
    ref_inds, ref_fg = kw["foreground_inds"][0], kw["foreground_score"]
    for mode, tol_score, swaps in (("fp32", 3e-5, 8), ("auto", 3e-4, 40)):
        pkg.gemm.MODE = mode
        with torch.no_grad():
            mem, aux = ours.forward_encoder(feats, masks, pos)
            plan = aux["plan"]
            assert plan.layer_num_query == [x.shape[1] for x in kw["foreground_inds"]]
            assert torch.equal(plan.focus_token_nums.long().cpu(), kw["focus_token_nums"].long().cpu())
            assert (aux["foreground_score"] - ref_fg).abs().max() < tol_score
            for i in range(2):
                n = int(plan.focus_host[i])
                a, w = set(aux["selected_inds"][i, :n].tolist()), set(ref_inds[i, :n].tolist())
                assert len(a & w) >= n - swaps, (mode, n - len(a & w))
            inj = ours.encoder(query=kw["query"], query_pos=kw["query_pos"], query_key_padding_mask=plan.mask_flat,
                               spatial_shapes=plan.spatial_shapes, level_start_index=plan.level_start_index,
                               valid_ratios=plan.valid_ratios, foreground_score=ref_fg,
                               focus_token_nums=plan.focus_token_nums,
                               foreground_inds=kw["foreground_inds"], multi_level_masks=masks)
        _check_sampled(z, "memory", inj, 1e-3, 0)
        if torch.equal(aux["selected_inds"], ref_inds):
            _check_sampled(z, "memory", mem, 1e-3, 0)
