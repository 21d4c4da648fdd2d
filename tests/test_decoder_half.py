"""Decoder half (SURVEY.md 8(f)-1) against outputs of the UNMODIFIED reference (tests/golden/decoder_*.npz, made by
``oracle/make_golden.py decoder`` with weights regenerated from a seed, see tests/test_dropin_reference.py): two-stage
proposal selection (salience_transformer.py:194-212, 249-295) and the decoder (:498-674) with 4-d reference boxes through
the fused sampling kernel."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import oracle as orc

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

GEO = dict(embed_dim=256, d_ffn=512, n_heads=8, n_levels=4, n_points=4, num_layers=2, num_classes=17,
           level_filter_ratio=(0.4, 0.8, 1.0, 1.0), layer_filter_ratio=(1.0, 0.5), topk_sa=100, max_num_embedding=100,
           num_proposals=300)
DEC_LAYERS = 3


class _Stop(Exception):
    pass


@pytest.fixture(scope="module")
def pkg():
    import salience_detr_b200 as p
    p.cabi.lib()
    return p


@pytest.fixture(autouse=True)
def _fp32(pkg):
    prev, mode = torch.backends.cuda.matmul.allow_tf32, pkg.gemm.MODE
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32 = prev
    pkg.gemm.MODE = mode


def _golden(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


def _sampled(z, name, got, seed):
    """-> (fixture's samples of `name`, `got` at the same positions)"""
    want = torch.from_numpy(z[name + "_sample"])
    return want, orc.sampled(got, want.numel(), seed)


def _ours(pkg, z):
    """This package's transformer, encoder and decoder, loaded with the reference model's full state_dict."""
    geo = json.loads(str(z["geo_json"]))
    assert geo["dec_layers"] == DEC_LAYERS and all(geo[k] == (list(v) if isinstance(v, tuple) else v)
                                                   for k, v in GEO.items() if k in geo)
    relu = torch.nn.ReLU(inplace=True)
    enc = pkg.SalienceTransformerEncoder(pkg.SalienceTransformerEncoderLayer(GEO["embed_dim"], GEO["d_ffn"], 0.0, GEO["n_heads"], relu,
                                                                            4, 4, topk_sa=GEO["topk_sa"]), GEO["num_layers"],
                                         GEO["max_num_embedding"])
    dec = pkg.SalienceTransformerDecoder(pkg.SalienceTransformerDecoderLayer(GEO["embed_dim"], GEO["d_ffn"], GEO["n_heads"], 0.0, relu,
                                                                            4, 4), DEC_LAYERS, GEO["num_classes"])
    ours = pkg.SalienceTransformer(enc, None, dec, GEO["num_classes"], 4, GEO["num_proposals"], GEO["level_filter_ratio"],
                                   GEO["layer_filter_ratio"])
    sd = orc.golden_state_dict(str(z["shapes_json"]), int(z["seed"]), str(z["aliases_json"]))
    sd.update({k: ours.state_dict()[k] for k in ("level_filter_ratio", "layer_filter_ratio")})  # config buffers
    ours.load_state_dict(sd, strict=True)  # every reference key, decoder half included
    return ours.to(DEV).eval()


def _inputs(ragged):
    sizes = [(480, 640), (400, 500)] if ragged else [(480, 640), (480, 640)]
    feats, masks, pos = orc.synthetic_inputs(sizes, (480, 640), GEO["embed_dim"], seed=13)
    return [f.to(DEV) for f in feats], [m.to(DEV) for m in masks], [p.to(DEV) for p in pos]


def test_nms_on_topk_index_matches_torchvision(pkg):
    """sdetr_nms_topk_index vs the reference's own nms_on_topk_index (torchvision.ops.batched_nms), index for index."""
    z = _golden("decoder_nms_topk.npz")
    g = torch.Generator().manual_seed(0)
    for i in range(3):
        shapes, k = [tuple(s) for s in z[f"shapes{i}"].tolist()], int(z[f"k{i}"])
        st = torch.tensor(shapes, device=DEV)
        lsi = torch.cat([st.new_zeros(1), st.prod(1).cumsum(0)[:-1]])
        nv = int(st.prod(1).sum())
        scores = torch.rand(2, nv, generator=g).to(DEV)  # distinct with probability 1: the order is unambiguous
        topk_scores, topk_index = torch.topk(scores, k, dim=1)
        want = torch.from_numpy(z[f"kept{i}"].astype(np.int64)).to(DEV)
        kept, count, flag = pkg.cabi.nms_topk_index(topk_index.contiguous(), shapes, 0.3)
        n = want.shape[1]
        assert int(count.min()) >= n and torch.equal(kept[:, :n], want)
        for b in range(2):  # the verdicts are a valid greedy NMS: no two kept 4-neighbours, every suppressed one has a kept better neighbour
            assert int(flag[b].sum()) == int(count[b])
    ours = pkg.SalienceTransformer(pkg.SalienceTransformerEncoder(pkg.SalienceTransformerEncoderLayer(64, 64, 0.0, 2), 1, 40), None, None,
                                   two_stage_num_proposals=900)
    assert torch.equal(ours.nms_on_topk_index(topk_scores, topk_index, st, lsi), want)


@pytest.mark.parametrize("ragged", [False, True])
def test_decoder_on_reference_inputs(pkg, ragged):
    """The decoder alone on the reference's own proposals, with the inputs the reference decoder was given: class logits and
    boxes of every layer within 1e-3 / 1e-4, in the strict fp32-GEMM mode and in the default tensor-core mode."""
    z = _golden("decoder_half_ragged.npz" if ragged else "decoder_half_even.npz")
    ours = _ours(pkg, z)
    feats, masks, pos = _inputs(ragged)
    plan = ours.make_plan(masks)
    b = feats[0].shape[0]
    kw = dict(query=ours.tgt_embed.weight.expand(b, -1, -1), value=pkg.flatten_levels(feats), key_padding_mask=plan.mask_flat,
              reference_points=torch.from_numpy(z["reference_points"]).to(DEV), spatial_shapes=plan.spatial_shapes,
              level_start_index=plan.level_start_index, valid_ratios=torch.from_numpy(z["valid_ratios"]).to(DEV), attn_mask=None)
    assert sorted(kw) == z["decoder_kwargs"].tolist()
    for mode in ("fp32", "auto"):
        pkg.gemm.MODE = mode
        n0 = pkg.cabi.launch_count()
        with torch.no_grad():
            cls, box = ours.decoder(**kw)
        assert pkg.cabi.launch_count() > n0 + 3 * DEC_LAYERS
        assert cls.shape == (DEC_LAYERS, b, GEO["num_proposals"], GEO["num_classes"]) and box.shape == cls.shape[:3] + (4,)
        w, a = _sampled(z, "dec_classes", cls, 4)
        assert (a - w).abs().max() < 1e-3 and abs(cls.abs().max().item() - float(z["dec_classes_absmax"])) < 1e-3, mode
        w, a = _sampled(z, "dec_coords", box, 5)
        assert (a - w).abs().max() < 1e-4, mode
    # denoising queries + attention mask pass through like in the reference (salience_transformer.py:218-221)
    nq = kw["query"].shape[1]
    g = torch.Generator().manual_seed(4)
    dn_q = torch.randn(b, 20, GEO["embed_dim"], generator=g).to(DEV)
    dn_b = torch.rand(b, 20, 4, generator=g).to(DEV) * 0.5 + 0.25
    mask = torch.zeros(nq + 20, nq + 20, dtype=torch.bool, device=DEV)
    mask[20:, :20] = True
    kw2 = dict(kw, query=torch.cat([dn_q, kw["query"]], 1), reference_points=torch.cat([dn_b, kw["reference_points"]], 1), attn_mask=mask)
    with torch.no_grad():
        pkg.gemm.MODE = "auto"
        g2 = ours.decoder(**kw2)
    (wc, ac), (wb, ab) = _sampled(z, "dec_dn_classes", g2[0], 4), _sampled(z, "dec_dn_coords", g2[1], 5)
    assert (ac - wc).abs().max() < 1e-3 and (ab - wb).abs().max() < 1e-4


@pytest.mark.parametrize("ragged", [False, True])
def test_full_transformer_forward_vs_reference(pkg, ragged):
    """Whole ``SalienceTransformer.forward`` (filter + encoder + two-stage selection + decoder), reference call signature and
    5-tuple of outputs.  Encoder memories differ by round-off, so near-tied proposals may swap: the proposal SETS must agree
    except for a few entries, and every query whose proposal agrees in position must agree in its outputs."""
    z = _golden("decoder_half_ragged.npz" if ragged else "decoder_half_even.npz")
    ours = _ours(pkg, z)
    feats, masks, pos = _inputs(ragged)
    with torch.no_grad():
        pkg.gemm.MODE = "fp32"
        got = ours(feats, masks, pos, None, None, None)
    want_coord = torch.from_numpy(z["enc_outputs_coord"]).to(DEV)
    assert len(got) == 5 and got[0].shape == (DEC_LAYERS,) + got[2].shape and got[3].shape == want_coord.shape
    assert [tuple(a.shape) for a in got[4]] == [(feats[0].shape[0], 1) + tuple(m.shape[-2:]) for m in masks]
    w, a = _sampled(z, "salience", torch.cat([s.flatten(1) for s in got[4]], 1), 3)  # salience score maps
    assert (a - w).abs().max() < 1e-4
    same = ((got[3] - want_coord).abs().amax(-1) < 1e-4)          # proposals equal position by position
    assert same.float().mean() > 0.9
    w, a = _sampled(z, "enc_outputs_class", got[2], 2)            # their class logits
    at_same = orc.sampled(same[..., None].expand_as(got[2]), w.numel(), 2)
    assert (a - w).abs()[at_same].max() < 1e-3
    if bool(same.all()):  # identical proposal lists: the decoder outputs must agree everywhere
        (wc, ac), (wb, ab) = _sampled(z, "outputs_classes", got[0], 0), _sampled(z, "outputs_coords", got[1], 1)
        assert (ac - wc).abs().max() < 2e-3 and (ab - wb).abs().max() < 2e-4


def test_neck_handoff_with_reference_repvgg(pkg):
    """SURVEY.md 8(f)-3: the encoder memory is handed to the neck in per-level NCHW maps and comes back as tokens
    (salience_transformer.py:185-192).  Layout kernels: exact round trip; then a neck (oracle.TopDownNeck, a stand-in for the
    RepVGG neck of models/necks/repnet.py: any module taking and returning {level: NCHW}) plugged into OUR transformer against
    the reference transformer with the same neck and weights: the memory that leaves the neck (captured at the decoder's
    `value` input) within 2e-3."""
    shapes = [(60, 80), (30, 40), (15, 20), (8, 10)]
    g = torch.Generator().manual_seed(1)
    tok = torch.randn(2, sum(h * w for h, w in shapes), 96, generator=g).to(DEV)
    maps = pkg.cabi.tokens_to_maps(tok, shapes)
    want = [t.transpose(1, 2).reshape(2, 96, h, w) for t, (h, w) in zip(tok.split([h * w for h, w in shapes], 1), shapes)]
    assert all(torch.equal(a, b) for a, b in zip(maps, want))
    assert torch.equal(pkg.cabi.maps_to_tokens(maps), tok)

    z = _golden("decoder_neck.npz")
    ours = _ours(pkg, z)
    ours.neck = orc.TopDownNeck(GEO["embed_dim"], 4).to(DEV).eval()
    feats, masks, pos = _inputs(False)
    cap = {}

    def spy(**kw):
        cap["value"] = kw["value"]
        raise _Stop()

    ours.decoder.forward = spy
    try:
        with torch.no_grad():
            pkg.gemm.MODE = "fp32"
            ours(feats, masks, pos, None, None, None)
    except _Stop:
        pass
    finally:
        del ours.decoder.forward
    scale = max(1.0, float(z["value_absmax"]))
    assert cap["value"].shape == (2, sum(m.shape[-2] * m.shape[-1] for m in masks), GEO["embed_dim"])
    w, a = _sampled(z, "value", cap["value"], 0)
    assert (a - w).abs().max() < 2e-3 * scale and abs(cap["value"].abs().max().item() - float(z["value_absmax"])) < 2e-3 * scale
