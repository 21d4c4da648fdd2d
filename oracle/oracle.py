"""TEST INFRASTRUCTURE ONLY -- CPU oracle for the Salience-DETR encoder hot path.

Two layers:

* ``lib()`` / the ``c_*`` wrappers: ctypes bindings of ``oracle/sdetr_oracle.c`` (plain-C restatement of the
  MSDA core, selection, gather/scatter, ...; see the header of that file for reference line numbers).
* the ``*_torch`` / module-level functions: a functional torch-CPU restatement of the reference's
  PyTorch path (what the reference actually executes on a CPU), driven by a ``state_dict`` that uses
  the reference's own parameter names.  This is also the "reference arm" timed by
  ``bench.py --impl reference`` and the ``cpu_baseline`` (kind "port").

Only tests/, ``__graft_entry__.smoke()`` and bench.py's CPU-baseline legs may import this module.
The oracle is pinned against outputs of the unmodified reference (``tests/golden/*.npz`` made by
``oracle/make_golden.py``; checked in ``tests/test_oracle_golden.py``) -- the reference itself ships
no tests or golden vectors.

All citations are relative to the reference root (xiuqhou/Salience-DETR).
"""
from __future__ import annotations

import ctypes
import math
import os
import subprocess
from typing import Dict, List, Sequence

import numpy as np
import torch
import torch.nn.functional as F

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def build(force: bool = False) -> str:
    """Compile oracle/sdetr_oracle.c -> oracle/liboracle.so (gcc; OpenMP when available)."""
    so = os.path.join(_HERE, "liboracle.so")
    src = os.path.join(_HERE, "sdetr_oracle.c")
    if not force and os.path.exists(so) and os.path.getmtime(so) >= os.path.getmtime(src):
        return so
    gcc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    base = [gcc, "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-o", so, src, "-lm"]
    try:
        subprocess.run(base[:1] + ["-fopenmp"] + base[1:], check=True, capture_output=True)
    except (subprocess.CalledProcessError, FileNotFoundError):
        subprocess.run(base, check=True, capture_output=True)
    return so


def lib():
    global _LIB
    if _LIB is None:
        _LIB = ctypes.CDLL(build())
    return _LIB


_KEEP: list = []  # tensors referenced by raw pointers of the ctypes call being assembled


def _p(t: torch.Tensor):
    """Raw pointer of a CPU tensor; the tensor is kept alive until the next _done()."""
    assert t.is_contiguous() and t.device.type == "cpu"
    _KEEP.append(t)
    return ctypes.c_void_p(t.data_ptr())


def _done():
    _KEEP.clear()


# --------------------------------------------------------------------------------------------------
# C oracle wrappers
# --------------------------------------------------------------------------------------------------
def c_msda_forward(value, shapes, lsi, loc, attn):
    """ms_deform_attn_forward semantics (.cu:12-72): value (b,Nv,M,D) f32 -> (b,Nq,M*D)."""
    b, nv, m, d = value.shape
    _, nq, _, l, p, _ = loc.shape
    out = torch.empty(b, nq, m * d, dtype=torch.float32)
    lib().oracle_msda_forward(_p(value.contiguous()), _p(shapes.contiguous()), _p(lsi.contiguous()),
                              _p(loc.contiguous()), _p(attn.contiguous()), _p(out), b, nv, m, d, l, nq, p)
    _done()
    return out


def c_msda_backward(value, shapes, lsi, loc, attn, grad_out):
    """ms_deform_attn_backward semantics (.cu:75-145) -> (grad_value, grad_loc, grad_attn)."""
    b, nv, m, d = value.shape
    _, nq, _, l, p, _ = loc.shape
    gv = torch.zeros_like(value)
    gl = torch.zeros_like(loc)
    ga = torch.zeros_like(attn)
    lib().oracle_msda_backward(_p(value.contiguous()), _p(shapes.contiguous()), _p(lsi.contiguous()),
                               _p(loc.contiguous()), _p(attn.contiguous()), _p(grad_out.contiguous()),
                               _p(gv), _p(gl), _p(ga), b, nv, m, d, l, nq, p)
    _done()
    return gv, gl, ga


def c_salience_select(raw_score, mask, lsi, hw, k: Sequence[int]):
    """(b,Nv) scores + mask -> selected_inds (b,K) i64, selected_score (b,K), foreground_score (b,Nv)."""
    b, nv = raw_score.shape
    levels = len(k)
    kk = torch.tensor(list(k), dtype=torch.int32)
    K = int(kk.sum())
    inds = torch.empty(b, K, dtype=torch.int64)
    sc = torch.empty(b, K, dtype=torch.float32)
    fg = torch.empty(b, nv, dtype=torch.float32)
    lib().oracle_salience_select(_p(raw_score.contiguous()), _p(mask.to(torch.uint8).contiguous()),
                                 _p(lsi.contiguous()), _p(hw.contiguous()), _p(kk), b, nv, levels,
                                 _p(inds), _p(sc), _p(fg))
    _done()
    return inds, sc, fg


def c_token_budgets(mask, lsi, hw, level_ratio, layer_ratio):
    b, nv = mask.shape
    levels, layers = len(level_ratio), len(layer_ratio)
    lr = torch.tensor(list(level_ratio), dtype=torch.float32)
    yr = torch.tensor(list(layer_ratio), dtype=torch.float32)
    ltn = torch.empty(levels, dtype=torch.int32)
    ftn = torch.empty(b, dtype=torch.int32)
    lnq = torch.empty(layers, dtype=torch.int64)
    lib().oracle_token_budgets(_p(mask.to(torch.uint8).contiguous()), _p(lsi), _p(hw), b, nv, levels,
                               _p(lr), layers, _p(yr), _p(ltn), _p(ftn), _p(lnq))
    _done()
    return ltn, ftn, lnq


def c_token_gather(tokens, pos, fg, valid_ratios, inds, shapes, lsi, num_query):
    b, nv, c = tokens.shape
    levels = shapes.shape[0]
    q = torch.empty(b, num_query, c)
    qp = torch.empty(b, num_query, c)
    fq = torch.empty(b, num_query)
    rq = torch.empty(b, num_query, levels, 2)
    assert inds.stride(1) == 1
    lib().oracle_token_gather(_p(tokens.contiguous()), _p(pos.contiguous()), _p(fg.contiguous()),
                              _p(valid_ratios.contiguous()), ctypes.c_void_p(inds.data_ptr()),
                              ctypes.c_int64(inds.stride(0)), _p(shapes), _p(lsi), b, nv, c, levels,
                              num_query, _p(q), _p(qp), _p(fq), _p(rq))
    _done()
    return q, qp, fq, rq


def c_token_scatter(tokens, query, inds, focus_token_nums):
    """In place on ``tokens``."""
    b, nv, c = tokens.shape
    nq = query.shape[1]
    assert tokens.is_contiguous() and inds.stride(1) == 1
    lib().oracle_token_scatter(_p(tokens), _p(query.contiguous()), ctypes.c_void_p(inds.data_ptr()),
                               ctypes.c_int64(inds.stride(0)), _p(focus_token_nums.to(torch.int32).contiguous()),
                               b, nv, c, nq)
    _done()
    return tokens


def c_background_embed(tokens, mask, last_inds, row_embed, col_embed, shapes, lsi):
    """In place on ``tokens``."""
    b, nv, c = tokens.shape
    assert tokens.is_contiguous() and last_inds.stride(1) == 1
    lib().oracle_background_embed(_p(tokens), _p(mask.to(torch.uint8).contiguous()),
                                  ctypes.c_void_p(last_inds.data_ptr()), ctypes.c_int64(last_inds.stride(0)),
                                  last_inds.shape[1], _p(row_embed.contiguous()), _p(col_embed.contiguous()),
                                  _p(shapes), _p(lsi), b, nv, c, shapes.shape[0])
    _done()
    return tokens


def c_score_modulate(mem, coarse, alpha: float, H, W, Hc, Wc):
    b, hw, c = mem.shape
    out = torch.empty_like(mem)
    lib().oracle_score_modulate(_p(mem.contiguous()), _p(coarse.contiguous()), ctypes.c_float(alpha), b, H, W,
                                Hc, Wc, c, _p(out))
    _done()
    return out


# --------------------------------------------------------------------------------------------------
# torch-CPU restatement of the reference's PyTorch path (functional, state_dict-driven)
# --------------------------------------------------------------------------------------------------
def msda_core_torch(value, shapes_list: List[Sequence[int]], loc, attn):
    """Restates multi_scale_deformable_attn_pytorch (models/bricks/ms_deform_attn.py:159-212)."""
    b, _, m, d = value.shape
    nq = loc.shape[1]
    grids = loc * 2 - 1
    sampled = []
    start = 0
    for lvl, (h, w) in enumerate(shapes_list):
        v = value[:, start:start + h * w].permute(0, 2, 3, 1).reshape(b * m, d, h, w)
        g = grids[:, :, :, lvl].permute(0, 2, 1, 3, 4).reshape(b * m, nq, -1, 2)
        sampled.append(F.grid_sample(v, g, mode="bilinear", padding_mode="zeros", align_corners=False))
        start += h * w
    a = attn.permute(0, 2, 1, 3, 4).reshape(b * m, 1, nq, -1)
    out = (torch.cat(sampled, dim=-1) * a).sum(-1)
    return out.view(b, m * d, nq).permute(0, 2, 1).contiguous()


def _lin(sd, name, x):
    return F.linear(x, sd[name + ".weight"], sd.get(name + ".bias"))


def _ln(sd, name, x):
    return F.layer_norm(x, (x.shape[-1],), sd[name + ".weight"], sd[name + ".bias"])


def msda_module(sd, pre, query, ref, value, shapes, lsi, mask, heads, levels, points, core="torch"):
    """Restates MultiScaleDeformableAttention.forward (ms_deform_attn.py:311-377), 2-d ref points."""
    b, nq, c = query.shape
    nv = value.shape[1]
    v = _lin(sd, pre + "value_proj", value)
    if mask is not None:
        v = v.masked_fill(mask[..., None], 0.0)
    v = v.view(b, nv, heads, c // heads)
    off = _lin(sd, pre + "sampling_offsets", query).view(b, nq, heads, levels, points, 2)
    w = _lin(sd, pre + "attention_weights", query).view(b, nq, heads, levels * points).softmax(-1)
    w = w.view(b, nq, heads, levels, points)
    norm = torch.stack([shapes[:, 1], shapes[:, 0]], -1)
    loc = ref[:, :, None, :, None, :] + off / norm[None, None, None, :, None, :]
    if core == "torch":
        out = msda_core_torch(v, shapes.tolist(), loc, w)
    elif callable(core):  # an operator with the `_C.ms_deform_attn_forward` contract (value, shapes, lsi, loc, attn)
        out = core(v, shapes, lsi, loc, w)
    else:
        out = c_msda_forward(v, shapes, lsi, loc, w)
    return _lin(sd, pre + "output_proj", out)


def mask_predictor(sd, pre, x):
    """Restates MaskPredictor.forward (salience_transformer.py:41-47)."""
    z = F.gelu(_lin(sd, pre + "layer1.1", _ln(sd, pre + "layer1.0", x)))
    h = z.shape[-1] // 2
    z = torch.cat([z[..., :h], z[..., h:].mean(1, keepdim=True).expand(-1, z.shape[1], -1)], -1)
    z = F.gelu(_lin(sd, pre + "layer2.0", z))
    z = F.gelu(_lin(sd, pre + "layer2.2", z))
    return _lin(sd, pre + "layer2.4", z)


def flatten_levels(xs):
    """base_transformer.py:21-26."""
    y = torch.cat([e.flatten(-2) for e in xs], -1)
    return y.transpose(1, 2).contiguous() if y.ndim == 3 else y


def level_misc(masks):
    """base_transformer.py:34-56 -> spatial_shapes (L,2) i64, level_start_index (L,), valid_ratios (b,L,2)."""
    shapes = torch.tensor([list(m.shape[-2:]) for m in masks], dtype=torch.int64)
    lsi = torch.cat([shapes.new_zeros(1), shapes.prod(1).cumsum(0)[:-1]])
    vr = []
    for m in masks:
        _, h, w = m.shape
        vh = (~m[:, :, 0]).sum(1).float() / h
        vw = (~m[:, 0, :]).sum(1).float() / w
        vr.append(torch.stack([vw, vh], -1))
    return shapes, lsi, torch.stack(vr, 1)


def proposal_keep_mask(mask_flat, shapes_list):
    """`~padding & output_proposals_valid` of gen_encoder_output_proposals (base_transformer.py:74-110)."""
    b = mask_flat.shape[0]
    keep = []
    cur = 0
    for lvl, (h, w) in enumerate(shapes_list):
        m = mask_flat[:, cur:cur + h * w].view(b, h, w)
        vh = (~m[:, :, 0]).sum(1)
        vw = (~m[:, 0, :]).sum(1)
        gy = (torch.arange(h, dtype=torch.float32) + 0.5)[None, :, None] / vh[:, None, None]
        gx = (torch.arange(w, dtype=torch.float32) + 0.5)[None, None, :] / vw[:, None, None]
        wh = 0.05 * 2.0 ** lvl
        ok = (gy > 0.01) & (gy < 0.99) & (gx > 0.01) & (gx < 0.99) & (0.01 < wh < 0.99)
        keep.append((ok & ~m).flatten(1))
        cur += h * w
    return torch.cat(keep, 1)


def salience_filter(sd, feat, lpos, mask_flat, masks, shapes, lsi, level_ratio, layer_ratio):
    """Restates salience_transformer.py:112-168.  Returns a dict of everything the encoder consumes."""
    shapes_list = shapes.tolist()
    L = len(shapes_list)
    b = feat.shape[0]
    keep = proposal_keep_mask(mask_flat, shapes_list)
    mem = _ln(sd, "enc_output_norm", _lin(sd, "enc_output", (feat + lpos) * keep[..., None]))
    valid = torch.stack([(~m).sum((1, 2)) for m in masks], -1)
    focus = (valid * torch.tensor(level_ratio, dtype=torch.float32)).int()
    level_token_nums = focus.max(0)[0]
    focus_token_nums = focus.sum(-1)
    raw = torch.empty(b, feat.shape[1])
    score = None
    for lvl in range(L - 1, -1, -1):
        h, w = shapes_list[lvl]
        s0 = int(lsi[lvl])
        m_l = mem[:, s0:s0 + h * w]
        if lvl != L - 1:
            up = F.interpolate(score, size=(h, w), mode="bilinear", align_corners=True)
            m_l = m_l + m_l * up.view(b, 1, h * w).transpose(1, 2) * sd["alpha"][lvl]
        s = mask_predictor(sd, "enc_mask_predictor.", m_l)
        raw[:, s0:s0 + h * w] = s.squeeze(-1)
        score = s.transpose(1, 2).reshape(b, 1, h, w)
    hw = shapes.prod(1)
    inds, sel_score, fg = c_salience_select(raw, mask_flat, lsi, hw, level_token_nums.tolist())
    K = inds.shape[1]
    nq = (K * torch.tensor(layer_ratio, dtype=torch.float32)).to(torch.int64).tolist()
    return dict(memory0=mem, raw_score=raw, selected_inds=inds, selected_score=sel_score,
                foreground_score=fg, level_token_nums=level_token_nums, focus_token_nums=focus_token_nums,
                layer_num_query=nq)


def reference_points(shapes_list, valid_ratios):
    """Restates SalienceTransformerEncoder.get_reference_points (salience_transformer.py:417-432)."""
    refs = []
    for lvl, (h, w) in enumerate(shapes_list):
        ys = (torch.arange(h, dtype=torch.float32) + 0.5)
        xs = (torch.arange(w, dtype=torch.float32) + 0.5)
        ry = ys[None, :, None].expand(1, h, w).reshape(1, -1) / (valid_ratios[:, None, lvl, 1] * h)
        rx = xs[None, None, :].expand(1, h, w).reshape(1, -1) / (valid_ratios[:, None, lvl, 0] * w)
        refs.append(torch.stack((rx, ry), -1))
    return torch.cat(refs, 1)[:, :, None] * valid_ratios[:, None]


def pre_attention(sd, pre, q, qp, cls, fg_q, heads, topk_sa):
    """Restates salience_transformer.py:366-379 (top-k salient tokens -> MHA -> LN -> scatter)."""
    b, nq, c = q.shape
    mc = cls.max(-1)[0] * fg_q
    # canonical tie order (score desc, position asc); the set is what matters (MHA is permutation-equivariant)
    order = torch.sort(mc, dim=1, descending=True, stable=True)[1][:, :topk_sa]
    ix = order[..., None].expand(-1, -1, c)
    t, tp = q.gather(1, ix), qp.gather(1, ix)
    x = t + tp
    wi, bi = sd[pre + "pre_attention.in_proj_weight"], sd[pre + "pre_attention.in_proj_bias"]
    qh = F.linear(x, wi[:c], bi[:c]).view(b, -1, heads, c // heads).transpose(1, 2)
    kh = F.linear(x, wi[c:2 * c], bi[c:2 * c]).view(b, -1, heads, c // heads).transpose(1, 2)
    vh = F.linear(t, wi[2 * c:], bi[2 * c:]).view(b, -1, heads, c // heads).transpose(1, 2)
    att = (qh @ kh.transpose(-1, -2) / math.sqrt(c // heads)).softmax(-1) @ vh
    att = _lin(sd, pre + "pre_attention.out_proj", att.transpose(1, 2).reshape(b, -1, c))
    t = _ln(sd, pre + "pre_norm", t + att)
    return q.scatter(1, ix, t), order


def encoder_layer(sd, pre, q, qp, value, ref_q, shapes, lsi, mask, cls, fg_q, heads, levels, points,
                  topk_sa, core="torch"):
    """Restates SalienceTransformerEncoderLayer.forward (salience_transformer.py:353-396)."""
    q, _ = pre_attention(sd, pre, q, qp, cls, fg_q, heads, topk_sa)
    a = msda_module(sd, pre + "self_attn.", q + qp, ref_q, value, shapes, lsi, mask, heads, levels, points, core)
    q = _ln(sd, pre + "norm1", q + a)
    f = _lin(sd, pre + "linear2", F.relu(_lin(sd, pre + "linear1", q)))
    return _ln(sd, pre + "norm2", q + f)


def encoder_forward(sd, feat, lpos, mask_flat, shapes, lsi, valid_ratios, filt, heads, points, topk_sa,
                    num_layers, core="torch", use_c_helpers=False, trace=None):
    """Restates SalienceTransformerEncoder.forward (salience_transformer.py:434-497)."""
    shapes_list = shapes.tolist()
    L = len(shapes_list)
    b, nv, c = feat.shape
    ref = reference_points(shapes_list, valid_ratios)
    out = feat.clone()
    inds_all = filt["selected_inds"]
    fg = filt["foreground_score"]
    focus = filt["focus_token_nums"]
    for j in range(num_layers):
        nq = filt["layer_num_query"][j]
        inds = inds_all[:, :nq]
        if use_c_helpers:
            q, qp, fq, rq = c_token_gather(out, lpos, fg, valid_ratios, inds, shapes, lsi, nq)
        else:
            ix = inds[..., None].expand(-1, -1, c)
            q, qp = out.gather(1, ix), lpos.gather(1, ix)
            fq = fg.gather(1, inds)
            rq = ref.view(b, nv, -1).gather(1, inds[..., None].expand(-1, -1, L * 2)).view(b, nq, L, 2)
        cls = _lin(sd, "encoder_class_head", q)
        q = encoder_layer(sd, f"encoder.layers.{j}.", q, qp, feat, rq, shapes, lsi, mask_flat, cls, fq, heads,
                          L, points, topk_sa, core)
        if trace is not None:
            trace.append(q)
        if use_c_helpers:
            c_token_scatter(out, q, inds, focus)
        else:
            for i in range(b):
                n = min(int(focus[i]), nq)
                out[i, inds[i, :n]] = q[i, :n]
    row, col = sd["encoder.background_embedding.row_embed.weight"], sd["encoder.background_embedding.col_embed.weight"]
    if use_c_helpers:
        c_background_embed(out, mask_flat, inds, row, col, shapes, lsi)
    else:
        bg = []
        for (h, w) in shapes_list:
            e = torch.cat([col[:w][None].expand(h, -1, -1), row[:h][:, None].expand(-1, w, -1)], -1)
            bg.append(e.reshape(1, h * w, c).expand(b, -1, -1))
        bg = torch.cat(bg, 1).clone()
        bg.scatter_(1, inds[..., None].expand(-1, -1, c), 0.0)
        bg = bg * (~mask_flat)[..., None]
        out = out + bg
    return out


def encoder_half_forward(sd, feats, masks, pos_embeds, cfg: Dict, core="torch", use_c_helpers=False, trace=None):
    """salience_transformer.py:106-183: (multi-level feats, masks, pos) -> encoder memory (b,Nv,C).

    cfg: heads, points, topk_sa, num_layers, level_filter_ratio, layer_filter_ratio.
    """
    feat = flatten_levels(feats)
    mask_flat = flatten_levels(masks)
    lpos = flatten_levels([p + l.view(1, -1, 1, 1) for p, l in zip(pos_embeds, sd["level_embeds"])])
    shapes, lsi, vr = level_misc(masks)
    filt = salience_filter(sd, feat, lpos, mask_flat, masks, shapes, lsi, cfg["level_filter_ratio"],
                           cfg["layer_filter_ratio"])
    mem = encoder_forward(sd, feat, lpos, mask_flat, shapes, lsi, vr, filt, cfg["heads"], cfg["points"],
                          cfg["topk_sa"], cfg["num_layers"], core, use_c_helpers, trace)
    return mem, filt


# --------------------------------------------------------------------------------------------------
# synthetic inputs (SURVEY.md 8(d)); shared by tests and bench (pure torch, no reference needed)
# --------------------------------------------------------------------------------------------------
def sine_pos_embed(mask, num_pos_feats, temperature=10000, scale=2 * math.pi, eps=1e-6, offset=-0.5):
    """Restates PositionEmbeddingSine.forward with normalize=True (position_encoding.py:48-65)."""
    nm = (~mask).to(torch.float32)
    y = nm.cumsum(1)
    x = nm.cumsum(2)
    y = (y + offset) / (y[:, -1:, :] + eps) * scale
    x = (x + offset) / (x[:, :, -1:] + eps) * scale
    dim_t = temperature ** (2 * torch.arange(num_pos_feats).div(2, rounding_mode="floor") / num_pos_feats)
    px = x[..., None] / dim_t
    py = y[..., None] / dim_t
    px = torch.stack((px[..., 0::2].sin(), px[..., 1::2].cos()), dim=4).flatten(3)
    py = torch.stack((py[..., 0::2].sin(), py[..., 1::2].cos()), dim=4).flatten(3)
    return torch.cat((py, px), dim=3).permute(0, 3, 1, 2).contiguous()


def level_shapes_for_image(h, w, strides=(8, 16, 32, 64)):
    """Feature-map sizes of the padded image (ceil division per stride; last level = 3x3 s2 conv)."""
    out = []
    for i, s in enumerate(strides):
        if i == len(strides) - 1 and len(out) and s == 2 * strides[i - 1]:
            ph, pw = out[-1]
            out.append(((ph - 1) // 2 + 1, (pw - 1) // 2 + 1))
        else:
            out.append((math.ceil(h / s), math.ceil(w / s)))
    return out


def synthetic_inputs(image_sizes, padded_hw, embed_dim=256, strides=(8, 16, 32, 64), seed=0):
    """Synthetic multi-level feats/masks/pos for images of ``image_sizes`` [(h,w)...] padded to ``padded_hw``."""
    g = torch.Generator().manual_seed(seed)
    b = len(image_sizes)
    H, W = padded_hw
    full = torch.ones(b, H, W, dtype=torch.bool)
    for i, (h, w) in enumerate(image_sizes):
        full[i, :h, :w] = False
    shapes = level_shapes_for_image(H, W, strides)
    feats, masks, pos = [], [], []
    for (h, w) in shapes:
        feats.append(torch.randn(b, embed_dim, h, w, generator=g))
        m = F.interpolate(full[None].float(), size=(h, w))[0].to(torch.bool)  # salience_detr.py:175
        masks.append(m)
        pos.append(sine_pos_embed(m, embed_dim // 2))
    return feats, masks, pos


def deterministic_state_dict(shapes: Dict[str, Sequence[int]], seed: int) -> Dict[str, torch.Tensor]:
    """Weights regenerated from (sorted name order, shape, seed) with the CPU generator, so that a golden fixture made
    from the reference need not carry a multi-megabyte state_dict: oracle/make_golden.py loads these into the reference
    model, the tests load the same tensors into the oracle / the CUDA modules.  Scales keep activations O(1):
    matrices ~ N(0, 1/fan_in), LayerNorm gains 1 + 0.1 N, biases 0.1 N, sampling-offset weights 0.05 N."""
    out = {}
    for i, name in enumerate(sorted(shapes)):
        g = torch.Generator().manual_seed(seed * 100003 + i)
        shp = tuple(int(v) for v in shapes[name])
        x = torch.randn(shp, generator=g)
        if len(shp) == 1:
            if name.endswith(".weight"):
                x = 1.0 + 0.1 * x
            elif name == "alpha":
                x = 0.3 * x
            elif name.endswith("sampling_offsets.bias"):
                x = 0.5 * x
            else:
                x = 0.1 * x
        elif name.endswith("sampling_offsets.weight"):
            x = 0.05 * x
        elif name.endswith("_embed.weight") or name == "level_embeds":
            x = 0.5 * x
        else:
            x = x / (shp[-1] ** 0.5)
        out[name] = x
    return out


def golden_state_dict(shapes_json: str, seed: int, aliases_json: str = "{}") -> Dict[str, torch.Tensor]:
    """The weights a golden fixture was made with: ``deterministic_state_dict`` of its stored shapes, with every key that is
    the same tensor as another one in the reference model (e.g. ``encoder.enhance_mcsp`` = ``encoder_class_head``, reference
    salience_transformer.py:79) set to the value that tensor ended up holding."""
    import json
    sd = deterministic_state_dict(json.loads(shapes_json), seed)
    for k, src in json.loads(aliases_json).items():
        sd[k] = sd[src]
    return sd


def sample_index(numel: int, n: int, seed: int) -> torch.Tensor:
    """Fixed, seeded positions at which a golden fixture stores a large output (flat indices, at most ``n``)."""
    return torch.randperm(numel, generator=torch.Generator().manual_seed(seed))[:n]


def sampled(t: torch.Tensor, n: int, seed: int) -> torch.Tensor:
    """``t`` (any device) at ``sample_index`` positions, on the CPU."""
    return t.detach().reshape(-1)[sample_index(t.numel(), n, seed).to(t.device)].cpu()


class TopDownNeck(torch.nn.Module):
    """A small stand-in for the detector's neck (any module taking and returning ``{level: (b, C, h, w)}``, reference
    salience_transformer.py:185-192): per level a channel mix, plus the nearest-upsampled result of the next coarser level,
    then SiLU.  Weights come from ``seed``; channel mixes are matrix products, so they run in fp32 on any device."""

    def __init__(self, channels: int, levels: int, seed: int = 3):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.weight = torch.nn.Parameter(torch.randn(levels, channels, channels, generator=g) / channels ** 0.5)
        self.bias = torch.nn.Parameter(0.1 * torch.randn(levels, channels, generator=g))

    def forward(self, feats):
        out, up = {}, None
        for i in sorted(feats, reverse=True):
            x = torch.einsum("oc,bchw->bohw", self.weight[i], feats[i]) + self.bias[i][None, :, None, None]
            if up is not None:
                x = x + F.interpolate(up, size=x.shape[-2:], mode="nearest")
            up = F.silu(x)
            out[i] = up
        return {i: out[i] for i in sorted(out)}
