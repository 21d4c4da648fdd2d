"""TEST INFRASTRUCTURE ONLY -- loader for the *unmodified* reference (xiuqhou/Salience-DETR).

Used in the build container to (a) generate the golden fixtures under ``tests/golden/`` and
(b) validate the oracle restatements in ``oracle/`` against the reference itself.  The
reference tree (``/root/reference``) does not travel to the GPU box, so nothing on a product,
bench or ``-m gpu`` path may import this module; callers must check :func:`available` first.

The only accommodation made is a stub for ``util.misc`` (its real module imports ``accelerate``,
which is not installed): ``models/bricks/salience_transformer.py:13`` needs only
``inverse_sigmoid`` (semantics of ``util/misc.py:31-35``), used by the decoder, not the encoder.
"""
from __future__ import annotations

import os
import sys
import types
import warnings

_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASELINE_REF = os.path.join(_REPO, "baseline", "_ref")  # git-ignored install of the reference's hot-path modules


def _has(root: str) -> bool:
    return os.path.isfile(os.path.join(root, "models", "bricks", "salience_transformer.py"))


def _resolve_root() -> str:
    env = os.environ.get("SDETR_REFERENCE_ROOT")
    if env:
        return env
    for root in ("/root/reference", BASELINE_REF):  # the tree itself in the build container, the install on the GPU box
        if _has(root):
            return root
    return "/root/reference"


REFERENCE_ROOT = _resolve_root()


def available() -> bool:
    return _has(REFERENCE_ROOT)


def _install_stub():
    import torch

    if "util.misc" in sys.modules:
        return
    pkg = types.ModuleType("util")
    pkg.__path__ = [os.path.join(REFERENCE_ROOT, "util")]
    misc = types.ModuleType("util.misc")

    def inverse_sigmoid(x, eps: float = 1e-3):  # util/misc.py:31-35
        x = x.clamp(min=0, max=1)
        return torch.log(x.clamp(min=eps) / (1 - x).clamp(min=eps))

    misc.inverse_sigmoid = inverse_sigmoid
    pkg.misc = misc
    sys.modules.setdefault("util", pkg)
    sys.modules["util.misc"] = misc


def load():
    """Return a namespace with the reference modules of the hot path (imported unmodified)."""
    if not available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    _install_stub()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        import models.bricks.ms_deform_attn as msda  # noqa
        import models.bricks.salience_transformer as st  # noqa
        import models.bricks.position_encoding as pe  # noqa
        import models.bricks.base_transformer as bt  # noqa
    ns = types.SimpleNamespace(msda=msda, st=st, pe=pe, bt=bt, repnet=None)
    try:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            import models.necks.repnet as repnet  # noqa
        ns.repnet = repnet
    except Exception:  # older installs without the neck modules
        pass
    return ns


class _Stop(Exception):
    pass


def run_encoder_half(tr, feats, masks, pos):
    """Run the reference ``SalienceTransformer.forward`` up to the end of the encoder (salience_transformer.py:106-183)
    and return (memory, kwargs the filter handed to the encoder).  The decoder half is cut off by an exception raised
    from a wrapper around ``encoder.forward`` -- the reference code itself is untouched."""
    import torch

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
    finally:
        del tr.encoder.forward  # drop the instance attribute: the class's forward is visible again
    return captured.pop("memory"), captured


def build_transformer(embed_dim=256, d_ffn=2048, n_heads=8, n_levels=4, n_points=4, num_layers=6,
                      num_classes=91, level_filter_ratio=(0.4, 0.8, 1.0, 1.0),
                      layer_filter_ratio=(1.0, 0.8, 0.6, 0.6, 0.4, 0.2), topk_sa=300,
                      max_num_embedding=200, num_proposals=900, seed=0):
    """Reference ``SalienceTransformer`` (neck=None) with default init under ``manual_seed(seed)``.

    Geometry defaults follow configs/salience_detr/salience_detr_resnet50_800_1333.py:22-29,44-81.
    """
    import torch
    from torch import nn

    ref = load()
    st = ref.st
    torch.manual_seed(seed)
    enc_layer = st.SalienceTransformerEncoderLayer(embed_dim, d_ffn, 0.0, n_heads, nn.ReLU(inplace=True),
                                                   n_levels, n_points, topk_sa=topk_sa)
    enc = st.SalienceTransformerEncoder(enc_layer, num_layers, max_num_embedding=max_num_embedding)
    dec_layer = st.SalienceTransformerDecoderLayer(embed_dim, d_ffn, n_heads, 0.0, nn.ReLU(inplace=True),
                                                   n_levels, n_points)
    dec = st.SalienceTransformerDecoder(dec_layer, 1, num_classes)
    tr = st.SalienceTransformer(enc, None, dec, num_classes, n_levels, num_proposals,
                                tuple(level_filter_ratio), tuple(layer_filter_ratio))
    return tr.eval()
