"""CPU tests of the host-side logic above the C-ABI: the EncoderPlan (token budgets, level tables, keep mask,
valid ratios) against the oracle and the reference-made golden fixtures.  Pure torch, no kernels."""
import torch

from conftest import load_golden
from oracle import oracle as orc


def _model(pkg, cfg_levels=(0.4, 0.8, 1.0, 1.0), layers=(1.0, 0.6, 0.3)):
    enc = pkg.SalienceTransformerEncoder(pkg.SalienceTransformerEncoderLayer(64, 128, 0.0, 2, topk_sa=20), len(layers), 40)
    return pkg.SalienceTransformer(enc, num_classes=11, level_filter_ratio=cfg_levels, layer_filter_ratio=layers).eval()


def test_plan_matches_reference_golden():
    import salience_detr_b200 as pkg
    for name in ("encoder_tiny_even", "encoder_tiny_ragged"):
        g, sd = load_golden(name)
        tr = _model(pkg)
        masks = [g[f"mask{i}"] for i in range(4)]
        plan = tr.make_plan(masks)
        assert torch.equal(plan.spatial_shapes, g["spatial_shapes"])
        assert torch.equal(plan.level_start_index, g["level_start_index"])
        assert torch.equal(plan.valid_ratios, g["valid_ratios"])
        assert torch.equal(plan.focus_token_nums.long(), g["focus_token_nums"].long())
        assert plan.layer_num_query == g["layer_num_query"].tolist()
        assert plan.num_selected == g["selected_inds"].shape[1]
        mask_flat = orc.flatten_levels(masks)
        keep = orc.proposal_keep_mask(mask_flat, plan.shapes_list)
        assert torch.equal(plan.keep[..., 0].bool(), keep)


def test_plan_budgets_config2_fp32_truncation():
    """800x1333 padded to 800x1344 (SURVEY.md 8(d)): K = 11363, Nq = [11363, 9090, 6817, 6817, 4545, 2272]."""
    import salience_detr_b200 as pkg
    enc = pkg.SalienceTransformerEncoder(pkg.SalienceTransformerEncoderLayer(64, 128, 0.0, 2), 6, 200)
    tr = pkg.SalienceTransformer(enc, level_filter_ratio=(0.4, 0.8, 1.0, 1.0),
                                 layer_filter_ratio=(1.0, 0.8, 0.6, 0.6, 0.4, 0.2))
    _, masks, _ = orc.synthetic_inputs([(800, 1333)] * 2, (800, 1344), embed_dim=8)
    plan = tr.make_plan(masks)
    assert plan.shapes_list == [(100, 168), (50, 84), (25, 42), (13, 21)]
    assert plan.level_token_nums == [6680, 3360, 1050, 273]
    assert plan.focus_host == [11363, 11363]
    assert plan.layer_num_query == [11363, 9090, 6817, 6817, 4545, 2272]
    mask_flat = orc.flatten_levels(masks)
    ltn, ftn, lnq = orc.c_token_budgets(mask_flat, plan.level_start_index, torch.tensor(plan.level_size),
                                        (0.4, 0.8, 1.0, 1.0), (1.0, 0.8, 0.6, 0.6, 0.4, 0.2))
    assert ltn.tolist() == plan.level_token_nums and ftn.tolist() == plan.focus_host
    assert lnq.tolist() == plan.layer_num_query
    # ragged second image (SURVEY.md 8(d)): focus = [11363, 6832]
    _, masks, _ = orc.synthetic_inputs([(800, 1333), (640, 1000)], (800, 1344), embed_dim=8)
    assert tr.make_plan(masks).focus_host == [11363, 6832]


def test_state_dict_names_match_reference():
    """A reference state_dict (encoder-half keys) loads with no missing and no unexpected key."""
    import salience_detr_b200 as pkg
    g, sd = load_golden("encoder_tiny_even")
    res = _model(pkg).load_state_dict(sd, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    # optimizer/param_dict.py:80 matches `sampling_offsets` by name
    assert any("self_attn.sampling_offsets.weight" in k for k in sd)


def test_msda_module_init_matches_reference_golden_shapes():
    import salience_detr_b200 as pkg
    m = pkg.MultiScaleDeformableAttention(256, 4, 8, 4)
    b = m.sampling_offsets.bias.view(8, 4, 4, 2)
    assert torch.allclose(b[0, 0, :, 0], torch.tensor([1.0, 2.0, 3.0, 4.0])) and b[0, 0, :, 1].abs().max() < 1e-6
    assert m.sampling_offsets.weight.abs().max() == 0 and m.attention_weights.weight.abs().max() == 0
    assert m.im2col_step == 64


def test_mha_transposed_weight_cache_follows_parameter_updates():
    """The fused pre-attention consumes in_proj_weight^T / out_proj.weight^T; the cache must refresh when the
    parameters are modified in place (optimizer step) or replaced (load_state_dict)."""
    import salience_detr_b200 as pkg
    layer = pkg.SalienceTransformerEncoderLayer(embed_dim=64, d_ffn=128, dropout=0.0, n_heads=2, n_levels=4, n_points=4, topk_sa=10)
    w_in_t, w_out_t = layer._mha_transposed()
    assert w_in_t.shape == (64, 192) and torch.equal(w_in_t, layer.pre_attention.in_proj_weight.detach().t())
    assert layer._mha_transposed()[0] is w_in_t  # cached
    with torch.no_grad():
        layer.pre_attention.in_proj_weight.add_(1.0)
        layer.pre_attention.out_proj.weight.mul_(2.0)
    w_in_t2, w_out_t2 = layer._mha_transposed()
    assert w_in_t2 is not w_in_t and torch.equal(w_in_t2, layer.pre_attention.in_proj_weight.detach().t())
    assert torch.equal(w_out_t2, layer.pre_attention.out_proj.weight.detach().t())


def test_salience_criterion_matches_reference_golden():
    """SalienceCriterion mirror (host restatement of the target maps + focal loss) against the reference class's loss,
    gradient and target maps (tests/golden/salience_criterion.npz, oracle/make_golden.py::make_salience_criterion)."""
    import salience_detr_b200 as pkg
    g, _ = load_golden("salience_criterion")
    shapes = [tuple(int(v) for v in r) for r in g["shapes"]]
    fg = [g[f"fg{i}"].clone().requires_grad_(True) for i in range(4)]
    targets = [{"boxes": g["boxes0"]}, {"boxes": g["boxes1"]}]
    sizes = [tuple(int(v) for v in r) for r in g["image_sizes"]]
    strides = [tuple(float(v) for v in r) for r in g["strides"]]
    crit = pkg.SalienceCriterion()
    assert torch.equal(crit.mask_targets(shapes, targets, strides, sizes, torch.device("cpu")), g["mask_targets"])
    loss = crit(fg, targets, strides, sizes)["loss_salience"]
    assert abs(loss.item() - g["loss"].item()) < 1e-6
    loss.backward()
    for i in range(4):
        assert (fg[i].grad - g[f"grad{i}"]).abs().max() < 1e-7
    # an image without boxes contributes zero targets
    assert crit.mask_targets(shapes, [{"boxes": torch.zeros(0, 4)}, targets[1]], strides, sizes, torch.device("cpu"))[0].abs().max() == 0


def test_load_reference_checkpoint_layouts():
    """Checkpoints as the reference writes them: bare state_dict, {"model": ...}, DDP `module.` prefix, whole-detector
    `transformer.` prefix, shape-mismatched entries skipped (util/utils.py:358-422)."""
    import salience_detr_b200 as pkg
    g, sd = load_golden("encoder_tiny_even")
    ref_sum = sum(float(v.double().sum()) for v in sd.values())

    def fresh():
        return _model(pkg)

    def total(m):
        return sum(float(v.double().sum()) for k, v in m.state_dict().items() if k in sd)

    for ckpt in (sd, {"model": sd, "epoch": 3}, {"model": {"module." + k: v for k, v in sd.items()}},
                 {"model": {**{"transformer." + k: v for k, v in sd.items()}, "backbone.conv1.weight": torch.zeros(3)}}):
        m = fresh()
        rep = pkg.load_reference_checkpoint(m, ckpt)
        assert not rep["missing"] and not rep["mismatched"] and abs(total(m) - ref_sum) < 1e-6
    bad = dict(sd)
    bad["alpha"] = torch.zeros(7)
    m = fresh()
    rep = pkg.load_reference_checkpoint(m, bad)
    assert rep["mismatched"] == ["alpha"] and m.alpha.shape == (3,)


def test_tensor_core_linears_context_on_cpu():
    """gemm.tensor_core_linears routes torch.nn.functional.linear through gemm.linear_train and restores it (also on an exception);
    tensors the kernel does not take (CPU, few rows, K % 64 != 0) fall back to the original F.linear with ordinary autograd."""
    import torch
    import salience_detr_b200 as pkg
    F = torch.nn.functional
    orig = F.linear
    lin = torch.nn.Linear(64, 8)
    x = torch.randn(5, 64, requires_grad=True)
    with pkg.gemm.tensor_core_linears():
        assert F.linear is pkg.gemm.linear_train
        y = lin(x)
    assert F.linear is orig
    assert "LinearF16x3" not in type(y.grad_fn).__name__ and torch.allclose(y, orig(x, lin.weight, lin.bias))
    y.sum().backward()
    assert x.grad is not None and lin.weight.grad is not None
    try:
        with pkg.gemm.tensor_core_linears():
            raise KeyError("boom")
    except KeyError:
        pass
    assert F.linear is orig


def test_masked_predictor_transposed_weight_cache_follows_updates():
    """MaskPredictor.transposed_weights (the (in, out) weights sdetr_mask_predictor_level streams) is rebuilt when a parameter changes."""
    import torch
    from salience_detr_b200.salience_transformer import MaskPredictor
    mp = MaskPredictor(256, 256)
    t0 = mp.transposed_weights()
    assert t0[0].shape == (256, 256) and t0[2].shape == (256, 128) and t0[4].shape == (128, 64) and t0[6].shape == (64,)
    assert torch.equal(t0[0], mp.layer1[1].weight.t()) and mp.transposed_weights() is t0
    with torch.no_grad():
        mp.layer2[0].weight.add_(1.0)
    t1 = mp.transposed_weights()
    assert t1 is not t0 and torch.equal(t1[2], mp.layer2[0].weight.t())


def test_bench_stdout_carries_only_the_result_line():
    """bench.py's stdout contract: ONE JSON line, whatever libraries print.  After `_claim_stdout()` file descriptor 1 points at stderr
    (NCCL writes its version banner there from C, past sys.stdout) and only `emit()` reaches the real stdout."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import os, sys; sys.path.insert(0, %r); import bench; bench._claim_stdout(); "
            "os.write(1, b'banner from a C library\\n'); print('a python print'); bench.emit('{\"ok\": 1}')" % root)
    p = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=300, cwd=root)
    assert p.returncode == 0, p.stderr.decode()[-800:]
    assert p.stdout.decode() == '{"ok": 1}\n'
    err = p.stderr.decode()
    assert "banner from a C library" in err and "a python print" in err


def test_bench_dump_outputs(tmp_path):
    """`bench.py --dump-outputs DIR`: every output as DIR/<name>.npy in float32, values unchanged; more than 64 MiB in all is
    refused before anything is written."""
    import numpy as np
    import pytest
    import bench
    mem = torch.randn(2, 37, 8, dtype=torch.float64)
    bench.dump_outputs(str(tmp_path / "out"), {"memory": mem})
    got = np.load(tmp_path / "out" / "memory.npy")
    assert got.dtype == np.float32 and np.array_equal(got, mem.float().numpy())
    with pytest.raises(SystemExit):
        bench.dump_outputs(str(tmp_path / "big"), {"memory": torch.empty(bench.DUMP_LIMIT_BYTES // 4 + 1)})
    assert not (tmp_path / "big").exists()
