"""Shared helpers of the parity tests: build a seeded case, run it through the CPU oracle and through the CUDA
path (via the C ABI behind the package classes), compare.

Tolerances (fp32 path, decoder contractions in 3xTF32 ~ fp32):
  indices            bit-exact
  feature            |d| <= 2e-6 + 1e-5 |ref|
  pred               |d| <= 2e-5 + 1e-5 |ref|
  loss               relative 2e-5
  table / dec grads  max|d| <= 2e-4 * max|ref| + 1e-10   (float atomics are order-nondeterministic)
With SHINE_FLAG_TF32X1 (plain TF32) pred is only good to ~2e-3 and is tested separately.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import shine_oracle as orc  # noqa: E402  (tests are allowed to import the oracle)

DEC_KEYS = ["layers.0.weight", "layers.0.bias", "layers.1.weight", "layers.1.bias", "lout.weight", "lout.bias"]


def make_config(feat_levels=2, world_level=12, leaf_vox=0.2, device="cpu", **kw):
    from shine_mapping_b200.config import SHINEConfig
    base = dict(tree_level_world=world_level, tree_level_feat=feat_levels, leaf_vox_size=leaf_vox, device=device,
                surface_sample_range_m=0.3, surface_sample_n=3, free_sample_begin_ratio=0.3,
                free_sample_end_dist_m=0.8, free_sample_n=3, min_range=3.0, pc_radius=30.0)
    base.update(kw)
    return SHINEConfig(**base)


def make_case(n_points=3000, n_batch=2048, feat_levels=2, seed=0, n_frames=1, poly=True, weighted=False,
              reduction="mean", world_level=12, n_azimuth=None, feature_dim=8):
    """Seeded synthetic case on the CPU: scans -> samples -> oracle octree -> batch (with out-of-map and
    out-of-cube stragglers appended to exercise the miss / clamp rules)."""
    from shine_mapping_b200 import synth
    torch.manual_seed(seed)
    cfg = make_config(feat_levels, world_level, poly_int_on=poly, loss_weight_on=weighted, loss_reduction=reduction,
                      feature_dim=feature_dim)
    gen = torch.Generator().manual_seed(seed)
    n_az = n_azimuth or max(8, n_points // 40)
    dirs = synth.lidar_directions(n_az)
    boxes = synth.default_boxes()
    oct_o = orc.OracleOctree(world_level, feat_levels, cfg.feature_dim, cfg.feature_std, poly)
    frames, coords, labels, weights = [], [], [], []
    for f in range(n_frames):
        origin = torch.tensor([2.0 * f, 0.0, 0.0])
        hits = synth.raycast_scene(origin, dirs, boxes, cfg.min_range, cfg.pc_radius)
        c, l, w = synth.sample_rays(hits * cfg.scale, origin * cfg.scale, cfg, gen)
        surf = c[w > 0]
        frames.append(surf.numpy().copy())
        oct_o.update(surf)
        coords.append(c); labels.append(l); weights.append(w)
    pool_c, pool_l, pool_w = torch.cat(coords), torch.cat(labels), torch.cat(weights)
    idx = torch.randint(0, pool_c.shape[0], (n_batch,), generator=gen)
    coord, label, weight = pool_c[idx], pool_l[idx], pool_w[idx]
    # stragglers: far from the map (miss on every level), on / beyond the cube faces (clamp rule), exact voxel corners
    extra = torch.tensor([[0.9, 0.9, 0.9], [-1.0, -1.0, -1.0], [1.0, 1.0, 1.0], [1.25, -1.5, 0.0],
                          [0.0, 0.0, 0.0], [2.0 ** -11, 2.0 ** -11, 2.0 ** -11]], dtype=torch.float32)
    coord = torch.cat((coord, extra, surf[:10]))
    label = torch.cat((label, torch.zeros(extra.shape[0]), torch.zeros(10)))
    weight = torch.cat((weight, torch.ones(extra.shape[0]), torch.ones(10)))
    if weighted:  # make the weights non-trivial
        weight = weight * (0.5 + torch.rand(weight.shape[0], generator=gen))
    dec = orc.make_decoder_params(cfg.feature_dim, 32, 2, True)
    return {
        "cfg": dict(tree_level_world=world_level, tree_level_feat=feat_levels, feature_dim=cfg.feature_dim,
                    poly_int_on=poly, leaf_vox_size=cfg.leaf_vox_size, sigma=float(cfg.sigma_sigmoid),
                    weighted=weighted, reduction=reduction),
        "frames": frames,
        "tables": [t.detach().numpy().copy() for t in oct_o.hier_features],
        "dec": {k: v.detach().numpy().copy() for k, v in dec.items()},
        "coord": coord.numpy().copy(), "label": label.numpy().copy(), "weight": weight.numpy().copy(),
    }


def sort_case_morton(case, level=12):
    """The same batch in Morton order of its coordinates (what the sorted sample pool hands out)."""
    from shine_mapping_b200.feature_octree import points_to_morton, quantize_points
    order = torch.argsort(points_to_morton(quantize_points(torch.from_numpy(case["coord"]), level)), stable=True).numpy()
    out = dict(case)
    for k in ("coord", "label", "weight"):
        out[k] = np.ascontiguousarray(case[k][order])
    return out


def drop_relu_kink_points(case, eps=2e-6):
    """Remove the (very few) batch points that have a decoder pre-activation within `eps` of zero.  At a ReLU kink two
    fp32-grade implementations that sum in a different order can land on different sides; the gradient of that one point
    then differs by O(1) although both are right.  Found with the tcgen05 kernel on point 31 624 of seed 44 (layer-2
    pre-activation 6.4e-8); the parity bar is for points where the function is differentiable."""
    o, dec = oracle_from_case(case)
    with torch.no_grad():
        f = o.query_feature(torch.from_numpy(case["coord"])).double()
        a1 = f @ dec["layers.0.weight"].double().T + dec["layers.0.bias"].double()
        a2 = torch.relu(a1) @ dec["layers.1.weight"].double().T + dec["layers.1.bias"].double()
        keep = ((a1.abs().min(1).values > eps) & (a2.abs().min(1).values > eps)).numpy()
    out = dict(case)
    for k in ("coord", "label", "weight"):
        out[k] = case[k][keep].copy()
    return out, int((~keep).sum())


def oracle_from_case(case):
    """Rebuild the oracle octree by replaying the frames, then overwrite its tables with the case's."""
    c = case["cfg"]
    o = orc.OracleOctree(c["tree_level_world"], c["tree_level_feat"], c["feature_dim"], 0.05, c["poly_int_on"])
    for fr in case["frames"]:
        o.update(torch.from_numpy(np.asarray(fr)))
    assert [tuple(t.shape) for t in o.hier_features] == [tuple(t.shape) for t in case["tables"]], \
        "oracle row counts differ from the case's tables"
    o.hier_features = [torch.from_numpy(np.asarray(t).copy()).requires_grad_(True) for t in case["tables"]]
    dec = {k: torch.from_numpy(np.asarray(v).copy()).requires_grad_(True) for k, v in case["dec"].items()}
    return o, dec


def run_oracle_step(case):
    o, dec = oracle_from_case(case)
    c = case["cfg"]
    coord = torch.from_numpy(case["coord"]); label = torch.from_numpy(case["label"])
    weight = torch.from_numpy(case["weight"])
    res = orc.train_step(o, dec, coord, label, weight, c["sigma"], c["weighted"], c["reduction"])
    return {
        "indices": [t.numpy() for t in o.hierarchical_indices],
        "feature": res["feature"].numpy(), "pred": res["pred"].numpy(), "loss": float(res["loss"]),
        "table_grads": [g.numpy() for g in res["table_grads"]],
        "dec_grads": {k: g.numpy() for k, g in res["dec_grads"].items()},
    }


def build_cuda_models(case, device="cuda:0", freeze_decoder=False):
    """FeatureOctree grown by the package's own update() on the device + Decoder, tables/weights copied from the
    case (the RNG streams of CPU and CUDA differ, so values are copied; SHAPES must already agree)."""
    from shine_mapping_b200 import Decoder, FeatureOctree
    c = case["cfg"]
    cfg = make_config(c["tree_level_feat"], c["tree_level_world"], c["leaf_vox_size"], device=device,
                      poly_int_on=c["poly_int_on"], feature_dim=c["feature_dim"], loss_weight_on=c["weighted"],
                      loss_reduction=c["reduction"])
    octree = FeatureOctree(cfg)
    for fr in case["frames"]:
        octree.update(torch.from_numpy(np.asarray(fr)).to(device))
    shapes = [tuple(p.shape) for p in octree.hier_features]
    assert shapes == [tuple(t.shape) for t in case["tables"]], f"row counts differ: {shapes}"
    with torch.no_grad():
        for p, t in zip(octree.hier_features, case["tables"]):
            p.copy_(torch.from_numpy(np.asarray(t)))
    dec = Decoder(cfg)
    sd = dec.state_dict()
    for k in DEC_KEYS:
        sd[k] = torch.from_numpy(np.asarray(case["dec"][k])).to(device)
    dec.load_state_dict(sd)
    if freeze_decoder:
        for p in dec.parameters():
            p.requires_grad = False
    return cfg, octree, dec


def run_cuda_step(case, device="cuda:0", single_pass=True, tf32x1=False, unfused=False, morton_ordered=False,
                  freeze_decoder=False):
    from shine_mapping_b200 import sdf_bce_loss, sdf_bce_step
    cfg, octree, dec = build_cuda_models(case, device, freeze_decoder=freeze_decoder)
    c = case["cfg"]
    coord = torch.from_numpy(case["coord"]).to(device); label = torch.from_numpy(case["label"]).to(device)
    weight = torch.from_numpy(case["weight"]).to(device)
    indices = [t.cpu().numpy() for t in octree.get_indices(coord)]
    feature = octree.query_feature(coord)
    if unfused:   # class-surface path: query kernel + torch MLP + torch loss
        pred = dec.sdf(feature)
        loss = sdf_bce_loss(pred, label, c["sigma"], torch.abs(weight), c["weighted"], c["reduction"])
    else:
        loss, pred = sdf_bce_step(octree, dec, coord, label, c["sigma"], weight, c["weighted"], c["reduction"],
                                  single_pass=single_pass, tf32x1=tf32x1, return_pred=True, morton_ordered=morton_ordered)
    loss.backward()
    torch.cuda.synchronize()
    return {
        "indices": indices, "feature": feature.detach().cpu().numpy(), "pred": pred.detach().cpu().numpy(),
        "loss": float(loss.detach()),
        "table_grads": [p.grad.cpu().numpy() for p in octree.hier_features],
        "dec_grads": {} if freeze_decoder else {k: dict(dec.named_parameters())[k].grad.cpu().numpy() for k in DEC_KEYS},
    }


def _close(got, want, atol, rtol):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    err = np.abs(got - want) - (atol + rtol * np.abs(want))
    return float(err.max()) if err.size else -1.0


def compare_step(got, want, pred_atol=2e-5, pred_rtol=1e-5, grad_rel=2e-4, check_trash=False):
    """Assert parity; returns a one-line report of the worst deviations."""
    for lvl, (a, b) in enumerate(zip(got["indices"], want["indices"])):
        assert a.shape == b.shape and np.array_equal(a, b), f"indices differ at level index {lvl}"
    e_feat = _close(got["feature"], want["feature"], 2e-6, 1e-5)
    assert e_feat <= 0, f"feature mismatch (excess {e_feat:.3e})"
    e_pred = _close(got["pred"], want["pred"], pred_atol, pred_rtol)
    assert e_pred <= 0, f"pred mismatch (excess {e_pred:.3e})"
    rel_loss = abs(got["loss"] - want["loss"]) / max(abs(want["loss"]), 1e-12)
    assert rel_loss <= 2e-5 or pred_atol > 1e-4, f"loss mismatch {got['loss']} vs {want['loss']}"
    worst = 0.0
    for k, (a, b) in enumerate(zip(got["table_grads"], want["table_grads"])):
        if not check_trash:   # the trash-bin row's gradient is don't-care (re-zeroed before every query)
            a, b = a[:-1], b[:-1]
        scale = max(float(np.abs(b).max()), 1e-30)
        d = float(np.abs(a.astype(np.float64) - b).max()) / scale
        worst = max(worst, d)
        assert d <= grad_rel + 1e-10 / scale, f"table grad level {k}: rel err {d:.3e}"
    worst_d = 0.0
    for k in want["dec_grads"]:
        a, b = got["dec_grads"][k], want["dec_grads"][k]
        scale = max(float(np.abs(b).max()), 1e-30)
        d = float(np.abs(a.astype(np.float64) - b).max()) / scale
        worst_d = max(worst_d, d)
        assert d <= grad_rel + 1e-10 / scale, f"decoder grad {k}: rel err {d:.3e}"
    dp = float(np.abs(got["pred"] - want["pred"]).max())
    return (f"N={got['pred'].shape[0]} idx=exact max|dpred|={dp:.2e} rel_loss={rel_loss:.1e} "
            f"table_grad_rel={worst:.1e} dec_grad_rel={worst_d:.1e}")


GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
GOLDEN_NAMES = ["ref_c1_l2_mean", "ref_c2_l4_pretrained_frozen", "ref_incre_l3_sum_weighted_linear"]


def live_golden_name(levels, frames, poly):
    """Golden of the reference classes run on a `make_case` case (oracle/make_golden.py::make_live)."""
    return f"ref_live_l{levels}_f{frames}_{'poly' if poly else 'linear'}"


def load_golden(name):
    """-> (case, expected) frozen from the unmodified reference by oracle/make_golden.py."""
    import json
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    cfg = json.loads(str(z["cfg_json"]))
    L = cfg["tree_level_feat"]
    case = {
        "cfg": cfg,
        "frames": [z[f"frame_{i}"] for i in range(cfg["n_frames"])],
        "tables": [z[f"table_{k}"] for k in range(L)],
        "dec": {k: z["dec_" + k] for k in DEC_KEYS},
        "coord": z["coord"], "label": z["label"], "weight": z["weight"],
    }
    exp = {
        "indices": [z[f"exp_indices_{i}"].astype(np.int64) for i in range(L)],
        "feature": z["exp_feature"], "pred": z["exp_pred"], "loss": float(z["exp_loss"]),
        "table_grads": [z[f"exp_tgrad_{k}"] for k in range(L)],
        "dec_grads": {k: z["exp_dgrad_" + k] for k in DEC_KEYS if ("exp_dgrad_" + k) in z.files},
    }
    return case, exp
