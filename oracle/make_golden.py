"""Mint tests/golden/*.npz from the UNMODIFIED reference classes.  *** TEST INFRASTRUCTURE ***

Runs only in the build container (needs /root/reference; kaolin is replaced by oracle/kaolin_shim).  Imports the
reference's own `FeatureOctree`, `Decoder`, `sdf_bce_loss`, `dataSampler`, `SHINEConfig` verbatim and drives
them exactly like the loop body of shine_batch.py:123-209 on the CPU; the inputs and every output are frozen so
that the oracle restatement (tests/test_oracle_golden.py) and the CUDA path (tests/test_gpu_parity.py) can be
checked against the reference itself on the GPU box, where /root/reference does not exist.

    python oracle/make_golden.py            # rewrites tests/golden/*.npz
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("SHINE_REFERENCE", "/root/reference")
DEC_KEYS = ["layers.0.weight", "layers.0.bias", "layers.1.weight", "layers.1.bias", "lout.weight", "lout.bias"]


def import_reference():
    sys.path.insert(0, os.path.join(ROOT, "oracle", "kaolin_shim"))
    sys.path.insert(0, REF)
    from model.decoder import Decoder
    from model.feature_octree import FeatureOctree
    from utils.config import SHINEConfig
    from utils.data_sampler import dataSampler
    from utils.loss import sdf_bce_loss
    return SHINEConfig, FeatureOctree, Decoder, dataSampler, sdf_bce_loss


def reference_config(SHINEConfig, feat_levels, leaf_vox, poly, weighted, reduction):
    c = SHINEConfig()
    c.device = "cpu"
    c.tree_level_world, c.tree_level_feat, c.leaf_vox_size = 12, feat_levels, leaf_vox
    c.poly_int_on, c.loss_weight_on, c.loss_reduction = poly, weighted, reduction
    c.surface_sample_range_m, c.surface_sample_n = 0.3, 3
    c.free_sample_begin_ratio, c.free_sample_end_dist_m, c.free_sample_n = 0.3, 0.8, 3
    c.sigma_sigmoid_m = 0.1
    c.calculate_world_scale()
    return c


def make(name, feat_levels, n_frames, n_azimuth, n_batch, seed, poly=True, weighted=False, reduction="mean",
         pretrained=False, leaf_vox=0.2):
    SHINEConfig, FeatureOctree, Decoder, dataSampler, sdf_bce_loss = import_reference()
    sys.path.insert(0, ROOT)
    from shine_mapping_b200 import synth   # scene ray-caster only (inputs); everything after is the reference

    torch.manual_seed(seed)
    cfg = reference_config(SHINEConfig, feat_levels, leaf_vox, poly, weighted, reduction)
    octree, decoder, sampler = FeatureOctree(cfg), Decoder(cfg), dataSampler(cfg)
    if pretrained:   # BASELINE config 2: frozen geo_decoder_8dim (reference shine_batch.py:45-49)
        loaded = torch.load(os.path.join(REF, "pretrained", "geo_decoder_8dim.pth"), weights_only=False,
                            map_location="cpu")
        decoder.load_state_dict(loaded["geo_decoder"])
        for child in decoder.children():
            for p in child.parameters():
                p.requires_grad = False
    dirs, boxes = synth.lidar_directions(n_azimuth), synth.default_boxes()
    frames, pools = [], []
    for f in range(n_frames):
        origin = torch.tensor([2.0 * f, 0.0, 0.0])
        hits = synth.raycast_scene(origin, dirs, boxes, 3.0, 30.0)
        coord, label, _, _, weight, _, _ = sampler.sample(hits * cfg.scale, origin * cfg.scale, None, None)
        surface = coord[weight > 0, :]
        octree.update(surface, False)              # dataset/lidar_dataset.py:212-218
        frames.append(surface.numpy().copy())
        pools.append((coord, label, weight))
    pc = torch.cat([p[0] for p in pools]); pl = torch.cat([p[1] for p in pools]); pw = torch.cat([p[2] for p in pools])
    index = torch.randint(0, pc.shape[0], (n_batch,))   # dataset/lidar_dataset.py:431-448
    coord, label, weight = pc[index], pl[index], pw[index]
    extra = torch.tensor([[0.9, 0.9, 0.9], [-1.0, -1.0, -1.0], [1.0, 1.0, 1.0], [1.25, -1.5, 0.0],
                          [0.0, 0.0, 0.0], [2.0 ** -11, 2.0 ** -11, 2.0 ** -11]])
    coord = torch.cat((coord, extra, torch.from_numpy(frames[-1][:10])))
    label = torch.cat((label, torch.zeros(16)))
    weight = torch.cat((weight, torch.ones(16)))
    if weighted:
        weight = weight * (0.5 + torch.rand(weight.shape[0]))
    sigma = cfg.logistic_gaussian_ratio * cfg.sigma_sigmoid_m * cfg.scale   # shine_batch.py:87

    tables_before = [p.detach().numpy().copy() for p in octree.hier_features]
    # ---- the loop body, shine_batch.py:123,128,172-174,209 ----
    feature = octree.query_feature(coord)
    pred = decoder.sdf(feature)
    loss = sdf_bce_loss(pred, label, sigma, torch.abs(weight), cfg.loss_weight_on, cfg.loss_reduction)
    loss.backward()

    out = {
        "cfg_json": np.array(json.dumps(dict(
            tree_level_world=12, tree_level_feat=feat_levels, feature_dim=cfg.feature_dim, poly_int_on=poly,
            leaf_vox_size=leaf_vox, sigma=float(sigma), weighted=weighted, reduction=reduction,
            decoder_frozen=pretrained, n_frames=n_frames))),
        "coord": coord.numpy(), "label": label.numpy(), "weight": weight.numpy(),
        "exp_feature": feature.detach().numpy(), "exp_pred": pred.detach().numpy(),
        "exp_loss": np.array(float(loss)),
    }
    for i, fr in enumerate(frames):
        out[f"frame_{i}"] = fr
    # set_zero() ran inside query_feature; tables_before already had zero trash rows (update writes them)
    for k, t in enumerate(tables_before):
        out[f"table_{k}"] = t
        out[f"exp_tgrad_{k}"] = octree.hier_features[k].grad.numpy()
    for i, idx in enumerate(octree.hierarchical_indices):
        out[f"exp_indices_{i}"] = idx.numpy().astype(np.int32)
    sd = decoder.state_dict()
    params = dict(decoder.named_parameters())
    for k in DEC_KEYS:
        out["dec_" + k] = sd[k].numpy()
        if params[k].grad is not None:
            out["exp_dgrad_" + k] = params[k].grad.numpy()
    path = os.path.join(ROOT, "tests", "golden", name + ".npz")
    np.savez_compressed(path, **out)
    print(f"{name}: N={coord.shape[0]} rows={[t.shape[0] for t in tables_before]} loss={float(loss):.6f} "
          f"-> {path} ({os.path.getsize(path) / 1e6:.2f} MB)")


def make_eikonal(name, feat_levels, n_azimuth, n_batch, seed, poly=True, weight_e=0.1):
    """Loop body with ekional_loss_on: the reference's get_gradient (utils/tools.py:175-185 — restated inline because
    utils/tools.py imports open3d) on the reference's own FeatureOctree / Decoder, shine_batch.py:119-120,137-142,172-185."""
    SHINEConfig, FeatureOctree, Decoder, dataSampler, sdf_bce_loss = import_reference()
    sys.path.insert(0, ROOT)
    from shine_mapping_b200 import synth
    torch.manual_seed(seed)
    cfg = reference_config(SHINEConfig, feat_levels, 0.2, poly, False, "mean")
    octree, decoder, sampler = FeatureOctree(cfg), Decoder(cfg), dataSampler(cfg)
    dirs, boxes = synth.lidar_directions(n_azimuth), synth.default_boxes()
    origin = torch.zeros(3)
    hits = synth.raycast_scene(origin, dirs, boxes, 3.0, 30.0)
    coord, label, _, _, weight, _, _ = sampler.sample(hits * cfg.scale, origin * cfg.scale, None, None)
    surface = coord[weight > 0, :]
    octree.update(surface, False)
    index = torch.randint(0, coord.shape[0], (n_batch,))
    coord, label, weight = coord[index].clone(), label[index], weight[index]
    sigma = cfg.logistic_gaussian_ratio * cfg.sigma_sigmoid_m * cfg.scale
    tables_before = [p.detach().numpy().copy() for p in octree.hier_features]
    coord.requires_grad_(True)                                             # shine_batch.py:119-120
    feature = octree.query_feature(coord)
    pred = decoder.sdf(feature)
    surface_mask = weight > 0
    g = torch.autograd.grad(outputs=pred, inputs=coord, grad_outputs=torch.ones_like(pred), create_graph=True,
                            retain_graph=True, only_inputs=True)[0] * sigma   # get_gradient(coord, pred) * sigma_sigmoid
    loss = sdf_bce_loss(pred, label, sigma, torch.abs(weight), False, "mean")
    eikonal = ((1.0 - g[surface_mask].norm(2, dim=-1)) ** 2).mean()          # shine_batch.py:183-185
    total = loss + weight_e * eikonal
    total.backward()
    out = {"cfg_json": np.array(json.dumps(dict(tree_level_world=12, tree_level_feat=feat_levels, feature_dim=cfg.feature_dim,
                                                 poly_int_on=poly, leaf_vox_size=0.2, sigma=float(sigma), weighted=False,
                                                 reduction="mean", decoder_frozen=False, n_frames=1, weight_e=weight_e))),
           "frame_0": surface.numpy().copy(), "coord": coord.detach().numpy(), "label": label.numpy(), "weight": weight.numpy(),
           "exp_g": g.detach().numpy(), "exp_eikonal": np.array(float(eikonal)), "exp_loss": np.array(float(total)),
           "exp_pred": pred.detach().numpy()}
    for k, t in enumerate(tables_before):
        out[f"table_{k}"] = t
        out[f"exp_tgrad_{k}"] = octree.hier_features[k].grad.numpy()
    sd, params = decoder.state_dict(), dict(decoder.named_parameters())
    for k in DEC_KEYS:
        out["dec_" + k] = sd[k].numpy()
        out["exp_dgrad_" + k] = params[k].grad.numpy()
    path = os.path.join(ROOT, "tests", "golden", name + ".npz")
    np.savez_compressed(path, **out)
    print(f"{name}: N={coord.shape[0]} eikonal={float(eikonal):.6f} loss={float(total):.6f} -> {path} "
          f"({os.path.getsize(path) / 1e6:.2f} MB)")


def make_live(levels, frames, poly, sample_rows=64):
    """The reference classes on a seeded `tests.parity_utils.make_case` case (the oracle's initial tables and decoder
    copied in), frozen for tests/test_reference_live.py.  The table gradients are kept small: per level the set of rows
    with a nonzero gradient (bit-packed), one weighted sum over the features of each of those rows (seeded weights), and
    a fixed seeded sample of whole rows plus the trash row."""
    SHINEConfig, FeatureOctree, Decoder, _, sdf_bce_loss = import_reference()
    sys.path.insert(0, ROOT)
    from tests.parity_utils import live_golden_name, make_case
    case = make_case(n_points=1200, n_batch=1000, feat_levels=levels, seed=77 + levels, n_frames=frames, poly=poly)
    c = SHINEConfig(); c.device = "cpu"
    c.tree_level_world, c.tree_level_feat, c.leaf_vox_size, c.poly_int_on = 12, levels, 0.2, poly
    c.calculate_world_scale()
    octree, dec = FeatureOctree(c), Decoder(c)
    for fr in case["frames"]:
        octree.update(torch.from_numpy(fr), False)
    assert [tuple(p.shape) for p in octree.hier_features] == [t.shape for t in case["tables"]]
    with torch.no_grad():
        for p, t in zip(octree.hier_features, case["tables"]):
            p.copy_(torch.from_numpy(t))
    sd = dec.state_dict()
    for k, v in case["dec"].items():
        sd[k] = torch.from_numpy(v)
    dec.load_state_dict(sd)
    coord, label = torch.from_numpy(case["coord"]), torch.from_numpy(case["label"])
    pred = dec.sdf(octree.query_feature(coord))
    loss = sdf_bce_loss(pred, label, case["cfg"]["sigma"], None, False, "mean")
    loss.backward()
    out = {"table_rows": np.array([p.shape[0] for p in octree.hier_features]),
           "exp_pred": pred.detach().numpy(), "exp_loss": np.array(float(loss.detach()))}
    rng = np.random.default_rng(0)
    out["tgrad_row_weights"] = w = rng.uniform(0.5, 1.5, case["cfg"]["feature_dim"])
    for k, p in enumerate(octree.hier_features):
        g = p.grad.numpy()
        touched = np.abs(g).sum(1) > 0
        nz = np.flatnonzero(touched)
        rows = np.union1d(rng.choice(nz, min(nz.size, sample_rows), replace=False), [g.shape[0] - 1])
        out[f"exp_tgrad_touched_{k}"] = np.packbits(touched)
        out[f"exp_tgrad_rows_{k}"] = rows.astype(np.int32)
        out[f"exp_tgrad_{k}"] = g[rows]
        out[f"exp_tgrad_rowsum_{k}"] = (g[nz].astype(np.float64) @ w).astype(np.float32)
    for i, idx in enumerate(octree.hierarchical_indices):
        assert int(idx.max()) < 2 ** 15
        out[f"exp_indices_{i}"] = idx.numpy().astype(np.int16)
    path = os.path.join(ROOT, "tests", "golden", live_golden_name(levels, frames, poly) + ".npz")
    np.savez_compressed(path, **out)
    print(f"{path}: N={coord.shape[0]} loss={float(loss.detach()):.6f} ({os.path.getsize(path) / 1e6:.3f} MB)")


if __name__ == "__main__":
    if not os.path.isdir(REF):
        sys.exit(f"{REF} not found: goldens can only be minted where the reference is mounted")
    make("ref_c1_l2_mean", feat_levels=2, n_frames=1, n_azimuth=14, n_batch=1500, seed=42)
    make("ref_c2_l4_pretrained_frozen", feat_levels=4, n_frames=1, n_azimuth=12, n_batch=1500, seed=43,
         pretrained=True)
    make("ref_incre_l3_sum_weighted_linear", feat_levels=3, n_frames=2, n_azimuth=10, n_batch=1200, seed=44,
         poly=False, weighted=True, reduction="sum")
    make_eikonal("ref_eikonal_l3", feat_levels=3, n_azimuth=10, n_batch=1000, seed=45)
    for levels, frames, poly in [(2, 1, True), (4, 2, True), (3, 2, False)]:
        make_live(levels, frames, poly)
