"""Comparison helpers shared by the parity tests, smoke() and bench.py."""
from __future__ import annotations

import hashlib
from typing import Dict

import numpy as np


def layer_digest(indices: np.ndarray, voxels: np.ndarray, updated: np.ndarray = None) -> str:
    """SHA-256 of a layer: its sorted block indices, the voxel bytes of those blocks in that order and, when
    given, their updated bits.  Equal digests mean bit-identical layers."""
    h = hashlib.sha256()
    h.update(np.ascontiguousarray(indices, dtype=np.int32).tobytes())
    h.update(np.ascontiguousarray(voxels).tobytes())
    if updated is not None:
        h.update(np.ascontiguousarray(updated, dtype=np.uint8).tobytes())
    return h.hexdigest()


def device_layer_digest(layer, with_updated: bool = False) -> str:
    """layer_digest of a GPU Layer (voxblox_b200.Layer)."""
    idx = layer.getAllAllocatedBlocks()
    vox, upd = layer.getBlocks(idx)
    return layer_digest(idx, vox, upd if with_updated else None)


def oracle_layer_digest(omap, layer: int = 0, with_updated: bool = False) -> str:
    """layer_digest of an oracle map's TSDF (0) or ESDF (1) layer."""
    idx = omap.block_indices(layer)
    blocks = [omap.block(i, layer) for i in idx]
    vox = np.stack([b[0] for b in blocks]) if blocks else np.zeros(0)
    upd = np.array([b[1] for b in blocks], dtype=np.uint8)
    return layer_digest(idx, vox, upd if with_updated else None)


def rel_err(a: np.ndarray, b: np.ndarray, floor: float) -> np.ndarray:
    """|a - b| / max(|b|, floor): relative error with an absolute floor for values near 0."""
    return np.abs(a.astype(np.float64) - b.astype(np.float64)) / np.maximum(np.abs(b.astype(np.float64)), floor)


def compare_tsdf(layer, omap, dist_floor: float = None) -> Dict:
    """GPU Layer (voxblox_b200.Layer) against an oracle map (oracle.pyoracle.OracleMap).

    Block sets must be identical (allocation is exact); distances and weights are
    compared relatively (north_star: 1e-4), colours exactly."""
    gi = layer.getAllAllocatedBlocks()
    oi = omap.block_indices()
    rep = {"gpu_blocks": int(len(gi)), "oracle_blocks": int(len(oi)),
           "blocks_equal": gi.shape == oi.shape and bool((gi == oi).all())}
    if not rep["blocks_equal"]:
        return rep
    gv, gupd = layer.getBlocks(gi)
    ov = np.stack([omap.block(i)[0] for i in oi]) if len(oi) else gv
    oupd = np.array([omap.block(i)[1] for i in oi], dtype=np.uint8)
    floor = dist_floor if dist_floor is not None else 1e-3 * layer.voxel_size()
    de = rel_err(gv["distance"], ov["distance"], floor)
    we = rel_err(gv["weight"], ov["weight"], 1e-12)
    obs = ov["weight"] > 0
    rep.update({
        "voxels_observed": int(obs.sum()),
        "observed_equal": bool(((gv["weight"] > 0) == obs).all()),
        "max_rel_err_distance": float(de.max()) if de.size else 0.0,
        "max_rel_err_weight": float(we.max()) if we.size else 0.0,
        "n_dist_over_1e-4": int((de > 1e-4).sum()),
        "n_bit_exact": int(((gv["distance"] == ov["distance"]) & (gv["weight"] == ov["weight"])).sum()),
        "n_voxels": int(gv.size),
        "color_mismatch": int((gv["color"] != ov["color"]).any(axis=-1).sum()),
        "updated_equal": bool((gupd == oupd).all()),
    })
    rep["max_rel_err"] = max(rep["max_rel_err_distance"], rep["max_rel_err_weight"])
    return rep


def compare_oracles(a, b) -> Dict:
    """Two oracle maps (e.g. the reference at 4 threads against the reference at 1 thread)."""
    ai, bi = a.block_indices(), b.block_indices()
    rep = {"blocks_equal": ai.shape == bi.shape and bool((ai == bi).all())}
    if not rep["blocks_equal"]:
        return rep
    av = np.stack([a.block(i)[0] for i in ai])
    bv = np.stack([b.block(i)[0] for i in bi])
    obs = bv["weight"] > 0
    de = rel_err(av["distance"], bv["distance"], 1e-3 * b.voxel_size)
    we = rel_err(av["weight"], bv["weight"], 1e-12)
    rep.update({"voxels_observed": int(obs.sum()),
                "frac_over_1e-4": float(((de > 1e-4) | (we > 1e-4))[obs].mean()) if obs.any() else 0.0,
                "max_abs_dist_diff": float(np.abs(av["distance"].astype(np.float64) - bv["distance"]).max()),
                "color_mismatch_frac": float((av["color"] != bv["color"]).any(axis=-1)[obs].mean()) if obs.any() else 0.0,
                "n_bit_exact": int(((av["distance"] == bv["distance"]) & (av["weight"] == bv["weight"])).sum()),
                "n_voxels": int(av.size)})
    return rep


def compare_esdf(layer, omap, max_distance: float) -> Dict:
    """GPU ESDF Layer against the oracle's ESDF layer (layer id 1)."""
    gi = layer.getAllAllocatedBlocks()
    oi = omap.block_indices(1)
    rep = {"gpu_blocks": int(len(gi)), "oracle_blocks": int(len(oi)),
           "blocks_equal": gi.shape == oi.shape and bool((gi == oi).all())}
    if not rep["blocks_equal"]:
        return rep
    gv, gupd = layer.getBlocks(gi)
    ov = np.stack([omap.block(i, 1)[0] for i in oi]) if len(oi) else gv
    oupd = np.array([omap.block(i, 1)[1] for i in oi], dtype=np.uint8)
    obs = ov["observed"] != 0
    d_g, d_o = gv["distance"][obs].astype(np.float64), ov["distance"][obs].astype(np.float64)
    err = np.abs(d_g - d_o)
    rel = err / np.maximum(np.abs(d_o), 1e-3 * layer.voxel_size())
    rep.update({
        "voxels_observed": int(obs.sum()),
        "observed_equal": bool(((gv["observed"] != 0) == obs).all()),
        "fixed_equal": bool((gv["fixed"][obs] == ov["fixed"][obs]).all()),
        "hallucinated_equal": bool((gv["hallucinated"] == ov["hallucinated"]).all()),
        "in_queue_gpu": int((gv["in_queue"] != 0).sum()), "in_queue_oracle": int((ov["in_queue"] != 0).sum()),
        "n_bit_exact": int((gv["distance"][obs] == ov["distance"][obs]).sum()),
        "n_over_1e-4": int((rel > 1e-4).sum()),
        "max_rel_err": float(rel.max()) if rel.size else 0.0,
        "max_abs_err": float(err.max()) if err.size else 0.0,
        "rmse": float(np.sqrt(np.mean(err ** 2))) if err.size else 0.0,
        "parent_mismatch": int((gv["parent"][obs] != ov["parent"][obs]).any(axis=-1).sum()),
        "updated_equal": bool((gupd == oupd).all()),
        "flag_bytes_clean": bool((gv["in_queue"] <= 1).all() and (gv["observed"] <= 1).all()),
    })
    return rep
