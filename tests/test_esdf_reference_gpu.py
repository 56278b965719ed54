"""-m gpu: the device ESDF against the REFERENCE's own EsdfIntegrator (oracle/_ref), at the
configurations the reference itself uses.  The reference's results on these inputs are stored by
tests/golden/make_reference_golden.py: its block set and the observed / fixed flags and distance signs of
every observed voxel exactly, its distances on a seeded sample of observed voxels (all of them on the small
room, 8192 of ~47 000 on the full one) from which the error statistics below are computed.

What can and cannot be identical (DESIGN.md "ESDF"): the reference's processOpenSet
(esdf_integrator.cc:371-496) is a sequential bucket-queue algorithm.
 * min_diff_m = 0 (its own tests, test_sdf_integrators.cc:200): same-sign propagation converges to
   the unique least fixed point of the relaxation rule whatever the visiting order -- the device must
   be BIT-EXACT there.  Where a voxel borders a voxel of the opposite sign the reference ASSIGNS
   sign*dist in pop order (cc:458-488, last writer wins); the device keeps the candidate nearest the
   surface.  Those voxels, and what is propagated from them, may differ by at most a few voxel steps.
 * min_diff_m = 1e-3 (ros_params.h default): a voxel keeps its value unless a candidate improves it
   by more than min_diff, so the reference's own result depends on its pop order at the millimetre
   level; the device result must stay inside that band (|difference| <= a few min_diff) except at the
   sign-conflict voxels above.
The numbers asserted below are measured values plus a margin; every run prints the measured ones.
Also checked: the reference's own acceptance criteria against analytic ground truth
(test_sdf_integrators.cc:247-272) on the device layers, with the reference's errors beside them."""
import math

import numpy as np
import pytest

import voxblox_b200 as vb
from tests.golden import make_reference_golden as mr
from tests.parity import device_layer_digest
from voxblox_b200 import scenes

pytestmark = pytest.mark.gpu


def _pair(voxel, trunc, ekw):
    cfg = vb.TsdfIntegratorConfig(default_truncation_distance=trunc, integrator_threads=1)
    tsdf = vb.Layer(voxel, 16)
    integ = vb.TsdfIntegratorFactory.create("merged", cfg, tsdf)
    esdf = vb.Layer(voxel, 16, voxel_type="esdf")
    eint = vb.EsdfIntegrator(vb.EsdfIntegratorConfig(**ekw), tsdf, esdf)
    return tsdf, integ, esdf, eint


def _diff_stats(esdf, ref, voxel, min_diff):
    """The device ESDF layer against the reference's stored one (mr.esdf_golden): flags and signs over every
    observed voxel, distance errors over the stored sample."""
    gi = esdf.getAllAllocatedBlocks()
    assert gi.shape == ref["blocks"].shape and (gi == ref["blocks"]).all()
    gv, _ = esdf.getBlocks(gi)
    obs = np.unpackbits(ref["observed"], count=gv.size).reshape(gv.shape).astype(bool)
    assert ((gv["observed"] != 0) == obs).all()
    assert (gv["fixed"][obs] == ref["fixed"]).all()
    dg_all = gv["distance"][obs].astype(np.float64)
    dg, do = dg_all[ref["sample"]], ref["distance"].astype(np.float64)
    err = np.abs(dg - do)
    rel = err / np.maximum(np.abs(do), 1e-3 * voxel)
    return {"observed": int(obs.sum()), "sampled": int(do.size), "bit_exact": float((dg == do).mean()),
            "within_1e-4_rel": float((rel <= 1e-4).mean()),
            "within_2_min_diff": float((err <= 2 * min_diff + 1e-7).mean()) if min_diff > 0 else None,
            "within_one_voxel": float((err <= voxel * 1.0001).mean()),
            "max_abs_err_m": float(err.max()), "rmse_m": float(np.sqrt((err ** 2).mean())),
            "sign_equal": float((np.sign(dg_all) == ref["sign"]).mean())}


def _run_incremental(config, scene, sc, ekw):
    name = f"{config}_{scene}"
    scans = sc["scans"]()
    mr.require_inputs(scans, mr.golden("esdf", name))
    tsdf, integ, esdf, eint = _pair(sc["voxel"], sc["trunc"], ekw)
    for s in scans:
        integ.integratePointCloud((s[2], s[3]), s[0], s[1])
        eint.updateFromTsdfLayer(True)
    assert device_layer_digest(tsdf) == mr.golden("esdf", name)["tsdf"]   # the TSDF maps are bit-identical
    return _diff_stats(esdf, mr.esdf_golden(name), sc["voxel"], ekw["min_diff_m"])


ROOM_SMALL = dict(voxel=0.1, trunc=0.4, scans=lambda: scenes.c3_room_sequence(n_scans=4, width=160, height=120))
ROOM_FULL = dict(voxel=0.05, trunc=0.2, scans=lambda: [scenes.c3_room_scan(i) for i in range(2)])


@pytest.mark.parametrize("scene", ["room_small", "room_full_640x480"])
def test_esdf_reference_test_config_min_diff_zero(scene):
    """The reference's own test configuration (min_diff 0, multi_queue): incremental update after every scan."""
    sc = ROOM_SMALL if scene == "room_small" else ROOM_FULL
    ekw = dict(max_distance_m=2.0, default_distance_m=2.0, min_distance_m=sc["trunc"] / 2, min_diff_m=0.0, multi_queue=1)
    st = _run_incremental("min_diff_zero", scene, sc, ekw)
    print(scene, "min_diff=0 incremental:", st)
    # measured on B200 (profiles/r2_esdf_parity.json; the device result varies a little from run to run where
    # two sources race for a sign-conflict voxel): room_small 95.7-95.9 % within 1e-4, 99.9 % within one voxel,
    # rmse 0.16-0.19 voxel, max 0.93 m; room_full 97.0-97.2 % / 99.99 % / 0.07-0.11 voxel / 0.36-0.94 m
    assert st["sign_equal"] == 1.0, st
    assert st["within_1e-4_rel"] >= 0.94, st
    assert st["within_one_voxel"] >= 0.995, st
    assert st["rmse_m"] <= 0.3 * sc["voxel"], st
    assert st["max_abs_err_m"] < 2.0, st   # a handful of voxels (which source wins a race): bounded by max_distance_m only


@pytest.mark.parametrize("scene", ["room_small", "room_full_640x480"])
def test_esdf_ros_default_config(scene):
    """voxblox_ros defaults (ros_params.h:129-160): min_diff_m 1e-3, single queue, min_distance = truncation / 2 --
    the configuration bench.py's `downstream` section times."""
    sc = ROOM_SMALL if scene == "room_small" else ROOM_FULL
    md = 1e-3
    ekw = dict(max_distance_m=2.0, default_distance_m=2.0, min_distance_m=sc["trunc"] / 2, min_diff_m=md, multi_queue=0)
    st = _run_incremental("ros_default", scene, sc, ekw)
    print(scene, "ROS default config incremental:", st)
    # measured on B200: room_small 95.9 % within 1e-4 relative, 96.2 % within 2 min_diff, 99.9 % within one voxel,
    # rmse 0.19 voxel, max 9.3 voxels; room_full 96.0 % / 96.7 % / 99.996 % / 0.057 voxel / 1.2 voxels
    assert st["sign_equal"] == 1.0, st
    assert st["within_2_min_diff"] >= 0.94, st
    assert st["within_one_voxel"] >= 0.995, st
    assert st["rmse_m"] <= 0.3 * sc["voxel"], st
    assert st["max_abs_err_m"] < 2.0, st   # a handful of voxels (which source wins a race): bounded by max_distance_m only


# ------------------------------------------------------------------ analytic ground truth
def _world_sdf(p):
    """Signed distance of the reference test's world (test_sdf_integrators.cc:28-47): a cylinder of radius 2 and
    height 4 standing on the ground plane z = 0 (negative inside the cylinder and below the ground)."""
    x, y, z = p[..., 0], p[..., 1], p[..., 2]
    r = np.sqrt(x * x + y * y) - 2.0
    h = np.abs(z - 2.0) - 2.0
    outside = np.sqrt(np.maximum(r, 0) ** 2 + np.maximum(h, 0) ** 2)
    inside = np.minimum(np.maximum(r, h), 0.0)
    cyl = outside + inside
    return np.minimum(cyl, z)


def _gt_scans(n_views=16, width=160, height=120):
    prims = [scenes.CylinderZ((0.0, 0.0), 2.0, 0.0, 4.0), scenes.Plane((0.0, 0.0, 1.0), 0.0)]
    fx = (width / 2) / math.tan(math.radians(150.0) / 2)   # fov_h 2.61799 rad, test_sdf_integrators.cc:36
    dirs = scenes.pinhole_dirs(width, height, fx, fx, width / 2, height / 2)
    out = []
    for i in range(n_views):
        ang = 2 * math.pi * i / n_views
        pos = np.array([6.0 * math.cos(ang), 6.0 * math.sin(ang), 2.0])
        q = scenes.look_at(pos, (0.0, 0.0, 1.4))            # facing the cylinder, pitched down a bit (cc:66-68)
        out.append(scenes.render(prims, dirs, q, pos, min_range=0.5, max_range=10.0))
    return out


def _gt_errors(layer_blocks, voxel, max_d):
    errs = []
    for idx, vox in layer_blocks.items():
        obs = vox["observed"] != 0
        if not obs.any():
            continue
        lin = np.nonzero(obs)[0]
        lx, ly, lz = lin & 15, (lin >> 4) & 15, lin >> 8
        centre = (np.stack([lx, ly, lz], 1) + np.asarray(idx) * 16 + 0.5) * voxel
        gt = np.clip(_world_sdf(centre), -max_d, max_d)
        errs.append(np.abs(vox["distance"][lin].astype(np.float64) - gt))
    e = np.concatenate(errs)
    return {"voxels": int(e.size), "min_error": float(e.min()), "max_error": float(e.max()), "rmse": float(np.sqrt((e ** 2).mean()))}


@pytest.mark.parametrize("voxel", [0.2, 0.1])
def test_esdf_reference_acceptance_criteria_vs_ground_truth(voxel):
    """SdfIntegratorsTest.EsdfIntegrators (test_sdf_integrators.cc:180-272) on the device: incremental and batch ESDF
    of a cylinder on a ground plane against the analytic distance field; the reference's own EsdfIntegrator is run
    beside it (its errors are stored) and must not be better than the device by more than a hair."""
    trunc, max_d = 4 * voxel, 4.0
    ekw = dict(max_distance_m=max_d, default_distance_m=max_d, min_distance_m=trunc / 2, min_diff_m=0.0, multi_queue=1)
    scans = _gt_scans()
    gold = mr.golden("esdf_ground_truth", str(voxel))
    mr.require_inputs(scans, gold)
    ref_inc, ref_bat = gold["incremental"], gold["batch"]
    tsdf, integ, esdf_inc, e_inc = _pair(voxel, trunc, ekw)
    for s in scans:
        integ.integratePointCloud((s[2], s[3]), s[0], s[1])
        e_inc.updateFromTsdfLayer(True)
    inc = _gt_errors(esdf_inc.blocks(), voxel, max_d)
    # batch, on a second ESDF layer over the same TSDF map
    tsdf2, integ2, esdf_b, e_b = _pair(voxel, trunc, ekw)
    for s in scans:
        integ2.integratePointCloud((s[2], s[3]), s[0], s[1])
    e_b.updateFromTsdfLayerBatch()
    bat = _gt_errors(esdf_b.blocks(), voxel, max_d)
    print("voxel", voxel, "device incremental", inc, "| reference incremental", ref_inc)
    print("voxel", voxel, "device batch", bat, "| reference batch", ref_bat)
    for r in (inc, bat):
        assert r["min_error"] <= 1e-4                      # EXPECT_NEAR(min_error, 0, 1e-4)
        assert r["max_error"] < max_d                      # EXPECT_LT(max_error, esdf_max_distance_)
        assert r["rmse"] < max_d * voxel                   # EXPECT_LT(rmse, esdf_max_distance_ * voxel_size_)
    assert inc["voxels"] == bat["voxels"]                  # EXPECT_EQ(num_overlapping_voxels)
    assert abs(inc["rmse"] - bat["rmse"]) <= 1e-2          # kKindaSimilar
    assert abs(inc["max_error"] - bat["max_error"]) <= 1.0  # kCloseEnough
    # and against the reference's own result on the same input
    assert inc["voxels"] == ref_inc["voxels"] and bat["voxels"] == ref_bat["voxels"]
    assert inc["rmse"] <= ref_inc["rmse"] * 1.02 + 1e-4
    assert bat["rmse"] <= ref_bat["rmse"] * 1.02 + 1e-4
