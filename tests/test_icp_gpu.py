"""-m gpu: ICP pose refinement (SURVEY.md section 8f N4) on the device against the REFERENCE's own
voxblox::ICP (src/alignment/icp.cc compiled where it lies, oracle/_ref) and against the restatement.

What is compared: the refined pose T_tsdf_sensor and the number of fused mini batches (runICP's return
value).  ICP is float work end to end (SVD, SE(3) log / exp with libm functions), a chain of thousands of
dependent fusions: the bound is the north-star float tolerance, 1e-4 -- absolute on the unit quaternion's
coefficients, relative to max(1, |t|) on the translation -- not bit identity.  The TSDF maps the two sides
match against ARE bit identical (Merged, asserted).

num_threads = 1 is the reference's only deterministic setting and is compared with the reference itself (its
map digest and refined poses, stored by tests/golden/make_reference_golden.py); num_threads = T > 1 is compared with the restatement's round-robin schedule (oracle/vbo_api.h), which the
device implements with T warps."""
import numpy as np
import pytest

import voxblox_b200 as vb
from oracle import pyoracle as po
from tests.golden import make_reference_golden as mr
from tests.parity import compare_tsdf, device_layer_digest
from voxblox_b200 import scenes

pytestmark = pytest.mark.gpu

TOL = 1e-4


def _device_map(voxel, trunc, scans):
    cfg = vb.TsdfIntegratorConfig(default_truncation_distance=trunc, integrator_threads=1)
    layer = vb.Layer(voxel, 16)
    integ = vb.TsdfIntegratorFactory.create("merged", cfg, layer)
    for s in scans:
        integ.integratePointCloud((s[2], s[3]), s[0], s[1])
    return layer


def _maps(which, voxel, trunc, scans):
    layer = _device_map(voxel, trunc, scans)
    omap = po.OracleMap(po.OracleLib(which), po.TsdfConfig(default_truncation_distance=trunc, integrator_threads=1), voxel, 16)
    for s in scans:
        omap.integrate(po.MERGED, s)
    rep = compare_tsdf(layer, omap)
    assert rep["blocks_equal"] and rep["n_bit_exact"] == rep["n_voxels"], rep
    return layer, omap


def _close(dev, ref):
    (nd, (qd, td)), (qr, tr, nr) = dev, ref
    dq = float(np.abs(qd - qr).max())
    dt = float(np.abs(td - tr).max() / max(1.0, float(np.abs(tr).max())))
    return {"updates": (nd, nr), "dq": dq, "dt_rel": dt}


def _perturbed(s, dt, yaw):
    """s's pose, translated by dt and rotated by `yaw` rad about the world z axis."""
    q = np.asarray(s[2], np.float64)
    h = np.array([np.cos(yaw / 2), 0.0, 0.0, np.sin(yaw / 2)])
    w = np.array([h[0] * q[0] - h[3] * q[3], h[0] * q[1] - h[3] * q[2], h[0] * q[2] + h[3] * q[1], h[0] * q[3] + h[3] * q[0]])
    return w.astype(np.float32), (np.asarray(s[3], np.float64) + np.asarray(dt)).astype(np.float32)


# (translation, yaw) added to the fourth scan's true pose before refinement
PERTURBATIONS = [((0, 0, 0), 0.0), ((0.03, -0.02, 0.01), 0.0), ((-0.02, 0.03, 0.0), 0.01)]


@pytest.mark.parametrize("refine_roll_pitch", [0, 1])
def test_icp_one_thread_against_the_reference(refine_roll_pitch):
    """640 x 480 room scans at 0.05 m (the bench workload): map of three scans, the fourth cloud refined from
    its true pose and from two perturbed ones."""
    ss = [scenes.c3_room_scan(i) for i in range(4)]
    gold = mr.golden("icp", f"refine_roll_pitch_{refine_roll_pitch}")
    mr.require_inputs(ss, gold)
    layer = _device_map(0.05, 0.2, ss[:3])
    assert device_layer_digest(layer) == gold["map"]   # bit-identical to the reference's map
    s = ss[3]
    for k, ((dt, yaw), g) in enumerate(zip(PERTURBATIONS, gold["runs"])):
        q0, t0 = _perturbed(s, dt, yaw)
        dev = vb.ICP(vb.ICPConfig(refine_roll_pitch=refine_roll_pitch)).runICP(layer, s[0], (q0, t0), seed=7 + k)
        ref = (np.array([float.fromhex(v) for v in g["q_wxyz"]], np.float32),
               np.array([float.fromhex(v) for v in g["t"]], np.float32), g["num_updates"])
        rep = _close(dev, ref)
        err0 = float(np.abs(t0 - s[3]).max())
        err1 = float(np.abs(dev[1][1] - s[3]).max())
        print("refine_roll_pitch", refine_roll_pitch, "perturbation", dt, yaw, rep, "translation error", err0, "->", err1)
        assert rep["dq"] <= TOL and rep["dt_rel"] <= TOL, rep
        assert abs(rep["updates"][0] - rep["updates"][1]) <= max(2, rep["updates"][1] // 1000), rep
        if err0 > 0.01:
            assert err1 < 0.5 * err0   # the refinement pulls the pose back


@pytest.mark.parametrize("threads", [1, 4, 32])
def test_icp_round_robin_threads_against_the_restatement(threads):
    ss = list(scenes.c3_room_sequence(n_scans=4, width=320, height=240))
    layer, omap = _maps("port", 0.1, 0.4, ss[:3])
    s = ss[3]
    q0, t0 = _perturbed(s, (0.05, -0.04, 0.02), 0.01)
    for mb, ratio in ((20, 0.8), (50, 0.5), (7, 0.9)):
        cfg = dict(num_threads=threads, mini_batch_size=mb, min_match_ratio=ratio, subsample_keep_ratio=0.7)
        dev = vb.ICP(vb.ICPConfig(**cfg)).runICP(layer, s[0], (q0, t0), seed=123)
        ref = omap.icp(po.IcpConfig(**cfg), s[0], q0, t0, 123)
        rep = _close(dev, ref)
        print("threads", threads, "mini batch", mb, rep)
        assert rep["dq"] <= TOL and rep["dt_rel"] <= TOL, rep
        assert abs(rep["updates"][0] - rep["updates"][1]) <= max(2, rep["updates"][1] // 1000), rep


def test_icp_edge_cases():
    ss = list(scenes.c3_room_sequence(n_scans=2, width=160, height=120))
    layer, omap = _maps("port", 0.1, 0.4, ss[:1])
    s = ss[1]
    icp = vb.ICP(vb.ICPConfig())
    # empty cloud: pose unchanged, nothing fused
    n, (q, t) = icp.runICP(layer, np.zeros((0, 3), np.float32), (s[2], s[3]), seed=1)
    assert n == 0 and (q == np.asarray(s[2], np.float32)).all() and (t == np.asarray(s[3], np.float32)).all()
    # a cloud nowhere near the map: no batch reaches min_match_ratio
    far = s[0] + np.float32(500.0)
    n, (q, t) = icp.runICP(layer, far, (s[2], s[3]), seed=1)
    assert n == 0 and (q == np.asarray(s[2], np.float32)).all() and (t == np.asarray(s[3], np.float32)).all()
    # fewer points than one mini batch: one (short) batch, which cannot reach 16 matches of 20
    few = s[0][:11]
    dev = icp.runICP(layer, few, (s[2], s[3]), seed=5)
    ref = omap.icp(po.IcpConfig(), few, s[2], s[3], 5)
    assert dev[0] == ref[2] == 0
    # the cloud already on the device gives the same answer as the host cloud
    import torch
    d = torch.from_numpy(np.ascontiguousarray(s[0])).cuda()
    a = icp.runICP(layer, s[0], (s[2], s[3]), seed=9)
    b = icp.runICPDevice(layer, d.data_ptr(), int(s[0].shape[0]), (s[2], s[3]), seed=9)
    assert a[0] == b[0] and (a[1][0] == b[1][0]).all() and (a[1][1] == b[1][1]).all()
    # invalid configurations are refused
    with pytest.raises(vb.VoxbloxError):
        vb.ICP(vb.ICPConfig(num_threads=33)).runICP(layer, s[0], (s[2], s[3]), seed=1)
    with pytest.raises(vb.VoxbloxError):
        vb.ICP(vb.ICPConfig(mini_batch_size=0)).runICP(layer, s[0], (s[2], s[3]), seed=1)
