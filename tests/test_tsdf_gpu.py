"""-m gpu parity: the CUDA TSDF path through the C-ABI against the CPU oracle."""
import numpy as np
import pytest

import voxblox_b200 as vb
from oracle import pyoracle as po
from tests.parity import compare_tsdf
from voxblox_b200 import scenes

pytestmark = pytest.mark.gpu

REL_TOL = 1e-4  # north_star: TSDF distance / weight within 1e-4 relative


def _run(kind, scans, voxel_size, trunc, order, **cfg_kw):
    cfg = vb.TsdfIntegratorConfig(default_truncation_distance=trunc, integrator_threads=1, **cfg_kw)
    layer = vb.Layer(voxel_size, 16)
    integ = vb.TsdfIntegratorFactory.create(kind, cfg, layer)
    ocfg = po.TsdfConfig(default_truncation_distance=trunc, integrator_threads=1, **cfg_kw)
    omap = po.OracleMap(po.OracleLib("port"), ocfg, voxel_size, 16)
    for s in scans:
        integ.integratePointCloud((s[2], s[3]), s[0], s[1])
        omap.integrate(kind, s, order=order)
        gc, oc = integ.counters(), omap.counters()
        for k in ("rays", "clear_rays", "updates", "voxels_touched", "blocks_touched", "blocks_allocated"):
            assert gc[k] == oc[k], (k, gc, oc)
    return compare_tsdf(layer, omap)


def _assert_parity(rep):
    assert rep["blocks_equal"], rep
    assert rep["observed_equal"], rep
    assert rep["max_rel_err"] <= REL_TOL, rep
    assert rep["color_mismatch"] == 0, rep
    assert rep["updated_equal"], rep


def test_c1_simple_planar_wall():
    rep = _run(1, [scenes.c1_planar_wall()], 0.2, 0.8, po.ORDER_REFERENCE)
    print(rep)
    _assert_parity(rep)


def test_c1_merged_planar_wall():
    rep = _run(2, [scenes.c1_planar_wall()], 0.2, 0.8, po.ORDER_REFERENCE)
    print(rep)
    _assert_parity(rep)


@pytest.mark.parametrize("kind,order", [(1, po.ORDER_REFERENCE), (2, po.ORDER_REFERENCE)])
def test_room_sequence_small(kind, order):
    scans = scenes.c3_room_sequence(n_scans=4, width=160, height=120)
    rep = _run(kind, scans, 0.1, 0.4, order)
    print(rep)
    _assert_parity(rep)


# ----------------------------------------------------------------------------- edge cases
def _small_scans(n=2, w=96, h=72):
    return scenes.c3_room_sequence(n_scans=n, width=w, height=h)


@pytest.mark.parametrize("kind,order", [(1, po.ORDER_REFERENCE), (2, po.ORDER_REFERENCE)])
@pytest.mark.parametrize("cfg_kw", [
    dict(use_const_weight=1),
    dict(voxel_carving_enabled=0),
    dict(use_weight_dropoff=0),
    dict(use_sparsity_compensation_factor=1, sparsity_compensation_factor=3.0),
    dict(max_ray_length_m=2.0),                    # far points become clearing rays (allow_clear)
    dict(max_ray_length_m=2.0, allow_clear=0),     # ... or are dropped
    dict(min_ray_length_m=1.5),
    dict(max_weight=5.0),                          # the weight clamp fires
    dict(integration_order_mode=1),                # "sorted"
], ids=lambda d: ",".join(f"{k}={v}" for k, v in d.items()))
def test_config_variants(kind, order, cfg_kw):
    if cfg_kw.get("integration_order_mode") == 1:
        # std::sort leaves ties unspecified; the room scans have no exact |p|^2 ties
        pass
    rep = _run(kind, _small_scans(), 0.1, 0.4, order, **cfg_kw)
    print(rep)
    _assert_parity(rep)


def test_merged_anti_grazing():
    rep = _run(2, _small_scans(), 0.1, 0.4, po.ORDER_REFERENCE, enable_anti_grazing=1)
    print(rep)
    _assert_parity(rep)


@pytest.mark.parametrize("kind,order", [(1, po.ORDER_REFERENCE), (2, po.ORDER_REFERENCE)])
def test_freespace_points(kind, order):
    """freespace_points=true: every ray is a clearing ray (tsdf_integrator.h:96-99)."""
    cfg = vb.TsdfIntegratorConfig(default_truncation_distance=0.4, integrator_threads=1)
    layer = vb.Layer(0.1, 16)
    integ = vb.TsdfIntegratorFactory.create(kind, cfg, layer)
    omap = po.OracleMap(po.OracleLib("port"), po.TsdfConfig(default_truncation_distance=0.4), 0.1, 16)
    for s in _small_scans():
        integ.integratePointCloud((s[2], s[3]), s[0], s[1], freespace_points=True)
        omap.integrate(kind, s, freespace=True, order=order)
    rep = compare_tsdf(layer, omap)
    print(rep)
    _assert_parity(rep)


def test_far_clearing_points():
    """Points far beyond max_ray_length become clearing bundles keyed by voxels thousands of voxels
    away: the bundle keys are packed relative to the scan's own bounding box, so they simply use
    more key bits."""
    s = _small_scans(1)[0]
    pts = s[0].copy()
    pts[::7] *= 40.0      # ~100 m away: clearing rays whose end voxels are thousands of voxels off
    scan = (pts, s[1], s[2], s[3])
    rep = _run(2, [scan], 0.1, 0.4, po.ORDER_REFERENCE)
    print(rep)
    _assert_parity(rep)


@pytest.mark.parametrize("kind,order,cfg_kw", [
    (1, po.ORDER_REFERENCE, {}), (2, po.ORDER_REFERENCE, {}),
    (2, po.ORDER_REFERENCE, dict(enable_anti_grazing=1)), (1, po.ORDER_REFERENCE, dict(integration_order_mode=1))])
def test_more_updates_than_one_pass_holds(kind, order, cfg_kw):
    """K > max_updates_per_pass: the call is applied in passes over contiguous ray ranges and
    must equal the one-pass result (= the oracle) bit for bit; a single ray that does not fit is
    refused loudly."""
    scans = _small_scans(2)
    cfg = vb.TsdfIntegratorConfig(default_truncation_distance=0.4, integrator_threads=1, **cfg_kw)
    small = vb.EngineOptions(max_updates_per_pass=4096 if kind == 2 else 60000)
    layer = vb.Layer(0.1, 16, engine_options=small)
    integ = vb.TsdfIntegratorFactory.create(kind, cfg, layer)
    omap = po.OracleMap(po.OracleLib("port"), po.TsdfConfig(default_truncation_distance=0.4, integrator_threads=1,
                                                           **cfg_kw), 0.1, 16)
    for s in scans:
        integ.integratePointCloud((s[2], s[3]), s[0], s[1])
        omap.integrate(kind, s, order=order)
        gc, oc = integ.counters(), omap.counters()
        assert gc["passes"] > 1, gc
        for k in ("rays", "clear_rays", "updates", "blocks_touched", "blocks_allocated"):
            assert gc[k] == oc[k], (k, gc, oc)
    rep = compare_tsdf(layer, omap)
    print(rep, gc)
    _assert_parity(rep)
    assert rep["n_bit_exact"] == rep["n_voxels"], rep
    tiny = vb.Layer(0.1, 16, engine_options=vb.EngineOptions(max_updates_per_pass=8))
    integ2 = vb.TsdfIntegratorFactory.create(kind, cfg, tiny)
    with pytest.raises(vb.VoxbloxError):
        integ2.integratePointCloud((scans[0][2], scans[0][3]), scans[0][0], scans[0][1])


def test_degenerate_clouds():
    cfg = vb.TsdfIntegratorConfig(default_truncation_distance=0.4)
    layer = vb.Layer(0.1, 16)
    integ = vb.TsdfIntegratorFactory.create("merged", cfg, layer)
    s = _small_scans(1)[0]
    # empty cloud
    integ.integratePointCloud((s[2], s[3]), np.zeros((0, 3), np.float32), np.zeros((0, 4), np.uint8))
    assert layer.getNumberOfAllocatedBlocks() == 0
    # every point invalid (closer than min_ray_length_m) or non-finite
    pts = np.full((100, 3), 0.01, np.float32)
    pts[50:] = np.nan
    pts[75:] = np.inf
    integ.integratePointCloud((s[2], s[3]), pts, np.zeros((100, 4), np.uint8))
    assert layer.getNumberOfAllocatedBlocks() == 0
    assert integ.counters()["rays"] == 0
    # mismatched sizes: CHECK_EQ(points_C.size(), colors.size()), tsdf_integrator.cc:312
    with pytest.raises(vb.VoxbloxError):
        integ.integratePointCloud((s[2], s[3]), s[0], s[1][:-1])
    # a cloud larger than the engine was sized for is refused, not truncated
    small = vb.Layer(0.1, 16, engine_options=vb.EngineOptions(max_points_per_scan=1024))
    integ2 = vb.TsdfIntegratorFactory.create("merged", cfg, small)
    with pytest.raises(vb.VoxbloxError):
        integ2.integratePointCloud((s[2], s[3]), s[0], s[1])


def test_voxels_per_side_8():
    cfg = vb.TsdfIntegratorConfig(default_truncation_distance=0.4, integrator_threads=1)
    layer = vb.Layer(0.1, 8)
    integ = vb.TsdfIntegratorFactory.create("merged", cfg, layer)
    omap = po.OracleMap(po.OracleLib("port"), po.TsdfConfig(default_truncation_distance=0.4), 0.1, 8)
    for s in _small_scans():
        integ.integratePointCloud((s[2], s[3]), s[0], s[1])
        omap.integrate(2, s, order=po.ORDER_REFERENCE)
    gi, oi = layer.getAllAllocatedBlocks(), omap.block_indices()
    assert gi.shape == oi.shape and (gi == oi).all()
    gv, _ = layer.getBlocks(gi)
    ov = np.stack([omap.block(i)[0] for i in oi])
    assert gv.tobytes() == ov.tobytes()


def test_fast_integrator_statistics():
    """The Fast integrator is approximate by design (lossy sets, racy in the reference with more
    than one thread): block set and per-voxel values are compared statistically."""
    cfg = vb.TsdfIntegratorConfig(default_truncation_distance=0.4, integrator_threads=1)
    layer = vb.Layer(0.1, 16)
    integ = vb.TsdfIntegratorFactory.create("fast", cfg, layer)
    omap = po.OracleMap(po.OracleLib("port"), po.TsdfConfig(default_truncation_distance=0.4), 0.1, 16)
    for s in scenes.c3_room_sequence(n_scans=4, width=160, height=120):
        integ.integratePointCloud((s[2], s[3]), s[0], s[1])
        omap.integrate(3, s)
    gb, ob = layer.blocks(), omap.blocks()
    common = set(gb) & set(ob)
    assert len(common) >= 0.9 * max(len(gb), len(ob))
    g = np.stack([gb[k] for k in sorted(common)])
    o = np.stack([ob[k] for k in sorted(common)])
    both = (g["weight"] > 0) & (o["weight"] > 0)
    either = (g["weight"] > 0) | (o["weight"] > 0)
    assert both.sum() >= 0.9 * either.sum()
    rmse = float(np.sqrt(np.mean((g["distance"][both] - o["distance"][both]) ** 2)))
    print("fast: blocks", len(gb), len(ob), "observed overlap", both.sum() / either.sum(), "rmse", rmse)
    assert rmse < 0.1  # one voxel


# ------------------------------------------------------------------ asynchronous submission
def _layer_bytes(layer):
    idx = layer.getAllAllocatedBlocks()
    vox, upd = layer.getBlocks(idx)
    return idx.tobytes(), vox.tobytes(), np.asarray(upd).tobytes()


@pytest.mark.parametrize("kind", [1, 2])
@pytest.mark.parametrize("pageable", [False, True])
@pytest.mark.parametrize("n_scans,rings", [(7, None), (23, None), (23, (2, 1))],
                         ids=["7_scans", "23_scans", "23_scans_2_sets_1_lane"])
def test_async_submission_equals_synchronous(kind, pageable, n_scans, rings, monkeypatch):
    """vbx_tsdf_integrate_async overlaps the front half of scan i+1 with the back half of scan i;
    the map must equal the synchronous calls' bit for bit (and so the oracle's).  With more scans
    than hand-off sets and front lanes every ring (sets, lanes, sort and copy streams) wraps at least
    twice: a submission waits for the scan that used its set, collects it and reuses the buffers."""
    if rings:
        monkeypatch.setenv("VBX_ASYNC_SETS", str(rings[0]))
        monkeypatch.setenv("VBX_ASYNC_LANES", str(rings[1]))
    cfg = vb.TsdfIntegratorConfig(default_truncation_distance=0.4, integrator_threads=1)
    scans = scenes.c3_room_sequence(n_scans=n_scans, width=160, height=120)
    la, ls = vb.Layer(0.1, 16), vb.Layer(0.1, 16)
    ia = vb.TsdfIntegratorFactory.create(kind, cfg, la)
    isync = vb.TsdfIntegratorFactory.create(kind, cfg, ls)
    keep = []
    for s in scans:
        isync.integratePointCloud((s[2], s[3]), s[0], s[1])
        if pageable:
            p, c = np.ascontiguousarray(s[0]), np.ascontiguousarray(s[1])
        else:
            p, c = la.hostBuffer(s[0].shape, np.float32), la.hostBuffer(s[1].shape, np.uint8)
            p[...] = s[0]
            c[...] = s[1]
        keep.append((p, c))
        ia.integratePointCloudAsync((s[2], s[3]), p, c)
    la.sync()
    assert ia.counters()["updates"] == isync.counters()["updates"]
    assert _layer_bytes(la) == _layer_bytes(ls)
    # a synchronous call after asynchronous ones continues the same map
    s = scans[0]
    ia.integratePointCloud((s[2], s[3]), s[0], s[1])
    isync.integratePointCloud((s[2], s[3]), s[0], s[1])
    assert _layer_bytes(la) == _layer_bytes(ls)


def test_async_far_points_are_integrated():
    """Round 1 dropped an asynchronously submitted scan whose clearing points overflowed the compact
    bundle keys.  Keys are now packed relative to the scan's bounding box: nothing overflows."""
    cfg = vb.TsdfIntegratorConfig(default_truncation_distance=0.4, integrator_threads=1)
    layer = vb.Layer(0.1, 16)
    integ = vb.TsdfIntegratorFactory.create("merged", cfg, layer)
    s = _small_scans(1)[0]
    pts = s[0].copy()
    pts[::7] *= 40.0
    integ.integratePointCloudAsync((s[2], s[3]), pts, s[1])
    integ.integratePointCloudAsync((s[2], s[3]), pts, s[1])
    layer.sync()
    ref = vb.Layer(0.1, 16)
    r = vb.TsdfIntegratorFactory.create("merged", cfg, ref)
    r.integratePointCloud((s[2], s[3]), pts, s[1])
    r.integratePointCloud((s[2], s[3]), pts, s[1])
    assert _layer_bytes(layer) == _layer_bytes(ref)


@pytest.mark.parametrize("kind", [1, 2])
def test_async_scan_with_more_updates_than_one_pass_is_redone_not_dropped(kind):
    """An asynchronously submitted scan whose update records exceed max_updates_per_pass cannot be
    chunked on the device.  It raises the hold flag; the scans queued behind it skip their back
    halves; the host then redoes all of them synchronously (in passes), in submission order.  The map
    must equal the all-synchronous map and no error may surface."""
    cfg = vb.TsdfIntegratorConfig(default_truncation_distance=0.4, integrator_threads=1)
    small = lambda: vb.EngineOptions(max_updates_per_pass=6000 if kind == 2 else 100000)
    la, ls = vb.Layer(0.1, 16, engine_options=small()), vb.Layer(0.1, 16, engine_options=small())
    ia, isync = vb.TsdfIntegratorFactory.create(kind, cfg, la), vb.TsdfIntegratorFactory.create(kind, cfg, ls)
    scans = scenes.c3_room_sequence(n_scans=9, width=96, height=72)
    keep = []
    for s in scans:   # fewer scans than the default ten hand-off sets: the recovery runs in la.sync()
        isync.integratePointCloud((s[2], s[3]), s[0], s[1])
        p, c = np.ascontiguousarray(s[0]), np.ascontiguousarray(s[1])
        keep.append((p, c))
        ia.integratePointCloudAsync((s[2], s[3]), p, c)
    la.sync()
    assert isync.counters()["passes"] > 1
    assert ia.counters()["async_redone_total"] >= len(scans) - 1
    assert _layer_bytes(la) == _layer_bytes(ls)


def test_pool_overflow_is_reported_and_does_not_poison_later_calls():
    """ADVICE r1: a call that runs out of pool slots left hash entries without a slot behind; a later
    call found them and wrote out of bounds.  Now the failing call reports VBX_E_CAPACITY, the hash
    is rebuilt from the slots that exist, and the map keeps working (here: after blocks are removed)."""
    cfg = vb.TsdfIntegratorConfig(default_truncation_distance=0.4, integrator_threads=1)
    layer = vb.Layer(0.1, 16, engine_options=vb.EngineOptions(max_blocks=8))
    integ = vb.TsdfIntegratorFactory.create("merged", cfg, layer)
    s = _small_scans(1)[0]
    with pytest.raises(vb.VoxbloxError):
        integ.integratePointCloud((s[2], s[3]), s[0], s[1])
    assert layer.getNumberOfAllocatedBlocks() <= 8
    with pytest.raises(vb.VoxbloxError):   # still full: fails again, cleanly
        integ.integratePointCloud((s[2], s[3]), s[0], s[1])
    vox, _ = layer.getBlocks(layer.getAllAllocatedBlocks())
    assert np.isfinite(vox["distance"]).all()
    # asynchronous submissions behind a failing scan must not write through slot-less entries either
    for _ in range(4):
        integ.integratePointCloudAsync((s[2], s[3]), np.ascontiguousarray(s[0]), np.ascontiguousarray(s[1]))
    with pytest.raises(vb.VoxbloxError):
        layer.sync()
    layer.removeAllBlocks()
    assert layer.getNumberOfAllocatedBlocks() == 0
    few = (s[0][:1], s[1][:1], s[2], s[3])    # one ray: a handful of blocks fits
    integ.integratePointCloud((few[2], few[3]), few[0], few[1])
    omap = po.OracleMap(po.OracleLib("port"), po.TsdfConfig(default_truncation_distance=0.4), 0.1, 16)
    omap.integrate(2, few)
    rep = compare_tsdf(layer, omap)
    assert rep["blocks_equal"] and rep["n_bit_exact"] == rep["n_voxels"], rep


def test_async_falls_back_for_map_dependent_front_halves():
    cfg = vb.TsdfIntegratorConfig(default_truncation_distance=0.4, integrator_threads=1, enable_anti_grazing=True)
    la, ls = vb.Layer(0.1, 16), vb.Layer(0.1, 16)
    ia = vb.TsdfIntegratorFactory.create("merged", cfg, la)
    isync = vb.TsdfIntegratorFactory.create("merged", cfg, ls)
    for s in _small_scans(3):
        ia.integratePointCloudAsync((s[2], s[3]), s[0], s[1])
        isync.integratePointCloud((s[2], s[3]), s[0], s[1])
    la.sync()
    assert _layer_bytes(la) == _layer_bytes(ls)
