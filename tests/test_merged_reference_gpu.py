"""-m gpu: the Merged integrator (BASELINE.json's metric path) against the REFERENCE ITSELF.

The reference's own MergedTsdfIntegrator (its translation units, oracle/_ref/libvbx_ref.so) is run with
integrator_threads = 1 on these inputs by tests/golden/make_reference_golden.py, which stores a digest of
its layer.  With one thread its result is deterministic: bundles are integrated in the iteration order of
its std::unordered_map (tsdf_integrator.cc:436-456).  The device reproduces that order (k_bundle_order),
so at FULL size -- C2 (both truncations), the bench / C4 cloud stream and C5 -- every voxel must be
bit-identical: distance, weight, colour, block set, updated bits.

With more threads the reference is not deterministic (a mutex per voxel decides, cc:186)."""
import pytest

import voxblox_b200 as vb
from tests.golden import make_reference_golden as mr
from tests.parity import device_layer_digest
from voxblox_b200 import scenes

pytestmark = pytest.mark.gpu

CASES = {
    "c2_trunc0.4": dict(voxel=0.1, scans=lambda: [scenes.c2_sphere_scan(i) for i in range(3)],
                        cfg=dict(default_truncation_distance=0.4), opts=None),
    "c2_trunc4.0": dict(voxel=0.1, scans=lambda: [scenes.c2_sphere_scan(i) for i in range(3)],
                        cfg=dict(default_truncation_distance=4.0), opts=None),
    "bench_c4_stream": dict(voxel=0.05, scans=lambda: [scenes.c3_room_scan(i) for i in range(3)],
                            cfg=dict(default_truncation_distance=0.2), opts=None),
    "c5_lidar": dict(voxel=0.05, scans=lambda: [scenes.c5_lidar_scan(i) for i in range(2)],
                     cfg=dict(default_truncation_distance=0.2, max_ray_length_m=10.0, use_const_weight=1),
                     opts=dict(max_blocks=8192, max_points_per_scan=1 << 19)),
}


@pytest.mark.parametrize("name", list(CASES))
def test_merged_bit_exact_against_reference_one_thread(name):
    case = CASES[name]
    scans = case["scans"]()
    gold = mr.golden("merged", name)
    mr.require_inputs(scans, gold)
    cfg = vb.TsdfIntegratorConfig(integrator_threads=1, **case["cfg"])
    opts = vb.EngineOptions(**case["opts"]) if case["opts"] else None
    layer = vb.Layer(case["voxel"], 16, engine_options=opts)
    integ = vb.TsdfIntegratorFactory.create("merged", cfg, layer)
    for s in scans:
        integ.integratePointCloud((s[2], s[3]), s[0], s[1])
    print(name, "device blocks", layer.getNumberOfAllocatedBlocks(), "reference blocks", gold["blocks"])
    assert layer.getNumberOfAllocatedBlocks() == gold["blocks"]
    assert device_layer_digest(layer, with_updated=True) == gold["digest"]
