"""Pins the CPU restatement (oracle/vbx_oracle.cc) -- the checker every GPU parity test
trusts -- against the reference itself:
  * bit-identical layers vs oracle/_ref (the reference's own integrator sources compiled
    against oracle/shim/), wherever that library exists (it travels to the GPU box);
  * the committed digests of tests/golden/digests.json and tests/golden/reference.json, generated
    from oracle/_ref by tests/golden/make_golden.py and make_reference_golden.py, everywhere;
  * the known-answer INDEXING vectors of the reference's test/test_tsdf_map.cc.
"""
import json
import os

import numpy as np
import pytest

from oracle import pyoracle as po
from tests.golden import make_golden as mg
from tests.golden import make_reference_golden as mr
from tests.parity import oracle_layer_digest
from voxblox_b200 import scenes

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = json.load(open(os.path.join(HERE, "golden", "digests.json")))


@pytest.mark.parametrize("name", sorted(mg.CASES))
def test_port_matches_committed_golden(name):
    scan_name = mg.CASES[name][1]
    if mg.scans_digest(scan_name) != GOLD["inputs"][scan_name]:
        pytest.skip("scan generator output differs on this machine (numpy / libm): inputs not comparable")
    got = mg.run_case(po.OracleLib("port"), name)
    for layer, (digest, nblocks) in GOLD["digests"][name].items():
        assert got[layer][1] == nblocks, (name, layer)
        assert got[layer][0] == digest, (name, layer)


@pytest.mark.skipif(not po.available("reference"), reason="oracle/_ref not built (no /root/reference here)")
@pytest.mark.parametrize("name", sorted(mg.CASES))
def test_port_matches_reference_library(name):
    ref = mg.run_case(po.OracleLib("reference"), name)
    port = mg.run_case(po.OracleLib("port"), name)
    assert ref == port, name


def voxelwise_with_esdf_maps(lib):
    """Simple / Merged / Fast, each followed by an incremental ESDF update, over four scans."""
    scans = scenes.c3_room_sequence(n_scans=4, width=128, height=96)
    cfg = po.TsdfConfig(default_truncation_distance=0.4, integrator_threads=1)
    ecfg = po.EsdfConfig(max_distance_m=4.0, default_distance_m=4.0, min_distance_m=0.2, min_diff_m=0.0, multi_queue=1)
    maps = {}
    for kind in (1, 2, 3):
        m = maps[kind] = po.OracleMap(lib, cfg, 0.1, 16)
        m.esdf_create(ecfg)
        for s in scans:
            m.integrate(kind, s)
            m.esdf_update(False, True)
    return maps


def esdf_blocks_and_setters_maps(lib):
    """updateFromTsdfBlocks on a block subset (map 1 of 2), then setEsdfMaxDistance / setFullEuclidean and a
    batch update (map 2 of 2)."""
    scans = scenes.c3_room_sequence(n_scans=3, width=96, height=72)
    cfg = po.TsdfConfig(default_truncation_distance=0.4, integrator_threads=1)
    ecfg = po.EsdfConfig(max_distance_m=2.0, default_distance_m=2.0, min_distance_m=0.2, min_diff_m=1e-3)
    maps = [po.OracleMap(lib, cfg, 0.1, 16) for _ in range(2)]
    for k, m in enumerate(maps):
        m.esdf_create(ecfg)
        for s in scans:
            m.integrate(2, s)
        blocks = m.block_indices(0)
        m.esdf_update_blocks(np.concatenate([blocks[::2], np.array([[77, 77, 77]], np.int32)]), incremental=False)
        if k == 1:
            m.esdf_set_max_distance(3.0)
            m.esdf_set_full_euclidean(True)
            m.esdf_update(True, True)
    return maps


def serialization_map(lib):
    scans = scenes.c3_room_sequence(n_scans=2, width=96, height=72)
    m = po.OracleMap(lib, po.TsdfConfig(default_truncation_distance=0.4, integrator_threads=1), 0.1, 16)
    m.esdf_create(po.EsdfConfig(max_distance_m=2.0, default_distance_m=2.0, min_distance_m=0.2))
    for s in scans:
        m.integrate(2, s)
    m.esdf_update(False, True)
    return m


def serialization_decoded(lib, words, indices):
    """A fresh map into which the serialized blocks of both layers were deserialized."""
    m = po.OracleMap(lib, po.TsdfConfig(default_truncation_distance=0.4, integrator_threads=1), 0.1, 16)
    m.esdf_create(po.EsdfConfig(max_distance_m=2.0, default_distance_m=2.0, min_distance_m=0.2))
    for layer in (0, 1):
        for i, w in zip(indices[layer], words[layer]):
            m.deserialize_block(i, w, layer)
    return m


def test_port_matches_reference_voxelwise_with_esdf():
    """Same comparison as the committed digests, incl. updated bits and an incremental ESDF, over more scans."""
    gold = mr.restatement_golden()["voxelwise_with_esdf"]
    for kind, m in voxelwise_with_esdf_maps(po.OracleLib("port")).items():
        for layer in (0, 1):
            assert oracle_layer_digest(m, layer, with_updated=True) == gold[str(kind)][layer], (kind, layer)


def test_port_matches_reference_esdf_blocks_and_setters():
    """updateFromTsdfBlocks on a block subset, setEsdfMaxDistance / setFullEuclidean, then batch."""
    gold = mr.restatement_golden()["esdf_blocks_and_setters"]
    for k, m in enumerate(esdf_blocks_and_setters_maps(po.OracleLib("port"))):
        assert oracle_layer_digest(m, 1) == gold[k], k


def test_port_matches_reference_block_serialization():
    """Block::serializeToIntegers / deserializeFromIntegers (src/core/block.cc) for both voxel types,
    incl. the sign-extension quirk of serializeDirection for negative parent components."""
    gold = mr.restatement_golden()["serialization"]
    port = po.OracleLib("port")
    m = serialization_map(port)
    indices = [m.block_indices(layer) for layer in (0, 1)]
    words = [[m.serialize_block(i, layer) for i in indices[layer]] for layer in (0, 1)]
    assert [mr.int32_digest(*w) for w in words] == gold["words"]
    assert any((m.block(i, 1)[0]["parent"] < 0).any() for i in indices[1])
    # round trip through a fresh map: the restatement decodes the words as the reference does
    decoded = serialization_decoded(port, words, indices)
    assert [oracle_layer_digest(decoded, layer) for layer in (0, 1)] == gold["decoded"]
    for i in indices[0]:  # TSDF serialisation is lossless
        assert decoded.block(i, 0)[0].tobytes() == m.block(i, 0)[0].tobytes()


def _integrate_single_point(point, voxel_size, vps):
    """One point, no carving: the ray covers only [p - T, p + T] (integrator_utils.cc:93-98)."""
    cfg = po.TsdfConfig(default_truncation_distance=voxel_size * 0.4, voxel_carving_enabled=0,
                        min_ray_length_m=0.0, max_ray_length_m=100.0, use_const_weight=1)
    m = po.OracleMap(po.OracleLib("port"), cfg, voxel_size, vps)
    pts = np.array([point], dtype=np.float32)
    cols = np.array([[255, 0, 0, 255]], dtype=np.uint8)
    # the sensor sits far away along +x so that the ray through the point is axis aligned in x
    q = np.array([1, 0, 0, 0], dtype=np.float32)
    t = np.zeros(3, dtype=np.float32)
    m.integrate(1, (pts, cols, q, t))
    return m


def test_known_answer_indexing_vectors():
    """test/test_tsdf_map.cc: vps 8, voxel 0.1 (:12-16); (-0.5,-0.2,0.5) m -> block (-1,-1,0)
    (:281-292); voxel (3,6,5) <-> linear 371, voxel (0,1,0) <-> linear 8 (:140-149, :303-309),
    i.e. lin = x + vps*(y + vps*z)."""
    vs, vps = np.float32(0.1), 8
    m = _integrate_single_point((-0.5, -0.2, 0.5), float(vs), vps)
    blocks = {tuple(int(v) for v in b) for b in m.block_indices()}
    assert (-1, -1, 0) in blocks
    # a point at the centre of global voxel (-5, -2, 5): block (-1,-1,0), local (3, 6, 5)
    # -> linear 3 + 8*(6 + 8*5) = 371
    m = _integrate_single_point((-0.45, -0.15, 0.55), float(vs), vps)
    vox, _ = m.block((-1, -1, 0))
    assert vox["weight"][371] > 0
    assert 371 == 3 + 8 * (6 + 8 * 5) and 8 == 0 + 8 * (1 + 8 * 0)
    # point inside voxel (0,1,0) of block (0,0,0): linear index 8
    m2 = _integrate_single_point((0.05, 0.15, 0.05), float(vs), vps)
    vox2, _ = m2.block((0, 0, 0))
    assert vox2["weight"][8] > 0


def test_block_origin_round_trip():
    """test_tsdf_map.cc:325-345: origin <-> block index round trip at block size 0.32 for +-50^3
    (getGridIndexFromOriginPoint rounds, core/common.h:178-184)."""
    bs = np.float32(0.32)
    inv = np.float32(1.0 / bs)
    idx = np.arange(-50, 51, dtype=np.int32)
    origin = idx.astype(np.float32) * bs
    back = np.round(origin * inv).astype(np.int32)
    assert (back == idx).all()
