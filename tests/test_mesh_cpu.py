"""Pins the meshing restatement (oracle/vbx_oracle.cc, generateMesh) and the generated marching-cubes
table (voxblox_b200/csrc/vbx_mc_tables.h) to the reference: MeshIntegrator<TsdfVoxel>
(mesh/mesh_integrator.h), MarchingCubes (mesh/marching_cubes.h, src/mesh/marching_cubes.cc) compiled
from the reference's sources into oracle/_ref, and committed digests where the reference is absent."""
import ctypes as C
import hashlib
import json
import os
import re

import numpy as np
import pytest

from oracle import pyoracle as po
from voxblox_b200 import scenes

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLD_PATH = os.path.join(HERE, "golden", "mesh_digests.json")


def _packed_tables():
    text = open(os.path.join(ROOT, "voxblox_b200", "csrc", "vbx_mc_tables.h")).read()
    words = [int(w, 16) for w in re.findall(r"0x([0-9a-f]{16})ull", text)]
    pairs = [(int(a), int(b)) for a, b in re.findall(r"\{(\d+), (\d+)\}", text)]
    assert len(words) == 256 and len(pairs) == 12
    rows = []
    for w in words:
        row = [(w >> (4 * k)) & 0xF for k in range(16)]
        rows.append([-1 if v == 0xF else v for v in row])
    return rows, pairs


def test_generated_table_is_well_formed():
    rows, pairs = _packed_tables()
    assert rows[0] == [-1] * 16 and rows[255] == [-1] * 16
    for case, row in enumerate(rows):
        n = row.index(-1)
        assert n % 3 == 0 and all(v == -1 for v in row[n:])
        # every edge a case uses joins a corner inside the surface with one outside
        for e in row[:n]:
            a, b = pairs[e]
            assert ((case >> a) & 1) != ((case >> b) & 1), (case, e)
    # complementary cases cut the same edges
    for case in range(256):
        assert sorted(set(v for v in rows[case] if v >= 0)) == sorted(set(v for v in rows[255 - case] if v >= 0))


def test_generated_table_equals_reference_table():
    """The packed tables against a digest of the reference's MarchingCubes::kTriangleTable / kEdgeIndexPairs
    (stored by tests/golden/make_reference_golden.py)."""
    from tests.golden import make_reference_golden as mr

    rows, pairs = _packed_tables()
    assert mr.int32_digest(rows, pairs) == mr.golden("restatement_pins", "mc_tables")


def _meshed_map(which, use_color=True, incremental=True):
    scans = scenes.c3_room_sequence(n_scans=3, width=96, height=72)
    m = po.OracleMap(po.OracleLib(which), po.TsdfConfig(default_truncation_distance=0.4, integrator_threads=1), 0.1, 16)
    for k, s in enumerate(scans):
        m.integrate(2, s)
        if incremental:
            # mesh the blocks the scan dirtied, clearing their kMesh bit (tsdf_server.cc:494-501)
            m.mesh_generate(use_color, 1e-4, only_mesh_updated_blocks=True, clear_updated_flag=True)
    if not incremental:
        m.mesh_generate(use_color, 1e-4, only_mesh_updated_blocks=False, clear_updated_flag=False)
    return m


def _mesh_digest(m):
    h = hashlib.sha256()
    idx = m.mesh_block_indices()
    h.update(idx.tobytes())
    nv = 0
    for i in idx:
        v, n, c, upd = m.mesh_block(i)
        h.update(v.tobytes())
        h.update(n.tobytes())
        h.update(b"" if c is None else c.tobytes())
        h.update(bytes([int(upd), 0 if c is None else 1]))
        nv += len(v)
    return h.hexdigest(), int(len(idx)), int(nv)


CASES = {"incremental_color": (True, True), "full_color": (True, False), "full_nocolor": (False, False)}


@pytest.mark.skipif(not po.available("reference"), reason="oracle/_ref not built")
@pytest.mark.parametrize("name", sorted(CASES))
def test_port_mesh_matches_reference(name):
    use_color, incremental = CASES[name]
    ref, port = _meshed_map("reference", use_color, incremental), _meshed_map("port", use_color, incremental)
    ia, ib = ref.mesh_block_indices(), port.mesh_block_indices()
    assert ia.shape == ib.shape and (ia == ib).all()
    total = 0
    for i in ia:
        va, na, ca, ua = ref.mesh_block(i)
        vb, nb, cb, ub = port.mesh_block(i)
        assert va.shape == vb.shape, tuple(i)
        assert va.tobytes() == vb.tobytes() and na.tobytes() == nb.tobytes(), tuple(i)
        assert (ca is None) == (cb is None) and (ca is None or ca.tobytes() == cb.tobytes()), tuple(i)
        assert ua == ub
        total += len(va)
    assert total > 1000
    # the kMesh bits were cleared the same way
    for i in ref.block_indices(0):
        assert ref.block(i)[1] == port.block(i)[1]


@pytest.mark.parametrize("name", sorted(CASES))
def test_port_mesh_matches_committed_golden(name):
    from tests.golden import make_golden as mg
    inputs = json.load(open(os.path.join(HERE, "golden", "digests.json")))["inputs"]
    if mg.scans_digest("room") != inputs["room"]:
        pytest.skip("scan generator output differs on this machine (numpy / libm): inputs not comparable")
    gold = json.load(open(GOLD_PATH))
    use_color, incremental = CASES[name]
    got = _mesh_digest(_meshed_map("port", use_color, incremental))
    assert list(got) == gold[name], name


if __name__ == "__main__":  # regenerate the digests from the REFERENCE library
    out = {name: list(_mesh_digest(_meshed_map("reference", *CASES[name]))) for name in CASES}
    json.dump(out, open(GOLD_PATH, "w"), indent=1, sort_keys=True)
    print("wrote", GOLD_PATH, out)
