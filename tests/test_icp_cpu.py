"""Pins the restatement's ICP (oracle/vbx_oracle.cc, the checker tests/test_icp_gpu.py trusts for
num_threads > 1) against the reference's own voxblox::ICP: directly where oracle/_ref exists, and against
the committed vectors of tests/golden/icp.json (generated from oracle/_ref by
tests/golden/make_icp_golden.py) everywhere.  Tolerance 1e-5: the two differ only in the 2 x 2 Procrustes
step (closed form here, JacobiSVD there) and in nothing at all for refine_roll_pitch = true."""
import json
import os

import numpy as np
import pytest

from oracle import pyoracle as po
from tests.golden import make_golden as mg
from tests.golden import make_icp_golden as mi
from tests.golden import make_reference_golden as mr

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = json.load(open(os.path.join(HERE, "golden", "icp.json")))
TOL = 1e-5


@pytest.mark.parametrize("name", sorted(mi.CASES))
def test_port_icp_matches_committed_golden(name):
    if mg.scans_digest("room") != GOLD["inputs"]["room"]:
        pytest.skip("scan generator output differs on this machine (numpy / libm): inputs not comparable")
    q, t, n = mi.run_case(po.OracleLib("port"), name)
    g = GOLD["cases"][name]
    gq = np.array([float.fromhex(v) for v in g["q_wxyz"]])
    gt = np.array([float.fromhex(v) for v in g["t"]])
    assert n == g["num_updates"]
    assert np.abs(q - gq).max() <= TOL and np.abs(t - gt).max() <= TOL, (q, gq, t, gt)


@pytest.mark.skipif(not po.available("reference"), reason="oracle/_ref not built (no /root/reference here)")
@pytest.mark.parametrize("name", sorted(mi.CASES))
def test_port_icp_matches_reference_library(name):
    rq, rt, rn = mi.run_case(po.OracleLib("reference"), name)
    pq, pt, pn = mi.run_case(po.OracleLib("port"), name)
    assert rn == pn
    assert np.abs(rq - pq).max() <= TOL and np.abs(rt - pt).max() <= TOL


def test_shuffle_is_the_library_shuffle():
    """both checkers call std::shuffle(std::default_random_engine(seed)) of the C++ library they are built with;
    the reference's permutations are stored as a digest by tests/golden/make_reference_golden.py"""
    port = po.OracleLib("port")
    for n, seed in mr.SHUFFLES:
        b = np.zeros(n, np.uint32)
        port.lib.vbo_icp_shuffle(n, seed, b.ctypes.data)
        assert sorted(b.tolist()) == list(range(n))
    assert mr.shuffle_digest(port) == mr.golden("restatement_pins", "shuffle")


def test_round_robin_schedule_with_one_thread_is_the_sequential_algorithm():
    """num_threads = T only changes WHICH pose a batch is matched against; with every thread alive the batches
    are the same ones in the same order, so the number of attempted batches is independent of T."""
    scans = mg.case_scans("room")
    omap = po.OracleMap(po.OracleLib("port"), po.TsdfConfig(default_truncation_distance=0.4), 0.1, 16)
    for s in scans[:2]:
        omap.integrate(po.MERGED, s)
    s = scans[2]
    base = omap.icp(po.IcpConfig(num_threads=1), s[0], s[2], s[3], 3)
    for T in (2, 8, 32):
        q, t, n = omap.icp(po.IcpConfig(num_threads=T), s[0], s[2], s[3], 3)
        assert abs(n - base[2]) <= max(3, base[2] // 20)
        assert np.abs(q - base[0]).max() < 5e-3 and np.abs(t - base[1]).max() < 5e-2   # same optimum, another path to it
