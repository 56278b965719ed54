"""Generates tests/golden/reference.json and tests/golden/esdf_reference.npz: what the REFERENCE's own
integrators (oracle/_ref/libvbx_ref.so, one thread) compute on the inputs of the device tests that compare
with it -- test_merged_reference_gpu, test_esdf_reference_gpu, test_tsdf_ground_truth_gpu and
test_icp_gpu -- and of the restatement pins of test_oracle_pin, test_mesh_cpu and test_icp_cpu, so that
those comparisons run wherever the tests do, with or without the reference.
Run it where the reference library is built:

    python tests/golden/make_reference_golden.py

Stored per case: a SHA-256 digest of the scans (the comparison is only meaningful on identical inputs),
digests of the reference's layers where the device must be bit-identical, the reference's ground-truth
error summaries, its ICP poses (exact hex floats) and, for the ESDF statistics, the reference's block
set, observed / fixed / sign flags of every observed voxel and its distances on a seeded sample of at
most ESDF_SAMPLE observed voxels per case.
"""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

HERE = os.path.dirname(os.path.abspath(__file__))
JSON_PATH = os.path.join(HERE, "reference.json")
NPZ_PATH = os.path.join(HERE, "esdf_reference.npz")
ESDF_SAMPLE = 8192


def scans_digest(scans) -> str:
    h = hashlib.sha256()
    for s in scans:
        for a in s:
            h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


_json = None
_npz = None


def golden(section: str, name: str) -> dict:
    global _json
    if _json is None:
        with open(JSON_PATH) as f:
            _json = json.load(f)
    return _json[section] if name is None else _json[section][name]


def pin_scans():
    """Every scan the restatement pins of restatement_pins() integrate."""
    from voxblox_b200 import scenes

    return (scenes.c3_room_sequence(n_scans=4, width=128, height=96)
            + scenes.c3_room_sequence(n_scans=3, width=96, height=72))


def restatement_golden() -> dict:
    """The reference's restatement pins; skips like require_inputs when the inputs are not reproduced."""
    gold = golden("restatement_pins", None)
    require_inputs(pin_scans(), gold)
    return gold


def esdf_golden(name: str) -> dict:
    global _npz
    if _npz is None:
        with np.load(NPZ_PATH) as z:
            _npz = {k: z[k] for k in z.files}
    return {k.split("/", 1)[1]: v for k, v in _npz.items() if k.split("/", 1)[0] == name}


def require_inputs(scans, entry):
    """Skips when this machine's scan generator (numpy / libm) does not reproduce the stored inputs."""
    import pytest

    if scans_digest(scans) != entry["inputs"]:
        pytest.skip("scan generator output differs on this machine (numpy / libm): inputs not comparable")


def esdf_case_arrays(omap, seed):
    idx = omap.block_indices(1)
    ov = np.stack([omap.block(i, 1)[0] for i in idx])
    obs = ov["observed"] != 0
    d = ov["distance"][obs]
    pos = np.arange(d.size, dtype=np.int32)
    if d.size > ESDF_SAMPLE:
        pos = np.sort(np.random.default_rng(seed).choice(d.size, ESDF_SAMPLE, replace=False)).astype(np.int32)
    return {"blocks": idx.astype(np.int32), "observed": np.packbits(obs.ravel()),
            "fixed": ov["fixed"][obs].astype(np.uint8), "sign": np.sign(d).astype(np.int8),
            "sample": pos, "distance": d[pos].astype(np.float32)}


def int32_digest(*arrays) -> str:
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a, dtype=np.int32).tobytes())
    return h.hexdigest()


SHUFFLES = ((0, 1), (1, 1), (1000, 42), (4099, 7))


def shuffle_digest(lib) -> str:
    """std::shuffle(std::default_random_engine(seed)) of 0..n-1 for every (n, seed) of SHUFFLES."""
    outs = []
    for n, seed in SHUFFLES:
        a = np.zeros(n, np.uint32)
        lib.lib.vbo_icp_shuffle(n, seed, a.ctypes.data)
        outs.append(a)
    return int32_digest(*outs)


def mc_tables(lib):
    tri = np.zeros(256 * 16, dtype=np.int32)
    edges = np.zeros(24, dtype=np.int32)
    assert lib.lib.vbo_mc_tables(tri.ctypes.data, edges.ctypes.data) == 0
    return tri, edges


def restatement_pins(lib) -> dict:
    """What tests/test_oracle_pin.py, test_mesh_cpu.py and test_icp_cpu.py compare the restatement with."""
    from tests import test_oracle_pin as tp
    from tests.parity import oracle_layer_digest

    out = {"inputs": scans_digest(pin_scans()), "mc_tables": int32_digest(*mc_tables(lib)),
           "shuffle": shuffle_digest(lib)}
    out["voxelwise_with_esdf"] = {str(kind): [oracle_layer_digest(m, layer, with_updated=True) for layer in (0, 1)]
                                  for kind, m in tp.voxelwise_with_esdf_maps(lib).items()}
    out["esdf_blocks_and_setters"] = [oracle_layer_digest(m, 1) for m in tp.esdf_blocks_and_setters_maps(lib)]
    m = tp.serialization_map(lib)
    words = [[m.serialize_block(i, layer) for i in m.block_indices(layer)] for layer in (0, 1)]
    decoded = tp.serialization_decoded(lib, words, [m.block_indices(layer) for layer in (0, 1)])
    out["serialization"] = {"words": [int32_digest(*w) for w in words],
                            "decoded": [oracle_layer_digest(decoded, layer) for layer in (0, 1)]}
    return out


def main():
    from oracle import pyoracle as po
    from tests import test_esdf_reference_gpu as te
    from tests import test_icp_gpu as ti
    from tests import test_merged_reference_gpu as tm
    from tests import test_tsdf_ground_truth_gpu as tt
    from tests.parity import oracle_layer_digest
    from voxblox_b200 import scenes

    ref = po.OracleLib("reference")

    def omap(voxel, **cfg):
        return po.OracleMap(ref, po.TsdfConfig(integrator_threads=1, **cfg), voxel, 16)

    out = {"generated_by": "oracle/_ref/libvbx_ref.so (the reference's integrator sources, integrator_threads = 1)",
           "merged": {}, "esdf": {}, "esdf_ground_truth": {}, "tsdf_ground_truth": {}, "icp": {}}
    arrays = {}

    for name, case in tm.CASES.items():
        scans = case["scans"]()
        m = omap(case["voxel"], **case["cfg"])
        for s in scans:
            m.integrate(po.MERGED, s)
        out["merged"][name] = {"inputs": scans_digest(scans), "blocks": int(len(m.block_indices())),
                               "digest": oracle_layer_digest(m, 0, with_updated=True)}
        print("merged", name, out["merged"][name], flush=True)

    for k, (config, min_diff, multi_queue) in enumerate((("min_diff_zero", 0.0, 1), ("ros_default", 1e-3, 0))):
        for scene, sc in (("room_small", te.ROOM_SMALL), ("room_full_640x480", te.ROOM_FULL)):
            name = f"{config}_{scene}"
            scans = sc["scans"]()
            m = omap(sc["voxel"], default_truncation_distance=sc["trunc"])
            m.esdf_create(po.EsdfConfig(max_distance_m=2.0, default_distance_m=2.0, min_distance_m=sc["trunc"] / 2,
                                        min_diff_m=min_diff, multi_queue=multi_queue))
            for s in scans:
                m.integrate(po.MERGED, s)
                m.esdf_update(batch=False, clear_updated_flag=True)
            out["esdf"][name] = {"inputs": scans_digest(scans), "tsdf": oracle_layer_digest(m, 0)}
            for key, a in esdf_case_arrays(m, seed=k).items():
                arrays[f"{name}/{key}"] = a
            print("esdf", name, out["esdf"][name], flush=True)

    gt_scans = te._gt_scans()
    for voxel in (0.2, 0.1):
        trunc, max_d = 4 * voxel, 4.0
        ekw = dict(max_distance_m=max_d, default_distance_m=max_d, min_distance_m=trunc / 2, min_diff_m=0.0,
                   multi_queue=1)
        res = {"inputs": scans_digest(gt_scans)}
        for mode in ("incremental", "batch"):
            m = omap(voxel, default_truncation_distance=trunc)
            m.esdf_create(po.EsdfConfig(**ekw))
            for s in gt_scans:
                m.integrate(po.MERGED, s)
                if mode == "incremental":
                    m.esdf_update(batch=False, clear_updated_flag=True)
            if mode == "batch":
                m.esdf_update(batch=True)
            res[mode] = te._gt_errors(m.blocks(1), voxel, max_d)
        out["esdf_ground_truth"][str(voxel)] = res
        res = {"inputs": scans_digest(gt_scans)}
        for kind in ("simple", "merged", "fast"):
            m = omap(voxel, default_truncation_distance=trunc)
            for s in gt_scans:
                m.integrate(tt.KIND_ID[kind], s)
            res[kind] = {"errors": tt._evaluate(m.blocks(), voxel, trunc), "digest": oracle_layer_digest(m, 0)}
        out["tsdf_ground_truth"][str(voxel)] = res
        print("ground truth", voxel, out["esdf_ground_truth"][str(voxel)], res, flush=True)

    ss = [scenes.c3_room_scan(i) for i in range(4)]
    m = omap(0.05, default_truncation_distance=0.2)
    for s in ss[:3]:
        m.integrate(po.MERGED, s)
    s = ss[3]
    for rrp in (0, 1):
        runs = []
        for k, (dt, yaw) in enumerate(ti.PERTURBATIONS):
            q0, t0 = ti._perturbed(s, dt, yaw)
            q, t, n = m.icp(po.IcpConfig(refine_roll_pitch=rrp), s[0], q0, t0, 7 + k)
            runs.append({"q_wxyz": [float(v).hex() for v in q], "t": [float(v).hex() for v in t], "num_updates": n})
        out["icp"][f"refine_roll_pitch_{rrp}"] = {"inputs": scans_digest(ss), "map": oracle_layer_digest(m, 0),
                                                  "runs": runs}
    print("icp", out["icp"], flush=True)

    out["restatement_pins"] = restatement_pins(ref)
    print("restatement pins", out["restatement_pins"], flush=True)

    with open(JSON_PATH, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    np.savez_compressed(NPZ_PATH, **arrays)
    print("wrote", JSON_PATH, NPZ_PATH)


if __name__ == "__main__":
    main()
