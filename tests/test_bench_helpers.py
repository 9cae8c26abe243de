"""bench.py's helpers (no GPU): byte model, checksum combination, group counting, roofline block arithmetic, the map
sample written by --dump-outputs."""
import argparse
import importlib.util
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_algorithmic_bytes_matches_design_model():
    b = _bench()
    # DESIGN.md §4: Nv (8 R + 8 W + 4 W) + Nsem (2*4*Lp + 4) + P*8 + Nblk*16
    nv, nsem, nblk, P = 117989, 25031, 325, 640 * 480
    got = b.algorithmic_bytes(nv, nsem, nblk, P)
    assert got == nv * 20 + nsem * 164 + P * 8 + nblk * 16
    assert abs(got / 1e6 - 8.95) < 0.05  # ~8.9-9.0 MB/frame (DESIGN.md §4, VERDICT r1)


def test_group_count_and_checksum_combination():
    b = _bench()
    assert [b.n_groups(n) for n in (1, 32, 33, 5000)] == [1, 1, 2, 157]
    parts = [((1 << 64) - 5, 0b1010, 3, 10), (9, 0b0110, 4, 20)]
    c = b.combine_checksums(parts)
    assert c == {"sum": "%016x" % 4, "xor": "%016x" % 0b1100, "blocks": 7, "observed_voxels": 30}


def test_roofline_block_fraction():
    b = _bench()
    args = argparse.Namespace(workload="hall640", small=False)
    # 157 groups of a 5000-frame lap at 8.98 MB/frame in 28 ms
    r = b.roofline_block(args, 32, 157, 28.0, 178.0, 117989 * 5000, 25031 * 5000, 325 * 5000, 5000, 640 * 480, 8)
    total = b.algorithmic_bytes(117989 * 5000, 25031 * 5000, 325 * 5000, 5000 * 640 * 480)
    assert abs(r["achieved"] - total / 28e-3 / 1e9) < 1e-6
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12 and 0.1 < r["frac"] < 0.5
    assert abs(r["launch_us"] - 28000.0 / 157) < 1e-9 and r["unit"] == "GB/s" and r["bound"] == "hbm"
    assert abs(r["algorithmic_bytes_per_launch"] - total / 157) < 1.0


def test_dump_outputs_is_a_sample_of_the_exported_map(oracle_lib, tmp_path, monkeypatch):
    """--dump-outputs on a map behind the same C ABI (the oracle's): every block index, and the voxels of the sampled
    blocks exactly as kb_export_blocks returns them; float32 / float64 only; the same sample on every run."""
    import numpy as np
    import harness as hs
    from khronos_b200 import synthetic as syn
    b = _bench()
    cam = hs.small_camera(4)
    poses, stamps = syn.orbit_trajectory(4, laps=0.05)
    h = hs.make_handle(oracle_lib, "ko_", cam=cam)
    hs.run_fusion(h, hs.render_frames(syn.room_scene(), cam, poses, stamps), poses, stamps, tracking=True)
    ex = h.export_blocks(likelihoods=False)
    monkeypatch.setattr(b, "DUMP_SAMPLE_BLOCKS", ex.n // 3)
    b.dump_outputs(h, str(tmp_path / "a"))
    b.dump_outputs(h, str(tmp_path / "b"))
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b")) and len(names) == 6
    d = {n[:-4]: np.load(tmp_path / "a" / n) for n in names}
    for n in names:
        np.testing.assert_array_equal(d[n[:-4]], np.load(tmp_path / "b" / n))
        assert d[n[:-4]].dtype in (np.float32, np.float64)
    np.testing.assert_array_equal(d["block_index"], ex.block_index)
    pos = [int(np.flatnonzero((ex.block_index == r).all(1))[0]) for r in d["sample_block_index"]]
    assert len(pos) == ex.n // 3 and pos == sorted(set(pos))
    np.testing.assert_array_equal(d["sample_distance"], ex.distance[pos])
    np.testing.assert_array_equal(d["sample_weight"], ex.weight[pos])
    np.testing.assert_array_equal(d["sample_last_observed_ns"], ex.last_observed[pos].astype(np.float64))
    lab = np.where(ex.semantic_empty[pos] != 0, -1, ex.semantic_label[pos].astype(np.int64))
    np.testing.assert_array_equal(d["sample_semantic_label"], lab)
    assert (d["sample_weight"] > 0).any() and (d["sample_semantic_label"] >= 0).any()
