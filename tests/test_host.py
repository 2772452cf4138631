"""CPU: host-side logic and the C-ABI surface (no compute calls without a GPU)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    g.build()
    import icp_slam_yolo_b200 as m
    return m


def test_cabi_exports_every_declared_symbol(pkg):
    header = open(os.path.join(ROOT, "include", "b200icp.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(b200icp_[a-z0-9_]+)\s*\(", header))
    assert {"b200icp_nn_batch", "b200icp_align_batch", "b200icp_polar_to_cartesian",
            "b200icp_version", "b200icp_last_error"} <= declared
    handle = ctypes.CDLL(pkg.library_path())
    for name in declared:
        assert hasattr(handle, name), f"{name} declared in b200icp.h but not exported"
    from icp_slam_yolo_b200 import _cabi
    assert set(_cabi.SYMBOLS) == declared
    assert pkg.lib().b200icp_version() == 3
    assert pkg.lib().b200icp_max_src_pitch() == 1024 and pkg.lib().b200icp_max_tgt_pitch() == 4096


def test_cabi_rejects_bad_arguments_without_touching_the_gpu(pkg):
    from icp_slam_yolo_b200 import _cabi
    L = pkg.lib()
    assert L.b200icp_nn_batch(None, 1, None, None, 0, None) == 1
    pr = _cabi.Problem()
    assert L.b200icp_nn_batch(ctypes.byref(pr), 1, None, None, 0, None) == 1
    assert b"NULL" in L.b200icp_last_error()
    pr.src_points = pr.tgt_points = 4096
    pr.src_pitch, pr.tgt_pitch, pr.dtype = 2000, 16, _cabi.F64
    assert L.b200icp_nn_batch(ctypes.byref(pr), 1, ctypes.c_void_p(4096), None, 0, None) == 2
    pr.src_pitch, pr.pairing, pr.n_rows = 16, _cabi.PAIR_TRIANGLE, 4
    assert L.b200icp_nn_batch(ctypes.byref(pr), 7, ctypes.c_void_p(4096), None, 0, None) == 1
    assert L.b200icp_align_batch(ctypes.byref(pr), 1, None, None, None) == 1
    assert L.b200icp_polar_to_cartesian(None, None, 1, 1, None, None, None, 1, None) == 1
    assert L.b200icp_s2m_search(None, None, None, None, 1, None, None, 1, 0, None, None, None) == 1
    assert L.b200icp_s2m_inbox_bytes(8192, 8) == 2 * 8 * 8192 * 32 + 17 * 8 and L.b200icp_s2m_inbox_bytes(8, 99) == -1
    assert L.b200icp_s2m_padded_chunks(1) == 32 and L.b200icp_s2m_padded_chunks(32 * 1024 + 1) == 64


def test_no_cpu_fallback(pkg):
    with pytest.raises(pkg.B200IcpError, match="CUDA tensor"):
        pkg.ScanTable(torch.zeros((2, 8, 2), dtype=torch.float64))
    if not torch.cuda.is_available():
        with pytest.raises(Exception):
            pkg.icp(np.random.rand(8, 2), np.random.rand(8, 2))


def test_missing_library_fails_loudly(pkg, monkeypatch, tmp_path):
    from icp_slam_yolo_b200 import _cabi, build
    monkeypatch.setattr(_cabi, "_lib", None)
    monkeypatch.setattr(build, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(pkg.B200IcpError, match="no CPU fallback"):
        _cabi.lib()


def test_product_never_imports_the_oracle():
    pkgdir = os.path.join(ROOT, "icp_slam-yolo_b200")
    for dirpath, _, files in os.walk(pkgdir):
        for f in files:
            if f.endswith((".py", ".cu", ".h", ".cuh")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f
                assert "scipy" not in text, f


def test_pack_host_and_shapes(pkg):
    scans = [np.arange(10.0).reshape(5, 2), np.zeros((0, 2)), np.ones((3, 3))]
    pts, lens = pkg.ScanTable.pack_host(scans, dtype=np.float32)
    assert pts.shape == (3, 5, 2) and pts.dtype == torch.float32 and lens.tolist() == [5, 0, 3]
    assert torch.equal(pts[0], torch.arange(10.0).reshape(5, 2))
    assert torch.all(pts[1] == 0) and torch.all(pts[2, :3] == 1) and torch.all(pts[2, 3:] == 0)
    with pytest.raises(ValueError):
        pkg.ScanTable.pack_host(scans, pitch=4)


def test_shard_range_partitions_exactly(pkg):
    for n in (0, 1, 7, 1830, 65536, 8386560):
        for w in (1, 2, 3, 4, 8):
            spans = [pkg.shard_range(n, r, w) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(w - 1))
            sizes = [e - b for b, e in spans]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        pkg.shard_range(10, 2, 2)


def test_triangle_enumeration(pkg):
    n = 9
    seen = [pkg.triangle_pair(q, n) for q in range(pkg.triangle_pair_count(n))]
    assert seen == [(i, j) for i in range(n) for j in range(i + 1, n)]
    assert pkg.triangle_pair_count(4096) == 8386560


def test_chain_poses(pkg):
    rng = np.random.default_rng(0)
    poses = []
    for _ in range(20):
        th = rng.uniform(-0.1, 0.1)
        poses.append([np.cos(th), -np.sin(th), np.sin(th), np.cos(th), *rng.uniform(-50, 50, 2)])
    chain = pkg.chain_poses(np.array(poses))
    T = np.eye(3)
    for p in poses:
        M = np.eye(3); M[:2, :2] = np.array(p[:4]).reshape(2, 2); M[:2, 2] = p[4:]
        T = T @ M
    assert chain.shape == (21, 6) and np.allclose(chain[-1, :4].reshape(2, 2), T[:2, :2])
    assert np.allclose(chain[-1, 4:], T[:2, 2]) and np.array_equal(chain[0], [1, 0, 0, 1, 0, 0])


def test_scan_io(pkg, raw_scans, tmp_path):
    # the bundled recording switches file-name case at scan 220 (SURVEY.md §8 a1)
    np.save(tmp_path / "Scan_data_1.npy", raw_scans[0])
    np.save(tmp_path / "scan_data_2.npy", raw_scans[2])
    np.save(tmp_path / "scan_data_3.npy", np.zeros((4, 5)))            # invalid shape -> skipped
    (tmp_path / "scan_data_4.npy").write_bytes(b"not an npy file")
    np.save(tmp_path / "scan_data_5.npy", np.ones((6, 2)))
    scans, numbers = pkg.scan_io.load_raw_sequence(str(tmp_path), 1, 6)
    assert numbers == [1, 2, 5] and np.array_equal(scans[1], raw_scans[2]) and scans[2].shape == (6, 2)
    assert pkg.scan_io.load_raw_scan(None) is None
    raw, lens = pkg.scan_io.raw_table(raw_scans[:4])
    assert raw.shape == (4, max(len(r) for r in raw_scans[:4]), 3) and lens.tolist() == [len(r) for r in raw_scans[:4]]
    fx = pkg.scan_io.unpack_fixture(os.path.join(ROOT, "tests", "golden", "scan_data_1_packed.npz"))
    assert len(fx) == 1831 and np.array_equal(fx[7], raw_scans[7])


def test_map_io_pcd_and_png_round_trip(tmp_path):
    """The reference's map outputs (slam_offline.py:445-453): binary x y z float32 PCD as Open3D
    writes it and an 8-bit RGB PNG as cv2.imwrite does."""
    import icp_slam_yolo_b200 as pkg
    rng = np.random.Generator(np.random.PCG64(3))
    pts = rng.normal(0, 3000, size=(257, 2))
    p = str(tmp_path / "map.pcd")
    pkg.map_io.write_pcd(p, pts)
    back = pkg.map_io.read_pcd(p)
    assert back.shape == (257, 3) and np.array_equal(back[:, :2], pts.astype(np.float32)) and not back[:, 2].any()
    blob = open(p, "rb").read()
    assert blob.startswith(b"# .PCD v0.7 - Point Cloud Data file format\nVERSION 0.7\nFIELDS x y z\nSIZE 4 4 4\n")
    assert b"\nWIDTH 257\nHEIGHT 1\nVIEWPOINT 0 0 0 1 0 0 0\nPOINTS 257\nDATA binary\n" in blob
    q = str(tmp_path / "again.pcd")                  # re-writing a map is the identity
    pkg.map_io.write_pcd(q, pkg.map_io.read_pcd(p))
    assert open(q, "rb").read() == blob

    img = rng.integers(0, 256, size=(37, 53, 3), dtype=np.uint8)
    f = str(tmp_path / "occ.png")
    pkg.map_io.write_png(f, img)
    assert np.array_equal(pkg.map_io.read_png(f), img)
    try:
        import cv2
    except ImportError:
        cv2 = None
    if cv2 is not None:
        assert np.array_equal(cv2.imread(f, cv2.IMREAD_UNCHANGED), img)          # OpenCV decodes our file
        g = str(tmp_path / "cv.png")
        cv2.imwrite(g, img)
        assert np.array_equal(pkg.map_io.read_png(g), img)                         # and we decode OpenCV's


def test_hostmem_topology_parsing_and_binding(pkg, tmp_path, monkeypatch):
    """hostmem.near_gpu: reads the GPU's NUMA node from sysfs, binds the thread for the block and restores it;
    degrades to a recorded no-op when the platform says nothing."""
    hm = pkg.hostmem
    assert hm.parse_cpulist("0-3,8,10-11") == {0, 1, 2, 3, 8, 10, 11} and hm.parse_cpulist("") == set()
    sysfs = tmp_path / "sys"
    dev = sysfs / "bus/pci/devices/0000:1b:00.0"
    dev.mkdir(parents=True)
    mine = sorted(os.sched_getaffinity(0))
    for node, cpus in ((0, mine[:1]), (1, mine[-1:])):
        d = sysfs / f"devices/system/node/node{node}"
        d.mkdir(parents=True)
        (d / "cpulist").write_text(",".join(map(str, cpus)) + "\n")
    (sysfs / "devices/system/node/online").write_text("0-1\n")
    monkeypatch.setattr(hm, "gpu_pci_address", lambda i: "0000:1b:00.0")
    monkeypatch.setattr(hm, "_set_mempolicy", lambda mode, node: False)
    (dev / "numa_node").write_text("-1\n")                       # VM without NUMA information
    with hm.near_gpu(0, sysfs=str(sysfs)) as rec:
        assert rec["node"] is None and not rec["bound"] and "no NUMA node" in rec["why"]
    (dev / "numa_node").write_text("1\n")
    before = os.sched_getaffinity(0)
    with hm.near_gpu(0, sysfs=str(sysfs)) as rec:
        assert rec["node"] == 1 and rec["host_nodes"] == [0, 1] and rec["bound"]
        assert os.sched_getaffinity(0) == {mine[-1]}
    assert os.sched_getaffinity(0) == before
    (sysfs / "devices/system/node/online").write_text("0\n")
    with hm.near_gpu(0, sysfs=str(sysfs)) as rec:
        assert not rec["bound"] and rec["why"] == "single NUMA node"


def test_host_pipeline_chunk_schedule(pkg):
    """HostPipeline's chunk sizes: cover the batch exactly, never exceed the staging buffers, ramp up
    by at most the growth factor from a short first chunk (the first copy is exposed) and end with
    shrinking chunks (the last kernel is exposed)."""
    from icp_slam_yolo_b200.registration import HostPipeline
    for n in (1, 2, 5, 100, 1830, 8192, 65536, 65537, 1 << 20):
        for chunks in (1, 2, 4, 8, 16):
            sizes = HostPipeline.chunk_schedule(n, chunks)
            big = max(1, -(-n // chunks))
            assert sum(sizes) == n and min(sizes) >= 1 and max(sizes) <= big, (n, chunks, sizes)
            if chunks == 1:
                assert sizes == [n]
    sizes = HostPipeline.chunk_schedule(65536, 8)
    big = 8192
    assert sizes[0] == big // 8 and sizes[-1] <= big // 4
    peak = sizes.index(big)
    for a, b in zip(sizes[:peak], sizes[1:peak + 1]):
        assert b <= int(a * 1.25) + 1 or b == big and a * 1.25 >= big * 0.9, (a, b)
    assert sizes[peak:] == sorted(sizes[peak:], reverse=True)
