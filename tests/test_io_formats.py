"""The host-side file formats (icp_variants_b200/io.py) against the reference's own readers where the reference build
is available (SimpleMesh::loadMesh through oracle/_ref), the bundled bunny files, and hand-written fixtures."""
import os

import numpy as np
import pytest

from icp_variants_b200 import io as fio
from icp_variants_b200 import synth
from oracle import ref as R

REF_DATA = os.path.join(R.REFERENCE_ROOT, "Data")


def test_off_round_trip_and_rules(tmp_path, bunny):
    src, tgt, _, _ = bunny
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "bunny.npz"))
    p = str(tmp_path / "m.off")
    v = z["target_vertices"].copy(); v[5, 1] = np.nan
    fio.write_off(p, v, z["target_colors"], z["target_faces"])
    v2, c2, f2 = fio.read_off(p)
    ok = np.isfinite(v).all(1)
    assert np.array_equal(v2[ok], v[ok]) and np.array_equal(f2, z["target_faces"])
    assert np.array_equal(v2[5], [0, 0, 0]) and np.array_equal(c2[5], [0, 0, 0, 0])       # SimpleMesh.h:245-246
    assert np.array_equal(c2[ok], z["target_colors"][ok])
    with open(p, "w") as f:
        f.write("OFF\n3 1 0\n0 0 0\n1 0 0\n0 1 0\n3 0 1 2\n")
    v3, c3, f3 = fio.read_off(p)
    assert v3.shape == (3, 3) and (c3 == [0, 0, 0, 255]).all() and f3.tolist() == [[0, 1, 2]]
    with open(p, "w") as f:
        f.write("PLY\n")
    with pytest.raises(ValueError):
        fio.read_off(p)
    with open(p, "w") as f:
        f.write("OFF\n4 1 0\n0 0 0\n1 0 0\n0 1 0\n1 1 0\n4 0 1 2 3\n")
    with pytest.raises(ValueError):
        fio.read_off(p)


@pytest.mark.skipif(not os.path.isdir(REF_DATA), reason="the reference's bundled .off files (ICP_REFERENCE_ROOT/Data) are absent")
def test_off_reader_equals_reference_loader(tmp_path, bunny):
    src, tgt, _, _ = bunny
    for name, cloud in (("bunny_part1.off", tgt), ("bunny_part2_trans.off", src)):
        v, c, f = fio.read_off(os.path.join(REF_DATA, name))
        pr, nr = R.cloud_from_off(os.path.join(REF_DATA, name))              # SimpleMesh::loadMesh + PointCloud(mesh)
        assert np.array_equal(v, pr) and np.array_equal(v, cloud.points)
        m = synth.mesh_to_cloud(v, f)
        assert np.array_equal(m.normals, nr)
        # and the reference reads back what write_off writes (COFF with colours)
        out = str(tmp_path / name)
        fio.write_off(out, v, c, f)
        pr2, nr2 = R.cloud_from_off(out)
        assert np.array_equal(pr2, pr) and np.array_equal(nr2, nr)


def test_tum_lists_trajectory_and_depth(tmp_path):
    p = str(tmp_path / "depth.txt")
    with open(p, "w") as f:
        f.write("# depth maps\n# file: 'x.bag'\n# timestamp filename\n1305031102.160407 depth/1305031102.160407.png\n1305031102.194330 depth/1305031102.194330.png\n")
    ts, names = fio.read_tum_file_list(p)
    assert ts.tolist() == [1305031102.160407, 1305031102.194330] and names[1] == "depth/1305031102.194330.png"
    g = str(tmp_path / "groundtruth.txt")
    with open(g, "w") as f:
        f.write("# ground truth trajectory\n# file: 'x.bag'\n# timestamp tx ty tz qx qy qz qw\n"
                "1305031098.6659 1.3563 0.6305 1.6380 0.6132 0.5962 -0.3311 -0.3986\n"
                "1305031098.6758 1.3543 0.6306 1.6360 0.6129 0.5966 -0.3316 -0.3980\n"
                "1305031098.6858 0 0 0 0 0 0 0\n"
                "1305031098.6958 1 1 1 0 0 0 1\n")
    tts, poses = fio.read_tum_trajectory(g)
    assert len(tts) == 2 and poses.shape == (2, 4, 4)                         # stops at the zero quaternion (VirtualSensor.h:241)
    # stored inverted: pose^-1 maps the camera origin to the recorded translation
    inv = np.linalg.inv(poses[0].astype(np.float64))
    assert np.allclose(inv[:3, 3], [1.3563, 0.6305, 1.6380], atol=1e-5)
    from scipy.spatial.transform import Rotation
    assert np.allclose(inv[:3, :3], Rotation.from_quat([0.6132, 0.5962, -0.3311, -0.3986]).as_matrix(), atol=2e-4)
    assert fio.nearest_trajectory_index(tts, 1305031098.6700) == 0 and fio.nearest_trajectory_index(tts, 1305031098.6720) == 1
    d = fio.tum_depth_to_float(np.array([[0, 5000], [2500, 65535]], np.uint16))
    assert np.isneginf(d[0, 0]) and d[0, 1] == 1.0 and d[1, 0] == 0.5 and d[1, 1] == np.float32(65535) / np.float32(5000)


def test_eth_pair_list(tmp_path):
    p = str(tmp_path / "apartment_global.csv")
    with open(p, "w") as f:
        f.write("id,reading,reference,t_overlap,T00,T01,T02,T03,T10,T11,T12,T13,T20,T21,T22,T23\n"
                "0,PointCloud1.pcd,PointCloud0.pcd,0.9,1,0,0,0.5,0,1,0,-0.25,0,0,1,2\n"
                "1,PointCloud2.pcd,PointCloud1.pcd,0.8,0,-1,0,0,1,0,0,0,0,0,1,0\n")
    rows = fio.read_eth_pairs(p)
    assert len(rows) == 2 and rows[0]["source"] == "PointCloud1.pcd" and rows[0]["target"] == "PointCloud0.pcd"
    assert rows[0]["pose"][:3, 3].tolist() == [0.5, -0.25, 2.0] and rows[1]["pose"][0, 1] == -1 and rows[1]["pose"][3].tolist() == [0, 0, 0, 1]


def test_pcd_ply_and_dump_round_trips(tmp_path):
    """PCD (pcl::io::loadPCDFile, ETHDataLoader.h:68,87), PLY (PointCloud::writeToFile, PointCloud.h:219-236) and the PointCloud binary
    dump (PointCloud.h:167-217): ascii and binary forms read back bit for bit, NaN points survive, extra fields come back by name."""
    rng = np.random.default_rng(0)
    p = rng.normal(size=(257, 3)).astype(np.float32); p[5] = np.nan
    n = rng.normal(size=(257, 3)).astype(np.float32)
    for binary in (False, True):
        f = str(tmp_path / f"c{int(binary)}.pcd"); fio.write_pcd(f, p, binary)
        q, extra = fio.read_pcd(f)
        assert np.array_equal(q, p, equal_nan=True) and extra == {}
        g = str(tmp_path / f"c{int(binary)}.ply"); fio.write_ply(g, p, n, binary)
        q, m, extra = fio.read_ply(g)
        assert np.array_equal(q, p, equal_nan=True) and np.array_equal(m, n) and extra == {}
    # a PCD as PCL writes clouds with normals (FIELDS x y z normal_x normal_y normal_z curvature), ascii
    f = str(tmp_path / "n.pcd")
    with open(f, "w") as fh:
        fh.write("# .PCD v0.7\nVERSION 0.7\nFIELDS x y z normal_x normal_y normal_z curvature\nSIZE 4 4 4 4 4 4 4\nTYPE F F F F F F F\n"
                 "COUNT 1 1 1 1 1 1 1\nWIDTH 2\nHEIGHT 1\nVIEWPOINT 0 0 0 1 0 0 0\nPOINTS 2\nDATA ascii\n1 2 3 0 0 1 0.5\n4 5 6 0 1 0 0.25\n")
    q, extra = fio.read_pcd(f)
    assert np.array_equal(q, np.array([[1, 2, 3], [4, 5, 6]], np.float32)) and np.array_equal(extra["curvature"], [0.5, 0.25])
    # the PLY layout of pcl::io::savePLYFile for PointXYZINormal: intensity between the point and the normal, curvature after it
    g = str(tmp_path / "pcl.ply")
    with open(g, "w") as fh:
        fh.write("ply\nformat ascii 1.0\ncomment PCL generated\nelement vertex 2\nproperty float x\nproperty float y\nproperty float z\n"
                 "property float intensity\nproperty float normal_x\nproperty float normal_y\nproperty float normal_z\nproperty float curvature\n"
                 "element camera 1\nproperty float view_px\nend_header\n1 2 3 1 0 0 1 0\n4 5 6 1 0 1 0 0\n0\n")
    q, m, extra = fio.read_ply(g)
    assert np.array_equal(q, np.array([[1, 2, 3], [4, 5, 6]], np.float32)) and np.array_equal(m, np.array([[0, 0, 1], [0, 1, 0]], np.float32))
    assert np.array_equal(extra["intensity"], [1, 1])
    for double in (False, True):
        d = str(tmp_path / f"d{int(double)}.bin"); fio.write_pointcloud_dump(d, p, n, double)
        q, m = fio.read_pointcloud_dump(d)
        assert np.array_equal(q, p, equal_nan=True) and np.array_equal(m, n)
