#!/usr/bin/env python3
"""Generate the committed golden input fixtures from the reference's own data files.

    python tests/golden/make_fixtures.py <fast_gicp checkout>/data

Reads  <data>/251370668.pcd (target), 251371071.pcd (source), relative.txt
Writes tests/golden/pair_0p1.npz   -- the reference's benchmark inputs: near-origin filter
                                      (src/align.cpp:128-133) + ApproximateVoxelGrid(0.1) (src/align.cpp:136-147)
       tests/golden/pair_0p2.npz   -- the reference's test inputs: VoxelGrid(0.2) (src/test/gicp_test.cpp:55-65)
       tests/golden/relative.txt   -- ground-truth pose (data/relative.txt), numbers only
       tests/golden/scan_window.npz -- a window of SCAN_WINDOW raw points of each scan and its ApproximateVoxelGrid(0.1) without
                                      and with the near-origin filter (the raw scans are too large to commit whole)

PCL is not vendored in the reference, so both filters are restated from the published PCL algorithm
(pcl/filters/approximate_voxel_grid.hpp, voxel_grid.hpp).  The restatement of ApproximateVoxelGrid (and of the PCD reader) is PINNED by
the point counts the reference prints in README.md:116 (target 17249 / source 17518), which it reproduces exactly when
the near-origin filter (added to align.cpp after the README run) is skipped: this script asserts them.  The committed
pair_0p1 follows the CURRENT align.cpp protocol (filter, then downsample): 17047 / 17334 points.
"""
import os
import sys
import numpy as np

OUT = os.path.dirname(os.path.abspath(__file__))
# raw points [start, start + 3072) of each scan: a stretch of the scan with many invalid returns at the origin
SCAN_WINDOW = slice(36864, 36864 + 3072)


def read_pcd_xyz(path):
    """Binary PCD reader (FIELDS x y z intensity, 4xF32) -> (N,3) float32."""
    with open(path, "rb") as f:
        raw = f.read()
    pos = 0
    fields, sizes, npts = None, None, None
    while True:
        end = raw.index(b"\n", pos)
        line = raw[pos:end].decode("ascii", "replace").strip()
        pos = end + 1
        if line.startswith("FIELDS"):
            fields = line.split()[1:]
        elif line.startswith("SIZE"):
            sizes = [int(s) for s in line.split()[1:]]
        elif line.startswith("POINTS"):
            npts = int(line.split()[1])
        elif line.startswith("DATA"):
            assert line.split()[1] == "binary", line
            break
    assert fields[:3] == ["x", "y", "z"] and all(s == 4 for s in sizes)
    stride = len(fields)
    data = np.frombuffer(raw, dtype=np.float32, count=npts * stride, offset=pos).reshape(npts, stride)
    return np.ascontiguousarray(data[:, :3])


def remove_near_origin(pts):
    """src/align.cpp:128-133 : drop points with squaredNorm() < 1e-3 (float arithmetic)."""
    p = pts.astype(np.float32)
    sq = (p[:, 0] * p[:, 0] + p[:, 1] * p[:, 1]) + p[:, 2] * p[:, 2]
    return pts[~(sq < np.float32(1e-3))]


def approximate_voxel_grid(pts, leaf, histsize=512):
    """pcl::ApproximateVoxelGrid<PointXYZ>::applyFilter restated (PCL 1.10+ approximate_voxel_grid.hpp).

    Streaming filter with a 512-entry hash history: a point goes to slot
    hash = (ix*7171 + iy*3079 + iz*4231) & (histsize-1); if the slot holds a different voxel it is flushed
    (centroid emitted) first.  ix = floor(x * inverse_leaf_size) in float.
    """
    inv = np.float32(1.0) / np.float32(leaf)
    ijk = np.floor(pts.astype(np.float32) * inv).astype(np.int64)
    hashes = ((ijk[:, 0] * 7171 + ijk[:, 1] * 3079 + ijk[:, 2] * 4231) & (histsize - 1)).astype(np.int64)
    h_ix = [(0, 0, 0)] * histsize
    h_cnt = [0] * histsize
    h_sum = np.zeros((histsize, 3), dtype=np.float32)
    out = []
    p32 = pts.astype(np.float32)
    ijk_l = [tuple(r) for r in ijk.tolist()]
    for i in range(len(pts)):
        h = hashes[i]
        key = ijk_l[i]
        if h_cnt[h] and h_ix[h] != key:
            out.append(h_sum[h] / np.float32(h_cnt[h]))
            h_cnt[h] = 0
            h_sum[h] = 0
        h_ix[h] = key
        h_cnt[h] += 1
        h_sum[h] += p32[i]          # float accumulation like Eigen::VectorXf centroid
    for h in range(histsize):
        if h_cnt[h]:
            out.append(h_sum[h] / np.float32(h_cnt[h]))
    return np.asarray(out, dtype=np.float32)


def voxel_grid(pts, leaf):
    """pcl::VoxelGrid<PointXYZ>::applyFilter restated (voxel_grid.hpp): exact centroid per leaf.

    ijk = floor(p * inverse_leaf) - min_b ; idx = ijk . (1, dx, dx*dy); output sorted by idx; centroid in float.
    """
    p = pts.astype(np.float32)
    inv = np.float32(1.0) / np.float32(leaf)
    min_p = p.min(axis=0)
    max_p = p.max(axis=0)
    min_b = np.floor(min_p * inv).astype(np.int64)
    max_b = np.floor(max_p * inv).astype(np.int64)
    div_b = max_b - min_b + 1
    mul = np.array([1, div_b[0], div_b[0] * div_b[1]], dtype=np.int64)
    ijk = np.floor(p * inv).astype(np.int64) - min_b
    idx = ijk @ mul
    order = np.argsort(idx, kind="stable")
    idx_s = idx[order]
    p_s = p[order]
    starts = np.flatnonzero(np.r_[True, idx_s[1:] != idx_s[:-1]])
    ends = np.r_[starts[1:], len(idx_s)]
    out = np.empty((len(starts), 3), dtype=np.float32)
    for n, (s, e) in enumerate(zip(starts, ends)):
        c = np.zeros(3, dtype=np.float32)
        for j in range(s, e):
            c += p_s[j]
        out[n] = c / np.float32(e - s)
    return out


def main(ref):
    tgt = read_pcd_xyz(os.path.join(ref, "251370668.pcd"))
    src = read_pcd_xyz(os.path.join(ref, "251371071.pcd"))
    assert tgt.shape == (69088, 3) and src.shape == (69792, 3)
    rel = np.loadtxt(os.path.join(ref, "relative.txt"))
    np.savetxt(os.path.join(OUT, "relative.txt"), rel, fmt="%.9g")

    # benchmark protocol (align.cpp): filter + ApproximateVoxelGrid(0.1)
    # PIN: the README numbers were produced before the near-origin filter was added to align.cpp; without
    # the filter the restated ApproximateVoxelGrid reproduces README.md:116 exactly.
    n_t, n_s = len(approximate_voxel_grid(tgt, 0.1)), len(approximate_voxel_grid(src, 0.1))
    print("ApproximateVoxelGrid(0.1), no origin filter: target", n_t, "source", n_s, "(README.md:116: 17249 / 17518)")
    assert (n_t, n_s) == (17249, 17518), "ApproximateVoxelGrid restatement no longer pinned"
    t1 = approximate_voxel_grid(remove_near_origin(tgt), 0.1)
    s1 = approximate_voxel_grid(remove_near_origin(src), 0.1)
    print("pair_0p1 (current align.cpp protocol, with origin filter): target", len(t1), "source", len(s1))
    assert (len(t1), len(s1)) == (17047, 17334)
    np.savez_compressed(os.path.join(OUT, "pair_0p1.npz"), target=t1, source=s1)

    # test protocol (gicp_test.cpp): VoxelGrid(0.2), no origin filter
    t2 = voxel_grid(tgt, 0.2)
    s2 = voxel_grid(src, 0.2)
    print("pair_0p2: target", len(t2), "source", len(s2))
    np.savez_compressed(os.path.join(OUT, "pair_0p2.npz"), target=t2, source=s2)

    win = {}
    for name, cloud in (("target", tgt), ("source", src)):
        raw = np.ascontiguousarray(cloud[SCAN_WINDOW])
        win[name + "_raw"] = raw
        win[name + "_avg"] = approximate_voxel_grid(raw, 0.1)
        win[name + "_avg_filtered"] = approximate_voxel_grid(remove_near_origin(raw), 0.1)
    print("scan_window: raw", len(win["target_raw"]), "/", len(win["source_raw"]), "-> target", len(win["target_avg"]), len(win["target_avg_filtered"]),
          "source", len(win["source_avg"]), len(win["source_avg_filtered"]))
    np.savez_compressed(os.path.join(OUT, "scan_window.npz"), **win)


if __name__ == "__main__":
    if len(sys.argv) != 2 or not os.path.isdir(sys.argv[1]):
        sys.exit(__doc__)
    main(sys.argv[1])
