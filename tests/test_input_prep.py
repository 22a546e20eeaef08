"""Input preparation (SURVEY.md 8f-2): near-origin filter + pcl::ApproximateVoxelGrid.

CPU part: the oracle restatement against the reference's goldens and against the numpy restatement that made the fixtures; the
parallel formulation the CUDA kernels implement (512 independent history chains, flushed centroids ranked by the index of the
flushing point) against the serial filter; the C ABI surface of lib/libvgicp_prep_b200.so.
GPU part (-m gpu): the CUDA library against the oracle, bit for bit (in a child process: a fault there cannot poison the CUDA
context of the other GPU tests)."""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, GOLDEN)


def raw_like_cloud(seed, n=40000):
    """A scan-ordered cloud with duplicates at the origin (invalid returns) and a long run of points in one voxel."""
    rng = np.random.default_rng(seed)
    az = np.sort(rng.uniform(-np.pi, np.pi, n))
    r = rng.uniform(2.0, 60.0, n) * (1.0 + 0.3 * np.sin(5 * az))
    pts = np.stack([r * np.cos(az), r * np.sin(az), rng.normal(0.0, 0.8, n) - 1.2], axis=1).astype(np.float32)
    pts[rng.choice(n, n // 15, replace=False)] = 0.0  # invalid returns, scattered
    if n > 1400:
        pts[1000:1400] = 0.0                          # ... and a long run of them
    if n > 5300:
        pts[5000:5300] = pts[5000] + rng.normal(0, 0.003, (300, 3)).astype(np.float32)  # > 16 matches of one entry in one tile
    return pts


def parallel_formulation(pts, leaf, remove_near_origin):
    """What fast_gicp_b200/csrc/prep/vgicp_prep.cu computes, restated with numpy bookkeeping: per history entry an independent
    sequential chain over the points that hash to it; a flushed centroid is stored at the index of the point that flushed it;
    output = those centroids by index, then the entries still holding a voxel in entry order."""
    p = pts.astype(np.float32)
    inv = np.float32(1.0) / np.float32(leaf)
    ijk = np.floor(p * inv).astype(np.int64)
    entry = (ijk[:, 0] * 7171 + ijk[:, 1] * 3079 + ijk[:, 2] * 4231) & 511
    if remove_near_origin:
        sq = (p[:, 0] * p[:, 0] + p[:, 1] * p[:, 1]) + p[:, 2] * p[:, 2]
        entry = np.where(sq < np.float32(1e-3), -1, entry)
    flushed = {}
    tail = []
    for h in range(512):
        idx = np.flatnonzero(entry == h)
        key, cnt, s = None, 0, np.zeros(3, np.float32)
        for i in idx:
            k = tuple(ijk[i])
            if cnt and k != key:
                flushed[i] = s / np.float32(cnt)
                cnt, s = 0, np.zeros(3, np.float32)
            key = k
            cnt += 1
            s = s + p[i]
        if cnt:
            tail.append(s / np.float32(cnt))
    out = [flushed[i] for i in sorted(flushed)] + tail
    return np.asarray(out, dtype=np.float32).reshape(-1, 3)


# k_prep_walk's bookkeeping restated step by step: tiles of 2048 staged points, per-entry lists of <= 16 tile-local indices
# filled in ARBITRARY order (shared-memory atomics) and sorted back, the scan fallback for longer runs, flushes stored at the
# flushing point's index
kHist, kTile, kCap = 512, 2048, 16
def emulate_walk_kernel(pts, leaf, flt, seed=0):
    rng = np.random.default_rng(seed)
    p = pts.astype(np.float32); n = len(p)
    inv = np.float32(1.0)/np.float32(leaf)
    ijk = np.floor(p*inv).astype(np.int64)
    ent = ((ijk[:,0]*7171 + ijk[:,1]*3079 + ijk[:,2]*4231) & 511).astype(np.int64)
    if flt:
        sq = (p[:,0]*p[:,0] + p[:,1]*p[:,1]) + p[:,2]*p[:,2]
        ent = np.where(sq < np.float32(1e-3), 0xFFFF, ent)
    flushed = np.zeros((n,4), np.float32)
    E = [dict(k=None,c=0,s=np.zeros(3,np.float32)) for _ in range(kHist)]
    def step(e,i):
        k = tuple(ijk[i])
        if e['c'] and e['k'] != k:
            flushed[i,:3] = e['s']/np.float32(e['c']); flushed[i,3] = 1
            e['c'] = 0; e['s'] = np.zeros(3,np.float32)
        e['k'] = k; e['c'] += 1; e['s'] = e['s'] + p[i]
    for base in range(0, n, kTile):
        cnt = np.zeros(kHist, int); lst = np.full((kHist,kCap), -1, int)
        sh = np.full(kTile, 0xFFFF, int)
        order = rng.permutation(kTile)   # arbitrary arrival order of the atomics
        for j in order:
            i = base + j
            t = ent[i] if i < n else 0xFFFF
            sh[j] = t
            if t != 0xFFFF:
                q = cnt[t]; cnt[t] += 1
                if q < kCap: lst[t,q] = j
        for h in range(kHist):
            c = cnt[h]
            if 0 < c <= kCap:
                for j in sorted(lst[h,:c]): step(E[h], base+j)
            elif c > kCap:
                for j in range(kTile):
                    if sh[j] == h: step(E[h], base+j)
    out = [flushed[i,:3] for i in range(n) if flushed[i,3] != 0]
    for h in range(kHist):
        if E[h]['c']: out.append(E[h]['s']/np.float32(E[h]['c']))
    return np.asarray(out, np.float32).reshape(-1,3)


# ------------------------------------------------------------------------------------------------------------------ CPU
def test_oracle_matches_the_numpy_restatement_and_the_fixture():
    import make_fixtures as mf

    pts = raw_like_cloud(1, 20000)
    for leaf in (0.1, 0.25, 1.0):
        assert np.array_equal(O.approximate_voxel_grid(pts, leaf), mf.approximate_voxel_grid(pts, leaf))
    kept = O.remove_near_origin(pts)
    assert np.array_equal(kept, mf.remove_near_origin(pts))
    assert len(kept) < len(pts) and not (np.abs(kept).sum(axis=1) == 0).any()


def test_oracle_pinned_by_the_reference_goldens():
    """A window of 3072 raw points of each scan of the reference's data/ pair (tests/golden/scan_window.npz), through
    ApproximateVoxelGrid(0.1) without and with the near-origin filter: bit for bit what make_fixtures.py's restatement gave, in
    the run where that restatement also reproduced README.md:116's full-scan counts (target 17249 / source 17518; produced before
    align.cpp gained its origin filter) and, with the filter (current align.cpp protocol), the committed benchmark fixture."""
    d = np.load(os.path.join(GOLDEN, "scan_window.npz"))
    for name in ("target", "source"):
        raw = d[name + "_raw"]
        assert (np.abs(raw).sum(axis=1) == 0).any()  # invalid returns at the origin: the filter has work to do
        assert np.array_equal(O.approximate_voxel_grid(raw, 0.1), d[name + "_avg"])
        assert np.array_equal(O.approximate_voxel_grid(O.remove_near_origin(raw), 0.1), d[name + "_avg_filtered"])


@pytest.mark.parametrize("flt", [False, True])
def test_parallel_formulation_equals_the_serial_filter(flt):
    pts = raw_like_cloud(2, 12000)
    want = O.approximate_voxel_grid(O.remove_near_origin(pts) if flt else pts, 0.25)
    assert np.array_equal(parallel_formulation(pts, 0.25, flt), want)


@pytest.mark.parametrize("n,leaf,flt", [(1, 0.1, True), (2048, 1.0, False), (9000, 0.1, True), (9000, 1.0, False)])
def test_walk_kernel_bookkeeping_equals_the_serial_filter(n, leaf, flt):
    c = raw_like_cloud(n + 7, n)  # n = 9000 holds both the origin run and a > 16-point run of one entry (scan fallback)
    want = O.approximate_voxel_grid(O.remove_near_origin(c) if flt else c, leaf)
    assert np.array_equal(emulate_walk_kernel(c, leaf, flt), want)


def test_prep_library_exports_its_abi():
    import ctypes

    import build_native

    path = build_native.build_prep()
    from fast_gicp_b200 import prep

    lib = ctypes.CDLL(path)
    hdr = open(os.path.join(ROOT, "include", "vgicp_prep_b200.h")).read()
    for sym in prep.EXPORTED_SYMBOLS:
        assert hasattr(lib, sym) and sym + "(" in hdr
    import re

    declared = set(re.findall(r"VGICP_PREP_API\s+[\w\s\*]+?\b(vgicp_prep_\w+)\s*\(", hdr))
    assert declared == set(prep.EXPORTED_SYMBOLS)


# ------------------------------------------------------------------------------------------------------------------ GPU
_CHILD = r"""
import sys, numpy as np
sys.path.insert(0, %r)
sys.path.insert(0, %r)
import oracle as O
from fast_gicp_b200.prep import InputPrep
from test_input_prep import raw_like_cloud
p = InputPrep(0)
d = np.load(%r)
clouds = [raw_like_cloud(3), raw_like_cloud(4, 3000), raw_like_cloud(5, 2048), raw_like_cloud(6, 1), np.repeat(d["target"], 4, axis=0)]
for c in clouds:
    for leaf, flt in ((0.1, True), (0.25, False), (1.0, True)):
        got = p.approximate_voxel_grid(c, leaf, flt)
        want = O.approximate_voxel_grid(O.remove_near_origin(c) if flt else c, leaf)
        assert got.shape == want.shape, (got.shape, want.shape)
        assert np.array_equal(got, want)
assert len(p.approximate_voxel_grid(np.zeros((0, 3), np.float32), 0.1)) == 0
print("prep ok")
"""


@pytest.mark.gpu
def test_gpu_input_prep_matches_the_oracle_bit_for_bit():
    code = _CHILD % (ROOT, os.path.join(ROOT, "tests"), os.path.join(GOLDEN, "pair_0p2.npz"))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "prep ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
