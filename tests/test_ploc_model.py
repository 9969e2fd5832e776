"""PLOC's merge rounds (csrc/bvh_device.cu, PTAP_ACCEL_BVH_DEVICE) restated in numpy: Morton keys of the triangle centroids
(k_lbvh_keys), fattened boxes (fatBox), the nearest neighbour within 16 positions by union area with a tie key (k_ploc_nearest) and the
merge of mutual pairs (k_ploc_merge), in binary32.

Every round is a host round trip, and the build gives up after 4096 rounds.  A tie rule that is not symmetric ("the lower position")
lets tied clusters point along a chain in which only the first pair is mutual: coincident triangles and long ribbons of equal quads
then merge one or a few pairs per round.  The symmetric key makes the globally best pair of every run of ties mutual.

The model stands apart from the kernel: it does not contract the centroid and box-corner arithmetic into FMAs as nvcc may, so its boxes
can differ from the device's in the last bit.  The round counts rest on exact ties of equal geometry, which both compute alike.
test_kernel_uses_the_symmetric_key ties the model's rule to the source of k_ploc_nearest."""
import os
import re

import numpy as np
import pytest

from test_gpu_degenerate_geometry import coincident_mesh, degenerate_mix_mesh, plane_mesh, ribbon_mesh, tube_mesh

RADIUS, TOP = 16, 4096          # kPlocRadius, kPlocTop
BAND = np.float32(0.0056)       # kBandEpsF
F = np.float32


def _expand(v):
    v = v.astype(np.uint64)
    v = (v * 0x00010001) & 0xFF0000FF
    v = (v * 0x00000101) & 0x0F00F00F
    v = (v * 0x00000011) & 0xC30C30C3
    v = (v * 0x00000005) & 0x49249249
    return v


def leaf_boxes(p, tri):
    """(lo, hi) float32 (n, 3) of the fattened triangles in Morton order, as k_lbvh_keys, the radix sort and k_lbvh_leaves make them."""
    v0 = p[tri[:, 0]].astype(F); e1 = (p[tri[:, 1]] - p[tri[:, 0]]).astype(F); e2 = (p[tri[:, 2]] - p[tri[:, 0]]).astype(F)
    lo_m, hi_m = p[tri].reshape(-1, 3).min(0).astype(F), p[tri].reshape(-1, 3).max(0).astype(F)
    minv = np.where(hi_m > lo_m, F(1023.999) / np.where(hi_m > lo_m, hi_m - lo_m, F(1)), F(0)).astype(F)
    c = v0 + (e1 + e2) * F(1.0 / 3.0)
    q = np.minimum(np.maximum((c - lo_m) * minv, F(0)), F(1023)).astype(np.uint32)
    key = (_expand(q[:, 0]) << 2) | (_expand(q[:, 1]) << 1) | _expand(q[:, 2])
    order = np.argsort(key, kind="stable")                   # cub's radix sort is stable: equal codes stay in triangle order
    ext = float(max(np.abs(lo_m).max(), np.abs(hi_m).max()))
    slack = F(ext * 4e-6 + 1e-6)
    uv = np.array([[-BAND, -BAND], [F(1) + F(2) * BAND, -BAND], [-BAND, F(1) + F(2) * BAND]], F)
    corners = v0[:, None, :] + uv[None, :, 0:1] * e1[:, None, :] + uv[None, :, 1:2] * e2[:, None, :]
    lo, hi = corners.min(1), corners.max(1)
    pad = slack + F(2e-6) * np.maximum(np.abs(lo), np.abs(hi))
    return (lo - pad)[order], (hi + pad)[order]


def tie_key_symmetric(i, j):
    """plocTieKey: the same aligned pair first, then the nearer position, then the lower one - the same from either end."""
    return (((i >> 1) != (j >> 1)).astype(np.uint64) << np.uint64(63)) | (np.abs(i - j).astype(np.uint64) << np.uint64(32)) | np.minimum(i, j).astype(np.uint64)


def tie_key_lower(i, j):
    """The rule before the symmetric key: ties go to the lower position j."""
    return j.astype(np.uint64)


def nearest(lo, hi, tie_key):
    n = len(lo)
    i = np.arange(n)
    best = np.full(n, F(3e38)); bj = np.full(n, -1); bkey = np.full(n, np.iinfo(np.uint64).max, np.uint64)
    for off in range(-RADIUS, RADIUS + 1):
        if off == 0:
            continue
        j = i + off
        ok = (j >= 0) & (j < n)
        jj = np.clip(j, 0, n - 1)
        d = np.maximum(hi, hi[jj]) - np.minimum(lo, lo[jj])
        a = d[:, 0] * d[:, 1] + d[:, 1] * d[:, 2] + d[:, 2] * d[:, 0]
        key = tie_key(i, jj)
        take = ok & ((a < best) | ((a == best) & (key < bkey)))
        best = np.where(take, a, best); bj = np.where(take, jj, bj); bkey = np.where(take, key, bkey)
    return bj


def merge_round(lo, hi, tie_key):
    """One k_ploc_nearest + k_ploc_merge + compaction: mutual pairs become one cluster at the lower position."""
    nb = nearest(lo, hi, tie_key)
    i = np.arange(len(lo))
    mutual = (nb >= 0) & (nb[np.maximum(nb, 0)] == i)
    first = mutual & (i < nb)
    lo, hi = lo.copy(), hi.copy()
    lo[first] = np.minimum(lo[first], lo[nb[first]]); hi[first] = np.maximum(hi[first], hi[nb[first]])
    keep = ~mutual | first
    return lo[keep], hi[keep]


def rounds_to(p, tri, target, tie_key, cap):
    """Merge rounds until at most `target` clusters remain (1: the root); None when `cap` rounds do not get there."""
    lo, hi = leaf_boxes(p, tri)
    for r in range(1, cap + 1):
        m = len(lo)
        lo, hi = merge_round(lo, hi, tie_key)
        assert len(lo) < m, "a round merged nothing"
        if len(lo) <= target:
            return r
    return None


MESHES = {
    "plane 96 x 96": lambda: plane_mesh(96),
    "tube 16 x 2000": lambda: tube_mesh(16, 2000),
    "ribbon 1 x 6000": lambda: ribbon_mesh(6000),
    "ribbon 1 x 20000": lambda: ribbon_mesh(20_000),
    "12000 coincident": lambda: coincident_mesh(12_000),
    "zero-area mix": lambda: degenerate_mix_mesh(),
}


@pytest.mark.parametrize("name", list(MESHES))
def test_rounds_to_top(name):
    """At most 16 rounds down to the kPlocTop clusters the host's SAH top takes over."""
    p, tri = MESHES[name]()
    if len(tri) <= TOP:
        pytest.fail(f"{name}: {len(tri)} triangles do not reach PLOC")
    r = rounds_to(p, tri, TOP, tie_key_symmetric, 16)
    assert r is not None, f"{name}: more than 16 rounds to {TOP} clusters"


@pytest.mark.parametrize("name", ["ribbon 1 x 20000", "12000 coincident"])
def test_rounds_to_root(name):
    """PTAP_PLOC_TOP=0, PLOC up to the root: a few rounds per halving, far from the 4096-round guard."""
    p, tri = MESHES[name]()
    assert rounds_to(p, tri, 1, tie_key_symmetric, 128) is not None


@pytest.mark.parametrize("name", ["ribbon 1 x 20000", "12000 coincident"])
def test_lower_position_rule_stalls(name):
    """The rule the symmetric key replaced does not get these meshes to kPlocTop in 64 rounds (it needs thousands, past the guard)."""
    p, tri = MESHES[name]()
    assert rounds_to(p, tri, TOP, tie_key_lower, 64) is None


def test_kernel_uses_the_symmetric_key():
    """k_ploc_nearest compares (area, plocTieKey) lexicographically, and plocTieKey is the key restated by tie_key_symmetric."""
    src = open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "pathtracerap_b200", "csrc", "bvh_device.cu")).read()
    key = re.search(r"plocTieKey\(int i, int j\)\s*\{\s*return ([^;]*);", src)
    assert key, "plocTieKey not found"
    assert re.sub(r"\s+", "", key.group(1)) == ("((unsignedlonglong)((i>>1)!=(j>>1))<<63)|((unsignedlonglong)abs(i-j)<<32)|(unsigned)min(i,j)")
    body = src[src.index("__global__ void k_ploc_nearest"):]
    body = body[:body.index("nearest[i] = bj;")]
    assert "plocTieKey(i, j)" in body and "a < best || (a == best && key < bkey)" in body
