"""Helpers shared by the BVH tests (tests/test_wide_bvh.py, tests/test_soup_traversal.py): reading the reference-order dump of
tcpt_get_bvh and the 4-wide records of tcpt_get_wide_bvh, and the reference's slab test restated in numpy float32."""
import numpy as np

LEAF, NONE, SLOT = 0x80000000, 0xFFFFFFFF, 0x07FFFFFF


def reference_leaves(ref):
    """(box bits [6], items) of every leaf of a tcpt_get_bvh dump, in DFS order; plus parent links of the flattened tree."""
    leaves, i = [], 0
    while i < len(ref):
        kind, value = int(ref[i, 0]), int(ref[i, 1])
        if kind == 1:
            leaves.append((ref[i, 2:8].copy(), [int(ref[i + 1 + k, 1]) for k in range(value)]))
            i += 1 + value
        else:
            i += 1
    return leaves


def wide_leaves(rec, first, root=0):
    """Leaf ranges of the wide layout in DFS order: (box bits [6], first slot, count)."""
    out = []

    def walk(r):
        for k in range(4):
            e = int(rec[r, 6, k])
            if e == NONE:
                assert np.isposinf(rec[r, 0, k].view(np.float32)) and np.isneginf(rec[r, 1, k].view(np.float32))
                continue
            box = rec[r, [0, 2, 4, 1, 3, 5], k]            # lo.xyz, hi.xyz like the reference dump
            if e & LEAF:
                cnt = ((e >> 27) & 15) + 1
                assert int(rec[r, 7, k]) == cnt
                out.append((box.copy(), e & SLOT, cnt))
            else:
                assert first <= e < first + len(rec) and int(rec[r, 7, k]) == 0
                walk(e - first)

    walk(root)
    return out


def check_collapse(scene, which, n_expected_items=None):
    ref = scene.get_bvh(which)
    rec, first, sbase = scene.get_wide_bvh(which)
    rl, wl = reference_leaves(ref), wide_leaves(rec, first)
    slot, j = sbase, 0
    for box, items in rl:                      # a reference leaf = one or more consecutive ranges (cut at 16 items) under the same box
        left = len(items)
        while left:
            wbox, wslot, wcnt = wl[j]; j += 1
            assert np.array_equal(wbox, box), "leaf box bits changed"
            assert wslot == slot and wcnt <= min(left, 16)
            slot += wcnt; left -= wcnt
    assert j == len(wl)
    if n_expected_items is not None:
        assert slot - sbase == n_expected_items
    return ref, rec, first


def slab_reference(lo, hi, o, inv_d, t_max):
    """Bounds::intersect in numpy float32, the reference's compare-selects spelled out (NaN comparisons are False).  Boxes, rays and
    t_max (a scalar or one value per ray) broadcast against each other."""
    shape = np.broadcast_shapes(lo.shape[:-1], o.shape[:-1], np.shape(t_max))
    t0 = np.zeros(shape, np.float32)
    t1 = np.broadcast_to(np.asarray(t_max, np.float32), shape).copy()
    with np.errstate(invalid="ignore", over="ignore"):
        for a in range(3):
            tn = (lo[..., a] - o[..., a]) * inv_d[..., a]
            tf = (hi[..., a] - o[..., a]) * inv_d[..., a]
            sw = tn > tf
            tn, tf = np.where(sw, tf, tn), np.where(sw, tn, tf)
            t0 = np.where(tn > t0, tn, t0)
            t1 = np.where(tf < t1, tf, t1)
        return ~(t0 > t1)
