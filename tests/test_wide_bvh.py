"""The device walks a 4-wide collapse of the reference's binary BVH (include/tcpt_flat.h).  CPU-side gates of that layout:

1. every reference LEAF survives the collapse with its box bits, its item order and its place in the DFS order (so the tie-break
   key "later leaf first, earlier item first" of scene/src/bvh.rs:384-388,413-420 is still readable from the slots);
2. containment, numerically: with the reference's own slab arithmetic (math/src/bounds.rs:27-55, numpy float32, the NaN rules
   of its compare-selects included) a ray that passes a leaf box passes every ancestor box, so "leaves whose own box passes" is
   exactly the set of leaves the reference's recursive traversal reaches -- whatever inner boxes a wide node skips;
3. the worst-case stack height the host reports bounds a simulated walk that pushes every sibling.
The bit-exact hit tests on the GPU (tests/test_gpu_parity.py) are the gate of the device code itself."""
import numpy as np
import pytest
from bvh_checks import LEAF, NONE, check_collapse, slab_reference


@pytest.mark.parametrize("scene_id", [1, 3, 7, 17, 19])
def test_every_reference_leaf_survives_the_collapse(bundle_factory, scene_id):
    b = bundle_factory(scene_id, 64, 48, require_gpu=False)
    check_collapse(b.scene, -1)
    used = {p[1] for p in b.scene.desc.primitives if p[0] == "geom"}
    assert used
    for g in used:
        check_collapse(b.scene, g, len(b.scene.desc.meshes[g].indices))


def test_big_leaves_are_cut_into_ranges_under_the_leaf_box(tables):
    """40 identical triangles: the reference builder cannot split them (every split costs more than the leaf), so the BLAS is one
    leaf of 40 items -> a wide record of three ranges (13 + 13 + 14) that all carry the leaf's box."""
    import toy_cpu_pathtracing_b200 as tp
    from toy_cpu_pathtracing_b200 import scene as S
    from toy_cpu_pathtracing_b200.assets import MeshData
    s = tp.Scene(device=0, require_gpu=False)
    cam = tp.Camera(45.0, 32, 32)
    cam.set_look_to([0, 0, 3], [0, 0, -1], [0, 1, 0])
    pos = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0]], np.float32)
    nrm = np.tile(np.array([[0, 0, 1]], np.float32), (3, 1))
    idx = np.tile(np.array([[0, 1, 2]], np.uint32), (40, 1))
    g = s.load_obj(MeshData(pos, nrm, None, idx))
    s.create_primitive(S.GeometryPrimitive(g, S.LambertMaterial.new(S.SpectrumParameter.constant(S.ConstantSpectrum(0.5)), S.NormalParameter.none())))
    lg = s.load_obj(MeshData(pos + 2, nrm, None, idx[:1]))
    s.create_primitive(S.GeometryPrimitive(lg, S.EmissiveMaterial.new(S.SpectrumParameter.constant(S.presets.cie_illum_d6500()), S.FloatParameter.constant(1.0))))
    s.build(cam)
    ref, rec, first = check_collapse(s, g, 40)
    assert ref[0, 0] == 1 and ref[0, 1] == 40
    assert len(rec) == 2 and [int(rec[1, 7, k]) for k in range(4)] == [13, 13, 14, 0]


@pytest.mark.parametrize("scene_id,which", [(3, -1), (3, 0), (19, -1), (19, 1), (17, 0)])
def test_a_ray_that_passes_a_leaf_box_passes_every_ancestor(bundle_factory, scene_id, which):
    b = bundle_factory(scene_id, 64, 48, require_gpu=False)
    ref = b.scene.get_bvh(which)
    nodes = [i for i in range(len(ref)) if ref[i, 0] != 2]
    boxes = ref[nodes][:, 2:8].view(np.float32)
    # parent of every node of the reference's flattened pre-order (bvh.rs:234-295)
    parent = {}
    for i in nodes:
        if ref[i, 0] == 0:
            parent[i + 1] = i
            parent[i + int(ref[i, 1])] = i
    order = {n: k for k, n in enumerate(nodes)}
    rng = np.random.default_rng(5)
    lo_all, hi_all = boxes[:, :3].min(0), boxes[:, 3:].max(0)
    n = 3000
    o = rng.uniform(lo_all - 0.5, hi_all + 0.5, (n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3)).astype(np.float32)
    # a third of the rays are axis-parallel (infinite reciprocals) and start ON box planes: the NaN cases of 0 * inf
    k = n // 3
    d[:k, rng.integers(0, 3)] = 0.0
    d[k // 2:k, rng.integers(0, 3)] = -0.0
    pick = boxes[rng.integers(0, len(boxes), k)]
    o[:k] = np.where(rng.random((k, 3)) < 0.5, pick[:, :3], pick[:, 3:])
    d /= np.maximum(np.linalg.norm(d, axis=1, keepdims=True), 1e-20).astype(np.float32)
    with np.errstate(divide="ignore"):
        inv = (np.float32(1.0) / d).astype(np.float32)
    t_max = np.float32(np.finfo(np.float32).max)
    passes = slab_reference(boxes[:, None, :3], boxes[:, None, 3:], o[None], inv[None], t_max)   # [node, ray]
    reach = passes.copy()
    for i in nodes:           # pre-order: a parent comes before its children
        if i in parent:
            reach[order[i]] &= reach[order[parent[i]]]
    leaves = [order[i] for i in nodes if ref[i, 0] == 1]
    assert passes[leaves].any() and not passes[leaves].all()
    assert np.array_equal(passes[leaves], reach[leaves]), "a leaf box passed while an ancestor box failed"


def test_reported_stack_bound_covers_the_worst_walk(bundle_factory):
    """max_bvh_depth (tcpt_stats / tcpt_flat_scene) = siblings waiting along the deepest TLAS path + 1 + the same in the deepest BLAS."""
    for scene_id in (3, 17, 19):
        b = bundle_factory(scene_id, 64, 48, require_gpu=False)

        def worst(rec, first, r=0):
            kids = [int(e) for e in rec[r, 6] if int(e) != NONE]
            deepest = 0
            for e in kids:
                if not e & LEAF:
                    deepest = max(deepest, worst(rec, first, e - first))
            return deepest + len(kids) - 1

        rec, first, _ = b.scene.get_wide_bvh(-1)
        total = worst(rec, first) + 1
        deepest = 0
        for g in {p[1] for p in b.scene.desc.primitives if p[0] == "geom"}:
            rec, first, _ = b.scene.get_wide_bvh(g)
            deepest = max(deepest, worst(rec, first))
        assert b.scene.ctx.stats()["max_bvh_depth"] == total + deepest < 96
