"""The one place where every VertexAlign entry point checks its inputs (functional.check_align_inputs / align_tables):
the host checks on shapes and counts (CPU), and on the device that each entry point raises before any kernel reads past
a map and that Cubify's per-vertex mesh ids are reused only for Cubify's own vertex counts."""
import pytest
import torch

from meshrcnn_b200.functional import check_align_inputs

SHP = [(2, 8, 12, 12), (2, 16, 6, 6)]
SIZES = [(224, 224)] * 2


def test_host_check_accepts_consistent_inputs():
    check_align_inputs(SHP, (50, 3), [20, 30], SIZES, [1, 1])
    check_align_inputs(SHP, (50, 3), [20, 10, 20], SIZES, [2, 1])            # several meshes per image (eval)
    check_align_inputs(SHP, (30, 3), [10, 20], SIZES + [(224, 224)], [1, 1, 0])   # an image beyond the maps without a mesh
    check_align_inputs(SHP, (0, 3), [0, 0], SIZES, [1, 1])


@pytest.mark.parametrize("case", [
    dict(shapes=SHP, pos=(50, 3), vpm=[20, 20, 10], sizes=SIZES + [(224, 224)], mi=[1, 1, 1]),    # image 2 has a mesh
    dict(shapes=[(2, 8, 12, 12), (1, 16, 6, 6)], pos=(50, 3), vpm=[20, 30], sizes=SIZES, mi=[1, 1]),   # one short map
    dict(shapes=SHP, pos=(50, 3), vpm=[60, -10], sizes=SIZES, mi=[1, 1]),       # negative vertex count
    dict(shapes=SHP, pos=(50, 3), vpm=[20, 30], sizes=SIZES, mi=[3, -1]),       # negative mesh count
    dict(shapes=SHP, pos=(50, 3), vpm=[20, 20], sizes=SIZES, mi=[1, 1]),        # vertex counts do not sum to SV
    dict(shapes=SHP, pos=(50, 3), vpm=[20, 30], sizes=SIZES, mi=[1, 2]),        # mesh counts do not sum to the meshes
    dict(shapes=SHP, pos=(50, 3), vpm=[20, 30], sizes=SIZES, mi=[2]),           # mesh_index and image_sizes differ
    dict(shapes=[(2, 8, 12, 10)], pos=(50, 3), vpm=[20, 30], sizes=SIZES, mi=[1, 1]),    # non-square map
    dict(shapes=[(2, 8, 12)], pos=(50, 3), vpm=[20, 30], sizes=SIZES, mi=[1, 1]),        # 3-D map
    dict(shapes=SHP, pos=(50, 2), vpm=[20, 30], sizes=SIZES, mi=[1, 1]),        # positions not SV x 3
])
def test_host_check_rejects(case):
    with pytest.raises(RuntimeError):
        check_align_inputs(case["shapes"], case["pos"], case["vpm"], case["sizes"], case["mi"])


def _entry_points(F_):
    w = torch.randn(8, 16, device="cuda")
    return {
        "vert_align": lambda f, p, v, s, m: F_.vert_align(f, p, v, s, m),
        "vert_align_bilinear": lambda f, p, v, s, m: F_.vert_align_bilinear(f, p, v, s, m),
        "vert_align_linear": lambda f, p, v, s, m: F_.vert_align_linear(f, p, v, s, m, w),
        "vert_align_linear_bilinear": lambda f, p, v, s, m: F_.vert_align_linear(f, p, v, s, m, w, bilinear=True),
        "TexelTerm": lambda f, p, v, s, m: F_.TexelTerm(f[0], p, v, s, m),
    }


@pytest.mark.gpu
def test_every_entry_point_rejects_a_mesh_on_an_image_past_the_maps(lib):
    from meshrcnn_b200 import functional as F_, synthetic
    fm = synthetic.feature_maps(2, [(16, 12, 12)], 1)[0].cuda()
    pos = synthetic.in_frustum_positions(50, 224, 2).cuda()
    for name, fn in _entry_points(F_).items():
        fn([fm], pos, [20, 30], SIZES, [1, 1])                                  # in range: accepted
        with pytest.raises(RuntimeError, match="image 2 holds a mesh"):
            fn([fm], pos, [20, 20, 10], SIZES + [(224, 224)], [1, 1, 1])
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_cubify_mesh_ids_are_reused_only_for_cubify_vertex_counts(lib, monkeypatch):
    from meshrcnn_b200 import _lib, functional as F_, synthetic
    from meshrcnn_b200.layers import Cubify
    verts, v_index, _, _, adj = Cubify(0.2)(synthetic.blob_voxels(2, 10, 3).cuda())
    SV = verts.shape[0]
    topo = F_.lookup(adj, SV)
    assert topo is not None and topo.v_index == v_index and len(v_index) == 2
    fm = synthetic.feature_maps(2, [(16, 12, 12)], 4)[0].cuda()
    pos = synthetic.in_frustum_positions(SV, 224, 5).cuda()
    called = []
    real = _lib.call
    monkeypatch.setattr(_lib, "call", lambda name, *a: (called.append(name), real(name, *a))[1])

    F_.vert_align([fm], pos, v_index, SIZES, [1, 1], topo=topo)
    assert "mrb_segment_ids" not in called
    # the same vertex total as one mesh per image 0, two meshes there: another mesh list, so the ids are rebuilt
    for vpm, mi in (([SV], [1, 0]), ([v_index[0] - 1, v_index[1] + 1], [1, 1]), ([v_index[0], 0, v_index[1]], [2, 1])):
        called.clear()
        got = F_.vert_align([fm], pos, vpm, SIZES, mi, topo=topo)
        assert "mrb_segment_ids" in called
        assert torch.equal(got, F_.vert_align([fm], pos, vpm, SIZES, mi))
        called.clear()
        tex = F_.TexelTerm(fm, pos, vpm, SIZES, mi, topo=topo)
        assert "mrb_segment_ids" in called
        assert torch.equal(tex.texrow, F_.TexelTerm(fm, pos, vpm, SIZES, mi).texrow)
