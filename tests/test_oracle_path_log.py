"""The forward, one-vertex oracle (oracle_path_vertex, walked over whole frames by oracle_path_log) against the
recursive trace() of oracle_render_sum, on the CPU.

tests/test_gpu_wavefront_paths.py compares the wavefront kernels with this forward form vertex by vertex.  That is
only worth something if the forward form IS the pinned oracle: trace() is pinned to the reference by
test_oracle_vs_ref.py and test_golden.py.  Summed per pixel, the contributions of the log equal trace()'s sums up
to the association of the throughput products (a few units of 2^-53 per vertex: 1e-12 of the pixel's absolute
sum), and the ray counts are equal exactly.
"""
import numpy as np
import pytest


def _scenes(api):
    W, H = 40, 23
    verts = api.heightfield_mesh(12, 20 * W / H * 0.98)
    return {
        "c1": (api.scene_default(W, H), W, H),
        "dielectric-mirror-field": (api.scene_sphere_field(300, W, H, mix=(0.2, 0.4, 0.4)), W, H),
        "mesh-room": (api.mesh_room(verts, W, H), W, H),
    }


@pytest.mark.parametrize("scene", ["c1", "dielectric-mirror-field", "mesh-room"])
@pytest.mark.parametrize("dielectric", ["stochastic", "split"])
@pytest.mark.parametrize("max_depth", [0, 1, 5, 64])
def test_path_log_sums_to_trace(api, ol, scene, dielectric, max_depth):
    if dielectric == "split" and max_depth == 64:
        max_depth = 12  # 2^(depth+1) rays per path: the split tree is intractable at 64 (the renderer allows 16)
    objs, W, H = _scenes(api)[scene]
    cam = ol.init_camera(W, H)
    spp, first = 3, 5
    log = ol.path_log(objs, cam, W, H, spp, dielectric=dielectric, max_depth=max_depth, sample_offset=first)
    want, (rays, _) = ol.render_sum(objs, cam, W, H, spp, dielectric=dielectric, max_depth=max_depth,
                                    sample_offset=first)
    want = want.reshape(-1, 3)
    got = np.zeros_like(want)
    mag = np.zeros_like(want)
    np.add.at(got, log["pixel"], log["contrib"])
    np.add.at(mag, log["pixel"], np.abs(log["contrib"]))
    err = np.abs(got - want)
    bad = np.flatnonzero((err > 1e-12 * mag).any(axis=1))
    assert len(bad) == 0, f"pixels {bad[:5]}: log {got[bad[:3]]} vs trace {want[bad[:3]]}"
    assert int(log["rays"].sum()) == rays
    # the log is complete: every (pixel, sample) starts with one camera vertex, and every traced child is logged
    assert np.count_nonzero(log["depth"] == 0) == W * H * spp
    assert np.array_equal(np.unique(log["sample"]), np.arange(first, first + spp))
    traced_children = int((log["n_children"] - log["cut"].sum(axis=1)).sum())
    assert traced_children == len(log) - W * H * spp
    assert log["depth"].max() <= max_depth
