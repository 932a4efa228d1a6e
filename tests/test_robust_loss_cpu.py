"""Host side of the robust losses: graphs.add_outliers and the Python constants (no GPU needed)."""
import numpy as np


def test_add_outliers_is_seeded_and_leaves_the_rest_alone():
    from slam_plus_plus_b200 import graphs
    g = graphs.ba_shape("small")
    z0 = g.z.copy()
    a, ia = graphs.add_outliers(g, 0.05, 3)
    b, ib = graphs.add_outliers(g, 0.05, 3)
    c, ic = graphs.add_outliers(g, 0.05, 4)
    assert np.array_equal(g.z, z0)  # the input graph is not modified
    assert np.array_equal(ia, ib) and np.array_equal(a.z, b.z) and not np.array_equal(ia, ic)
    assert len(ia) == round(0.05 * g.n_obs) and np.all(np.diff(ia) > 0)
    keep = np.ones(g.n_obs, bool)
    keep[ia] = False
    assert np.array_equal(a.z[keep], g.z[keep]) and np.all(a.z[ia] != g.z[ia])
    assert a.z[ia].min() >= 0.0 and a.z[ia].max() < 800.0
    for x, y in ((a.vtype, g.vtype), (a.cams, g.cams), (a.pts, g.pts), (a.obs_pt, g.obs_pt), (a.obs_cam, g.obs_cam),
                 (a.info, g.info)):
        assert np.array_equal(x, y)


def test_loss_constants_match_the_header():
    import os
    import re
    from slam_plus_plus_b200 import capi
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, "include", "spp_b200.h")) as f:
        h = f.read()
    for name in ("NONE", "HUBER", "CAUCHY"):
        m = re.search(r"#define SPP_LOSS_%s (\d+)" % name, h)
        assert m and int(m.group(1)) == getattr(capi, "LOSS_" + name)
    assert "spp_ba_set_robust_loss" in capi.EXPORTED_SYMBOLS and "spp_ba_get_observation_errors" in capi.EXPORTED_SYMBOLS
