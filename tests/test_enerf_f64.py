"""oracle/enerf_f64.py (the float64 restatement of the ENeRF cascade: K1 cost volumes, a3 depth hypotheses, K2 depth
regression) against the golden vectors of the UNMODIFIED reference (tests/golden/enerf_ops.npz), on the CPU.

The golden outputs are float32, so the bar is float32 accuracy: |f64 - golden| <= 1e-5 * (max |golden| + |golden|) per
element, as in tests/test_mvsnerf_f64.py."""
import numpy as np
import torch

from conftest import load_golden
from oracle import enerf_f64 as E

RTOL = 1e-5
TRIPLE = [0, 1, 2]


def close(a, b, what, rtol=RTOL):
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    b = np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    err = np.abs(a - b)
    bad = err > rtol * (np.abs(b).max() + np.abs(b))
    assert not bad.any(), f"{what}: {int(bad.sum())}/{a.size} outside {rtol:g}; max abs err {err.max():.3e}"


def test_cost_volumes_restate_the_reference():
    g = load_golden("enerf_ops.npz")
    for lvl in (0, 1):
        planes = g.t(f"planes_l{lvl}")[0]
        r = E.cost_volume_var(g.t(f"in_feat{lvl}")[0], TRIPLE, g.t(f"proj_mats_l{lvl}")[0], planes)
        assert r["var"].dtype == torch.float64
        close(r["var"], g.np(f"volume_l{lvl}")[0], f"volume l{lvl}")
        if lvl == 0:
            close(r["feat"][1], g.np("warped_l0_view1")[0], "warped view 1, l0")
            # shared (D,) planes and row / plane subsets are slices of the full volume
            rows, pidx = [0, 3, 7], [0, 1, 31, 63]
            sub = E.cost_volume_var(g.t("in_feat0")[0], TRIPLE, g.t("proj_mats_l0")[0], planes[:, 0, 0], rows=rows,
                                    plane_idx=pidx, hw=planes.shape[1:])
            assert torch.equal(sub["var"], r["var"][:, pidx][:, :, rows])
            assert torch.equal(sub["coord"], r["coord"][:, pidx][:, :, rows])
    # the golden views are in front of every camera: no voxel at the 1e-6 clamp
    assert float(r["cz"].min()) > 0.1


def test_depth_hypotheses_restate_the_reference():
    g = load_golden("enerf_ops.npz")
    f = E.depth_planes_first(g.t("in_near_far")[0], 64, True)
    close(f["planes"], g.np("planes_l0")[0, :, 0, 0], "planes l0")
    close(f["nf"][:, None, None].expand(2, 8, 12), g.np("near_far_l0")[0], "near_far l0")
    n = E.depth_planes_next(g.t("depth_l0"), g.t("std_l0"), g.t("near_far_l0"), 8, 32, 48, False)
    close(n["planes"], g.np("planes_l1"), "planes l1")
    close(n["nf"], g.np("near_far_l1"), "near_far l1")
    # shared near / far (2,h0,w0) is the same as the per-chain form
    n2 = E.depth_planes_next(g.t("depth_l0"), g.t("std_l0"), g.t("near_far_l0")[0], 8, 32, 48, False)
    assert torch.equal(n2["planes"], n["planes"])
    # the upsample reproduces its source on the coincident grid points (x4 - 1 = 3 * (w0 - 1) / (w - 1) steps)
    up = n["up_depth"][0][0]
    assert torch.allclose(up[0, 0], g.t("depth_l0")[0, 0, 0].double()) and torch.allclose(up[-1, -1], g.t("depth_l0")[0, -1, -1].double())


def test_depth_regression_restates_the_reference():
    g = load_golden("enerf_ops.npz")
    for lvl, inv in ((0, True), (1, False)):
        r = E.depth_regression(g.t(f"in_logits{lvl}"), g.t(f"planes_l{lvl}"), inv)
        close(r["depth"], g.np(f"depth_l{lvl}"), f"depth l{lvl}")
        close(r["std"], g.np(f"std_l{lvl}"), f"std l{lvl}")
        assert (r["p_max"] <= 1).all() and (r["p_max"] >= 1.0 / r["prob"].shape[1] - 1e-12).all()
        assert torch.allclose(r["prob"].sum(1), torch.ones_like(r["depth"]))
