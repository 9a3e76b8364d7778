"""Parity of the kernels either side of the solve: Euler <-> R, projection, the synthetic
workload generator, error reporting, classification and the two-pass statistics."""
import os

import numpy as np
import pytest
import torch

from conftest import load_golden
from gpu_util import dev, to_np
from oracle import oracle as orc
from pnp_solver_test_b200 import patterns as pt

pytestmark = pytest.mark.gpu


def test_euler_kernels_match_reference_fixture_and_oracle():
    import pnp_solver_test_b200 as pnp
    g = load_golden("euler_fixture")
    R = pnp.R_from_euler_batch(dev(g["roll_yaw_pitch_deg"]), is_degree=True).cpu().numpy()
    assert np.abs(R - g["R"]).max() < 1e-12                         # the reference's own fixture
    e = pnp.euler_from_R_batch(dev(g["R"]), is_degree=True).cpu().numpy()
    assert np.abs(e - g["roll_yaw_pitch_deg"]).max() < 1e-9
    rng = np.random.default_rng(0)
    ang = rng.uniform(-3.0, 3.0, (5000, 3))
    R = pnp.R_from_euler_batch(dev(ang), is_degree=False).cpu().numpy()
    Ro = np.array([orc.R_from_euler(*a, is_degree=False) for a in ang])
    assert np.abs(R - Ro).max() < 1e-14
    e = pnp.euler_from_R_batch(dev(Ro), is_degree=False).cpu().numpy()
    eo = np.array([orc.euler_from_R(r, False) for r in Ro])
    assert np.abs(e - eo).max() < 1e-12
    # gimbal-lock branch (PNP_SOLVER_LIB.py:4482)
    Rg = np.array([orc.R_from_euler(0.3, 0.0, np.pi / 2, False), orc.R_from_euler(-1.0, 0.0, -np.pi / 2, False)])
    eg = pnp.euler_from_R_batch(dev(Rg), False).cpu().numpy()
    assert np.abs(eg - np.array([orc.euler_from_R(r, False) for r in Rg])).max() < 1e-12
    f32 = pnp.euler_from_R_batch(dev(Ro, torch.float32), False).cpu().numpy()
    assert np.median(np.abs(f32 - eo)) < 1e-5


def test_projection_matches_oracle_including_rounding():
    import pnp_solver_test_b200 as pnp
    P = pt.pattern_array(pt.synthetic_pattern(68))
    K = pt.default_camera_matrix()
    w = orc.synth(0, 512, P, K)
    for quant, q in ((False, 1.0), (True, 1.0), (True, 30.0 / 112.0)):
        got = pnp.project_batch(dev(P), K, dev(w["R_gt"]), dev(w["t_gt"]), quant, q).cpu().numpy()
        ref = np.array([orc.project(P, K, w["R_gt"][b], w["t_gt"][b], quant, q) for b in range(512)])
        if quant:
            assert (np.abs(got - ref) > 1e-9).mean() < 1e-4         # a tie may round the other way
        else:
            assert np.abs(got - ref).max() < 1e-10
    # behind the camera: divide by |z| (PNP_SOLVER_LIB.py:4548) -> homogeneous coordinate -1
    t_neg = w["t_gt"].copy(); t_neg[:, 2] *= -1
    got = pnp.project_batch(dev(P), K, dev(w["R_gt"]), dev(t_neg), False, 1.0).cpu().numpy()
    assert np.allclose(got[..., 2], -1.0)


def test_synthetic_workload_matches_oracle_and_is_shard_invariant():
    import pnp_solver_test_b200 as pnp
    from pnp_solver_test_b200 import workload as wl
    P = pt.pattern_array(pt.synthetic_pattern(68))
    K = pt.default_camera_matrix()
    for cfg_kw in (dict(is_quantized=0), dict(is_quantized=1), dict(is_quantized=0, noise_sigma_px=1.5),
                   dict(is_quantized=1, quantize_q=30.0 / 112.0, noise_sigma_px=0.5),
                   dict(is_quantized=1, quantize_q=30.0 / 112.0, noise_sigma_px=0.4, angle_range_deg=0.0, yaw_center_deg=38.5,
                        depth_min_m=1.0, depth_max_m=1.0, fov_max_deg=0.0)):      # LM_noise_test.py's fixed pose
        ref = orc.synth(5, 4000, P, K, orc.default_synth(seed=9, **{k: v for k, v in cfg_kw.items()}))
        got = wl.synth_batch(5, 4000, P, K, cfg=pnp.default_synth(seed=9, **cfg_kw), want_pose=True)
        assert np.abs(got["gt"].cpu().numpy() - ref["gt"]).max() < 1e-12
        assert np.abs(got["R_gt"].cpu().numpy() - ref["R_gt"]).max() < 1e-14
        d = np.abs(got["uv"].cpu().numpy() - ref["uv"])
        assert (d > 1e-8).mean() < 1e-4, (cfg_kw, d.max())
    full = wl.synth_batch(0, 3000, P, K)["uv"]
    parts = torch.cat([wl.synth_batch(0, 1000, P, K)["uv"], wl.synth_batch(1000, 2000, P, K)["uv"]])
    assert torch.equal(full, parts)
    f32 = wl.synth_batch(0, 3000, P, K, dtype=torch.float32)["uv"]
    assert torch.equal(f32.double(), full)                          # integer pixels are exact in FP32


def test_report_classification_and_statistics_match_reference():
    from pnp_solver_test_b200 import workload as wl
    g = load_golden("stress_report")
    rep = wl.report_batch(g["pattern"], dev(g["uv"]), g["K"], dev(g["R"]), dev(g["t"]), dev(g["euler"]), dev(g["gt"]))
    assert np.abs(rep["report"].cpu().numpy() - g["report"]).max() < 1e-10
    assert rep["report"][:, 3].is_contiguous() and rep["report"].shape == (g["uv"].shape[0], 16)     # column layout
    rows = wl.report_batch(g["pattern"], dev(g["uv"]), g["K"], dev(g["R"]), dev(g["t"]), dev(g["euler"]), dev(g["gt"]), layout="rows")
    assert rows["report"].is_contiguous() and torch.equal(rows["report"], rep["report"])
    assert torch.equal(rows["flags"], rep["flags"]) and torch.equal(rows["max_idx"], rep["max_idx"])
    one = wl.report_batch(g["pattern"], dev(g["uv"][:1]), g["K"], dev(g["R"][:1]), dev(g["t"][:1]), dev(g["euler"][:1]), dev(g["gt"][:1]))
    assert torch.equal(one["report"], rep["report"][:1])
    assert np.array_equal(rep["flags"].cpu().numpy(), g["flags"])
    assert np.array_equal(rep["max_idx"].cpu().numpy(), g["max_idx"])
    cls = wl.classify(dev(g["gt"])[:, 0], wl.CLASS_BINS["depth"], scale=100.0)
    assert np.array_equal(cls.cpu().numpy(), g["depth_class"])
    st = wl.error_statistics(rep["report"], dev(g["gt"]), distributed=False)
    for q, name in enumerate(("depth", "roll", "pitch", "yaw")):
        np.testing.assert_allclose(st[name]["all"].numpy(), g["stats_all"][q], rtol=1e-11, atol=1e-13)
        ref = g["stats_by_depth"][q]
        has = ~np.isnan(ref[:, 0])
        np.testing.assert_allclose(st[name]["by_depth"].numpy()[has], ref[has], rtol=1e-11, atol=1e-13)


def test_report_on_cuda_solution_matches_oracle_report():
    import pnp_solver_test_b200 as pnp
    from pnp_solver_test_b200 import workload as wl
    pat15 = pt.get_golden_pattern()
    P, K = pt.pattern_array(pat15), pt.default_camera_matrix()
    w = orc.synth(0, 5000, P, K)
    idx = [list(pat15).index(k) for k in pt.LM_KEY_LIST_6]
    out = pnp.solve_batch("qeif", dev(w["uv"]), dev(P)[None], K, point_index=idx)
    rep = wl.report_batch(P, dev(w["uv"]), K, out["R"], out["t"], out["euler"], dev(w["gt"]))
    o = to_np(out)
    ref = orc.report_batch(P, w["uv"], K, o["R"], o["t"], o["euler"], w["gt"])
    assert np.abs(rep["report"].cpu().numpy() - ref["report"]).max() < 1e-9
    assert np.array_equal(rep["flags"].cpu().numpy(), ref["flags"])
    assert (rep["max_idx"].cpu().numpy() == ref["max_idx"]).mean() > 0.999
    assert ref["flags"].all(axis=1).mean() > 0.95


def test_report_warp_kernel_for_large_patterns():
    """n = 1024: the 32-row tile no longer fits, the one-warp-per-problem report kernel runs."""
    from pnp_solver_test_b200 import workload as wl
    P, K = pt.pattern_array(pt.synthetic_pattern(1024)), pt.default_camera_matrix()
    w = orc.synth(0, 200, P, K)
    s = orc.solve_batch("linear_f2", w["uv"], P, K)
    ref = orc.report_batch(P, w["uv"], K, s["R"], s["t"], s["euler"], w["gt"])
    rep = wl.report_batch(P, dev(w["uv"]), K, dev(s["R"]), dev(s["t"]), dev(s["euler"]), dev(w["gt"]))
    assert np.abs(rep["report"].cpu().numpy() - ref["report"]).max() < 1e-9
    assert np.array_equal(rep["flags"].cpu().numpy(), ref["flags"])
    assert (rep["max_idx"].cpu().numpy() == ref["max_idx"]).mean() > 0.99


@pytest.mark.parametrize("n_class,nq", [(1, 1), (13, 4), (64, 4), (40, 2)])
def test_statistics_kernels_both_paths_match_numpy(n_class, nq):
    """Lane-private tables (few classes) and the turn-taking kernel (tables too large for shared
    memory) against the NumPy restatement of get_statistic_of_result, ragged B, empty classes."""
    from pnp_solver_test_b200 import workload as wl
    rng = np.random.default_rng(n_class * 10 + nq)
    B = 70001
    est = rng.normal(1.0, 0.3, (B, nq)) + 3.0
    gt = rng.normal(1.0, 0.1, (B, nq)) + 3.0
    cls = rng.integers(0, n_class + 2, B).astype(np.int32) - 1          # -1 and n_class: outside every class
    cls[cls == 2] = 3 if n_class > 3 else cls[cls == 2]                 # leave class 2 empty when there is room
    d_est, d_gt = dev(est), dev(gt)
    st = wl.statistics([d_est[:, q] for q in range(nq)], [d_gt[:, q] for q in range(nq)],
                       torch.from_numpy(cls).cuda(), n_class, distributed=False).numpy()
    assert st.shape == (nq, n_class + 1, 7)
    for q in range(nq):
        for c in list(range(n_class)) + [-1]:
            sel = np.ones(B, bool) if c == -1 else (cls == c)
            row = st[q, c]
            if sel.sum() == 0:
                assert row[0] == 0
                continue
            ref = np.array(orc.stats_of(est[sel, q], gt[sel, q]), dtype=np.float64)
            assert row[0] == ref[0]
            assert np.abs(row[1:] - ref[1:]).max() < 1e-11 * max(1.0, np.abs(ref[1:]).max()), (q, c, row, ref)


def test_drpy_class_combination_statistics_match_reference(tmp_path):
    """classify_drpy + the many-class statistics kernels (1500 classes, global FP64 reductions)
    against the oracle on the reference's own result rows, the tables they produce against the
    reference's files, and a large synthetic batch against the oracle (ragged B, dense classes)."""
    from pnp_solver_test_b200 import workload as wl
    import pnp_solver_test_b200 as pnp
    g = load_golden("stress_report")
    bins = [wl.CLASS_BINS[q] for q in wl.DRPY_ORDER]
    rep, gt = dev(g["report"]), dev(g["gt"])
    cls = wl.classify_drpy(gt).cpu().numpy()
    ref_cls = np.ravel_multi_index([np.digitize(g["gt"][:, q] * (100.0 if q == 0 else 1.0), np.asarray(bins[q])) for q in range(4)],
                                   wl.drpy_shape())
    assert (cls == ref_cls).all()
    st = wl.drpy_statistics(rep, gt, distributed=False)
    ref = orc.drpy_stats(g["report"], g["gt"], bins)
    for k in ref:
        a = st[k].numpy()
        assert (a[..., 0] == ref[k][..., 0]).all()
        m = ref[k][..., 0] > 0
        assert np.abs(a[m] - ref[k][m]).max() < 1e-11 * max(1.0, np.abs(ref[k][m]).max()), k
    paths = wl.drpy_analysis_and_saving(rep, gt, str(tmp_path) + "/", "stat_", "data.txt", distributed=False)
    import csv, io
    for p in paths:
        key = "drpy_csv_" + os.path.basename(p)[len("stat_data_drpy_to_"):-4]
        mine = list(csv.reader(io.StringIO(open(p, newline="").read())))
        want = list(csv.reader(io.StringIO(str(g[key]))))
        assert len(mine) == len(want) and mine[0] == want[0], key
        for ra, rb in zip(mine, want):
            assert len(ra) == len(rb)
            for x, y in zip(ra, rb):
                try:
                    fy = float(y)
                except ValueError:
                    assert x == y, (key, x, y)
                    continue
                assert abs(float(x) - fy) <= 1e-9 * max(1.0, abs(fy)), (key, x, y)
    # dense classes: a synthetic batch, every combination hit many times
    B = 200003
    w = wl.synth_batch(0, B, g["pattern"], g["K"], cfg=pnp.default_synth(seed=5))
    rng = np.random.default_rng(3)
    gt_h = w["gt"].cpu().numpy()
    rep_h = np.zeros((B, 16))
    rep_h[:, 10] = gt_h[:, 0] * (1.0 + 0.01 * rng.normal(size=B)); rep_h[:, 11] = gt_h[:, 0]
    for q in range(3):
        rep_h[:, 12 + q] = gt_h[:, 1 + q] + rng.normal(size=B)
    rep_h[:, 4] = np.abs(rng.normal(size=B))
    st = wl.drpy_statistics(dev(rep_h), w["gt"], distributed=False)
    ref = orc.drpy_stats(rep_h, gt_h, bins)
    for k in ref:
        a = st[k].numpy()
        assert (a[..., 0] == ref[k][..., 0]).all() and a[..., 0].sum() == B
        m = ref[k][..., 0] > 0
        assert np.abs(a[m] - ref[k][m]).max() < 1e-10 * max(1.0, np.abs(ref[k][m]).max()), k


def test_face_variation_workload_and_fragility_analysis_match_reference():
    """face_variation_test.py: perturbed-pattern generator vs the oracle; device top-10 % selection,
    fragile-point counts and perturbation directions vs the script's own function (golden) and, on a
    larger batch with ties, vs its NumPy restatement."""
    from pnp_solver_test_b200 import workload as wl
    import pnp_solver_test_b200 as pnp
    g = load_golden("fragility")
    keys = [str(k) for k in g["keys"]]
    fixed = int(g["fixed_index"])
    w = wl.synth_face_variation(0, 600, g["pattern"], g["K"], fixed, 0.02, cfg=pnp.default_synth(seed=int(g["seed"])))
    assert np.abs(w["perturb"].cpu().numpy() - g["perturb"]).max() < 1e-15
    assert (np.abs(w["uv"].cpu().numpy() - g["uv"]) > 1e-8).mean() < 1e-3
    assert np.abs(w["gt"].cpu().numpy() - g["gt"]).max() < 1e-12
    err = dev(np.abs(g["err"]))
    res = wl.fragility_analysis([err[:, q] for q in range(4)], dev(g["perturb"]), keys=keys)
    for q, name in enumerate(("depth", "roll", "pitch", "yaw")):
        r = res[q]
        assert r["n_selected"] == 60
        assert np.array_equal(r["fragile_point_count"], g[name + "_count"])
        assert [k for _, k in r["fragile_point_sorted_list"]] == [str(k) for k in g[name + "_sorted_keys"]]
        assert np.abs(r["top_similarity"] - g[name + "_similarity"]).max() < 1e-12
        for i in range(5):
            d, ref = r["top_perturbation"][i], g[name + "_directions"][i]
            assert min(np.abs(d - ref).max(), np.abs(d + ref).max()) < 1e-8
        assert r["value_max"] == g[name + "_value_max"] and abs(r["top_value_mean"] - g[name + "_value_mean"]) < 1e-14
    # larger batch, 68 landmarks, quantised errors (many exact ties at the selection threshold), shard offset
    rng = np.random.default_rng(3)
    B, n = 50000, 68
    e = np.round(rng.gamma(2.0, 1.0, (B, 2)), 1)                    # ties by construction
    pert = rng.normal(size=(B, n, 3)) * rng.uniform(0.1, 1.0, (B, n, 1))
    res = wl.fragility_analysis([dev(e)[:, 0], dev(e)[:, 1]], dev(pert), idx0=0)
    kk = ["k%03d" % i for i in range(n)]
    for q in range(2):
        ref = orc.fragility_of(e[:, q], pert, kk)
        assert res[q]["n_selected"] == 5000
        assert np.array_equal(res[q]["fragile_point_count"], np.array([ref["fragile_point_count_dict"][k] for k in kk]))
        assert np.abs(res[q]["top_similarity"] / ref["top_similarity"] - 1).max() < 1e-10
        assert res[q]["value_max"] == ref["value_max"] and abs(res[q]["top_value_mean"] - ref["top_value_mean"]) < 1e-12


@pytest.mark.parametrize("method,n,dtype,subset", [("lm", 68, torch.float64, False), ("linear_f2", 68, torch.float64, False),
                                                 ("lm", 15, torch.float64, False), ("lm", 68, torch.float32, False),
                                                 ("lm_plus", 68, torch.float64, False), ("qeif", 15, torch.float64, True),
                                                 ("lm", 1024, torch.float64, False), ("eif2", 15, torch.float64, False),
                                                 ("lm", 68, torch.float64, "skew"), ("linear_f2", 68, torch.float64, "skew"),
                                                 ("lm", 68, torch.float32, "skew"), ("lm", 95, torch.float64, False),
                                                 ("linear_f2", 190, torch.float32, False)])
def test_fused_solve_report_equals_the_two_calls(method, n, dtype, subset):
    """pnpb200_solve_report_batch (the residual pass of the moment mapping folded into the report kernel, the pixel rows
    read twice instead of three times) returns what pnpb200_solve_batch followed by pnpb200_report_batch_strided return --
    bit for bit, for a ragged batch, for every method and shape (those that cannot fuse run the two calls inside).
    subset = "skew": all landmarks, K with a nonzero skew, so the fused kernel normalises the pixels with both FMAs
    (k_report_chunk<T, RES, SKEW = true>); n = 95 (FP64) and 190 (FP32) are the largest n that fuse."""
    import pnp_solver_test_b200 as pnp
    from pnp_solver_test_b200 import workload as wl
    pat = pt.get_golden_pattern() if n == 15 else pt.synthetic_pattern(n)
    P, K = pt.pattern_array(pat), pt.default_camera_matrix()
    B = 3 * 1024 + 45 if n < 1024 else 77
    _fused_case(method, n, dtype, subset, B)
    if n == 68 and dtype == torch.float64:
        for small in (1, 33):
            _fused_case(method, n, dtype, subset, small)


def _fused_case(method, n, dtype, subset, B):
    import pnp_solver_test_b200 as pnp
    from pnp_solver_test_b200 import workload as wl
    pat = pt.get_golden_pattern() if n == 15 else pt.synthetic_pattern(n)
    P, K = pt.pattern_array(pat), pt.default_camera_matrix()
    if subset == "skew":
        K = K.copy()
        K[0, 1] = 1.75
    w = wl.synth_batch(7, B, P, K, dtype=dtype)
    idx = [list(pat).index(k) for k in pt.LM_KEY_LIST_6] if subset is True else None
    patd = dev(P, dtype)[None]
    a = pnp.solve_batch(method, w["uv"], patd, K, point_index=idx)
    r = wl.report_batch(P, w["uv"], K, a["R"], a["t"], a["euler"], w["gt"])
    f = wl.solve_report_batch(method, w["uv"], patd, K, w["gt"], point_index=idx)
    torch.cuda.synchronize()
    bits = lambda x: x.contiguous().view(torch.int64 if x.element_size() == 8 else torch.int32)
    for k in ("R", "t", "euler", "res_norm", "iters"):
        assert torch.equal(bits(f[k]), bits(a[k])), k
    for k in ("report", "flags", "max_idx"):
        assert torch.equal(bits(f[k]), bits(r[k])), k
    # res_norm against the oracle where parity is well-posed (LM: first 512 problems)
    if dtype == torch.float64 and method in ("lm", "linear_f2") and n < 1024 and B >= 512:
        from gpu_util import oracle_stability
        uv = w["uv"][:512].cpu().numpy()
        ref, stable, _ = oracle_stability(method, uv, P, K)
        d = np.abs(f["res_norm"][:512].cpu().numpy() - ref["res_norm"])[stable] / ref["res_norm"][stable]
        assert d.max() < 1e-9
