"""The solution check without ground truth (pnpb200_check_batch, pnpb200_solve_check_batch_host): its reprojection
distance is the error report's, its status bits are what their definitions say, and on the stress workload they
separate the failures of LM from its successes as include/pnpb200.h states."""
import numpy as np
import pytest
import torch

from oracle import oracle as orc
from pnp_solver_test_b200 import patterns as pt

from gpu_util import dev

pytestmark = pytest.mark.gpu

B_STRESS = 1 << 16
NONFINITE, DEPTH, BEHIND, REPROJ = 1, 2, 4, 8


def _solve(method, n, dtype=torch.float64, B=B_STRESS, seed=42, subset=False):
    """A seeded random_stress_test workload (quantised pixels) solved on the device; everything back as NumPy."""
    import pnp_solver_test_b200 as pnp
    from pnp_solver_test_b200 import workload as wl
    pat = pt.get_golden_pattern() if n == 15 else pt.synthetic_pattern(n)
    P, K = pt.pattern_array(pat), pt.default_camera_matrix()
    w = wl.synth_batch(0, B, P, K, cfg=pnp.default_synth(seed=seed), dtype=dtype)
    Pd = dev(P, dtype)
    idx = [list(pat).index(k) for k in pt.LM_KEY_LIST_6] if subset else None
    out = pnp.solve_batch(method, w["uv"], Pd[None], K, point_index=idx)
    return dict(P=P, Pd=Pd, K=K, uv=w["uv"], gt=w["gt"], out=out)


@pytest.fixture(scope="module")
def lm68():
    return _solve("lm", 68)


def _np(x):
    return x.detach().double().cpu().numpy() if x.is_floating_point() else x.detach().cpu().numpy()


def _check(s, limit=1.0, with_res=True):
    import pnp_solver_test_b200 as pnp
    o = s["out"]
    c = pnp.check_batch(s["uv"], s["Pd"], s["K"], o["R"], o["t"], res_norm=o["res_norm"] if with_res else None,
                        reproj_limit_px=limit)
    torch.cuda.synchronize()
    return _np(c["status"]), _np(c["reproj"])


def _report(s, unit_distance):
    from pnp_solver_test_b200 import workload as wl
    gt = s["gt"].clone()
    if unit_distance:
        gt[:, 0] = 1.0
    o = s["out"]
    r = wl.report_batch(s["P"], s["uv"], s["K"], o["R"], o["t"], o["euler"], gt)
    torch.cuda.synchronize()
    return _np(r["report"]), _np(r["flags"])


def _oracle_reproj(s):
    """(mean, max) of the oracle's report columns 6, 7 divided by column 11, on the same pose and pixels widened to FP64"""
    o = s["out"]
    rep = orc.report_batch(_np(s["Pd"]), _np(s["uv"]), s["K"], _np(o["R"]).reshape(-1, 3, 3), _np(o["t"]), _np(o["euler"]),
                           _np(s["gt"]))["report"]
    return np.stack([rep[:, 6] / rep[:, 11], rep[:, 7] / rep[:, 11]], axis=1)


def _numpy_status(s, reproj, limit):
    """The bits recomputed from the returned R, t: (status, mask of problems where BEHIND and REPROJ are well-posed)"""
    o = s["out"]
    R, t = _np(o["R"]).reshape(-1, 3, 3), _np(o["t"])
    P = _np(s["Pd"])
    z = np.einsum("bj,nj->bn", R[:, 2, :], P) + t[:, 2:3]     # K's last row is (0, 0, 1): the depth of every landmark
    st = np.zeros(len(t), np.int32)
    fin = np.isfinite(R).reshape(len(t), -1).all(1) & np.isfinite(t).all(1) & np.isfinite(_np(o["res_norm"])) & np.isfinite(reproj).all(1)
    st |= np.where(~fin, NONFINITE, 0)
    st |= np.where(t[:, 2] <= 0, DEPTH, 0)
    st |= np.where((z < 0).any(1), BEHIND, 0)
    st |= np.where(reproj[:, 0] > limit, REPROJ, 0)
    posed = (np.abs(z).min(1) >= 1e-9) & (np.abs(reproj[:, 0] - limit) > 1e-9 * limit)
    return st, posed


def _rel(a, b):
    return np.abs(a - b) / np.maximum(np.abs(b), 1e-300)


def _within_oracle(s, reproj, ref):
    """1e-12 relative where every landmark's depth is well-conditioned.  A landmark almost in the camera plane has a depth
    that is a difference of nearly equal terms; the report's projection (K folded into R, t) and the oracle's (R, then K)
    round it differently, and its reprojection (up to 1e7 px) carries that rounding: there the bound is 1e-15 times the
    depth's condition number.  Returns the number of well-conditioned problems."""
    o = s["out"]
    R, t = _np(o["R"]).reshape(-1, 3, 3), _np(o["t"])
    P = _np(s["Pd"])
    z = np.einsum("bj,nj->bn", R[:, 2, :], P) + t[:, 2:3]
    scale = np.einsum("bj,nj->bn", np.abs(R[:, 2, :]), np.abs(P)) + np.abs(t[:, 2:3])
    kappa = (scale / np.maximum(np.abs(z), 1e-300)).max(1)
    fin = np.isfinite(ref).all(1)
    rel = _rel(reproj[fin], ref[fin]).max(1)
    good = kappa[fin] <= 1e3
    assert rel[good].max() <= 1e-12, rel[good].max()
    assert (rel <= 1e-12 + 1e-15 * kappa[fin]).all()
    return int(good.sum())


@pytest.mark.parametrize("case", ["lm68", "qeif15"])
def test_reprojection_is_the_reports(case, lm68):
    s = lm68 if case == "lm68" else _solve("qeif", 15, subset=True)
    status, reproj = _check(s)
    rep, _ = _report(s, unit_distance=True)
    assert np.array_equal(reproj[:, 0], rep[:, 6], equal_nan=True)      # bit for bit: report columns 6, 7 at distance_GT = 1
    assert np.array_equal(reproj[:, 1], rep[:, 7], equal_nan=True)
    ref = _oracle_reproj(s)
    assert np.isfinite(ref).all(1).mean() > 0.99
    assert _within_oracle(s, reproj, ref) > 0.9 * len(ref)
    st_np, posed = _numpy_status(s, reproj, 1.0)
    assert posed.mean() > 0.99
    assert np.array_equal(status[posed], st_np[posed])


def test_depth_bit_fails_the_reports_depth_test(lm68):
    status, _ = _check(lm68)
    _, flags = _report(lm68, unit_distance=False)
    d = (status & DEPTH) != 0
    assert (flags[d, 0] == 0).all()


def test_bits_separate_the_failures_of_lm_and_lm_plus(lm68):
    """Margins around the oracle figures quoted in include/pnpb200.h (8 192 problems there, 65 536 here: LM-68 30.6 % fail,
    every BEHIND problem fails, 7.1 % of the unflagged fail, 85 % of the failures flagged; LM+-68 none unflagged fail)."""
    status, _ = _check(lm68)
    _, flags = _report(lm68, unit_distance=False)
    fail = ~flags.all(1).astype(bool)
    behind = (status & BEHIND) != 0
    assert 0.2 < fail.mean() < 0.45 and behind.mean() > 0.05
    assert fail[behind].mean() >= 0.99
    clear = status == 0
    assert fail[clear].mean() <= 0.09
    assert fail[~clear].sum() >= 0.8 * fail.sum()
    s = _solve("lm_plus", 68)
    status, _ = _check(s)
    _, flags = _report(s, unit_distance=False)
    fail = ~flags.all(1).astype(bool)
    assert fail[status == 0].mean() <= 0.001


def test_limit_zero_never_sets_reproj(lm68):
    st1, rp1 = _check(lm68, limit=1.0)
    st0, rp0 = _check(lm68, limit=0.0)
    assert np.array_equal(rp0, rp1)
    assert ((st0 & REPROJ) == 0).all() and ((st1 & REPROJ) != 0).any()
    assert np.array_equal(st0, st1 & ~REPROJ)
    stn, _ = _check(lm68, limit=float("nan"))
    assert np.array_equal(stn, st0)


def test_nonfinite_inputs_flag_exactly_their_problems(lm68):
    import pnp_solver_test_b200 as pnp
    o = lm68["out"]
    n = 4096
    R, t, res = o["R"][:n].clone(), o["t"][:n].clone(), o["res_norm"][:n].clone()
    base = pnp.check_batch(lm68["uv"][:n], lm68["Pd"], lm68["K"], R, t, res_norm=res)
    hit = {5: ("R", (5, 1, 2), float("nan")), 38: ("t", (38, 0), float("inf")), 70: ("res", (70,), float("nan")),
           100: ("t", (100, 2), float("-inf")), 101: ("R", (101, 0, 0), float("-inf"))}
    for b, (name, ix, v) in hit.items():
        {"R": R, "t": t, "res": res}[name][ix] = v
    got = pnp.check_batch(lm68["uv"][:n], lm68["Pd"], lm68["K"], R, t, res_norm=res)
    st0, st = _np(base["status"]), _np(got["status"])
    assert ((st0 & NONFINITE) == 0).all()
    flagged = np.nonzero(st & NONFINITE)[0]
    assert sorted(flagged.tolist()) == sorted(hit)
    rest = np.setdiff1d(np.arange(n), list(hit))
    assert np.array_equal(st[rest], st0[rest])
    assert np.array_equal(_np(got["reproj"])[rest], _np(base["reproj"])[rest])
    assert np.isfinite(_np(got["reproj"])[70]).all()                  # res_norm enters the status word only


def test_check_follows_best_pattern():
    import pnp_solver_test_b200 as pnp
    from conftest import load_golden
    g = load_golden("solve_pnp_two_patterns")
    uv, pats, K = dev(g["uv"]), dev(g["patterns"]), g["K"]
    out = pnp.solve_batch("qeif", uv, pats, K, point_index=g["key_index"])
    B = uv.shape[0]
    rng = np.random.default_rng(7)
    for best in (out["best_pattern"], torch.from_numpy(rng.integers(0, 2, B).astype(np.int32)).cuda()):
        both = pnp.check_batch(uv, pats, K, out["R"], out["t"], res_norm=out["res_norm"], best_pattern=best)
        bn = _np(best)
        assert (bn == 0).any() and (bn == 1).any()
        for p in (0, 1):
            one = pnp.check_batch(uv, pats[p], K, out["R"], out["t"], res_norm=out["res_norm"])
            m = bn == p
            assert np.array_equal(_np(both["status"])[m], _np(one["status"])[m])
            assert np.array_equal(_np(both["reproj"])[m], _np(one["reproj"])[m])
    bad = out["best_pattern"].clone()
    bad[3], bad[17] = 2, -1
    c = pnp.check_batch(uv, pats, K, out["R"], out["t"], best_pattern=bad)
    st, rp = _np(c["status"]), _np(c["reproj"])
    assert (st[[3, 17]] & NONFINITE).all() and np.isnan(rp[[3, 17]]).all()


def test_fp32_within_rounding_of_the_oracle():
    """FP32 inputs are widened and checked in FP64; the outputs are that result rounded once to FP32."""
    s = _solve("lm", 68, dtype=torch.float32)
    status, reproj = _check(s)
    ref = _oracle_reproj(s)
    fin = np.isfinite(ref).all(1)
    assert fin.mean() > 0.99
    r32 = ref[fin].astype(np.float32).astype(np.float64)
    ulp = np.spacing(np.abs(ref[fin]).astype(np.float32)).astype(np.float64)
    assert (np.abs(reproj[fin] - ref[fin]) <= 0.5 * ulp * 1.001).all()
    assert (reproj[fin] == r32).mean() > 0.999
    st_np, posed = _numpy_status(s, reproj, 1.0)
    assert np.array_equal(status[posed], st_np[posed])


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_large_pattern_path(dtype):
    s = _solve("lm", 1024, dtype=dtype, B=4096)
    status, reproj = _check(s)
    ref = _oracle_reproj(s)
    fin = np.isfinite(ref).all(1)
    assert fin.mean() > 0.99
    if dtype == torch.float64:
        assert _within_oracle(s, reproj, ref) > 0.9 * len(ref)
    else:
        ulp = np.spacing(np.abs(ref[fin]).astype(np.float32)).astype(np.float64)
        assert (np.abs(reproj[fin] - ref[fin]) <= 0.5 * ulp * 1.001).all()
    st_np, posed = _numpy_status(s, reproj, 1.0)
    assert np.array_equal(status[posed], st_np[posed])


@pytest.mark.parametrize("pix", ["f64", "int16", "float32"])
def test_host_entry_adds_the_check_and_changes_nothing_else(pix):
    import pnp_solver_test_b200 as pnp
    P, K = pt.pattern_array(pt.synthetic_pattern(68)), pt.default_camera_matrix()
    chunk = 4096
    B = 3 * chunk + 123                                                 # several chunks, the last one ragged
    w = orc.synth(11, B, P, K)
    uv = {"f64": w["uv"], "int16": w["uv"].astype(np.int16), "float32": w["uv"].astype(np.float32)}[pix]
    assert np.array_equal(uv.astype(np.float64), w["uv"])
    solver = pnp.PNP_SOLVER(K, [pt.synthetic_pattern(68)], verbose=False, method="lm")
    plain = solver.solve_pnp_batch_host(uv, chunk_problems=chunk)
    got = solver.solve_pnp_batch_host(uv, chunk_problems=chunk, check=1.0)
    assert sorted(got) == sorted(list(plain) + ["status", "reproj"])
    for k in plain:
        assert np.array_equal(got[k], plain[k], equal_nan=True), k
    c = pnp.check_batch(dev(w["uv"]), dev(P), K, dev(got["R"]), dev(got["t"]), res_norm=dev(got["res_norm"]),
                        best_pattern=torch.from_numpy(got["best_pattern"]).cuda(), reproj_limit_px=1.0)
    assert np.array_equal(got["status"], _np(c["status"]))
    assert np.array_equal(got["reproj"], _np(c["reproj"]), equal_nan=True)
    again = solver.solve_pnp_batch_host(uv, chunk_problems=chunk)
    assert sorted(again) == sorted(plain)
