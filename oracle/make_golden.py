"""TEST INFRASTRUCTURE ONLY (oracle/): generates the committed fixtures under tests/golden/.

Run once, with COCONS_REFERENCE naming the reference package's source tree (for its data/ and oracle/_ref):
    python -m oracle.make_golden            # everything
    python -m oracle.make_golden --quick    # skip the full-size holes / stripes values

Outputs
  tests/golden/datasets.npz      the reference's holes / stripes / holes_bm data (data/*.rda,
                                 GPL >= 3, R/data.R:1-55) as plain float64 matrices
  tests/golden/cov_cases.npz     covariance matrices produced by the REFERENCE's own compiled
                                 source (oracle/_ref) for the inputs stored beside them
  tests/golden/taper_cases.npz   the same for the tapered model (src/cocons_taper.cpp): entries on
                                 nearest.dist patterns, objective and prediction values
  tests/golden/n2ll_cases.json   -2 loglik values: reference-compiled covariance + the literal
                                 numpy/LAPACK restatement of the R objectives (oracle/rmirror.py)
  tests/golden/fresh_cases.npz   the reference's results on the seeded inputs of oracle/fresh_inputs.py
"""
import argparse
import json
import os
import time

import numpy as np

from . import cov, fresh_inputs, rmirror
from .rda import frame_to_matrix, read_rda

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
REF = os.path.join(cov.REFERENCE, "data")
KIND = "reference"  # oracle/_ref: the reference's src/cocons_full.cpp / cocons_taper.cpp compiled here


def load_datasets():
    holes = read_rda(os.path.join(REF, "holes.rda"))["holes"]
    stripes = read_rda(os.path.join(REF, "stripes.rda"))["stripes"]
    bm = read_rda(os.path.join(REF, "holes_bm.rda"))["holes_bm"]
    d = {}
    d["holes_training"], hc = frame_to_matrix(holes["training"])
    d["holes_test"], _ = frame_to_matrix(holes["test"])
    d["stripes_training"], sc = frame_to_matrix(stripes["training"])
    d["stripes_test"], _ = frame_to_matrix(stripes["test"])
    d["holes_bm_training"], bc = frame_to_matrix(bm[0]["training"])
    d["holes_bm_training_z"] = np.asarray(bm[0]["training.z"], dtype=np.float64)
    d["holes_columns"] = np.array(hc)
    d["stripes_columns"] = np.array(sc)
    d["holes_bm_columns"] = np.array(bc)
    return d


def design(M, cov_cols, stats=None):
    X = np.column_stack([np.ones(M.shape[0])] + [M[:, c] for c in cov_cols])
    if stats is None:
        return rmirror.get_scale(X)
    return rmirror.get_scale(X, stats["mean.vector"], stats["sd.vector"])


def theta_block(p, **kw):
    """aspect -> length-p vector; unspecified aspects are zero vectors (fixed at 0)."""
    th = {k: np.zeros(p) for k in rmirror.ASPECT_ORDER}
    for k, v in kw.items():
        v = np.atleast_1d(np.asarray(v, dtype=np.float64))
        th[k.replace("_", ".")][: len(v)] = v
    return th


TH_A3 = dict(std_dev=[0.2, 0.15, 0.1], scale=[-1.6, 0.2, -0.15], nugget=[-np.inf])
TH_B3 = dict(std_dev=[0.2, 0.15, 0.1], scale=[-1.6, 0.2, -0.15], aniso=[0.1, 0.2, -0.1], tilt=[0.3, -0.2, 0.1],
             smooth=[0.2, 0.3, -0.2], nugget=[-4, 0.1, 0.1])
TH_B4 = dict(std_dev=[0.2, 0.15, 0.1, -0.05], scale=[-1.6, 0.2, -0.15, 0.1], aniso=[0.1, 0.2, -0.1, 0.05],
             tilt=[0.3, -0.2, 0.1, 0.1], smooth=[0.2, 0.3, -0.2, 0.1], nugget=[-4, 0.1, 0.1, 0.0])


def cov_cases(d):
    H, HT, S = d["holes_training"], d["holes_test"], d["stripes_training"]
    out = {}

    def add(name, fn, **inputs):
        t = time.time()
        out[name + "__out"] = fn()
        for k, v in inputs.items():
            out[name + "__" + k] = np.asarray(v)
        print("  cov case %-22s %.2fs" % (name, time.time() - t))

    n = 120
    idx = np.arange(n)
    sc = design(H[idx], [2, 3])
    X, locs = sc["std.covs"], H[idx, :2]

    def square(name, th, lim, X=X, locs=locs, classic=False):
        t6 = cov.pack_theta(th, X.shape[1])
        if classic:
            add(name, lambda: cov.cov_rns_classic(th, locs, X, kind=KIND), theta6=t6, locs=locs, X=X)
        else:
            add(name, lambda: cov.cov_rns(th, locs, X, lim, kind=KIND), theta6=t6, locs=locs, X=X, limits=lim)

    square("nu15_vignette", theta_block(3, **TH_A3), [1.5, 1.5])
    square("nu05_fixed", theta_block(3, **TH_A3), [0.5, 0.5])
    square("nu25_fixed", theta_block(3, **TH_A3), [2.5, 2.5])
    square("general_all_aspects", theta_block(3, **TH_B3), [0.5, 2.5])
    square("degenerate_nu1_fixed", theta_block(3, **TH_A3), [1.0, 1.0])  # SURVEY App. B-1
    thc = theta_block(3, **TH_B3)
    thc["smooth"] = np.array([0.1, 0.2, -0.1])
    square("classic_all_aspects", thc, None, classic=True)
    # tilt / aniso fixed at 0 but smoothness covariate-driven: cos(pi/2) = 6.1e-17 path
    square("general_no_aniso", theta_block(3, std_dev=[0.2, 0.15, 0.1], scale=[-1.6, 0.2, -0.15],
                                           smooth=[0.2, 0.3, -0.2], nugget=[-3.0]), [0.5, 2.5])
    # smoothness slopes zero but limits differ -> general branch with constant nu
    square("general_const_nu", theta_block(3, std_dev=[0.2, 0.15, 0.1], scale=[-1.6, 0.2, -0.15],
                                           smooth=[0.4], nugget=[-3.0]), [0.5, 2.5])
    # tiny ranges: Q spans the Hankel band and the >= 706 tail
    square("general_far_pairs", theta_block(3, std_dev=[0.2, 0.15, 0.1], scale=[-6.5, 0.2, -0.15],
                                            aniso=[0.1, 0.2, -0.1], tilt=[0.3, -0.2, 0.1], smooth=[0.2, 0.3, -0.2],
                                            nugget=[-4, 0.1, 0.1]), [0.5, 2.5])
    # large ranges: most pairs in the Temme band (Q < 2)
    square("general_near_pairs", theta_block(3, std_dev=[0.2, 0.15, 0.1], scale=[1.0, 0.2, -0.15],
                                             aniso=[0.1, 0.2, -0.1], tilt=[0.3, -0.2, 0.1], smooth=[0.2, 0.3, -0.2],
                                             nugget=[-4, 0.1, 0.1]), [0.5, 2.5])
    # wide smoothness limits (nu up to 4.5: beyond the Hankel nu cap)
    square("general_wide_nu", theta_block(3, **TH_B3), [0.2, 4.5])
    # duplicated locations (different covariates): coincident rule, SURVEY App. B-2
    locs_dup = locs.copy()
    locs_dup[90] = locs_dup[5]
    locs_dup[17] = locs_dup[100]
    square("general_duplicates", theta_block(3, **TH_B3), [0.5, 2.5], locs=locs_dup)
    square("nu15_duplicates", theta_block(3, **TH_A3), [1.5, 1.5], locs=locs_dup)
    # intercept-only design (p = 1)
    X1 = np.ones((n, 1))
    square("intercept_only", theta_block(1, std_dev=[0.3], scale=[-1.2], smooth=[0.3], nugget=[-2.0]), [0.5, 2.5],
           X=X1)
    # stripes, p = 4, ragged size (not a multiple of the 128 tile)
    ns = 203
    scs = design(S[:ns], [2, 3, 4])
    square("stripes_general_p4", theta_block(4, **TH_B4), [0.5, 2.5], X=scs["std.covs"], locs=S[:ns, :2])
    # prediction cross-covariance incl. three prediction sites sitting on training sites
    m = 70
    lp = HT[:m, :2].copy()
    lp[3], lp[40], lp[69] = locs[10], locs[77], locs[119]
    Xp = design(HT[:m], [2, 3], sc)["std.covs"]
    for nm, th, lim in (("pred_general", theta_block(3, **TH_B3), [0.5, 2.5]),
                        ("pred_nu15_fixed", theta_block(3, **TH_A3), [1.5, 1.5]),
                        ("pred_nu1_fixed", theta_block(3, **TH_A3), [1.0, 1.0])):
        add(nm, lambda th=th, lim=lim: cov.cov_rns_pred(th, locs, lp, X, Xp, lim, kind=KIND),
            theta6=cov.pack_theta(th, 3), locs=locs, X=X, locs_pred=lp, X_pred=Xp, limits=lim)
    return out


def taper_cases(d):
    """Sparse (tapered) model: entries produced by the REFERENCE's own compiled src/cocons_taper.cpp on
    brute-force nearest.dist patterns, and objective / prediction values from oracle/rmirror.py (LAPACK on the
    dense expansion standing in for spam's sparse Cholesky)."""
    H, HT, S = d["holes_training"], d["holes_test"], d["stripes_training"]
    out = {}
    n, delta = 500, 0.25
    sc = design(H[:n], [2, 3])
    X, locs = sc["std.covs"], H[:n, :2].copy()
    dist, ci, rp = rmirror.nearest_dist(locs, delta=delta)
    taper = rmirror.cov_wend1(dist, (delta, 1))
    print("  taper pattern: n=%d nnz=%d density=%.3f" % (n, len(ci), len(ci) / n / n))
    TH_T = dict(std_dev=[0.2, 0.15, 0.1], scale=[-2.6, 0.2, -0.15], smooth=[0.2, 0.3, -0.2], nugget=[-4, 0.1, 0.1])
    TH_TF = dict(std_dev=[0.2, 0.15, 0.1], scale=[-2.6, 0.2, -0.15], nugget=[-4, 0.1, 0.1])

    def square(name, th, lim, locs=locs, X=X, ci=ci, rp=rp):
        out[name + "__out"] = cov.cov_rns_taper(th, locs, X, ci, rp, lim, kind=KIND)
        for k, v in dict(theta6=cov.pack_theta(th, X.shape[1]), locs=locs, X=X, limits=lim, colindices=ci,
                         rowpointers=rp).items():
            out[name + "__" + k] = np.asarray(v)

    square("taper_general", theta_block(3, **TH_T), [0.5, 2.5])
    square("taper_nu05", theta_block(3, **TH_TF), [0.5, 0.5])
    square("taper_nu15", theta_block(3, **TH_TF), [1.5, 1.5])
    square("taper_nu25", theta_block(3, **TH_TF), [2.5, 2.5])
    square("taper_degenerate_nu1", theta_block(3, **TH_TF), [1.0, 1.0])
    square("taper_wide_nu", theta_block(3, **TH_T), [0.2, 4.5])
    # tiny ranges: Q runs through the Hankel band into the >= 706 tail inside the taper radius
    square("taper_far_pairs", theta_block(3, std_dev=[0.2, 0.15, 0.1], scale=[-9.5, 0.2, -0.15],
                                          smooth=[0.2, 0.3, -0.2], nugget=[-4, 0.1, 0.1]), [0.5, 2.5])
    locs_dup = locs.copy()
    locs_dup[90], locs_dup[17] = locs_dup[5], locs_dup[100]
    dd, cid, rpd = rmirror.nearest_dist(locs_dup, delta=delta)
    square("taper_duplicates", theta_block(3, **TH_T), [0.5, 2.5], locs=locs_dup, ci=cid, rp=rpd)
    ns = 331
    scs = design(S[:ns], [2, 3, 4])
    ds, cis, rps = rmirror.nearest_dist(S[:ns, :2], delta=0.08)
    square("taper_stripes_p4", theta_block(4, std_dev=[0.2, 0.15, 0.1, -0.05], scale=[-2.6, 0.2, -0.15, 0.1],
                                           smooth=[0.2, 0.3, -0.2, 0.1], nugget=[-4, 0.1, 0.1, 0.0]), [0.5, 2.5],
           locs=S[:ns, :2], X=scs["std.covs"], ci=cis, rp=rps)
    # prediction pattern, incl. prediction sites sitting on training sites
    m = 90
    lp = HT[:m, :2].copy()
    lp[3], lp[40] = locs[10], locs[77]
    Xp = design(HT[:m], [2, 3], sc)["std.covs"]
    dp, cip, rpp = rmirror.nearest_dist(lp, locs, delta=delta)
    for nm, th, lim in (("taper_pred_general", theta_block(3, **TH_T), [0.5, 2.5]),
                        ("taper_pred_nu15", theta_block(3, **TH_TF), [1.5, 1.5])):
        out[nm + "__out"] = cov.cov_rns_taper_pred(th, locs, lp, X, Xp, cip, rpp, lim, kind=KIND)
        for k, v in dict(theta6=cov.pack_theta(th, 3), locs=locs, X=X, locs_pred=lp, X_pred=Xp, limits=lim,
                         colindices=cip, rowpointers=rpp).items():
            out[nm + "__" + k] = np.asarray(v)
    # objectives and prediction at one theta (all-free aspects but aniso / tilt, which the tapered model ignores)
    pp = par_pos_free(3)
    pp["aniso"], pp["tilt"] = 0.0, 0.0
    tl = theta_block(3, **TH_T)
    tl["mean"] = np.array([0.1, 0.3, -0.2])
    theta = theta_vector_from_lists(tl, pp)
    z = np.column_stack([H[:n, 4], H[:n, 4] ** 2 - 1.0])
    out["obj__theta"], out["obj__z"], out["obj__delta"] = theta, z, np.array(delta)
    out["obj__ml"] = np.array(rmirror.neg2loglik_taper(theta, pp, taper, ci, rp, locs, X, [0.5, 2.5], z, n,
                                                       (0.0, 0.0, 0.0), cov_kind=KIND))
    out["obj__ml_pen"] = np.array(rmirror.neg2loglik_taper(theta, pp, taper, ci, rp, locs, X, [0.5, 2.5], z, n,
                                                           (0.05, 0.02, 0.3), cov_kind=KIND))
    ppp = dict(pp)
    ppp["std.dev"] = np.array([False, True, True])
    theta_p = np.delete(theta, 3)  # drop the std.dev intercept slot (R/optim.R:570-576)
    out["obj__theta_profile"] = theta_p
    out["obj__profile"] = np.array(rmirror.neg2loglik_taper_profile(theta_p, ppp, taper, ci, rp, locs, X, [0.5, 2.5],
                                                                    z, n, (0.0, 0.0, 0.0), cov_kind=KIND))
    back = rmirror.get_model_lists(theta, pp, "diff")
    pr = rmirror.predict_taper(back, delta, locs, lp, X, Xp, [0.5, 2.5], z[:, 0], "pred", cov_kind=KIND)
    out["obj__pred_stochastic"], out["obj__pred_sd"] = pr["stochastic"], pr["sd.pred"]
    # not positive definite: a pattern whose row 8 lost its diagonal entry (zero pivot) -> 1e6 under safe = TRUE
    k = int(rp[7] - 1 + np.flatnonzero(ci[rp[7] - 1:rp[8] - 1] == 8)[0])
    ci_bad, taper_bad = np.delete(ci, k), np.delete(taper, k)
    rp_bad = rp.copy()
    rp_bad[8:] -= 1
    out["obj__notpd_colindices"], out["obj__notpd_rowpointers"], out["obj__notpd_taper"] = ci_bad, rp_bad, taper_bad
    out["obj__notpd"] = np.array(rmirror.neg2loglik_taper(theta, pp, taper_bad, ci_bad, rp_bad, locs, X, [0.5, 2.5], z,
                                                          n, (0.0, 0.0, 0.0), cov_kind=KIND))
    print("  taper objectives: ml %.10f  profile %.10f  notpd %g" % (out["obj__ml"], out["obj__profile"],
                                                                    out["obj__notpd"]))
    return out


def par_pos_free(p, mean_free=True):
    pp = {k: np.ones(p, dtype=bool) for k in rmirror.ASPECT_ORDER}
    if not mean_free:
        pp["mean"] = 0.0
    return pp


def theta_vector_from_lists(tl, par_pos):
    """Inverse of getModelLists(type='diff') for all-free aspects (so the stored input is the
    optimiser-level theta vector the R objective receives)."""
    tl = {k: np.array(v, dtype=np.float64) for k, v in tl.items()}
    sd, sc = tl["std.dev"].copy(), tl["scale"].copy()
    a, b = sd + sc, sd - sc
    tl["std.dev"], tl["scale"] = a, b
    parts = []
    for k in rmirror.ASPECT_ORDER:
        pos = par_pos[k]
        if isinstance(pos, np.ndarray):
            parts.append(tl[k][pos])
    return np.concatenate(parts)


def n2ll_cases(d, quick):
    H, S = d["holes_training"], d["stripes_training"]
    cases = []

    def run(name, M, cov_cols, n, th, lim, mean, z, lam=(0.0, 0.0, 0.0), kinds=("ml", "profile", "reml")):
        t0 = time.time()
        sc = design(M[:n], cov_cols)
        X, locs = sc["std.covs"], M[:n, :2]
        p = X.shape[1]
        tl = theta_block(p, **th)
        tl["mean"] = np.zeros(p)
        tl["mean"][: len(mean)] = mean
        # nugget intercept -Inf cannot pass through the (a+b)/2 re-parameterisation as a free
        # parameter; such aspects are fixed in par.pos, exactly as a coco model.list would have it
        pp = par_pos_free(p)
        for k in ("aniso", "tilt", "smooth", "nugget"):
            if not np.any(tl[k][1:]) and (tl[k][0] == 0 or not np.isfinite(tl[k][0])):
                pp[k] = float(tl[k][0])
        theta = theta_vector_from_lists(tl, pp)
        back = rmirror.get_model_lists(theta, pp, "diff")
        for k in rmirror.ASPECT_ORDER:
            assert np.allclose(back[k], tl[k], rtol=0, atol=1e-15, equal_nan=True) or not np.all(np.isfinite(tl[k]))
        z = np.asarray(z, dtype=np.float64).reshape(n, -1)
        Sigma = cov.cov_rns(back, locs, X, lim, kind=KIND)
        rec = {"name": name, "n": n, "p": p, "r": z.shape[1], "limits": list(lim), "lambda": list(lam),
               "theta": theta.tolist(),
               "par_pos": {k: (v.tolist() if isinstance(v, np.ndarray) else v) for k, v in pp.items()},
               "values": {}}
        if "ml" in kinds:
            rec["values"]["ml"] = rmirror.neg2loglik(theta, pp, locs, X, lim, z, n, lam, Sigma=Sigma)
        ppm = dict(pp)
        ppm["mean"] = np.zeros(p, dtype=bool)
        theta_nomean = theta[p:]
        if "profile" in kinds:
            rec["values"]["profile"] = rmirror.neg2loglik_profile(theta_nomean, ppm, locs, X, lim, z, n, X, lam,
                                                                  Sigma=Sigma)
            rec["values"]["betas"] = rmirror.profile_betas(back, locs, X, lim, X, z, cov_kind=KIND).tolist() \
                if n <= 2500 else None
        if "reml" in kinds:
            zc = rmirror.reml_contrast(X, z) if n <= 6000 else z - X @ np.linalg.solve(X.T @ X, X.T @ z)
            rec["values"]["reml"] = rmirror.neg2loglik_reml(theta_nomean, ppm, locs, X, X, lim, zc, n, lam,
                                                            Sigma=Sigma)
        rec["dataset_rows"] = n
        cases.append(rec)
        print("  n2ll case %-28s n=%d %s  %.1fs" % (name, n, {k: v for k, v in rec["values"].items() if k != "betas"},
                                                   time.time() - t0))
        return rec

    mean3 = [0.1, 0.3, -0.2]
    run("holes1500_nu15", H, [2, 3], 1500, TH_A3, [1.5, 1.5], mean3, H[:1500, 4])["dataset"] = "holes"
    run("holes1500_general", H, [2, 3], 1500, TH_B3, [0.5, 2.5], mean3, H[:1500, 4])["dataset"] = "holes"
    run("holes1500_general_pen", H, [2, 3], 1500, TH_B3, [0.5, 2.5], mean3, H[:1500, 4],
        lam=(0.05, 0.02, 0.3))["dataset"] = "holes"
    run("holes777_ragged", H, [2, 3], 777, TH_B3, [0.5, 2.5], mean3, H[:777, 4])["dataset"] = "holes"
    bm, bz = d["holes_bm_training"], d["holes_bm_training_z"]
    run("holesbm1000_r10", bm, [2, 3], 1000, TH_B3, [0.5, 2.5], mean3, bz[:1000])["dataset"] = "holes_bm"
    run("stripes2000_p4", S, [2, 3, 4], 2000, TH_B4, [0.5, 2.5], [0.1, 0.3, -0.2, 0.1],
        S[:2000, 5])["dataset"] = "stripes"
    # not positive definite: the degenerate fixed-nu quirk makes Sigma singular -> 1e6
    run("holes300_notpd", H, [2, 3], 300, TH_A3, [1.0, 1.0], mean3, H[:300, 4], kinds=("ml",))["dataset"] = "holes"
    if not quick:
        run("holes_full_nu15", H, [2, 3], H.shape[0], TH_A3, [1.5, 1.5], [0.0], H[:, 4])["dataset"] = "holes"
        run("holes_full_general", H, [2, 3], H.shape[0], TH_B3, [0.5, 2.5], mean3, H[:, 4])["dataset"] = "holes"
        run("stripes_full_general", S, [2, 3, 4], S.shape[0], TH_B4, [0.5, 2.5], [0.1, 0.3, -0.2, 0.1],
            S[:, 5])["dataset"] = "stripes"
    return cases


def fresh_cases():
    """The reference's result of every call of oracle/fresh_inputs.py, under the call's key."""
    return {call[0]: np.asarray(fresh_inputs.run(call, KIND))
            for call in list(fresh_inputs.dense_calls()) + list(fresh_inputs.taper_calls())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--only", choices=["datasets", "cov", "n2ll", "taper", "fresh"], default=None)
    args = ap.parse_args()
    if not cov._reference_source_present():
        raise SystemExit("oracle.make_golden: no reference source under '%s' - set COCONS_REFERENCE to the cocons "
                         "source tree" % cov.REFERENCE)
    if args.only != "fresh" and not os.path.isdir(REF):
        raise SystemExit("oracle.make_golden: the reference's data sets are not at '%s' - set COCONS_REFERENCE to the "
                         "cocons source tree" % REF)
    os.makedirs(GOLD, exist_ok=True)
    cov.build(force=True)
    if args.only in (None, "fresh"):
        np.savez_compressed(os.path.join(GOLD, "fresh_cases.npz"), **fresh_cases())
    if args.only == "fresh":
        return
    d = load_datasets()
    if args.only in (None, "datasets"):
        np.savez_compressed(os.path.join(GOLD, "datasets.npz"), **d)
    if args.only in (None, "cov"):
        np.savez_compressed(os.path.join(GOLD, "cov_cases.npz"), **cov_cases(d))
    if args.only in (None, "taper"):
        np.savez_compressed(os.path.join(GOLD, "taper_cases.npz"), **taper_cases(d))
    if args.only in (None, "n2ll"):
        cases = n2ll_cases(d, args.quick)
        with open(os.path.join(GOLD, "n2ll_cases.json"), "w") as f:
            json.dump({"generator": "oracle/make_golden.py", "covariance": "oracle/_ref (reference source compiled)",
                       "algebra": "oracle/rmirror.py on scipy/OpenBLAS LAPACK", "cases": cases}, f, indent=1)


if __name__ == "__main__":
    main()
