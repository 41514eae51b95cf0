"""TEST INFRASTRUCTURE ONLY -- generate ``tests/golden/*`` from the UNMODIFIED reference.

Run in the authoring container (needs ``/root/reference``):

    python -m oracle.make_golden

It (1) copies the reference's own data fixtures the parity tests need on the GPU
box (``test_partim_small`` par/tim, the libstempo golden npz, the ng15 noise
dictionary -- data, not source), and (2) runs the reference's hot functions,
byte-for-byte as shipped, under the ``sys.modules`` stubs of ``oracle/refstubs.py``
and stores inputs + outputs as small npz files:

``ref_small.npz``   the libstempo recipe of ``tests/test_against_libstempo.py:19-53``
                    on JPSR00-02 (per-signal delays with TOAs frozen at their ideal
                    epochs; plus the summed, TOA-shifting run that reproduces the
                    golden vector).
``ref_flags.npz``   4 synthetic multi-backend pulsars with sub-banded epochs and
                    unsorted TOAs: the per-backend ``flags`` paths, ``tnequad``,
                    1-second ECORR buckets, default Fourier convention, GWB options
                    (turnover, no_correlations, userSpec, lmax=2), CGW branches --
                    none of which the reference's own test covers (SURVEY.md section 4).
``ref_orf.npz``     ``spharmORFbasis.correlated_basis`` for lmax<=6 incl. coincident and
                    antipodal pairs.
``ref_recipe8.npz`` one realization of the 15-yr recipe on 8 synthetic ng15-full pulsars
                    (what ``oracle/recipe.py``, the numpy port, must reproduce).
"""
from __future__ import annotations

import glob
import json
import os
import shutil

import numpy as np

from oracle import refstubs
from pta_replicator_b200 import partim

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(os.path.dirname(HERE), "tests", "golden")
REF = refstubs.REFERENCE_ROOT


def _copy_data_fixtures():
    os.makedirs(os.path.join(GOLD, "partim_small", "par"), exist_ok=True)
    os.makedirs(os.path.join(GOLD, "partim_small", "tim"), exist_ok=True)
    for f in glob.glob(os.path.join(REF, "test_partim_small", "par", "*.par")):
        shutil.copy(f, os.path.join(GOLD, "partim_small", "par"))
    for f in glob.glob(os.path.join(REF, "test_partim_small", "tim", "*.tim")):
        shutil.copy(f, os.path.join(GOLD, "partim_small", "tim"))
    shutil.copy(os.path.join(REF, "tests", "libstempo_test_residuals_efac_ecorr_rn_gwb_cgw.npz"),
                os.path.join(GOLD, "libstempo_golden.npz"))
    with open(os.path.join(REF, "noise_dicts", "ng15_dict.json")) as fh:
        nd = json.load(fh)
    pkgdata = os.path.join(os.path.dirname(HERE), "pta_replicator_b200", "data")
    os.makedirs(pkgdata, exist_ok=True)
    with open(os.path.join(pkgdata, "ng15_noise_dict.json"), "w") as fh:
        json.dump({k: float(v) for k, v in sorted(nd.items())}, fh, indent=0)


def _load_small(freeze):
    pars = sorted(glob.glob(os.path.join(REF, "test_partim_small", "par", "*.par")))
    tims = sorted(glob.glob(os.path.join(REF, "test_partim_small", "tim", "*.tim")))
    out = []
    for p, t in zip(pars, tims):
        par = partim.read_par(p)
        c = partim.read_tim(t)
        out.append(refstubs.StubPulsar(par["_name"], par["_loc"], c["mjd"], c["err_us"], c["flags"], freeze_toas=freeze))
    return out


def _reference_nf(psrs, npts=600, howml=10):
    start = float(np.min([p.toas.first_MJD.value * 86400 for p in psrs]) - 86400)
    stop = float(np.max([p.toas.last_MJD.value * 86400 for p in psrs]) + 86400)
    dur = stop - start
    return len(np.arange(0, 1 / (2 * (dur / npts)), 1 / (dur * howml)))


CGW_TEST = dict(gwtheta=np.pi / 2, gwphi=2.5, mc=1e9, dist=5.0, fgw=1e-8, phase0=0.5, psi=1.5, inc=np.pi / 4,
                pdist=1.0, pphase=None, psrTerm=True, evolve=True, phase_approx=False, tref=53000 * 86400)
LAST_MJD_NUDGE = 1e-8  # days; makes len(arange) == 3000 like the PINT run behind the golden npz


def _libstempo_recipe(ref, psrs):
    ref.red_noise.add_gwb(psrs, -14, 4.33, seed=123456)
    for ii, p in enumerate(psrs):
        ref.white_noise.add_measurement_noise(p, efac=1.0, log10_equad=None, seed=54321 + ii, tnequad=False)
        ref.white_noise.add_jitter(p, log10_ecorr=np.log10(3e-7), seed=54321 + ii)
    for ii, p in enumerate(psrs):
        ref.red_noise.add_red_noise(p, -15, 4.2, components=30, Tspan=None, seed=12345 + ii, libstempo_convention=True)
    for p in psrs:
        ref.deterministic.add_cgw(p, **CGW_TEST)


def make_small(ref):
    out = {}
    for freeze in (True, False):
        psrs = _load_small(freeze)
        lm = max(p.toas.last_MJD.value for p in psrs)
        for p in psrs:
            p.toas.last_override = lm + LAST_MJD_NUDGE
        nf = _reference_nf(psrs)
        assert nf == 3000, nf
        _libstempo_recipe(ref, psrs)
        if freeze:
            for sig in ("gwb", "measurement_noise", "jitter", "red_noise", "cw"):
                out[sig] = np.array([p.signal_seconds(f"{p.name}_{sig}") for p in psrs])
        else:
            out["residuals_shifting"] = np.array([p.resids_value for p in psrs])
    out["nf"] = np.array(3000)
    out["last_mjd_nudge_days"] = np.array(LAST_MJD_NUDGE)
    gold = np.load(os.path.join(GOLD, "libstempo_golden.npz"))["residuals"]
    dev = [np.max(np.abs(out["residuals_shifting"][i] - gold[i])) / np.sqrt(np.mean(gold[i] ** 2)) for i in range(3)]
    print("stub-harness vs libstempo golden, max|d|/rms per psr:", dev)
    assert max(dev) < 1e-3
    np.savez(os.path.join(GOLD, "ref_small.npz"), **out)


def synth_flag_pulsars(seed=20250922, npsr=4):
    """Small multi-backend, sub-banded, unsorted data set (float64-exact MJDs)."""
    rng = np.random.default_rng(seed)
    psrs = []
    for i in range(npsr):
        nb = 2 + i % 2
        backends = [f"BE{i}{k}" for k in range(nb)]
        nep = 36 + 5 * i
        ep = np.sort(rng.uniform(53000, 58800, nep))
        mj, er, fl = [], [], []
        for e, t0 in enumerate(ep):
            nsub = int(rng.integers(3, 12))
            off = rng.uniform(0, 0.5, nsub) / 86400.0
            for o in off:
                mj.append(float(np.float64(t0 + o)))
                er.append(float(rng.uniform(0.1, 3.0)))
                fl.append({"f": backends[e % nb], "pta": "SYN"})
        perm = rng.permutation(len(mj))
        mj = np.asarray(mj)[perm]
        er = np.asarray(er)[perm]
        fl = [fl[k] for k in perm]
        loc = {"RAJ": float(rng.uniform(0, 24)), "DECJ": float(np.degrees(np.arcsin(rng.uniform(-1, 1))))}
        psrs.append(dict(name=f"J{1000 + 137 * i:04d}+{10 + i:02d}", loc=loc, mjd=mj, err_us=er, flags=fl, backends=backends))
    return psrs


def make_flags(ref):
    spec = synth_flag_pulsars()
    rng = np.random.default_rng(7)
    store = {"npsr": np.array(len(spec))}
    params = []
    for i, s in enumerate(spec):
        nb = len(s["backends"])
        params.append(dict(efac=rng.uniform(0.8, 1.4, nb), l10_equad=rng.uniform(-7.5, -6.0, nb),
                           l10_ecorr=rng.uniform(-7.5, -6.2, nb), rn_l10A=float(rng.uniform(-14.5, -13.0)),
                           rn_gamma=float(rng.uniform(1.5, 5.0))))
        store[f"mjd_{i}"] = s["mjd"]
        store[f"err_{i}"] = s["err_us"]
        store[f"flag_{i}"] = np.array([f["f"] for f in s["flags"]])
        store[f"backends_{i}"] = np.array(s["backends"])
        store[f"raj_decj_{i}"] = np.array([s["loc"]["RAJ"], s["loc"]["DECJ"]])
        store[f"name_{i}"] = np.array(s["name"])
        for k, v in params[i].items():
            store[f"{k}_{i}"] = np.asarray(v)

    def fresh():
        return [refstubs.StubPulsar(s["name"], s["loc"], s["mjd"].astype(np.longdouble), s["err_us"], s["flags"]) for s in spec]

    # --- per-backend white noise, t2equad and tnequad; ECORR with flags at 1 s and scalar at 0.1 d
    psrs = fresh()
    for i, p in enumerate(psrs):
        pr, be = params[i], np.array(spec[i]["backends"])
        ref.white_noise.add_measurement_noise(p, efac=pr["efac"], log10_equad=pr["l10_equad"], flagid="f", flags=be, seed=10660 + i)
        ref.white_noise.add_jitter(p, log10_ecorr=pr["l10_ecorr"], flagid="f", flags=be, coarsegrain=1.0 / 86400.0, seed=17763 + i)
        ref.red_noise.add_red_noise(p, pr["rn_l10A"], pr["rn_gamma"], components=30, seed=19870 + i)
        store[f"wn_flags_{i}"] = p.signal_seconds(f"{p.name}_measurement_noise")
        store[f"jit_flags_{i}"] = p.signal_seconds(f"{p.name}_jitter")
        store[f"rn_default_{i}"] = p.signal_seconds(f"{p.name}_red_noise")
    psrs = fresh()
    for i, p in enumerate(psrs):
        pr, be = params[i], np.array(spec[i]["backends"])
        ref.white_noise.add_measurement_noise(p, efac=pr["efac"], log10_equad=pr["l10_equad"], flagid="f", flags=be, seed=333 + i, tnequad=True)
        ref.white_noise.add_jitter(p, log10_ecorr=-6.7, seed=444 + i)  # scalar, default 0.1 d buckets
        ref.red_noise.add_red_noise(p, -13.7, 3.1, components=12, seed=555 + i, libstempo_convention=True)
        store[f"wn_tn_{i}"] = p.signal_seconds(f"{p.name}_measurement_noise")
        store[f"jit_scalar_{i}"] = p.signal_seconds(f"{p.name}_jitter")
        store[f"rn_ls12_{i}"] = p.signal_seconds(f"{p.name}_red_noise")
    psrs = fresh()
    for i, p in enumerate(psrs):  # scalar efac + equad, modes given explicitly
        ref.white_noise.add_measurement_noise(p, efac=1.1, log10_equad=-6.5, seed=777 + i)
        modes = np.array([1e-9, 3.3e-9, 7.7e-9, 2.1e-8, 5e-8])
        ref.red_noise.add_red_noise(p, -14.0, 2.5, modes=modes, seed=888 + i)
        store[f"wn_scalar_{i}"] = p.signal_seconds(f"{p.name}_measurement_noise")
        store[f"rn_modes_{i}"] = p.signal_seconds(f"{p.name}_red_noise")
    store["rn_modes"] = modes

    # --- GWB variants
    uspec = np.stack([np.logspace(-9.5, -7.2, 9), 1e-15 * np.logspace(-9.5, -7.2, 9) ** (-0.6) / (1e-8) ** (-0.6)], axis=1)
    store["gwb_userspec"] = uspec
    rng2 = np.random.default_rng(11)
    clm2 = np.concatenate([[np.sqrt(4 * np.pi)], 0.3 * rng2.standard_normal(8)])
    store["gwb_clm_l2"] = clm2
    variants = {
        "hd": dict(log10_amplitude=-14.2, spectral_index=13.0 / 3.0, seed=16672),
        "turnover": dict(log10_amplitude=-14.0, spectral_index=4.0, seed=16673, turnover=True, f0=3e-9, beta=1.2, power=1.5),
        "nocorr": dict(log10_amplitude=-14.3, spectral_index=3.0, seed=16674, no_correlations=True),
        "userspec": dict(log10_amplitude=-14.0, spectral_index=4.0, seed=16675, userSpec=uspec),
        "aniso_l2": dict(log10_amplitude=-14.1, spectral_index=13.0 / 3.0, seed=16676, clm=list(clm2), lmax=2),
        "npts300": dict(log10_amplitude=-14.1, spectral_index=13.0 / 3.0, seed=16677, npts=300, howml=4),
    }
    for tag, kw in variants.items():
        psrs = fresh()
        store[f"gwb_{tag}_nf"] = np.array(_reference_nf(psrs, kw.get("npts", 600), kw.get("howml", 10)))
        ref.red_noise.add_gwb(psrs, **kw)
        for i, p in enumerate(psrs):
            store[f"gwb_{tag}_{i}"] = p.signal_seconds(f"{p.name}_gwb")

    # --- CGW branches
    base = dict(gwtheta=1.1, gwphi=4.0, mc=3e9, dist=40.0, fgw=2.2e-8, phase0=1.3, psi=0.4, inc=1.0, tref=53000 * 86400)
    cvar = {
        "evolve": dict(base, pdist=1.3, psrTerm=True, evolve=True),
        "earth": dict(base, psrTerm=False, evolve=True),
        "approx": dict(base, pdist=0.9, psrTerm=True, evolve=False, phase_approx=True),
        "mono": dict(base, pdist=0.9, psrTerm=True, evolve=False, phase_approx=False),
        "pphase": dict(base, pphase=2.0, psrTerm=True, evolve=True),
    }
    for tag, kw in cvar.items():
        psrs = fresh()
        for i, p in enumerate(psrs):
            ref.deterministic.add_cgw(p, signal_name="cw", **kw)
            store[f"cgw_{tag}_{i}"] = p.signal_seconds(f"{p.name}_cw")
    np.savez(os.path.join(GOLD, "ref_flags.npz"), **store)


def make_catalog(ref):
    """``add_catalog_of_cws`` (deterministic.py:188-318; numba loops :321-561) on the 4 synthetic pulsars with a
    300-source catalog; source 7 has already merged at the late TOAs (negative frequency -> NaN -> masked)."""
    spec = synth_flag_pulsars()
    rng = np.random.default_rng(21)
    n = 300
    cat = dict(gwtheta=np.arccos(rng.uniform(-1, 1, n)), gwphi=rng.uniform(0, 2 * np.pi, n),
               mc=10 ** rng.uniform(8.0, 9.8, n), dist=10 ** rng.uniform(1.0, 3.0, n), fgw=10 ** rng.uniform(-8.8, -7.3, n),
               phase0=rng.uniform(0, 2 * np.pi, n), psi=rng.uniform(0, np.pi, n), inc=np.arccos(rng.uniform(-1, 1, n)))
    cat["mc"][7], cat["fgw"][7] = 3e10, 4e-7          # merges inside the data span
    store = {f"cat_{k}": v for k, v in cat.items()}
    variants = {"evolve": dict(pdist=1.2, psrTerm=True, evolve=True), "earth": dict(psrTerm=False, evolve=True),
                "approx": dict(pdist=0.8, psrTerm=True, evolve=False, phase_approx=True),
                "mono": dict(pdist=0.8, psrTerm=True, evolve=False, phase_approx=False),
                "pphase": dict(pphase=1.5, psrTerm=True, evolve=True)}
    for tag, kw in variants.items():
        for i, s in enumerate(spec):
            p = refstubs.StubPulsar(s["name"], s["loc"], s["mjd"].astype(np.longdouble), s["err_us"], s["flags"])
            ref.deterministic.add_catalog_of_cws(p, cat["gwtheta"].copy(), cat["gwphi"].copy(), cat["mc"].copy(), cat["dist"].copy(),
                                                 cat["fgw"].copy(), cat["phase0"].copy(), cat["psi"].copy(), cat["inc"].copy(),
                                                 tref=53000 * 86400, **kw)
            store[f"cat_{tag}_{i}"] = p.signal_seconds(f"{p.name}_cw_catalog")
    assert any(np.isnan(v).sum() == 0 for v in store.values())
    np.savez(os.path.join(GOLD, "ref_catalog.npz"), **store)


def _fixtures_module():
    import importlib.util
    # by path: the reference tree on sys.path has a ``tests`` package of its own
    sp = importlib.util.spec_from_file_location("ptar_test_fixtures", os.path.join(os.path.dirname(GOLD), "fixtures.py"))
    fx = importlib.util.module_from_spec(sp)
    sp.loader.exec_module(fx)
    return fx


def make_outliers(ref):
    """``add_gwb_plus_outlier_cws`` (deterministic.py:565-715) on the 4 synthetic pulsars with a 4000-sample population,
    3 outliers per bin.  holodeck / astropy.constants are stand-ins (oracle/refstubs.py); everything else is the
    unmodified reference: binning, ranking, free spectrum, add_gwb(userSpec), the global-stream draws, the catalog."""
    fx = _fixtures_module()
    vals, weights, fobs, T_obs = fx.outlier_population()
    spec = synth_flag_pulsars()
    psrs = [refstubs.StubPulsar(s["name"], s["loc"], s["mjd"].astype(np.longdouble), s["err_us"], s["flags"]) for s in spec]
    ret = ref.deterministic.add_gwb_plus_outlier_cws(psrs, vals, weights, fobs, T_obs, outlier_per_bin=3, seed=4242)
    names = ("f_centers", "free_spec", "outlier_fo", "outlier_hs", "outlier_mc", "outlier_dl", "gwthetas", "gwphis", "phases",
             "psis", "incs")
    store = {k: np.asarray(v) for k, v in zip(names, ret)}
    for i, p in enumerate(psrs):
        store[f"gwb_{i}"] = p.signal_seconds(f"{p.name}_gwb")
        store[f"cw_{i}"] = p.signal_seconds(f"{p.name}_cw_catalog")
    assert len(store["outlier_fo"]) == 18
    np.savez(os.path.join(GOLD, "ref_outliers.npz"), **store)


def make_f4(ref):
    """``add_burst`` (deterministic.py:718-793, with and without ``remove_quad``), ``add_noise_transient`` (:796-819)
    and ``add_gw_memory`` (:822-884) on the 4 synthetic pulsars; the waveforms live in tests/fixtures.py."""
    fx = _fixtures_module()
    spec = synth_flag_pulsars()
    store = {}
    for i, s in enumerate(spec):
        def fresh():
            return refstubs.StubPulsar(s["name"], s["loc"], s["mjd"].astype(np.longdouble), s["err_us"], s["flags"])
        for tag, quad in (("burst", False), ("burstq", True)):
            p = fresh()
            ref.deterministic.add_burst(p, 1.1, 4.0, fx.burst_plus, fx.burst_cross, psi=0.7, tref=fx.F4_TREF, remove_quad=quad)
            store[f"{tag}_{i}"] = p.signal_seconds(f"{p.name}_burst")
        p = fresh()
        ref.deterministic.add_noise_transient(p, fx.transient_waveform, tref=fx.F4_TREF)
        store[f"transient_{i}"] = p.signal_seconds(f"{p.name}_noise_transient")
        p = fresh()
        ref.deterministic.add_gw_memory(p, 3.0e-14, 0.9, 2.2, 0.4, fx.F4_T0_MJD)
        store[f"memory_{i}"] = p.signal_seconds(f"{p.name}_gw_memory")
    np.savez(os.path.join(GOLD, "ref_f4.npz"), **store)


def make_fourier(ref):
    """create_fourier_design_matrix_red with the options the injection path never uses: pshift (random phases from the
    global stream), logf / fmin / fmax, Tspan (red_noise.py:61-101)."""
    rng = np.random.default_rng(31)
    t = np.sort(rng.uniform(53000, 58800, 120)) * 86400.0
    out = {"t": t}
    np.random.seed(4242)
    out["F_pshift"], out["f_pshift"] = ref.red_noise.create_fourier_design_matrix_red(t, nmodes=20, pshift=True)
    np.random.seed(4243)
    out["F_pshift_ls"], _ = ref.red_noise.create_fourier_design_matrix_red(t, nmodes=20, pshift=True, libstempo_convention=True)
    out["F_logf"], out["f_logf"] = ref.red_noise.create_fourier_design_matrix_red(t, nmodes=20, logf=True, fmin=2e-9, fmax=3e-7)
    out["F_lin"], out["f_lin"] = ref.red_noise.create_fourier_design_matrix_red(t, nmodes=20, fmin=2e-9, fmax=3e-7)
    out["F_tspan"], out["f_tspan"] = ref.red_noise.create_fourier_design_matrix_red(t, nmodes=20, Tspan=6.0e8)
    np.savez(os.path.join(GOLD, "ref_fourier.npz"), **out)


def make_real(ref):
    """The reference's real NANOGrav 15-yr files (test_partim: B1855+09, B1937+21, J1909-3744; unsorted TOAs, 7.8k / 23k /
    35k TOAs, ELONG/ELAT positions, -f backend flags): the columns the hot path reads, stored compactly (the tim files
    are 26 MB of text), the bucket counts of the unmodified ``quantize_fast`` and every 40th TOA of the unmodified
    white / ECORR / red-noise injections with the 15-yr noise dictionary."""
    from pta_replicator_b200 import noise_dict as nd
    out = {}
    names = ["B1855+09", "B1937+21", "J1909-3744"]
    noise = nd.load_noise_dict()
    psrs = []
    for i, name in enumerate(names):
        par = partim.read_par(os.path.join(REF, "test_partim", "par", name + ".par"))
        c = partim.read_tim(os.path.join(REF, "test_partim", "tim", name + ".tim"))
        fl = np.array([f.get("f", "") for f in c["flags"]])
        be, inv = np.unique(fl, return_inverse=True)
        mjd = np.asarray(c["mjd"], dtype=np.longdouble)
        hi = mjd.astype(np.float64)
        out[f"name_{i}"] = np.array(name)
        out[f"elong_elat_{i}"] = np.array([par["_loc"]["ELONG"], par["_loc"]["ELAT"]])
        out[f"mjd_hi_{i}"], out[f"mjd_lo_{i}"] = hi, (mjd - hi.astype(np.longdouble)).astype(np.float64)
        out[f"err_us_{i}"] = np.asarray(c["err_us"], np.float64)
        out[f"flag_idx_{i}"], out[f"backends_{i}"] = inv.astype(np.uint8), be
        psrs.append(refstubs.StubPulsar(name, par["_loc"], mjd, c["err_us"], c["flags"]))
        for tag, width in (("1s", 1.0 / 86400.0), ("0p1d", 0.1)):
            ave, U = ref.white_noise.quantize_fast(np.asarray(mjd, dtype=float), dt=width)
            out[f"nbucket_{tag}_{i}"] = np.array(U.shape[1])
        pp = nd.per_pulsar(noise, name)
        pbe = np.array(pp["backends"])
        out[f"dict_backends_{i}"] = pbe
        p = psrs[-1]
        ref.white_noise.add_measurement_noise(p, efac=np.asarray(pp["efac"]), log10_equad=np.asarray(pp["log10_equad"]), flagid="f",
                                              flags=pbe, seed=10660 + i)
        ref.white_noise.add_jitter(p, log10_ecorr=np.asarray(pp["log10_ecorr"]), flagid="f", flags=pbe, coarsegrain=1.0 / 86400.0,
                                   seed=17763 + i)
        ref.red_noise.add_red_noise(p, pp["rn_log10_A"], pp["rn_gamma"], components=30, seed=19870 + i)
        for sig in ("measurement_noise", "jitter", "red_noise"):
            out[f"{sig}_{i}"] = p.signal_seconds(f"{p.name}_{sig}")[::40]
    np.savez_compressed(os.path.join(GOLD, "ref_real3.npz"), **out)


RECIPE_STRIDE = 4   # every 4th TOA of each pulsar: keeps the fixture small (76k TOAs in all)


def make_recipe(ref):
    """One realization (seed 5) of the 15-yr recipe through the unmodified ``add_measurement_noise`` / ``add_jitter`` /
    ``add_red_noise`` / ``add_gwb`` (oracle/refrecipe.py) on the first 8 pulsars of the synthetic ng15-full set: every
    ``RECIPE_STRIDE``-th TOA of each pulsar and the rms of the whole realization per pulsar."""
    from oracle import refrecipe
    from pta_replicator_b200 import synthetic
    psrs, noise = synthetic.make_ng15_like("full", npsr=8)
    out = refrecipe.realization(refrecipe.dataset_from_pulsars(psrs, noise), 5)
    store = {"npsr": np.array(len(out)), "seed": np.array(5), "stride": np.array(RECIPE_STRIDE)}
    for i, d in enumerate(out):
        store[f"delay_{i}"] = d[::RECIPE_STRIDE]
        store[f"rms_{i}"] = np.array(np.sqrt(np.mean(d * d)))
        store[f"ntoa_{i}"] = np.array(len(d))
    np.savez_compressed(os.path.join(GOLD, "ref_recipe8.npz"), **store)


def make_orf(ref):
    rng = np.random.default_rng(3)
    n = 9
    phi = rng.uniform(0, 2 * np.pi, n)
    th = np.arccos(rng.uniform(-1, 1, n))
    phi[4], th[4] = phi[1], th[1]                        # coincident pair  -> zeta == 0 off the diagonal
    phi[6], th[6] = (phi[2] + np.pi) % (2 * np.pi), np.pi - th[2]   # antipodal pair (zeta ~ pi)
    locs = np.stack([phi, th], axis=1)
    basis = np.array(ref.orf.correlated_basis(locs, 6))
    rng = np.random.default_rng(5)
    n2 = 24
    locs2 = np.stack([rng.uniform(0, 2 * np.pi, n2), np.arccos(rng.uniform(-1, 1, n2))], axis=1)
    basis2 = np.array(ref.orf.correlated_basis(locs2, 0))
    np.savez(os.path.join(GOLD, "ref_orf.npz"), locs=locs, basis_l6=basis, locs_hd=locs2, basis_hd=basis2)


def main():
    os.makedirs(GOLD, exist_ok=True)
    _copy_data_fixtures()
    ref = refstubs.reference_modules()
    from oracle import refnumpy
    assert refnumpy.SOLAR2S == ref.constants.SOLAR2S and refnumpy.KPC2S == ref.constants.KPC2S
    assert refnumpy.MPC2S == ref.constants.MPC2S and refnumpy.YEAR == ref.constants.YEAR_IN_SEC
    make_small(ref)
    make_flags(ref)
    make_orf(ref)
    make_fourier(ref)
    make_real(ref)
    make_catalog(ref)
    make_f4(ref)
    make_outliers(ref)
    make_recipe(ref)
    print("golden fixtures written to", GOLD)


if __name__ == "__main__":
    main()
