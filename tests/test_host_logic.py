"""CPU tests of the host-side logic: readers, bucketing, the epoch/tile planner, the noise
dictionary, the ORF closed form, ledger semantics, and that the C-ABI library loads and exports
every symbol include/ptar.h declares (no kernel is launched here)."""
import os
import re
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from oracle import refnumpy as O
from tests.fixtures import GOLD, load_flags_case

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_cabi_exports_every_declared_symbol():
    from pta_replicator_b200 import _cabi
    hdr = open(os.path.join(ROOT, "include", "ptar.h")).read()
    declared = set(re.findall(r"\b(ptar_[a-z_0-9]+)\s*\(", hdr))
    assert declared == set(_cabi.EXPORTS), declared ^ set(_cabi.EXPORTS)
    L = _cabi.lib()
    for name in declared:
        assert hasattr(L, name)
    assert L.ptar_version() == 200


def test_no_cpu_fallback_without_a_gpu():
    """In a child process with every GPU hidden (CUDA_VISIBLE_DEVICES=""), so that it runs on GPU machines too."""
    code = textwrap.dedent(f"""
        import os
        import pytest
        import torch
        assert not torch.cuda.is_available()
        import pta_replicator_b200 as P
        from pta_replicator_b200 import _cabi
        p = P.load_pulsar(os.path.join({GOLD!r}, "partim_small", "par", "JPSR00.par"),
                          os.path.join({GOLD!r}, "partim_small", "tim", "fake_JPSR00_noiseonly.tim"))
        P.make_ideal(p)
        with pytest.raises(_cabi.PtarError, match="no CPU fallback"):
            P.add_measurement_noise(p, efac=1.0)
        assert p.added_signals == {{}}
    """)
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr


def test_product_does_not_import_the_oracle():
    pkg = os.path.join(ROOT, "pta_replicator_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), fn


def test_par_tim_readers_and_loader():
    import pta_replicator_b200 as P
    psrs = P.load_from_directories(os.path.join(GOLD, "partim_small", "par"), os.path.join(GOLD, "partim_small", "tim"),
                                   num_psrs=2)
    assert [p.name for p in psrs] == ["JPSR00", "JPSR01"]
    p = psrs[0]
    assert p.toas.ntoas == 122 and p.added_signals is None
    assert abs(p.loc["RAJ"] - (9 + 19 / 60 + 49.05 / 3600)) < 1e-12 and abs(p.loc["DECJ"] + (75 + 42 / 60 + 35.3 / 3600)) < 1e-12
    assert p.toas.table["tdbld"].dtype == np.longdouble and p.toas.table["flags"].data[0] == {"pta": "PPTA"}
    assert np.allclose(p.toas.get_errors().to("s").value, 0.5e-6)
    with pytest.raises(FileNotFoundError):
        P.load_from_directories("/nonexistent", "/nonexistent")
    with pytest.raises(ValueError, match="make_ideal"):
        p.update_added_signals("x", {})
    P.make_ideal(p)
    p.update_added_signals("x", {"a": 1}, P.simulate.TimeArray(np.ones(122) * 1e-6, "s"))
    with pytest.raises(ValueError, match="already exists"):
        p.update_added_signals("x", {})
    assert p.added_signals_time["x"].to_value("us")[0] == pytest.approx(1.0)
    p.toas.adjust_TOAs(p.added_signals_time["x"].to("day"))
    p.update_residuals()
    assert np.allclose(p.residuals.resids_value, 0.0, atol=1e-18)      # constant delay is absorbed by the mean


def test_greedy_buckets_match_quantize_rule():
    from pta_replicator_b200.engine import greedy_buckets
    from pta_replicator_b200.white_noise import quantize_fast, quantize_index
    rng = np.random.default_rng(0)
    for width in (1.0 / 86400.0, 0.1, 1.0, 30.0):
        t = np.sort(np.concatenate([rng.uniform(53000, 53400, 300), 53100 + np.arange(40) * width, [53000.0, 53000.0]]))
        ref, firsts = O.epoch_buckets(t, width)
        assert np.array_equal(greedy_buckets(t, width), ref)
    t = rng.permutation(t)
    b, firsts = quantize_index(t, 0.1)
    rb, rf = O.epoch_buckets(t, 0.1)
    assert np.array_equal(b, rb) and np.array_equal(np.sort(t[firsts]), np.sort(t[rf]))
    ave, U = quantize_fast(t, dt=0.1)
    assert U.shape == (len(t), len(firsts)) and np.all(U.sum(axis=1) == 1) and np.allclose(U.T @ t / U.sum(axis=0), ave)


def _plan_invariants(b, pl):
    tiles = pl["tiles"]
    covered = np.zeros(b.ld, dtype=int)
    for (ts, nt, tl0, es, ne, psr, nd, _) in tiles:
        assert 0 < nt <= 1024 and 0 < ne <= 64 and ts % 4 == 0 and 1 <= nd <= 3
        assert ts - b.toa_off[psr] == tl0
        covered[ts:ts + nt] += 1
        el = pl["eloc"][ts:ts + nt]
        assert el.min() == 0 and el.max() == ne - 1 and np.all(np.diff(el.astype(int)) >= 0)
    for i in range(b.n_psr):
        assert np.all(covered[b.toa_off[i]:b.toa_off[i] + b.ntoa[i]] == 1)
    assert covered.sum() == b.n_toa_total
    assert np.all(pl["dtau"] >= 0)


def test_planner_epochs_and_tiles():
    import pta_replicator_b200 as P
    from pta_replicator_b200.engine import PulsarBatch
    _, spec = load_flags_case()
    psrs = []
    for s in spec:
        p = P.pulsar_from_arrays(s["name"], s["loc"], s["mjd"].astype(np.longdouble), s["err_us"],
                                 flags=[{"f": f} for f in s["flag"]])
        P.make_ideal(p)
        psrs.append(p)
    for exact in (False, True):
        b = PulsarBatch(psrs, plan_only=True, exact_epochs=exact, rn_taylor_tol=1e-14)   # 1e-14: three Taylor terms
        for i, s in enumerate(spec):
            b.set_white(i, efac=s["efac"], log10_equad=s["l10_equad"], flags=np.array(s["backends"]))
            b.set_ecorr(i, s["l10_ecorr"], flags=np.array(s["backends"]), coarsegrain=1.0 / 86400.0)
            b.set_red(i, s["rn_l10A"], s["rn_gamma"])
        b.set_gwb(-14.5, 13 / 3)
        pl = b.plan()
        _plan_invariants(b, pl)
        if exact:
            assert pl["n_epochs"] == b.n_toa_total and np.all(pl["dtau"] == 0) and pl["tiles"][:, 6].max() == 1
        else:
            assert pl["n_epochs"] == pl["n_bucket_total"]            # sub-banded epochs == 1-second ECORR buckets here
            assert pl["dtau"].max() < 0.51 and pl["tiles"][:, 6].max() == 3
            # white: w1 = efac * sigma in engine order
            i = 1
            s = spec[i]
            ef = O.per_toa_params(s["efac"], s["backends"], s["flag"], len(s["mjd"]))
            sl = slice(b.toa_off[i], b.toa_off[i] + b.ntoa[i])
            assert np.array_equal(pl["w1"][sl], (ef * (s["err_us"] * 1e-6))[b.order[i]])
        with pytest.raises(Exception, match="plan_only"):
            b.compile()
    # an epoch is never allowed to straddle a GWB grid knot
    mj = np.sort(np.concatenate([53000 + np.arange(0, 3000, 0.37)]))
    p = P.pulsar_from_arrays("JX", {"RAJ": 1.0, "DECJ": 2.0}, mj.astype(np.longdouble), np.ones(len(mj)))
    P.make_ideal(p)
    b = PulsarBatch([p], plan_only=True, rn_taylor_tol=1e-3)     # huge window: only buckets / knots cut epochs
    b.set_ecorr(0, -6.5, coarsegrain=5.0)
    b.set_red(0, -14, 3.0, components=5)
    b.set_gwb(-14.5, 13 / 3)
    pl = b.plan()
    _plan_invariants(b, pl)
    g = b._gwb
    gj = np.clip(np.searchsorted(g["ut"], b.mjd[0] * 86400, side="right") - 1, 0, g["npts"] - 2)
    ep = np.zeros(b.ld, dtype=int)
    for t in pl["tiles"]:
        ep[t[0]:t[0] + t[1]] = t[3] + pl["eloc"][t[0]:t[0] + t[1]]
    ep = ep[:len(mj)]
    for e in np.unique(ep):
        assert len(np.unique(gj[ep == e])) == 1
        assert pl["knots"][pl["ep_gidx"][e]] == gj[ep == e][0]          # compact-grid column -> knot
        assert pl["knots"][pl["ep_gidx"][e] + 1] == gj[ep == e][0] + 1
    assert pl["g_ld"] % 2 == 0 and np.all(pl["syn_tiles"][:, 2] <= 64) and np.all(np.diff(pl["syn_tiles"][:, 3]) <= 0)


def test_noise_dict_and_synthetic_dataset():
    from pta_replicator_b200 import noise_dict as nd
    from pta_replicator_b200 import synthetic
    d = nd.load_noise_dict()
    assert len(d) == 785 and abs(d["gw_log10_A"] + 14.6733) < 0.01
    names = nd.pulsar_names(d)
    assert len(names) == 67 and "J0614-3329" not in names and "B1855+09" in names
    pp = nd.per_pulsar(d, "B1855+09")
    assert pp["backends"] == ["430_ASP", "430_PUPPI", "L-wide_ASP", "L-wide_PUPPI"] and len(pp["efac"]) == 4
    assert pp["rn_gamma"] == d["B1855+09_red_noise_gamma"]
    pp = nd.per_pulsar(d, "J1751-2857")           # the one backend with equad + ecorr but no efac
    assert 1.0 in pp["efac"]
    psrs, noise = synthetic.make_ng15_like("epoch")
    assert len(psrs) == 67 and 6700 <= sum(p.toas.ntoas for p in psrs) <= 33500
    psrs2, _ = synthetic.make_ng15_like("epoch")
    assert np.array_equal(psrs[5].toas.table["tdbld"], psrs2[5].toas.table["tdbld"])
    assert all(p.added_signals == {} for p in psrs)


def test_orf_l0_matches_reference_fixture():
    from pta_replicator_b200 import orf
    z = np.load(os.path.join(GOLD, "ref_orf.npz"))
    assert np.max(np.abs(orf.correlated_basis(z["locs_hd"], 0)[0] - z["basis_hd"][0])) < 1e-15
    assert np.max(np.abs(orf.correlated_basis(z["locs"], 0)[0] - z["basis_l6"][0])) < 1e-15   # incl. coincident / antipodal pairs
    ra, dec = orf.ecliptic_to_equatorial(0.0, 0.0)
    assert abs(ra) < 1e-12 and abs(dec) < 1e-12
    ra, dec = orf.ecliptic_to_equatorial(90.0, 0.0)
    assert abs(ra - np.pi / 2) < 1e-12 and abs(dec - np.radians(23.4392911)) < 1e-12


def test_orf_anisotropic_basis_matches_reference_fixture():
    """lmax = 6 on 9 pulsars incl. a coincident and an antipodal pair, against the reference's own
    ``correlated_basis`` (tests/golden/ref_orf.npz).  The computational-frame sums alternate with
    factorial-sized terms; for one close pair the reference's own rounding noise is ~2e-11."""
    from pta_replicator_b200 import orf
    z = np.load(os.path.join(GOLD, "ref_orf.npz"))
    got = np.array(orf.correlated_basis(z["locs"], 6))
    assert got.shape == (49, 9, 9)
    assert np.max(np.abs(got - z["basis_l6"])) < 1e-10
    assert np.median(np.abs(got - z["basis_l6"])) < 1e-15
    for k in range(49):
        assert np.array_equal(got[k], got[k].T)


def test_shard_bounds_cover_everything():
    from pta_replicator_b200.distributed import shard_bounds
    for nreal in (0, 1, 3, 4, 1000, 100000, 1003):
        for world in (1, 2, 3, 8):
            got = [shard_bounds(nreal, world, r) for r in range(world)]
            pos = 0
            for s, c in got:
                assert s == pos or c == 0
                assert s % 4 == 0 or c == 0
                pos = s + c if c else pos
            assert sum(c for _, c in got) == nreal


def test_population_partition_matches_the_reference_function():
    """SURVEY.md 8f row f2: the realization-independent half of add_gwb_plus_outlier_cws (deterministic.py:616-689)
    against the arrays the unmodified reference returned (tests/golden/ref_outliers.npz; holodeck helpers stood in by
    the same published formulas on both sides, see population.py)."""
    import os

    from pta_replicator_b200.population import partition_population, z_to_dcom
    from tests import fixtures as fx
    z = np.load(os.path.join(fx.GOLD, "ref_outliers.npz"))
    vals, weights, fobs, T_obs = fx.outlier_population()
    f_centers, free_spec, o_fo, o_hs, o_mc, o_dl = partition_population(vals, weights, fobs, T_obs, outlier_per_bin=3)
    for got, key in ((f_centers, "f_centers"), (free_spec, "free_spec"), (o_fo, "outlier_fo"), (o_hs, "outlier_hs"),
                     (o_mc, "outlier_mc"), (o_dl, "outlier_dl")):
        assert np.array_equal(got, z[key]), key
    # per bin the kept sources are the loudest, in descending order
    assert all(np.all(np.diff(o_hs[3 * k:3 * k + 3]) <= 0) for k in range(6))
    # fewer members than slots: empty slots are dropped, nothing is left for the free spectrum
    f2, fs2, fo2, hs2, _, _ = partition_population(vals[:, :5], weights[:5], fobs, T_obs, outlier_per_bin=3)
    assert len(fo2) == 5 and np.all(fs2 == 1e-100)
    # comoving distance: Hubble law at low z, monotonic, ~ 3.3 Gpc at z = 1 for this cosmology
    d = z_to_dcom(np.array([1e-3, 0.5, 1.0]))
    mpc = 3.0856775814913674e24
    assert abs(d[0] / mpc - 1e-3 * 2.99792458e5 / 69.32) < 2e-3 and d[0] < d[1] < d[2] and 3200 < d[2] / mpc < 3500


def test_radix256_digit_slices_of_the_tensor_core_synthesis():
    """engine.PulsarBatch.radix256_digits (the host restatement of the digit slicing in csrc/ptar_gwb_i8.cuh): six signed
    int8 digits reproduce round(x 2^48) exactly for |x| <= 1/4, digits stay in [-128, 127], |x| > 1/4 is refused."""
    from pta_replicator_b200.engine import PulsarBatch
    rng = np.random.default_rng(12)
    x = np.r_[rng.uniform(-0.25, 0.25, 4000), 0.25, -0.25, 0.0, 2.0 ** -48, -2.0 ** -49, 127 / 256 * 0.5]
    d = PulsarBatch.radix256_digits(x)
    assert d.dtype == np.int8 and d.shape == (6, len(x))
    rec = sum(d[s].astype(np.int64) * 256 ** (5 - s) for s in range(6))
    assert np.array_equal(rec, np.rint(x * 2.0 ** 48).astype(np.int64))
    assert np.abs(rec * 2.0 ** -48 - x).max() <= 2.0 ** -49
    with pytest.raises(ValueError):
        PulsarBatch.radix256_digits(np.array([0.6]))
