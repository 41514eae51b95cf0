"""CPU tests of the pieces around the hot path that round 1 left untested or unpinned (VERDICT round 1):
write_partim / read_tim round trip, simulate_pulsar, the ELONG/ELAT conversion against catalogued positions,
the PINT bridge wiring (against the astropy / PINT stand-ins of the stub harness; the real-PINT test skips with a
reason), the oracle's Fourier-matrix options and the oracle on the reference's real NANOGrav files."""
import os
import sys

import numpy as np
import pytest

from oracle import refnumpy as O
from tests.fixtures import GOLD


# ------------------------------------------------------------------------------------------ writers / simulate_pulsar
def test_write_partim_round_trip(tmp_path):
    """simulate.py:71-77: the shifted TOAs written by write_partim read back bit for bit (long-double MJDs, errors to
    1e-5 us, every flag), and the par file is carried through."""
    import pta_replicator_b200 as P
    from pta_replicator_b200 import partim
    par = os.path.join(GOLD, "partim_small", "par", sorted(os.listdir(os.path.join(GOLD, "partim_small", "par")))[0])
    tim = os.path.join(GOLD, "partim_small", "tim", sorted(os.listdir(os.path.join(GOLD, "partim_small", "tim")))[0])
    psr = P.load_pulsar(par, tim)
    P.make_ideal(psr)
    rng = np.random.default_rng(1)
    shift = rng.normal(0, 1e-6, psr.toas.ntoas)
    psr.toas.adjust_TOAs(shift)                      # seconds, like TimeDelta
    psr.toas.table["flags"][3]["be"] = "GUPPI"
    outpar, outtim = str(tmp_path / "o.par"), str(tmp_path / "o.tim")
    psr.write_partim(outpar, outtim, tempo2=True)
    back = partim.read_tim(outtim)
    assert np.array_equal(np.asarray(back["mjd"], np.longdouble), np.asarray(psr.toas.table["tdbld"], np.longdouble))
    assert np.allclose(back["err_us"], psr.toas.err_us, rtol=0, atol=1e-5)
    assert back["flags"] == [dict(f) for f in psr.toas.table["flags"]]
    assert back["site"] == list(psr.toas.site) and np.allclose(back["freq"], psr.toas.freq)
    assert partim.read_par(outpar)["_name"] == psr.name
    again = P.load_pulsar(outpar, outtim)
    assert again.name == psr.name and again.loc == psr.loc and again.toas.ntoas == psr.toas.ntoas


def test_simulate_pulsar_from_a_par_file():
    """simulate.py:98-135: fake TOAs at given MJDs; scalar or per-TOA errors / frequencies; flags; missing file."""
    import pta_replicator_b200 as P
    par = os.path.join(GOLD, "partim_small", "par", sorted(os.listdir(os.path.join(GOLD, "partim_small", "par")))[1])
    mjd = np.linspace(53000, 57000, 50)
    psr = P.simulate_pulsar(par, mjd, 0.5, freq=1440.0, observatory="AXIS", flags={"f": "sim", "pta": "X"})
    assert psr.toas.ntoas == 50 and psr.name.startswith("JPSR") and set(psr.loc) == {"RAJ", "DECJ"}
    assert np.allclose(psr.toas.get_errors().to("s").value, 0.5e-6) and np.allclose(psr.toas.get_mjds().value, mjd)
    assert psr.toas.table["flags"][7] == {"f": "sim", "pta": "X"} and psr.added_signals is None
    err = np.linspace(0.1, 1.0, 50)
    psr2 = P.simulate_pulsar(par, mjd, err, freq=np.full(50, 820.0))
    assert np.allclose(psr2.toas.get_errors().to("us").value, err)
    with pytest.raises(ValueError, match="make_ideal"):
        psr.update_added_signals("x", {})
    P.make_ideal(psr)
    psr.update_added_signals("x", {})
    with pytest.raises(FileNotFoundError):
        P.simulate_pulsar("/nonexistent.par", mjd, 1.0)


# ------------------------------------------------------------------------------------------ ELONG / ELAT
def _sep_arcsec(ra1, dec1, ra2, dec2):
    c = np.sin(dec1) * np.sin(dec2) + np.cos(dec1) * np.cos(dec2) * np.cos(ra1 - ra2)
    return float(np.degrees(np.arccos(np.clip(c, -1, 1))) * 3600)


def _hms(h, m, s):
    return (h + m / 60 + s / 3600) * np.pi / 12


def _dms(sign, d, m, s):
    return sign * (d + m / 60 + s / 3600) * np.pi / 180


REAL3 = {   # ELONG / ELAT of the reference's real NG15 par files (test_partim/par/*.par:19-20), catalogued J2000 and B1950 positions
    "B1855+09": dict(ecl=(286.863485782621126, 32.321482985635249), j2000=(_hms(18, 57, 36.3906), _dms(+1, 9, 43, 17.207)),
                     b1950=(_hms(18, 55, 13.7), _dms(+1, 9, 39, 13.0))),
    "B1937+21": dict(ecl=(301.973244484302029, 42.296752077547630), j2000=(_hms(19, 39, 38.5612), _dms(+1, 21, 34, 59.126)),
                     b1950=(_hms(19, 37, 28.72), _dms(+1, 21, 28, 1.3))),
    "J1909-3744": dict(ecl=(284.220845879968067, -15.155533209547460), j2000=(_hms(19, 9, 47.4336), _dms(-1, 37, 44, 14.516)),
                       b1950=None),
}


def test_ecliptic_positions_against_catalogued_coordinates():
    """red_noise.py:210-221 / deterministic.py:79-88 call PyEphem (absent here): ``Equatorial(Ecliptic(str(ELONG),
    str(ELAT)), epoch='1950' if 'B' in name else '2000')``.  Pinned to what that call must return: the catalogued J2000
    positions of the three real pulsars to 0.5 arcsec (proper motion between position epochs is ~0.2 arcsec), the
    catalogued B1950 positions (from which the B names derive) to 3 arcsec for the epoch-1950 quirk, and the B-name
    digits themselves (hhmm, +-dd of the 1950 position)."""
    from pta_replicator_b200 import orf
    for name, d in REAL3.items():
        ra, dec = orf.ecliptic_to_equatorial(*d["ecl"], "2000")
        assert _sep_arcsec(ra, dec, *d["j2000"]) < 0.5, (name, _sep_arcsec(ra, dec, *d["j2000"]))
        if d["b1950"] is not None:
            ra, dec = orf.ecliptic_to_equatorial(*d["ecl"], "1950")
            assert _sep_arcsec(ra, dec, *d["b1950"]) < 3.0, (name, _sep_arcsec(ra, dec, *d["b1950"]))
            hh, mm = int(ra * 12 / np.pi), int((ra * 12 / np.pi % 1) * 60)
            assert f"B{hh:02d}{mm:02d}{'+' if dec >= 0 else '-'}{int(abs(np.degrees(dec))):02d}" == name

    class P:   # psrlocs_from_pulsars applies the B-name rule of the reference
        def __init__(self, name, loc):
            self.name, self.loc = name, loc
    locs = orf.psrlocs_from_pulsars([P(n, {"ELONG": d["ecl"][0], "ELAT": d["ecl"][1]}) for n, d in REAL3.items()])
    assert _sep_arcsec(locs[0, 0], locs[0, 1], *REAL3["B1855+09"]["b1950"]) < 3.0
    assert _sep_arcsec(locs[2, 0], locs[2, 1], *REAL3["J1909-3744"]["j2000"]) < 0.5


# ------------------------------------------------------------------------------------------ PINT bridge
def test_pint_bridge_without_pint_raises_with_a_reason():
    from pta_replicator_b200 import pint_bridge
    import pta_replicator_b200 as P
    if pint_bridge.have_pint():
        pytest.skip("PINT is installed: the unavailable-path test does not apply")
    psr = P.pulsar_from_arrays("J0000+00", {"RAJ": 1.0, "DECJ": 2.0}, np.linspace(53000, 54000, 5).astype(np.longdouble), np.ones(5))
    for call in (lambda: psr.fit(), lambda: psr.to_enterprise(), lambda: pint_bridge.load_pulsar_pint(__file__, __file__)):
        with pytest.raises(pint_bridge.PintUnavailable):
            call()


def test_pint_bridge_applies_delays_through_the_pint_api():
    """``apply_delay`` / ``apply_realization`` do what every ``add_*`` of the reference does with its dt
    (white_noise.py:111-125): ledger entry with a Quantity in seconds, ``toas.adjust_TOAs(TimeDelta(dt))``,
    ``update_residuals()``.  Run against the astropy / PINT stand-ins of the stub harness (oracle/refstubs.py) in a
    subprocess-free way: the stand-ins are installed only if the real packages are absent."""
    from oracle import refstubs
    from pta_replicator_b200 import pint_bridge
    saved = {k: sys.modules.get(k) for k in ("astropy", "astropy.units", "astropy.time")}
    try:
        if not pint_bridge.have_pint():
            refstubs._module("astropy.units", s=refstubs._Unit("s"), day=refstubs._Unit("day"), us=refstubs._Unit("us"),
                             Quantity=refstubs._Quantity)
            refstubs._module("astropy.time", TimeDelta=refstubs._TimeDelta)
            refstubs._module("astropy", units=sys.modules["astropy.units"], time=sys.modules["astropy.time"])
        mjd = np.linspace(53000, 54000, 11).astype(np.longdouble)
        psrs = [refstubs.StubPulsar(f"J000{i}+00", {"RAJ": 1.0 + i, "DECJ": 2.0}, mjd[::-1].copy() if i else mjd, np.ones(11),
                                    [{"f": "x"}] * 11, freeze_toas=False) for i in range(2)]

        class FakeBatch:       # unpack() contract of PulsarBatch: engine order (time-sorted) -> table order
            ld = 24
            order = [np.argsort(np.asarray(p.toas.table["tdbld"], float), kind="stable") for p in psrs]

            def unpack(self, row, i):
                out = np.empty(11)
                out[self.order[i]] = row[12 * i:12 * i + 11]
                return out
        row = np.arange(24, dtype=float) * 1e-7
        pint_bridge.apply_realization(FakeBatch(), psrs, row, "b200_batch", {"seed": 3})
        for i, p in enumerate(psrs):
            want = FakeBatch().unpack(row, i)
            assert np.allclose(p.toas.delta, want, rtol=0, atol=1e-20)
            assert np.allclose(p.signal_seconds(f"{p.name}_b200_batch"), want) and p.added_signals[f"{p.name}_b200_batch"] == {"seed": 3}
            shifted = np.asarray(p.toas.table["tdbld"] - p.toas.mjd0, float) * 86400
            assert np.allclose(shifted, want, atol=2e-9)          # MJD long-double resolution
        with pytest.raises(ValueError, match="already exists"):
            pint_bridge.apply_delay(psrs[0], np.zeros(11), f"{psrs[0].name}_b200_batch")
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def test_pint_bridge_with_real_pint():
    from pta_replicator_b200 import pint_bridge
    if not pint_bridge.have_pint():
        pytest.skip("pint-pulsar / astropy are not installed in this image (no network): the real-PINT round trip cannot run here")
    par = os.path.join(GOLD, "partim_small", "par", sorted(os.listdir(os.path.join(GOLD, "partim_small", "par")))[0])
    tim = os.path.join(GOLD, "partim_small", "tim", sorted(os.listdir(os.path.join(GOLD, "partim_small", "tim")))[0])
    psr = pint_bridge.load_pulsar_pint(par, tim)
    pint_bridge.make_ideal_pint(psr)
    before = np.asarray(psr.toas.get_mjds().value, float)
    pint_bridge.apply_delay(psr, np.full(psr.toas.ntoas, 1e-6), f"{psr.name}_test")
    assert np.allclose((np.asarray(psr.toas.get_mjds().value, float) - before) * 86400, 1e-6, atol=2e-7)


# ------------------------------------------------------------------------------------------ oracle pins
def test_oracle_fourier_matrix_options_against_the_unmodified_reference():
    """pshift (phases drawn from the global legacy stream at red_noise.py:83), logf / fmin / fmax, Tspan."""
    z = np.load(os.path.join(GOLD, "ref_fourier.npz"))
    t = z["t"]
    np.random.seed(4242)
    F, f = O.fourier_basis(t, nmodes=20, ranphase=np.random.uniform(0.0, 2 * np.pi, 20))
    assert np.array_equal(f, z["f_pshift"]) and np.max(np.abs(F - z["F_pshift"])) < 1e-15
    np.random.seed(4243)
    F, _ = O.fourier_basis(t, nmodes=20, ranphase=np.random.uniform(0.0, 2 * np.pi, 20), libstempo_convention=True)
    assert np.max(np.abs(F - z["F_pshift_ls"])) < 1e-15
    F, f = O.fourier_basis(t, nmodes=20, logf=True, fmin=2e-9, fmax=3e-7)
    assert np.array_equal(f, z["f_logf"]) and np.max(np.abs(F - z["F_logf"])) < 1e-15
    F, f = O.fourier_basis(t, nmodes=20, fmin=2e-9, fmax=3e-7)
    assert np.array_equal(f, z["f_lin"]) and np.max(np.abs(F - z["F_lin"])) < 1e-15
    F, f = O.fourier_basis(t, nmodes=20, Tspan=6.0e8)
    assert np.array_equal(f, z["f_tspan"]) and np.max(np.abs(F - z["F_tspan"])) < 1e-15


def real3_pulsars():
    """(specs, npz) of tests/golden/ref_real3.npz: the reference's real NG15 TOAs (unsorted, 7.8k / 23k / 35k)."""
    from pta_replicator_b200 import noise_dict as nd
    z = np.load(os.path.join(GOLD, "ref_real3.npz"))
    noise = nd.load_noise_dict()
    out = []
    for i in range(3):
        name = str(z[f"name_{i}"])
        be = [str(s) for s in z[f"backends_{i}"]]
        mjd = z[f"mjd_hi_{i}"].astype(np.longdouble) + z[f"mjd_lo_{i}"].astype(np.longdouble)
        out.append(dict(name=name, loc={"ELONG": float(z[f"elong_elat_{i}"][0]), "ELAT": float(z[f"elong_elat_{i}"][1])}, mjd=mjd,
                        err_us=z[f"err_us_{i}"].astype(np.float64), flag=[be[k] for k in z[f"flag_idx_{i}"]],
                        pp=nd.per_pulsar(noise, name)))
    return out, z


def test_oracle_on_the_real_ng15_files():
    """Bucket counts of quantize_fast (360 / 629 / 831 at 1 s, 147 / 446 / 566 at 0.1 d) and every 40th TOA of the
    unmodified white / ECORR / red-noise injections with the 15-yr noise dictionary, same legacy seeds."""
    spec, z = real3_pulsars()
    for i, s in enumerate(spec):
        n, pp = len(s["mjd"]), s["pp"]
        mjd = np.asarray(s["mjd"], dtype=float)
        assert [str(x) for x in z[f"dict_backends_{i}"]] == list(pp["backends"])
        for tag, width in (("1s", 1.0 / 86400.0), ("0p1d", 0.1)):
            bk, firsts = O.epoch_buckets(mjd, width)
            assert len(firsts) == int(z[f"nbucket_{tag}_{i}"])
        flag = np.array(s["flag"])
        ef = O.per_toa_params(pp["efac"], pp["backends"], flag, n)
        eq = O.per_toa_params(10 ** np.asarray(pp["log10_equad"]), pp["backends"], flag, n)
        z1, z2 = O.legacy_randn(10660 + i, n, n)
        wn = O.white_noise(s["err_us"] * 1e-6, ef, eq, z1, z2)
        assert np.max(np.abs(wn[::40] - z[f"measurement_noise_{i}"])) < 1e-14 * np.sqrt(np.mean(wn ** 2)) + 1e-30
        bk, firsts = O.epoch_buckets(mjd, 1.0 / 86400.0)
        ec = O.ecorr_per_bucket(10 ** np.asarray(pp["log10_ecorr"]), pp["backends"], flag, firsts)
        (zb,) = O.legacy_randn(17763 + i, len(firsts))
        jit = O.jitter(bk, ec, zb)
        assert np.max(np.abs(jit[::40] - z[f"jitter_{i}"])) < 1e-14 * np.sqrt(np.mean(jit ** 2)) + 1e-30
        (zr,) = O.legacy_randn(19870 + i, 60)
        rn = O.red_noise(mjd, pp["rn_log10_A"], pp["rn_gamma"], zr)
        assert np.max(np.abs(rn[::40] - z[f"red_noise_{i}"])) < 1e-12 * np.sqrt(np.mean(rn ** 2))


def test_unmodified_reference_recipe_equals_the_port():
    """oracle/refrecipe.py (the UNMODIFIED functions under the stub harness: the CPU arm of bench.py) and
    oracle/recipe.py (the numpy port) produce the same realization from the same seeds, 8 pulsars of ng15-full.
    The reference's side is tests/golden/ref_recipe8.npz (oracle/make_golden.py: every 4th TOA and the rms)."""
    from oracle import recipe
    from pta_replicator_b200 import synthetic
    z = np.load(os.path.join(GOLD, "ref_recipe8.npz"))
    psrs, noise = synthetic.make_ng15_like("full", npsr=int(z["npsr"]))
    b = recipe.realization(recipe.dataset_from_pulsars(psrs, noise), int(z["seed"]))
    k = int(z["stride"])
    assert [len(y) for y in b] == [int(z[f"ntoa_{i}"]) for i in range(len(b))]
    worst = max(np.max(np.abs(z[f"delay_{i}"] - y[::k])) / np.sqrt(np.mean(y * y)) for i, y in enumerate(b))
    assert worst < 1e-13, worst
    assert max(abs(float(z[f"rms_{i}"]) / np.sqrt(np.mean(y * y)) - 1.0) for i, y in enumerate(b)) < 1e-13
