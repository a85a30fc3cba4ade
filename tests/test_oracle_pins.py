"""CPU: pin the oracle (oracle/blah2_oracle.py).

Three anchors, strongest first:
  1. the reference's own known-answer tests (TestHammingNumber.cpp:15-17,
     TestAmbiguity.cpp:87-92,110-115);
  2. committed golden fixtures produced by the reference's UNMODIFIED sources
     (tests/golden/*.npz, made by oracle/gen_golden.py from oracle/_ref);
  3. the reference's outputs on more inputs (tests/golden/live_ref.npz, made by oracle/gen_golden_live.py from
     oracle/_ref), and live comparisons on those inputs when oracle/_ref/libblah2ref.so is present.
"""
import ctypes as C
import os

import numpy as np
import pytest

from blah2_b200.scene import make_scene, random_iq, Target
from oracle import blah2_oracle as O
from oracle import refpath as R
from oracle.fixture import errors as fixture_errors

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
# the FFT shim the reference library is linked with, built alone (no reference sources needed) by `make -C oracle shim`
SHIM_PATH = os.path.join(os.path.dirname(R.LIB_PATH), "libfftshim.so")


def gold(name):
    return np.load(os.path.join(GOLD, name + ".npz"))


# ---- 1. reference known answers ------------------------------------------------------
def test_next_hamming_known_answers():
    assert O.next_hamming(104) == 108 and O.next_hamming(3322) == 3375 and O.next_hamming(19043) == 19200


def test_constructor_known_answers():
    g = O.ambiguity_geometry(-10, 300, -300, 300, 2000000, 1000000)
    assert (g.nCorr, g.nDelayBins, g.nDopplerBins, g.nfft, g.dopplerMiddle) == (3322, 311, 301, 6643, 0)
    assert abs(g.cpi - 0.5) < 0.02
    assert O.ambiguity_geometry(-10, 300, -300, 300, 2000000, 1000000, True).nfft == 6750


def test_survey_geometry_table():
    # SURVEY.md s8 size table (BASELINE configs)
    rows = {(0, 299, -128, 128, 2000000, 2000000): (300, 257, 7782, 15625),
            (0, 511, -256, 256, 10000000, 20000000): (512, 1025, 19512, 39366),
            (0, 511, -512, 512, 10000000, 10000000): (512, 1025, 9756, 19683),
            (0, 511, -512, 512, 20000000, 80000000): (512, 4097, 19526, 39366)}
    for k, v in rows.items():
        g = O.ambiguity_geometry(*k, True)
        assert (g.nDelayBins, g.nDopplerBins, g.nCorr, g.nfft) == v


# ---- 2. golden fixtures ----------------------------------------------------------------
def test_golden_hamming():
    d = gold("hamming")
    for v, n in zip(d["value"], d["next"]):
        assert O.next_hamming(int(v)) == int(n)


def test_golden_geometry():
    for row in gold("geometry")["rows"]:
        g = O.ambiguity_geometry(*[int(v) for v in row[:6]], bool(row[6]))
        assert (g.nDelayBins, g.nDopplerBins, g.nCorr, g.nfft) == tuple(int(v) for v in row[7:11])
        assert g.cpi == row[11] and g.dopplerMiddle == row[12]


@pytest.mark.parametrize("name", ["caf_a", "caf_b", "caf_c"])
def test_golden_ambiguity(name, relerr):
    d = gold(name)
    geom = tuple(int(v) for v in d["geom"][:6]) + (bool(d["geom"][6]),)
    x, y = random_iq(geom[5], int(d["seed"]))
    g = O.ambiguity_geometry(*geom)
    m, lx, ly = O.ambiguity_process(x, y, g)
    assert relerr(m, d["map"])[0] < 1e-12
    assert np.array_equal(g.delay, d["delay"]) and np.array_equal(g.doppler, d["doppler"])
    assert (lx, ly) == tuple(int(v) for v in d["leftover"])
    noise, mx = O.set_metrics(m)
    assert abs(noise - d["metrics"][0]) < 1e-9 and abs(mx - d["metrics"][1]) < 1e-9
    # the FFT-free statement agrees too
    Rd = O.range_matrix_direct(O.ambiguity_prerotate(np.asarray(x, np.complex128), g), np.asarray(y, np.complex128), g)
    assert relerr(O.doppler_transform(Rd, g), d["map"])[0] < 1e-12


@pytest.mark.parametrize("name", ["wh_a", "wh_b"])
def test_golden_wienerhopf(name, relerr):
    d = gold(name)
    n, dm, dM, seed = (int(v) for v in d["params"])
    sc = make_scene(n, 2e6, seed=seed, targets=[Target(25, 300.0, -40.0)])
    ok, y = O.wienerhopf_process(sc.x, sc.y, dm, dM)
    assert ok == bool(d["ok"])
    assert relerr(y, d["y"])[0] < 1e-10


def test_golden_chain(relerr):
    d = gold("chain_a")
    geom = tuple(int(v) for v in d["geom"][:6]) + (bool(d["geom"][6]),)
    pfa, nGuard, nTrain, minDelay, minDoppler, nCentroid = d["det"]
    det = dict(pfa=float(pfa), nGuard=int(nGuard), nTrain=int(nTrain), minDelay=int(minDelay),
               minDoppler=float(minDoppler), nCentroid=int(nCentroid))
    sc = make_scene(geom[5], geom[4], seed=int(d["seed"]), targets=[Target(17, 300.0, -25.0), Target(41, -200.0, -28.0)])
    g = O.ambiguity_geometry(*geom)
    out = O.chain(sc.x, sc.y, g, clutter=tuple(int(v) for v in d["clutter"]), det=det)
    assert relerr(out["map"], d["map"])[0] < 1e-10
    # stage by stage on the REFERENCE map: bit-exact positions, snr to 1e-9 dB
    m, noise = d["map"], float(d["metrics"][0])
    d1 = O.cfar_1d(m, d["delay"], d["doppler"], noise, det["pfa"], det["nGuard"], det["nTrain"], det["minDelay"],
                   det["minDoppler"])
    assert np.array_equal(np.array(d1)[:2], d["cfar"][:2]) and np.allclose(d1[2], d["cfar"][2], atol=1e-9, rtol=0)
    d2 = O.centroid(*d["cfar"], det["nCentroid"], det["nCentroid"], 1.0 / (geom[5] / geom[4]))
    assert np.array_equal(np.array(d2), d["centroid"])
    d3 = O.interpolate(*d["centroid"], m, d["delay"], d["doppler"], noise, True, True)
    assert np.allclose(np.array(d3), d["interp"], atol=1e-9, rtol=0)
    assert len(d3[0]) >= 2


# ---- 3. against the compiled reference: its stored outputs, and live where it is built -----------
@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 7, 8, 12, 15, 60, 64, 73, 97, 100, 127, 131, 243, 257, 400, 625, 1001,
                               4096, 6643, 6750, 15625])
def test_fft_shim_matches_numpy(n):
    lib = C.CDLL(SHIM_PATH, mode=os.RTLD_LOCAL)
    rng = np.random.default_rng(n)
    x = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    for sign, ref in ((-1, np.fft.fft(x)), (+1, np.fft.ifft(x) * n)):
        out = np.empty(n, dtype=np.complex128)
        lib.b200dd_shim_fft(C.c_int(n), x.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p), C.c_int(sign))
        assert np.max(np.abs(out - ref)) <= 5e-13 * max(1.0, np.max(np.abs(ref)))


def test_live_ambiguity_unit_test_geometry(relerr):
    geom = (-10, 300, -300, 300, 2000000, 1000000, True)
    x, y = random_iq(geom[5], 4)
    g = O.ambiguity_geometry(*geom)
    m, lx, ly = O.ambiguity_process(x, y, g)
    d = gold("live_ref")
    assert max(fixture_errors(m, d, "amb_map")) < 1e-12
    assert (lx, ly) == tuple(int(v) for v in d["amb_leftover"])
    assert d["amb_metrics"][1] > 0 and d["amb_metrics"][0] > 0      # Process_Simple, TestAmbiguity.cpp:142-143
    if R.available():
        r = R.ambiguity_process(x, y, *geom)
        assert relerr(m, r["map"])[0] < 1e-12
        assert (lx, ly) == r["leftover"]
        assert r["maxPower"] > 0 and r["noisePower"] > 0


def test_live_wienerhopf_and_failure(relerr):
    sc = make_scene(30011, 2e6, seed=3, targets=[Target(25, 300.0, -40.0)])
    ok_o, y_o = O.wienerhopf_process(sc.x, sc.y, -10, 40)
    d = gold("live_ref")
    assert bool(d["wh_ok"]) and ok_o and max(fixture_errors(y_o, d, "wh_y")) < 1e-10
    assert not bool(d["wh_fail_ok"])
    assert not O.wienerhopf_process(np.zeros(512), np.ones(512), -2, 10)[0]
    if R.available():
        ok_r, y_r = R.wienerhopf_process(sc.x, sc.y, -10, 40)
        assert ok_r and relerr(y_o, y_r)[0] < 1e-10
        assert not R.wienerhopf_process(np.zeros(512), np.ones(512), -2, 10)[0]


def test_live_detection_quirks():
    # int8 narrowing and the uint16 wrap in Centroid, on a synthetic map
    rng = np.random.default_rng(0)
    m = (rng.standard_normal((41, 60)) + 1j * rng.standard_normal((41, 60))) * 10
    m[20, 30] = 500
    m[5, 3] = 400
    delay = np.arange(-5, 55, dtype=np.int32)
    doppler = (np.arange(41) - 20) * 2.5
    noise, _ = O.set_metrics(m)
    d = gold("live_ref")   # what the compiled reference returns for each call below
    assert abs(noise - float(d["quirk_noise"])) < 1e-12
    for k, (pfa, g_, t_, md, mf) in enumerate([(1e-3, 2, 6, 5, 3.0), (1e-2, 258, 4, 300, 0.0), (1e-2, 1, 3, -128, 0.0),
                                               (1e-3, 0, 0, 0, 0.0)]):
        a = d[f"quirk_cfar{k}"]
        b = O.cfar_1d(m, delay, doppler, noise, pfa, g_, t_, md, mf)
        assert all(np.array_equal(u, v) for u, v in zip(a[:2], b[:2])) and np.allclose(a[2], b[2], atol=1e-12, rtol=0)
    a = d["quirk_cfar2"]   # pfa 1e-2, nGuard 1, nTrain 3, minDelay -128, minDoppler 0
    c1, c2 = d["quirk_centroid"], O.centroid(*a, 6, 6, 2.5)
    assert all(np.array_equal(u, v) for u, v in zip(c1, c2))
    i1 = d["quirk_interp"]
    i2 = O.interpolate(*c1, m, delay, doppler, noise, True, True)
    assert all(np.allclose(u, v, atol=1e-12, rtol=0) for u, v in zip(i1, i2)) and len(i1[0]) == len(i2[0])


def test_live_wienerhopf_positive_delay_min_uint32_wrap(relerr):
    """WienerHopf.cpp:67 subtracts an int32 from a uint32: for delayMin > 0 the first samples
    wrap modulo 2^32, not modulo N.  The oracle must reproduce the reference, not 'fix' it."""
    sc = make_scene(10007, 2e6, seed=5, targets=[Target(25, 300.0, -40.0)])
    ok_o, y_o = O.wienerhopf_process(sc.x, sc.y, 2, 30)
    d = gold("live_ref")
    assert bool(d["wrap_ok"]) == ok_o
    if ok_o:
        assert max(fixture_errors(y_o, d, "wrap_y")) < 1e-10
    if R.available():
        ok_r, y_r = R.wienerhopf_process(sc.x, sc.y, 2, 30)
        assert ok_r == ok_o
        if ok_r:
            assert relerr(y_o, y_r)[0] < 1e-10


# ---- SpectrumAnalyser (src/process/spectrum/SpectrumAnalyser.cpp) ----------------------
def test_spectrum_geometry_like_blah2_cpp():
    # blah2.cpp:198-199: SpectrumAnalyser(nSamples, 2000) -> SpectrumAnalyser.cpp:16-18
    assert O.spectrum_geometry(2000000, 2000.0) == (1000, 2000, 2000000)
    assert O.spectrum_geometry(20000000, 2000.0) == (10000, 2000, 20000000)
    assert O.spectrum_geometry(5003, 97.0) == (51, 98, 4998)       # nfft < n
    assert O.spectrum_geometry(3999, 2000.0) == (1, 3999, 3999)    # decimation 1


@pytest.mark.parametrize("name", ["spectrum_a", "spectrum_b", "spectrum_c", "spectrum_d"])
def test_golden_spectrum(name, relerr):
    d = gold(name)
    n, bw, seed = int(d["params"][0]), float(d["params"][1]), int(d["params"][2])
    x, _ = random_iq(n, seed)
    spec, freq = O.spectrum_process(x, n, bw)
    assert spec.shape == d["spectrum"].shape
    assert relerr(spec, d["spectrum"])[0] < 1e-13
    # the reference's uint32_t loop counter leaves the frequency vector EMPTY (SpectrumAnalyser.cpp:34,64)
    assert d["frequency"].shape == (0,) and freq.shape == (0,)
    assert int(d["leftover"]) == n     # process() reads the FIFO, it does not consume it


def test_live_spectrum_vs_reference():
    d = gold("live_ref")
    for k, (n, bw, seed) in enumerate([(4000, 100.0, 5), (10000, 2500.0, 6), (7777, 1234.5, 7)]):
        assert np.array_equal(d[f"spec{k}_params"], [n, bw, seed])
        x, _ = random_iq(n, seed)
        s, f, left = d[f"spec{k}_s"], d[f"spec{k}_f"], int(d[f"spec{k}_left"])
        so, fo = O.spectrum_process(x, n, bw)
        assert s.shape == so.shape and f.shape == fo.shape == (0,) and left == n
        assert np.max(np.abs(s - so)) / np.max(np.abs(s)) < 1e-13


@pytest.mark.parametrize("name", ["wh_a", "wh_b"])
def test_golden_wienerhopf_against_lapack_cholesky(name, relerr):
    """VERDICT r1, weak point 2: the compiled reference's linear algebra comes from oracle/shim/armadillo (Armadillo /
    LAPACK are absent from the image).  Cross-check the golden WienerHopf outputs -- produced by the reference's
    source + that shim -- against an INDEPENDENT solve of the same Hermitian Toeplitz systems by LAPACK's zpotrf /
    zpotrs (scipy cho_factor / cho_solve, the routines Armadillo itself calls) and by numpy's general solver."""
    import scipy.linalg as sla
    d = gold(name)
    n, dm, dM, seed = (int(v) for v in d["params"])
    sc = make_scene(n, 2e6, seed=seed, targets=[Target(25, 300.0, -40.0)])
    ok, w, a, b, xs = O.wienerhopf_weights(sc.x, sc.y, dm, dM)
    assert ok == bool(d["ok"])
    nb = dM - dm
    ii, jj = np.meshgrid(np.arange(nb), np.arange(nb), indexing="ij")
    A = a[np.abs(ii - jj)]
    A = np.where(ii > jj, np.conj(A), A)                    # WienerHopf.cpp:85-97
    assert np.allclose(A, A.conj().T, rtol=0, atol=1e-9 * abs(a[0]))
    w_lapack = sla.cho_solve(sla.cho_factor(A, lower=False), b)
    w_lu = np.linalg.solve(A, b)
    assert relerr(w_lapack, w)[0] < 1e-10 and relerr(w_lu, w)[0] < 1e-9
    y = O.wienerhopf_apply(xs, sc.y, w_lapack)
    assert relerr(y, d["y"])[0] < 1e-9                       # the fixture: reference source + shim Cholesky
    # the residual of the normal equations, the statement that does not depend on any factorisation
    assert np.linalg.norm(A @ w - b) / np.linalg.norm(b) < 1e-10
