"""GPU: the C++ drop-in classes (blah2_b200/dropin, same names/signatures as the reference's
src/process classes) driven through the SAME harness source as the reference
(oracle/ref_capi.cpp compiled unchanged against our headers -> oracle/_ref/libdropin_harness.so), compared
with the reference's stored outputs (tests/golden/dropin_ref.npz, oracle/gen_golden_live.py) and with the
reference library (oracle/_ref) or, where that is absent, the numpy oracle."""
import importlib.util
import os

import numpy as np
import pytest

from blah2_b200.scene import make_scene, random_iq, Target
from oracle import blah2_oracle as O
from oracle import refpath as R
from oracle.fixture import errors as fixture_errors

pytestmark = pytest.mark.gpu

HARNESS = os.path.join(os.path.dirname(R.LIB_PATH), "libdropin_harness.so")
GEOMS = [(-10, 300, -300, 300, 2000000, 1000000, True),   # Process_Simple geometry
         (0, 31, -20, 60, 10000, 5000, True)]             # off-centre Doppler window


@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "dropin_ref.npz"))


@pytest.fixture(scope="module")
def D():
    """A second instance of the refpath binding, pointed at the drop-in harness."""
    if not os.path.exists(HARNESS):
        pytest.fail(f"{HARNESS} missing: run `make -C oracle dropin` where the blah2 sources are")
    spec = importlib.util.spec_from_file_location("dropin_binding", R.__file__)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.LIB_PATH = HARNESS
    return mod


def test_constructor_getters_like_testambiguity_cpp(D):
    g = D.ambiguity_geometry(-10, 300, -300, 300, 2000000, 1000000, False)   # TestAmbiguity.cpp:73-93
    assert (g["nCorr"], g["nDelayBins"], g["nDopplerBins"], g["nfft"], g["dopplerMiddle"]) == (3322, 311, 301, 6643, 0)
    assert abs(g["cpi"] - 0.5) < 0.02
    assert D.ambiguity_geometry(-10, 300, -300, 300, 2000000, 1000000, True)["nfft"] == 6750
    assert D.next_hamming(104) == 108 and D.next_hamming(3322) == 3375 and D.next_hamming(19043) == 19200


@pytest.mark.parametrize("geom", GEOMS)
def test_ambiguity_class_matches_reference_class(D, geom, relerr, gold):
    x, y = random_iq(geom[5], 21)
    d = D.ambiguity_process(x, y, *geom)
    k = GEOMS.index(geom)
    e = fixture_errors(d["map"], gold, f"amb{k}_map")
    assert max(e) < 1e-5, e
    assert d["leftover"] == tuple(int(v) for v in gold[f"amb{k}_leftover"])
    assert np.max(np.abs(np.array([d["noisePower"], d["maxPower"]]) - gold[f"amb{k}_metrics"])) < 1e-3
    if R.available():
        r = R.ambiguity_process(x, y, *geom)
        ref_map, left, noise, mx = r["map"], r["leftover"], r["noisePower"], r["maxPower"]
    else:
        g = O.ambiguity_geometry(*geom)
        ref_map, lx, ly = O.ambiguity_process(x, y, g)
        left = (lx, ly)
        noise, mx = O.set_metrics(ref_map)
    e = relerr(d["map"], ref_map)
    assert e[0] < 1e-5 and e[1] < 1e-5, e
    assert d["leftover"] == left                      # the FIFOs are consumed like the reference's
    assert d["maxPower"] > 0 and d["noisePower"] > 0  # Process_Simple, TestAmbiguity.cpp:142-143
    assert abs(d["noisePower"] - noise) < 1e-3 and abs(d["maxPower"] - mx) < 1e-3


def test_wienerhopf_class_matches_reference_class(D, relerr, gold):
    sc = make_scene(60011, 2e6, seed=4, targets=[Target(25, 300.0, -40.0)])
    ok, y = D.wienerhopf_process(sc.x, sc.y, -10, 60)
    assert ok and bool(gold["wh_ok"]) and max(fixture_errors(y, gold, "wh_y")) < 1e-9
    ok_ref, y_ref = (R.wienerhopf_process if R.available() else O.wienerhopf_process)(sc.x, sc.y, -10, 60)
    assert ok and ok_ref
    assert relerr(y, y_ref)[0] < 1e-9
    ok, y = D.wienerhopf_process(np.zeros(2048), np.ones(2048), -2, 10)   # chol failure -> false, y untouched
    assert not ok and np.array_equal(y, np.ones(2048))


def test_whole_loop_body_with_dropin_classes(D, relerr, gold):
    """src/blah2.cpp:268-287 through the class API: filter -> ambiguity -> set_metrics (the reference's
    own Map code) -> CFAR -> Centroid -> Interpolate."""
    # geometry inside the reference's own valid domain: its Doppler work buffer has nfft entries but the
    # Doppler FFT nDopplerBins points (Ambiguity.cpp:72,79-80), so nDopplerBins <= nfft is required or the
    # reference overflows its heap (found the hard way; the CUDA path has no such limit)
    fs, n = 2000000, 200000
    args = dict(delayMin=-10, delayMax=120, dopplerMin=-1000, dopplerMax=1000, fs=fs, n=n, roundHamming=True,
                clutter=(-10, 60), pfa=1e-5, nGuard=2, nTrain=6, minDelay=5, minDoppler=15.0, nCentroid=6)
    sc = make_scene(n, fs, seed=5, targets=[Target(37, 600.0, -30.0), Target(92, -400.0, -35.0)])
    d = D.Chain(**args).run(sc.x, sc.y)
    assert not d["skipped"]
    e = fixture_errors(d["map"], gold, "chain_map")
    assert max(e) < 1e-5, e
    assert abs(d["noisePower"] - float(gold["chain_metrics"][0])) < 1e-3
    assert len(d["detections"][0]) == gold["chain_detections"].shape[1] >= 2
    for a, b in zip(d["detections"], gold["chain_detections"]):
        assert np.max(np.abs(a - b)) < 1e-2
    if R.available():
        r = R.Chain(**args).run(sc.x, sc.y)
        ref_map, ref_det, noise = r["map"], r["detections"], r["noisePower"]
    else:
        g = O.ambiguity_geometry(-10, 120, -1000, 1000, fs, n, True)
        o = O.chain(sc.x, sc.y, g, clutter=(-10, 60), det=dict(pfa=1e-5, nGuard=2, nTrain=6, minDelay=5,
                                                                  minDoppler=15.0, nCentroid=6))
        ref_map, ref_det, noise = o["map"], o["detections"], o["noisePower"]
    assert not d["skipped"]
    e = relerr(d["map"], ref_map)
    assert e[0] < 1e-5 and e[1] < 1e-5, e
    assert abs(d["noisePower"] - noise) < 1e-3
    assert len(d["detections"][0]) == len(ref_det[0]) >= 2
    for a, b in zip(d["detections"], ref_det):
        assert np.max(np.abs(a - b)) < 1e-2
