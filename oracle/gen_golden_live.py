"""oracle/gen_golden_live.py -- TEST INFRASTRUCTURE ONLY.

Runs the reference's UNMODIFIED sources (oracle/_ref/libblah2ref.so, built by `make -C oracle` where the blah2
sources are) on the inputs of the tests that compare with it live, and stores what those tests compare against:

  tests/golden/live_ref.npz    tests/test_oracle_pins.py  test_live_*
  tests/golden/dropin_ref.npz  tests/test_dropin_gpu.py

Maps and filtered channels are stored as oracle/fixture.py summaries (seeded sample, max-abs, Frobenius norm,
projection); detection lists and spectra whole.

    python oracle/gen_golden_live.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import refpath as R  # noqa: E402
from oracle.fixture import summarise  # noqa: E402
from blah2_b200.scene import make_scene, random_iq, Target  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")

# the synthetic map of test_live_detection_quirks and the (pfa, nGuard, nTrain, minDelay, minDoppler) it runs
QUIRK_CFAR = [(1e-3, 2, 6, 5, 3.0), (1e-2, 258, 4, 300, 0.0), (1e-2, 1, 3, -128, 0.0), (1e-3, 0, 0, 0, 0.0)]


def quirk_map():
    rng = np.random.default_rng(0)
    m = (rng.standard_normal((41, 60)) + 1j * rng.standard_normal((41, 60))) * 10
    m[20, 30] = 500
    m[5, 3] = 400
    return m, np.arange(-5, 55, dtype=np.int32), (np.arange(41) - 20) * 2.5


DROPIN_CHAIN = dict(delayMin=-10, delayMax=120, dopplerMin=-1000, dopplerMax=1000, fs=2000000, n=200000,
                    roundHamming=True, clutter=(-10, 60), pfa=1e-5, nGuard=2, nTrain=6, minDelay=5, minDoppler=15.0,
                    nCentroid=6)
DROPIN_GEOMS = [(-10, 300, -300, 300, 2000000, 1000000, True), (0, 31, -20, 60, 10000, 5000, True)]


def live_ref():
    out = {}
    # test_live_ambiguity_unit_test_geometry
    x, y = random_iq(1000000, 4)
    r = R.ambiguity_process(x, y, -10, 300, -300, 300, 2000000, 1000000, True)
    out.update(summarise("amb_map", r["map"]))
    out["amb_leftover"] = np.array(r["leftover"])
    out["amb_metrics"] = np.array([r["noisePower"], r["maxPower"]])
    # test_live_wienerhopf_and_failure
    sc = make_scene(30011, 2e6, seed=3, targets=[Target(25, 300.0, -40.0)])
    ok, yf = R.wienerhopf_process(sc.x, sc.y, -10, 40)
    out.update(summarise("wh_y", yf))
    out["wh_ok"] = ok
    out["wh_fail_ok"] = R.wienerhopf_process(np.zeros(512), np.ones(512), -2, 10)[0]
    # test_live_detection_quirks
    m, delay, doppler = quirk_map()
    noise = R.set_metrics(m)[0]
    out["quirk_noise"] = noise
    for k, (pfa, g_, t_, md, mf) in enumerate(QUIRK_CFAR):
        out[f"quirk_cfar{k}"] = np.array(R.cfar_1d(m, delay, doppler, noise, pfa, g_, t_, md, mf))
    a = R.cfar_1d(m, delay, doppler, noise, 1e-2, 1, 3, -128, 0.0)
    c = R.centroid(*a, 6, 6, 2.5)
    out["quirk_centroid"] = np.array(c)
    out["quirk_interp"] = np.array(R.interpolate(*c, m, delay, doppler, noise, True, True))
    # test_live_wienerhopf_positive_delay_min_uint32_wrap
    sc = make_scene(10007, 2e6, seed=5, targets=[Target(25, 300.0, -40.0)])
    ok, yf = R.wienerhopf_process(sc.x, sc.y, 2, 30)
    out.update(summarise("wrap_y", yf))
    out["wrap_ok"] = ok
    # test_live_spectrum_vs_reference
    for k, (n, bw, seed) in enumerate([(4000, 100.0, 5), (10000, 2500.0, 6), (7777, 1234.5, 7)]):
        x, _ = random_iq(n, seed)
        s, f, left = R.spectrum_process(x, n, bw)
        out[f"spec{k}_params"] = np.array([n, bw, seed])
        out[f"spec{k}_s"], out[f"spec{k}_f"], out[f"spec{k}_left"] = s, f, left
    return out


def dropin_ref():
    out = {}
    for k, geom in enumerate(DROPIN_GEOMS):   # test_ambiguity_class_matches_reference_class
        x, y = random_iq(geom[5], 21)
        r = R.ambiguity_process(x, y, *geom)
        out.update(summarise(f"amb{k}_map", r["map"]))
        out[f"amb{k}_leftover"] = np.array(r["leftover"])
        out[f"amb{k}_metrics"] = np.array([r["noisePower"], r["maxPower"]])
    # test_wienerhopf_class_matches_reference_class
    sc = make_scene(60011, 2e6, seed=4, targets=[Target(25, 300.0, -40.0)])
    ok, yf = R.wienerhopf_process(sc.x, sc.y, -10, 60)
    out.update(summarise("wh_y", yf))
    out["wh_ok"] = ok
    # test_whole_loop_body_with_dropin_classes
    a = DROPIN_CHAIN
    sc = make_scene(a["n"], a["fs"], seed=5, targets=[Target(37, 600.0, -30.0), Target(92, -400.0, -35.0)])
    r = R.Chain(**a).run(sc.x, sc.y)
    assert not r["skipped"]
    out.update(summarise("chain_map", r["map"]))
    out["chain_metrics"] = np.array([r["noisePower"], r["maxPower"]])
    out["chain_detections"] = np.array(r["detections"])
    return out


def main():
    if not R.available():
        raise SystemExit(f"{R.LIB_PATH} missing: run `make -C oracle` where the blah2 sources are")
    os.makedirs(OUT, exist_ok=True)
    np.savez_compressed(os.path.join(OUT, "live_ref.npz"), **live_ref())
    np.savez_compressed(os.path.join(OUT, "dropin_ref.npz"), **dropin_ref())
    print("golden fixtures written to", OUT)


if __name__ == "__main__":
    main()
