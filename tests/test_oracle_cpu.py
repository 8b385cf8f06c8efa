"""CPU tests (no GPU): the oracles against the live reference pieces available in this image
(cv2.calcOpticalFlowFarneback, cv2.resize/remap/getGaussianKernel) and against ground truth."""
import numpy as np
import cv2
import pytest

from oracle import synth, metrics, tvl1_cpu, tvl1_gpu_model as gm, farneback_gpu_model as fm


def test_level_sizes_match_survey():
    # SURVEY.md §8: 1080p TV-L1 levels (saturate_cast<int> = round half to even)
    sizes, ns = gm.level_sizes(1080, 1920, 5, 0.8)
    assert ns == 5
    assert sizes == [(1080, 1920), (864, 1536), (691, 1229), (553, 983), (442, 786)]
    sizes, ns = gm.level_sizes(2160, 3840, 5, 0.8)
    assert sizes == [(2160, 3840), (1728, 3072), (1382, 2458), (1106, 1966), (885, 1573)]
    # <16 px stop rule (tvl1flow.cpp:243-247)
    sizes, ns = gm.level_sizes(40, 40, 8, 0.5)
    assert ns == 2 and sizes[-1] == (10, 10)


def test_cv_round_half_even():
    assert [gm.cv_round(v) for v in (2.5, 7.5, 67.5, 3.5, -0.5)] == [2, 8, 68, 4, 0]


def test_tvl1_cpu_oracle_recovers_known_flow():
    # criterion of the reference's CPU regression test (test_tvl1optflow.cpp:114-142):
    # >= 95 % of pixels with EPE <= 0.1 -- here against exact synthetic ground truth.
    I0, I1, gt = synth.make_pair(120, 160, seed=0, kind="const")
    P = tvl1_cpu.TVL1Params(warps=5, epsilon=0.0, innerIterations=1, outerIterations=30, medianFiltering=1)
    f = tvl1_cpu.calc(I0, I1, P)
    st = metrics.epe_stats(f, gt, border=16)
    assert st["frac_le_0.1"] >= 0.95 and st["mean"] < 0.05, st


def test_tvl1_cpu_oracle_defaults_with_median_and_early_exit():
    I0, I1, gt = synth.make_pair(96, 128, seed=1, kind="const")
    f = tvl1_cpu.calc(I0, I1, tvl1_cpu.TVL1Params())  # defaults: median 5, eps 0.01, 10 x 30
    st = metrics.epe_stats(f, gt, border=16)
    assert st["frac_le_0.1"] >= 0.95, st


def test_tvl1_cuda_semantics_model_close_to_cpu_oracle():
    # the reference's own GPU-vs-CPU test maps iterations the same way (test_optflow.cpp:456-460)
    I0, I1, gt = synth.make_pair(120, 160, seed=2, kind="affine")
    fc = tvl1_cpu.calc(I0, I1, tvl1_cpu.TVL1Params(warps=5, epsilon=0.0, innerIterations=1, outerIterations=30,
                                                   medianFiltering=1))
    fg = gm.calc(I0, I1, gm.TVL1Params(warps=5, epsilon=0.0, iterations=30))
    st = metrics.epe_stats(fc, fg, border=16)
    assert st["frac_le_0.1"] >= 0.95 and st["mean"] < 0.1, st


def test_tvl1_model_gamma_and_f32_run():
    I0, I1, gt = synth.make_pair(64, 80, seed=3, kind="const", dtype="f32")
    f = gm.calc(I0, I1, gm.TVL1Params(nscales=3, warps=2, epsilon=0.0, iterations=10, gamma=1.0))
    assert np.isfinite(f).all()


def test_tvl1_model_error_cadence_trace():
    I0, I1, _ = synth.make_pair(64, 80, seed=4, kind="const")
    tr = []
    gm.calc(I0, I1, gm.TVL1Params(nscales=2, warps=2, epsilon=0.05, iterations=50), trace=tr)
    # sampled only on odd n -> a warp that exits early stops after an even number of iterations
    for lvl in tr:
        for n in lvl:
            assert n == 50 or n % 2 == 0


@pytest.mark.parametrize("kw,ncc_tol,epe_tol", [
    (dict(), 1e-4, 0.02),                      # box filter: reference tolerance 1e-4 (test_optflow.cpp:341-348)
    (dict(polyN=7, polySigma=1.5, pyrScale=0.8, numLevels=3), 1e-4, 0.02),
    (dict(flags=256), 2e-2, 0.2),              # gaussian: reference tolerance 2e-2
])
def test_farneback_model_vs_live_cv2(kw, ncc_tol, epe_tol):
    I0, I1, gt = synth.make_pair(160, 200, seed=5, kind="smooth")
    f = fm.calc(I0, I1, fm.FarnebackParams(**kw))
    c = cv2.calcOpticalFlowFarneback(I0, I1, None, kw.get("pyrScale", 0.5), kw.get("numLevels", 5), 13, 10,
                                     kw.get("polyN", 5), kw.get("polySigma", 1.1), kw.get("flags", 0))
    assert metrics.ncc_dissimilarity(f, c) <= ncc_tol
    assert metrics.epe_stats(f, c)["mean"] <= epe_tol


def test_farneback_prepare_gaussian_closed_form():
    g, xg, xxg, ig11, ig03, ig33, ig55 = fm.prepare_gaussian(5, 1.1)
    assert abs(float(g[0] + 2 * g[1:].sum()) - 1.0) < 1e-6
    assert ig11 > 0 and ig33 > 0 and ig55 > 0 and ig03 < 0


def test_pyr_down_model_is_cv2():
    a = synth.texture(37, 51, 0)
    d = fm.pyr_down(a)
    assert d.shape == (19, 26)


def test_synth_pair_sign_convention():
    # I0(x) ~= I1(x + flow): cv2 Farneback on a constant shift must recover (+2.5, -1.25)
    I0, I1, gt = synth.make_pair(120, 160, seed=0, kind="const")
    c = cv2.calcOpticalFlowFarneback(I0, I1, None, 0.5, 3, 15, 5, 5, 1.1, 0)
    med = np.median(c[20:-20, 20:-20].reshape(-1, 2), axis=0)
    assert abs(med[0] - 2.5) < 0.2 and abs(med[1] + 1.25) < 0.2


def test_golden_fixtures_pin_the_oracles():
    """tests/golden/farneback_*.npz were produced by the live CPU reference (make_golden.py);
    the cv2 on this box and the CUDA-semantics model must both agree with them."""
    import os
    gold = os.path.join(os.path.dirname(__file__), "golden")
    names = sorted(n for n in os.listdir(gold) if n.startswith("farneback_") and n.endswith(".npz"))
    assert len(names) >= 4
    for n in names:
        z = np.load(os.path.join(gold, n))
        kw = {k[3:]: z[k].item() for k in z.files if k.startswith("kw_")}
        live = cv2.calcOpticalFlowFarneback(z["I0"], z["I1"], None, kw.get("pyrScale", 0.5), kw.get("numLevels", 5),
                                            13, 10, kw.get("polyN", 5), kw.get("polySigma", 1.1), kw.get("flags", 0))
        assert metrics.ncc_dissimilarity(live, z["flow"]) <= 1e-6, n
        model = fm.calc(z["I0"], z["I1"], fm.FarnebackParams(**kw))
        assert metrics.ncc_dissimilarity(model, z["flow"]) <= float(z["ncc_tol"]), n


@pytest.fixture(scope="module")
def native():
    import subprocess, os
    from oracle import tvl1_cpu_native as nat
    if not nat.available():
        subprocess.run(["make", "-C", os.path.dirname(nat.__file__)], check=True)
    return nat


def test_native_port_primitives_pinned_to_cv2(native):
    """oracle/tvl1_cpu.c restates cv::resize(INTER_LINEAR) and cv::remap(INTER_CUBIC); pin both
    against the live cv2 functions (the reference's own external primitives)."""
    rng = np.random.default_rng(0)
    a = synth.texture(211, 307, 3)
    for (dh, dw) in [(169, 246), (264, 384), (211, 307)]:
        r = native.resize_linear(a, dh, dw)
        c = cv2.resize(a, (dw, dh), interpolation=cv2.INTER_LINEAR)
        assert np.abs(r - c).max() <= 1e-4      # <= 2 ulp at 255 (cv2 uses a fused vertical pass)
    ys, xs = np.mgrid[0:211, 0:307].astype(np.float32)
    mx = xs + rng.uniform(-9, 9, xs.shape).astype(np.float32)
    my = ys + rng.uniform(-9, 9, xs.shape).astype(np.float32)
    assert np.array_equal(native.remap_cubic(a, mx, my), cv2.remap(a, mx, my, cv2.INTER_CUBIC))  # bit exact


def test_native_port_agrees_with_numpy_restatement(native):
    I0, I1, gt = synth.make_pair(120, 160, seed=0, kind="smooth")
    P = tvl1_cpu.TVL1Params(nscales=4, warps=5, epsilon=0.0, innerIterations=1, outerIterations=30,
                            medianFiltering=1)
    a, b = tvl1_cpu.calc(I0, I1, P), native.calc(I0, I1, P)
    st = metrics.epe_stats(a, b)
    assert st["mean"] <= 0.01 and st["frac_le_0.1"] >= 0.995, st


# ---- the reference's own CPU TV-L1 source, compiled unmodified (oracle/_ref) ----------------------------
def _golden_tvl1():
    import os
    gold = os.path.join(os.path.dirname(__file__), "golden")
    for n in sorted(os.listdir(gold)):
        if n.startswith("tvl1_ref_") and n.endswith(".npz"):
            z = np.load(os.path.join(gold, n))
            kw = {k[3:]: z[k].item() for k in z.files if k.startswith("kw_")}
            yield n, z, tvl1_cpu.TVL1Params(**kw)


def test_native_median_blur_pinned_to_cv2(native):
    """cv::medianBlur (float, 3 and 5) is the third external primitive tvl1flow.cpp calls (:1379-1383)."""
    import ctypes as C
    a = synth.texture(97, 131, 5) + np.random.default_rng(1).normal(0, 3, (97, 131)).astype(np.float32)
    fp = C.POINTER(C.c_float)
    for k in (3, 5):
        out = np.empty_like(a)
        native.lib().tvl1_cpu_median_blur(a.ctypes.data_as(fp), 97, 131, out.ctypes.data_as(fp), k)
        assert np.array_equal(out, cv2.medianBlur(a, k))


def test_golden_tvl1_vectors_pin_both_restatements(native):
    """tests/golden/tvl1_ref_*.npz come from the reference's own tvl1flow.cpp (oracle/_ref, make_golden.py).
    The C port must reproduce them bit for bit (same primitives, same arithmetic); the numpy restatement calls
    cv2's resize (<= 2 ulp away from the C primitive), which TV-L1's thresholding amplifies at a few pixels."""
    n_cases = 0
    for name, z, P in _golden_tvl1():
        n_cases += 1
        if P.gamma == 0 and P.medianFiltering <= 1:
            assert np.array_equal(native.calc(z["I0"], z["I1"], P), z["flow"]), name
        st = metrics.epe_stats(tvl1_cpu.calc(z["I0"], z["I1"], P), z["flow"])
        # fixed work: mean <= 0.01 px; with the data-dependent early exit (epsilon > 0) a 1-ulp difference can move
        # a warp's exit by an iteration pair, measured 0.013 px
        tol = (0.01, 0.99) if P.epsilon == 0 else (0.02, 0.97)
        assert st["mean"] <= tol[0] and st["frac_le_0.1"] >= tol[1], (name, st)
    assert n_cases >= 4


def test_reference_build_reproduces_golden_and_c_port(native):
    """tests/golden/tvl1_second_input.npz holds the unmodified reference source's output on a second input
    (oracle/_ref, make_golden.py): the C port is bit-identical to it (so the 1080p / 4K parity tests, which use the
    port, rest on the reference's own arithmetic).  Where the reference build is present (oracle/_ref), it must
    give every committed vector again."""
    import os
    from oracle import tvl1_ref
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "tvl1_second_input.npz"))
    I0, I1 = z["I0"], z["I1"]
    P = tvl1_cpu.TVL1Params(**{k[3:]: z[k].item() for k in z.files if k.startswith("kw_")})
    assert np.array_equal(native.calc(I0, I1, P), z["flow"])
    # useInitialFlow is honoured by the reference build (the port refuses it); the numpy restatement follows it
    P2 = tvl1_cpu.TVL1Params(**{k[7:]: z[k].item() for k in z.files if k.startswith("kwinit_")})
    assert P2.useInitialFlow
    assert np.abs(z["flow_init"][..., 0].mean() - 1.5) < 0.5
    st = metrics.epe_stats(tvl1_cpu.calc(I0, I1, P2, z["init"]), z["flow_init"])
    assert st["mean"] <= 0.01 and st["frac_le_0.1"] >= 0.99, st
    if tvl1_ref.available():
        assert tvl1_ref.source().endswith("modules/optflow/src/tvl1flow.cpp")
        for name, g, Pg in _golden_tvl1():
            assert np.array_equal(tvl1_ref.calc(g["I0"], g["I1"], Pg), g["flow"]), name
        assert np.array_equal(tvl1_ref.calc(I0, I1, P), z["flow"])
        assert np.array_equal(tvl1_ref.calc(I0, I1, P2, z["init"]), z["flow_init"])
