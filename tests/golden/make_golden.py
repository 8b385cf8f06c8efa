"""Generates the committed golden fixtures in the BUILD container (the only place /root/reference exists):
  farneback_*.npz  live CPU reference cv2.calcOpticalFlowFarneback (cv2 4.13.0 = opencv/opencv
                   modules/video/src/optflowgf.cpp, the function modules/optflow/src/interfaces.cpp:154-157 forwards to)
  tvl1_ref_*.npz   the reference's OWN CPU Dual TV-L1, /root/reference/modules/optflow/src/tvl1flow.cpp compiled
                   unmodified into oracle/_ref/libtvl1_ref.so (oracle/Makefile, oracle/ref_shim/)
  tvl1_second_input.npz   the same reference build on a second input, once with fixed work (what the C port must
                   reproduce bit for bit) and once from an initial flow (which the port refuses)
  brox_720p.npz, denselk_1080p.npz   BASELINE-size outputs of the numpy restatements oracle/brox_model.py and
                   oracle/denselk_model.py (no CPU implementation exists upstream: "parity unpinned"), stored as float32
                   on a stride-4 grid plus full-resolution means -- 2 minutes (brox) / 27 minutes (denselk) of numpy
python tests/golden/make_golden.py [farneback] [tvl1] [tvl1_second] [brox] [denselk]   (no argument = farneback + tvl1)"""
import os
import sys

import numpy as np
import cv2

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import synth  # noqa: E402

CASES = {
    "box": (dict(), 1e-4, 0.02),
    "poly7": (dict(polyN=7, polySigma=1.5), 1e-4, 0.02),
    "gauss": (dict(flags=256), 2e-2, 0.2),
    "scale08": (dict(pyrScale=0.8, numLevels=3), 1e-4, 0.02),
}
WHAT = {a.split(":", 1)[0] for a in sys.argv[1:]} or {"farneback", "tvl1"}   # "tvl1:<case>" regenerates one TV-L1 case
for name, (kw, ncc_tol, epe_tol) in (CASES.items() if "farneback" in WHAT else ()):
    I0, I1, _ = synth.make_pair(144, 192, seed=11, kind="smooth")
    flow = cv2.calcOpticalFlowFarneback(I0, I1, None, kw.get("pyrScale", 0.5), kw.get("numLevels", 5), 13, 10,
                                        kw.get("polyN", 5), kw.get("polySigma", 1.1), kw.get("flags", 0))
    out = {"I0": I0, "I1": I1, "flow": flow.astype(np.float32), "ncc_tol": ncc_tol, "epe_tol": epe_tol,
           "cv2_version": cv2.__version__}
    out.update({"kw_" + k: v for k, v in kw.items()})
    np.savez_compressed(os.path.join(HERE, f"farneback_{name}.npz"), **out)
    print(name, flow.shape)

if "tvl1" in WHAT:
    from oracle import tvl1_cpu, tvl1_ref  # noqa: E402
    TV = {
        # the mapping the reference's GPU-vs-CPU test uses (cudaoptflow/test/test_optflow.cpp:456-460)
        "gpu_twin": dict(nscales=4, warps=5, epsilon=0.0, innerIterations=1, outerIterations=30, medianFiltering=1),
        "defaults": dict(),                                             # median 5, eps 0.01, 10 x 30
        "gamma": dict(gamma=0.5, medianFiltering=1, epsilon=0.0, innerIterations=5, outerIterations=4),
        "f32_median3": dict(medianFiltering=3, warps=2),
        # fixed work with the median filter on: what the engine's MEDIAN_FILTERING / MEDIAN_PERIOD knobs are checked against
        "median5_fixed": dict(nscales=3, warps=3, epsilon=0.0, innerIterations=10, outerIterations=3, medianFiltering=5),
    }
    only = {a.split(":", 1)[1] for a in sys.argv[1:] if a.startswith("tvl1:")}
    for name, kw in TV.items():
        if only and name not in only:
            continue
        I0, I1, gt = synth.make_pair(120, 160, seed=21, kind="affine", dtype="f32" if name.startswith("f32") else "u8")
        flow = tvl1_ref.calc(I0, I1, tvl1_cpu.TVL1Params(**kw))
        out = {"I0": I0, "I1": I1, "flow": flow, "gt": gt.astype(np.float32), "source": tvl1_ref.source()}
        out.update({"kw_" + k: v for k, v in kw.items()})
        np.savez_compressed(os.path.join(HERE, f"tvl1_ref_{name}.npz"), **out)
        print("tvl1", name, flow.shape, float(np.abs(flow).mean()))

if "tvl1_second" in WHAT:
    from oracle import tvl1_cpu, tvl1_ref  # noqa: E402
    fixed = dict(warps=10, epsilon=0.0, innerIterations=1, outerIterations=30, medianFiltering=1)
    from_init = dict(nscales=1, warps=1, epsilon=0.0, innerIterations=1, outerIterations=2, medianFiltering=1,
                     useInitialFlow=True)
    I0, I1, _ = synth.make_pair(150, 190, seed=9, kind="smooth")
    flow = tvl1_ref.calc(I0, I1, tvl1_cpu.TVL1Params(**fixed))
    init = np.zeros(I0.shape + (2,), np.float32)
    init[..., 0] = 1.5
    flow_init = tvl1_ref.calc(I0, I1, tvl1_cpu.TVL1Params(**from_init), init)
    out = {"I0": I0, "I1": I1, "flow": flow, "init": init, "flow_init": flow_init}
    out.update({"kw_" + k: v for k, v in fixed.items()})
    out.update({"kwinit_" + k: v for k, v in from_init.items()})
    np.savez_compressed(os.path.join(HERE, "tvl1_second_input.npz"), **out)
    print("tvl1_second", flow.shape, float(np.abs(flow).mean()), float(flow_init[..., 0].mean()))


def _model_fixture(name, I0, I1, flow, kw, seed, kind, dtype):
    import hashlib
    out = {"flow_s4": flow[::4, ::4].astype(np.float32), "shape": np.array(flow.shape[:2]), "seed": seed, "kind": kind,
           "dtype": dtype, "sha1_I0": hashlib.sha1(np.ascontiguousarray(I0).tobytes()).hexdigest(),
           "sha1_I1": hashlib.sha1(np.ascontiguousarray(I1).tobytes()).hexdigest(),
           "mean_u": float(flow[..., 0].mean(dtype=np.float64)), "mean_v": float(flow[..., 1].mean(dtype=np.float64)),
           "mean_abs": float(np.abs(flow).mean(dtype=np.float64))}
    out.update({"kw_" + k: v for k, v in kw.items()})
    np.savez_compressed(os.path.join(HERE, name), **out)
    print(name, flow.shape, out["mean_u"], out["mean_v"])


if "brox" in WHAT:  # BASELINE configs[3]: 1280x720, create(0.197, 50, 0.8, 10, 77, 10) (cudaoptflow/test/test_optflow.cpp:75-76)
    from oracle import brox_model  # noqa: E402
    kw = dict(alpha=0.197, gamma=50.0, scale_factor=0.8, inner_iterations=10, outer_iterations=77, solver_iterations=10)
    I0, I1, _ = synth.make_pair(720, 1280, seed=0, kind="smooth", dtype="f32")
    _model_fixture("brox_720p.npz", I0, I1, brox_model.calc(I0, I1, brox_model.BroxParams(**kw)), kw, 0, "smooth", "f32")

if "denselk" in WHAT:  # DensePyrLK defaults at 1080p: 13x13, maxLevel 3, 30 iterations (cudaoptflow.hpp:245-249)
    from oracle import denselk_model  # noqa: E402
    I0, I1, _ = synth.make_pair(1080, 1920, seed=0, kind="smooth")
    flow = denselk_model.calc(I0, I1, (13, 13), 3, 30)
    _model_fixture("denselk_1080p.npz", I0, I1, flow, dict(win_w=13, win_h=13, maxLevel=3, iters=30), 0, "smooth", "u8")
