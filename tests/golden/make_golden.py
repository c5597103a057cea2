"""Generates the committed golden vectors from the third-party code the reference calls
(OpenCV, via the cv2 4.13 wheel in this container).  Run from the repo root:
    python tests/golden/make_golden.py [match|orb|pnp|all|run_vo_symbols|run_vo]
The reference ships no fixtures of its own (SURVEY.md §4); these pin the oracle.  Two makers read a checkout of the reference
that MVO_REFERENCE_DIR names and are not part of `all`: `run_vo_symbols` stores the symbols the reference's own run_vo.cpp,
compiled against the adapter headers, needs from elsewhere; `run_vo` stores the trajectory it writes on libmvo (it needs a B200
and oracle/_ref/run_vo_reference, which __graft_entry__.build() makes)."""
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent.parent
sys.path.insert(0, str(ROOT / "monocular-visual-odometry_b200" / "python"))
sys.path.insert(0, str(ROOT))
OUT = Path(__file__).resolve().parent


def make_match():
    import cv2
    import mvo_synth
    d1 = mvo_synth.random_descriptors(101, 211, dup_every=9)
    d2 = mvo_synth.random_descriptors(102, 197, dup_every=6)
    d1[::4] = d2[(np.arange(0, 211, 4) * 5) % 197]
    bf = cv2.BFMatcher(cv2.NORM_HAMMING)
    nn = bf.match(d1, d2)
    kn = bf.knnMatch(d1, d2, k=2)
    np.savez_compressed(OUT / "match_golden.npz", d1=d1, d2=d2,
                        nn_train=np.array([m.trainIdx for m in nn], np.int32),
                        nn_dist=np.array([m.distance for m in nn], np.float32),
                        knn_train=np.array([[m.trainIdx for m in mm] for mm in kn], np.int32),
                        knn_dist=np.array([[m.distance for m in mm] for mm in kn], np.float32),
                        cv_version=cv2.__version__)


def make_orb():
    """cv::ORB detect (feature_match.cpp:22-23,34) -> selectUniformKptsByGrid restatement -> compute (:45,48)."""
    import cv2
    import mvo_synth
    from oracle import oracle_lib
    scenes = {"rect0": mvo_synth.gray_to_bgr(mvo_synth.rect_scene(0)), "color1": mvo_synth.color_scene(1),
              "noise0": mvo_synth.gray_to_bgr(mvo_synth.noise_scene(0))}
    for name, img in scenes.items():
        kps = cv2.ORB_create(8000, 1.2, 4, 31, 0, 2, cv2.ORB_HARRIS_SCORE, 31, 20).detect(img, None)
        det = np.array([(k.pt[0], k.pt[1], k.size, k.angle, k.response, k.octave, k.class_id) for k in kps],
                       oracle_lib.KEYPOINT_DTYPE)
        sel = oracle_lib.select_uniform_kpts_by_grid(det, img.shape[0], img.shape[1], 2000, 16, 8)
        ck = [cv2.KeyPoint(float(k["x"]), float(k["y"]), float(k["size"]), float(k["angle"]), float(k["response"]),
                           int(k["octave"]), int(k["class_id"])) for k in sel]
        ck2, desc = cv2.ORB_create(8000, 1.2, 4).compute(img, ck)
        assert len(ck2) == len(sel)
        extra = {} if name == "noise0" else {"image": img}      # the noise image is regenerated from its seed
        np.savez_compressed(OUT / f"orb_{name}.npz", detect=det, selected=sel, descriptors=desc,
                            cv_version=cv2.__version__, **extra)


def make_pnp():
    """cv::solvePnPRansac exactly as called at src/vo/vo.cpp:318-320 on the config-3 instance."""
    import cv2
    import mvo_synth
    P, uv, rvec_true, tvec_true, is_out = mvo_synth.pnp_problem(0)
    K = mvo_synth.K_DEFAULT
    ok, rvec, tvec, inl = cv2.solvePnPRansac(P, uv, K, None, None, None, False, 100, 2.0, 0.999)
    assert ok
    inl = inl.ravel().astype(np.int32)
    ok2, r2, t2 = cv2.solvePnP(P[inl], uv[inl], K, None, flags=cv2.SOLVEPNP_ITERATIVE)
    np.savez_compressed(OUT / "pnp_config3.npz", P=P, uv=uv, K=K, rvec=rvec.ravel(), tvec=tvec.ravel(), inliers=inl,
                        rvec_refit=r2.ravel(), tvec_refit=t2.ravel(), rvec_true=rvec_true, tvec_true=tvec_true,
                        cv_version=cv2.__version__)


def make_run_vo_symbols():
    """The undefined symbols of the reference's run_vo.cpp compiled against my_slam_adapter/include + tests/cvshim, one per line."""
    import subprocess
    import tempfile
    from oracle import reference_run_vo
    src = reference_run_vo.source()
    assert src is not None, "MVO_REFERENCE_DIR must name a checkout of the reference"
    with tempfile.TemporaryDirectory() as tmp:
        obj = Path(tmp) / "run_vo.o"
        subprocess.run(reference_run_vo.command(src, obj, compile_only=True), check=True)
        nm = subprocess.run(["nm", "-P", "-u", str(obj)], capture_output=True, text=True, check=True).stdout
    syms = sorted({line.split()[0] for line in nm.splitlines() if line.split()[1:2] == ["U"]})
    (OUT / "run_vo_reference_undefined.txt").write_text("".join(s + "\n" for s in syms))


def make_run_vo():
    """run_vo.cpp of the reference on libmvo over the 14-frame PNG dataset of tests/test_run_vo_reference_source.py."""
    import subprocess
    import tempfile
    sys.path.insert(0, str(ROOT / "tests"))
    import test_run_vo_reference_source as t
    from oracle import reference_run_vo
    assert reference_run_vo.OUT.exists(), "build oracle/_ref/run_vo_reference first (MVO_REFERENCE_DIR + __graft_entry__.build())"
    with tempfile.TemporaryDirectory() as tmp:
        child = t.reference_child(tmp, reference_run_vo.OUT, save=t.GOLDEN_TRAJ)
        r = subprocess.run([sys.executable, "-c", child], capture_output=True, text=True)
        assert r.returncode == 0 and "reference run_vo child ok" in r.stdout, (r.stdout[-1500:], r.stderr[-3000:])


if __name__ == "__main__":
    what = sys.argv[1] if len(sys.argv) > 1 else "all"
    if what in ("match", "all"):
        make_match()
    if what in ("orb", "all") and "make_orb" in globals():
        make_orb()
    if what in ("pnp", "all") and "make_pnp" in globals():
        make_pnp()
    if what == "run_vo_symbols":
        make_run_vo_symbols()
    if what == "run_vo":
        make_run_vo()
