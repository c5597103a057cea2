"""north_star: 'keeping the my_slam::vo Frame/Map/MapPoint API surface so run_vo.cpp links unchanged'.  The original project's own
run_vo.cpp (compiled from a checkout of it that MVO_REFERENCE_DIR names, never copied into this repository; oracle/reference_run_vo.py)
against my_slam_adapter/include (Frame / Map / MapPoint / VisualOdometry over libmvo) + the stand-ins of tests/cvshim for what this
image lacks (OpenCV value types and highgui calls, PCL viewer, the original's basics/yaml/vo_io on the product's C ABI), linked with
vo_mvo.cpp and libmvo.so.  CPU tier: every symbol its object needs (stored in tests/golden/run_vo_reference_undefined.txt)
links against the adapter layer and libmvo, and with a checkout at hand the file itself compiles and links, unmodified.  GPU
tier: the trajectory that binary wrote for a PNG dataset and a config file in the original's dialect is stored (tests/golden/run_vo_reference_traj.txt, make_golden.py run_vo);
the ctypes path over the same config must write the same trajectory, and so must the binary where __graft_entry__.build() made it
(oracle/_ref/run_vo_reference)."""
import os
import re
import subprocess
import sys
from pathlib import Path

import pytest

from conftest import GOLDEN, have_cv2

ROOT = Path(__file__).resolve().parent.parent
PKG = ROOT / "monocular-visual-odometry_b200"
GOLDEN_TRAJ = GOLDEN / "run_vo_reference_traj.txt"
GOLDEN_SYMS = GOLDEN / "run_vo_reference_undefined.txt"
_TIMEOUT_SCALE = float(os.environ.get("MVO_TEST_TIMEOUT_SCALE", "1"))
_LINKER_DEFINED = {"_GLOBAL_OFFSET_TABLE_", "__dso_handle"}      # the static linker provides these to every executable


def _check_vo_symbols(exe):
    """The VO symbols come from the adapter layer, mvo_vo_add_frame from libmvo.so at run time."""
    syms = subprocess.run(["nm", "-C", str(exe)], capture_output=True, text=True).stdout
    assert "my_slam::vo::VisualOdometry::addFrame" in syms and "my_slam::vo::Frame::createFrame" in syms
    assert re.search(r"U mvo_vo_add_frame", syms)


def test_reference_run_vo_compiles_and_links_unmodified(built, tmp_path):
    from oracle import reference_run_vo
    # Every symbol the original run_vo.cpp needs from elsewhere (stored from a compile of it against the adapter headers,
    # make_golden.py run_vo_symbols), referenced from one translation unit and linked exactly as the original is linked.
    need = GOLDEN_SYMS.read_text().split()
    assert "_ZN7my_slam2vo14VisualOdometry8addFrameESt10shared_ptrINS0_5FrameEE" in need
    stub = tmp_path / "run_vo_needs.cpp"
    refs = "".join(f".quad {s}\\n" for s in need if s not in _LINKER_DEFINED)
    stub.write_text(f'asm(".section .data.rel.ro,\\"aw\\"\\n.balign 8\\n{refs}.text\\n");\nint main() {{ return 0; }}\n')
    out = tmp_path / "run_vo_needs"
    r = subprocess.run(reference_run_vo.command(stub, out), capture_output=True, text=True)
    assert r.returncode == 0 and out.exists(), r.stderr[-3000:]
    _check_vo_symbols(out)
    r = subprocess.run([str(out)], capture_output=True, text=True, env=dict(os.environ, LD_LIBRARY_PATH=str(PKG)))
    assert r.returncode == 0, r.stderr[-2000:]

    src = reference_run_vo.source()
    if src is None:
        return
    # with a checkout of the original at hand: the original file itself, unmodified
    out = tmp_path / "run_vo_reference"
    cmd = reference_run_vo.command(src, out)
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0 and out.exists(), r.stderr[-3000:]
    assert str(src) in cmd and not any(Path(c).name == "run_vo.cpp" and str(ROOT) in c for c in cmd)
    _check_vo_symbols(out)
    # wrong usage ends like the original's does (run_vo.cpp:64: assert(checkInputArguments(...)))
    r = subprocess.run([str(out)], capture_output=True, text=True, env=dict(os.environ, LD_LIBRARY_PATH=str(PKG)))
    assert r.returncode != 0 and "Lack arguments" in r.stdout


# {app}: the original's run_vo binary, or "" to check the ctypes path against the stored trajectory alone.  {save}: where to
# store the binary's trajectory instead of comparing with the stored one (make_golden.py run_vo), or "".
GPU_CHILD = r'''
import re, shutil, subprocess, sys, os
import numpy as np
sys.path.insert(0, r"{root}"); sys.path.insert(0, r"{root}/monocular-visual-odometry_b200/python")
import mvo_b200, mvo_synth
n = 14
frames, _ = mvo_synth.room_sequence(0, n)
imgs = [mvo_synth.gray_to_bgr(f) for f in frames]
cfg = open(r"{fixture}").read()
cfg = cfg.replace('dataset_name: "fr1_desk"', 'dataset_name: "matlab"').replace("dataset_dir: data/dataset_images_matlab", 'dataset_dir: "{tmp}"')
cfg = re.sub(r"num_images: 150", "num_images: %d" % n, cfg, count=1).replace("save_predicted_traj_to: data/test_data/cam_traj.txt", 'save_predicted_traj_to: "{tmp}/traj.txt"')
cfg = cfg.replace('is_draw_true_traj: "true"', 'is_draw_true_traj: "false"')
cfg = re.sub(r"(?m)^(output_folder|is_pcl_wait_for_keypress|cv_waitkey_time):[^\n]*\n", "", cfg)        # the display keys run_vo.cpp reads
cfg += '\noutput_folder: "{tmp}/out"\nis_pcl_wait_for_keypress: "false"\ncv_waitkey_time: 1\n'
open(r"{tmp}/config.yaml", "w").write(cfg)
lib = mvo_b200.load_library()
import ctypes as C

def read_traj(path):
    got, cnt = np.zeros((n, 16)), C.c_int(0)
    assert lib.mvo_read_pose_file(path.encode(), got.ctypes.data, n, C.byref(cnt)) == 0 and cnt.value == n
    return got.reshape(n, 4, 4)

trajs = []
if r"{app}":
    import cv2
    for i, im in enumerate(imgs):
        assert cv2.imwrite(r"{tmp}/rgb_%05d.png" % i, im)
    r = subprocess.run([r"{app}", r"{tmp}/config.yaml"], capture_output=True, text=True, timeout=200 * float(os.environ.get("MVO_TEST_TIMEOUT_SCALE", "1")))
    assert r.returncode == 0, (r.stdout[-1500:], r.stderr[-1500:])
    trajs.append(read_traj(r"{tmp}/traj.txt"))
    if r"{save}":
        shutil.copyfile(r"{tmp}/traj.txt", r"{save}")
if not r"{save}":
    trajs.append(read_traj(r"{golden}"))
h = C.c_void_p()
assert lib.mvo_config_load(r"{tmp}/config.yaml".encode(), C.byref(h)) == 0
p, vp, K = mvo_b200.Params(), mvo_b200.VoParams(), np.zeros(9)
lib.mvo_default_params(C.byref(p)); lib.mvo_vo_default_params(C.byref(vp))
assert lib.mvo_config_apply(h, C.byref(p), None, K.ctypes.data) == 0 and lib.mvo_config_apply_vo(h, C.byref(vp)) == 0
ctx = mvo_b200.Context(0, params=p)
vh = C.c_void_p()
assert lib.mvo_vo_create(ctx.h, K.ctypes.data, 480, 640, C.byref(vp), C.byref(vh)) == 0
poses = []
for im in imgs:
    T = np.zeros(16)
    assert lib.mvo_vo_add_frame(vh, im.ctypes.data, 3, 640 * 3, T.ctypes.data, None) == 0
    poses.append(T.reshape(4, 4))
for got in trajs:
    assert np.abs(got - np.stack(poses)).max() < 2e-5         # 6 significant digits in the file
assert lib.mvo_vo_is_initialized(vh) == 1
print("reference run_vo child ok (%d trajectories compared)" % len(trajs))
'''


def reference_child(tmp, app="", save=""):
    return GPU_CHILD.format(root=str(ROOT), tmp=str(tmp), app=str(app), save=str(save), golden=str(GOLDEN_TRAJ),
                            fixture=str(GOLDEN / "config_fixture.yaml"))


@pytest.mark.gpu
def test_reference_run_vo_runs_on_libmvo(built, tmp_path):
    from oracle import reference_run_vo
    app = reference_run_vo.OUT if reference_run_vo.OUT.exists() and have_cv2() else ""    # cv2 writes the PNG dataset
    r = subprocess.run([sys.executable, "-c", reference_child(tmp_path, app)], capture_output=True, text=True, timeout=300 * _TIMEOUT_SCALE)
    assert r.returncode == 0 and "reference run_vo child ok" in r.stdout, (r.stdout[-1500:], r.stderr[-3000:])
