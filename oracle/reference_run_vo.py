"""The original project's own run_vo.cpp, compiled UNMODIFIED and from where it lies, against the my_slam adapter headers
(my_slam_adapter/include first, then the stand-ins for OpenCV / PCL / the original's basics of tests/cvshim) and linked with
vo_mvo.cpp + libmvo.so into oracle/_ref/run_vo_reference.

The original project (felixchenfy/Monocular-Visual-Odometry) is never copied into this repository: MVO_REFERENCE_DIR names a
checkout of it.  Without one nothing is built, and tests/test_run_vo_reference_source.py checks what was stored from it
instead: the symbols its object needs (tests/golden/run_vo_reference_undefined.txt) and the trajectory the binary wrote
(tests/golden/run_vo_reference_traj.txt)."""
from __future__ import annotations

import os
import subprocess
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
PKG = ROOT / "monocular-visual-odometry_b200"
OUT = ROOT / "oracle" / "_ref" / "run_vo_reference"


def source() -> Path | None:
    """run_vo.cpp of the checkout MVO_REFERENCE_DIR names, or None when there is none (or it cannot be read)."""
    d = os.environ.get("MVO_REFERENCE_DIR")
    if not d:
        return None
    p = Path(d) / "run_vo.cpp"
    return p if os.path.isfile(p) and os.access(p, os.R_OK) else None


def command(src: Path, out: Path, compile_only: bool = False) -> list[str]:
    """g++ command linking src with the adapter layer and libmvo; with compile_only, src alone compiled to the object out."""
    flags = ["g++", "-O1", "-std=c++17", "-I", str(PKG / "my_slam_adapter" / "include"), "-I", str(ROOT / "tests" / "cvshim"), "-I", str(ROOT / "include"),
             "-I", str(PKG / "my_slam_adapter"), "-I", str(PKG / "apps")]
    if compile_only:
        return flags + ["-c", str(src), "-o", str(out)]
    return flags + [str(src), str(PKG / "my_slam_adapter" / "mvo_context.cpp"),
                    str(PKG / "my_slam_adapter" / "vo_mvo.cpp"), str(PKG / "apps" / "png_reader.cpp"), "-L", str(PKG), "-lmvo", "-lz",
                    "-Wl,-rpath,$ORIGIN/../../" + PKG.name, "-o", str(out)]


def build() -> Path | None:
    """oracle/_ref/run_vo_reference where the original project is present; None otherwise."""
    src = source()
    if src is None:
        return None
    OUT.parent.mkdir(parents=True, exist_ok=True)
    r = subprocess.run(command(src, OUT), capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("the original run_vo.cpp no longer compiles against my_slam_adapter/: " + r.stderr[-2000:])
    return OUT
