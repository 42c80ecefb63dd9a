"""TEST INFRASTRUCTURE ONLY — recipe that compiles the reference's own lateral post-process sources, where
they lie under ref_import.REFERENCE_ROOT, into oracle/_ref/libref_lateral.so (git-ignored):

  g++ -O2 -ffp-contract=off -shared -fPIC  -I oracle/cvstub  -I <ref>/include
      oracle/ref_lateral_harness.cpp  <ref>/src/lane_filtering/lane_filter.cpp
      <ref>/src/lane_tracking/lane_tracking.cpp  <ref>/src/path_planning/{estimator,poly_fit,path_finder}.cpp

The reference's build system (cmake + OpenCV + Eigen + TensorRT) is NOT run; the OpenCV and Eigen names these five
files use are provided by the minimal stand-ins oracle/cvstub/opencv2/opencv.hpp and oracle/cvstub/Eigen/Dense.
Returns the path of the library, or None when the reference sources are absent or the compile fails."""
from __future__ import annotations

import os
import subprocess
from typing import Optional

from oracle import ref_import

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.path.join(ref_import.REFERENCE_ROOT, "VisionPilot", "production_release")
OUT = os.path.join(HERE, "_ref", "libref_lateral.so")


def build(force: bool = False) -> Optional[str]:
    srcs = [os.path.join(REF, "src", p) for p in ("lane_filtering/lane_filter.cpp", "lane_tracking/lane_tracking.cpp",
                                                  "path_planning/estimator.cpp", "path_planning/poly_fit.cpp",
                                                  "path_planning/path_finder.cpp")]
    if not all(os.path.exists(s) for s in srcs):
        return OUT if os.path.exists(OUT) else None
    harness = os.path.join(HERE, "ref_lateral_harness.cpp")
    stubs = [os.path.join(HERE, "cvstub", "opencv2", "opencv.hpp"), os.path.join(HERE, "cvstub", "Eigen", "Dense")]
    if not force and os.path.exists(OUT) and os.path.getmtime(OUT) >= max(os.path.getmtime(f) for f in srcs + [harness] + stubs):
        return OUT
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    cmd = ["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-I", os.path.join(HERE, "cvstub"),
           "-I", os.path.join(REF, "include"), harness] + srcs + ["-o", OUT]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        print("oracle/_ref build failed:\n" + r.stderr[-3000:])
        return None
    return OUT


if __name__ == "__main__":
    print(build(force=True))
