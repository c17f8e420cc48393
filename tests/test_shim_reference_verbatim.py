"""The drop-in claim of the boundary, checked on the reference's own text: `initialize_trackers()` (ref:
src/auto_tracking.cpp:181-259), the class typedefs it relies on (ref :139-156) and the scene filters
(ref :536-575) are read AT TEST TIME from the checkout of cmaestre/pcl_tracking that PCL_TRACKING_REFERENCE names
(nothing of them is committed here; without it the test skips) and compiled
verbatim against include/pft/pcl_shim.hpp, with boost::shared_ptr and Eigen::Affine3f as the reference spells
them.  Boost and Eigen are not installed in this image: two tiny stand-in headers written by the test provide
`boost::shared_ptr` (= std::shared_ptr) and an `Eigen::Affine3f` with Identity(), operator()(r, c) and
matrix().data() -- the operations the shim needs from them.  g++ -fsyntax-only: no GPU, nothing runs."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(os.environ.get("PCL_TRACKING_REFERENCE", ""), "src", "auto_tracking.cpp")

STANDIN_BOOST = """#pragma once
#include <memory>
namespace boost { using std::shared_ptr; using std::make_shared; using std::static_pointer_cast; using std::dynamic_pointer_cast; }
"""
STANDIN_EIGEN = """#pragma once
#include <cstring>
namespace Eigen {
struct Matrix4f { float m[16]; const float* data() const { return m; } float* data() { return m; } };
struct Affine3f {
  Matrix4f mat;
  Affine3f() { std::memset(mat.m, 0, sizeof(mat.m)); mat.m[0] = mat.m[5] = mat.m[10] = mat.m[15] = 1.f; }
  static Affine3f Identity() { return Affine3f(); }
  float& operator()(int r, int c) { return mat.m[c * 4 + r]; }
  float operator()(int r, int c) const { return mat.m[c * 4 + r]; }
  const Matrix4f& matrix() const { return mat; }
};
}  // namespace Eigen
"""


def ref_lines(first, last):
    with open(REF) as f:
        lines = f.readlines()
    return "".join(lines[first - 1:last])


@pytest.mark.skipif(not os.environ.get("PCL_TRACKING_REFERENCE") or not os.path.exists(REF),
                    reason="needs the reference's src/auto_tracking.cpp: set PCL_TRACKING_REFERENCE to a checkout of cmaestre/pcl_tracking")
def test_reference_initialize_trackers_and_filters_compile_verbatim(tmp_path):
    inc = tmp_path / "standins"
    (inc / "boost").mkdir(parents=True)
    (inc / "Eigen").mkdir()
    for name in ("shared_ptr.hpp", "make_shared.hpp", "pointer_cast.hpp"):
        (inc / "boost" / name).write_text(STANDIN_BOOST)
    (inc / "Eigen" / "Geometry").write_text(STANDIN_EIGEN)
    src = tmp_path / "reference_verbatim.cpp"
    src.write_text(
        "#include <cmath>\n#include <map>\n#include <string>\n#include <vector>\n"
        "#include <boost/shared_ptr.hpp>\n#include <Eigen/Geometry>\n"
        "#define PFT_SHIM_USE_BOOST\n#define PFT_SHIM_USE_EIGEN\n"
        "#include <pft/pcl_shim.hpp>\n"
        "using namespace pcl::tracking;\n"                       # ref :133
        "#define FPS_CALC_BEGIN\n#define FPS_CALC_END(_WHAT_)\n"  # (the reference's fps printing macros, ref :111-131)
        "template <typename PointType>\nclass OpenNISegmentTracking\n{\npublic:\n"
        + ref_lines(139, 156)                                    # the typedefs, verbatim
        + "    pcl::NormalEstimationOMP<PointType, pcl::Normal> ne_;\n"  # members the two excerpts touch (ref :784-812)
          "    std::map<int, boost::shared_ptr<ParticleFilter> > tracker_dict;\n"
          "    int nb_objects;\n    bool use_fixed_;\n    int thread_nr_;\n    double downsampling_time_;\n"
        + ref_lines(181, 259)                                    # initialize_trackers(), verbatim
        + ref_lines(536, 575)                                    # filterPassThrough / gridSample / gridSampleApprox, verbatim
        + "};\ntemplate class OpenNISegmentTracking<pcl::PointXYZRGBA>;\nint main() { return 0; }\n")
    r = subprocess.run(["g++", "-std=c++11", "-fsyntax-only", "-I", str(inc), "-I", os.path.join(ROOT, "include"), str(src)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[:4000]
