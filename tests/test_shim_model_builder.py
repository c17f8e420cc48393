"""The model builder's C++ surface compiles without a GPU: examples/create_model_offline.cpp, the
pcl::transformPointCloud overloads of include/pft/pcl_shim.hpp (pft::Affine3f; Eigen::Affine3f and Eigen::Matrix4f
under PFT_SHIM_USE_EIGEN, with the stand-in Eigen header of test_shim_reference_verbatim.py) and
ParticleFilterTracker::getResultCloud.  g++ -fsyntax-only: nothing runs."""
import os
import subprocess

import pytest

from tests.test_shim_reference_verbatim import STANDIN_EIGEN

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INCLUDE = os.path.join(ROOT, "include")

USES = r'''
  typedef pcl::PointXYZRGBA P;
  pcl::PointCloud<P>::Ptr c(new pcl::PointCloud<P>());
  pcl::PointCloud<P> out;
  pft::Affine3f a = pft::Affine3f::Identity();
  pcl::transformPointCloud(*c, out, a);
  pcl::transformPointCloud(out, out, a, true);                                 // in place
  pcl::tracking::KLDAdaptiveParticleFilterOMPTracker<P, pcl::tracking::ParticleXYZRPY> t(8);
  pcl::PointCloud<P>::Ptr r = t.getResultCloud();                              // ref: src/auto_tracking.cpp:309-316
  pcl::PointCloud<P>::Ptr r2 = t.getResultCloud(0.f);
  int n = (int)r->size() + (int)r2->size();
'''


def _syntax(src, *extra):
    r = subprocess.run(["/usr/bin/g++", "-std=c++17", "-fsyntax-only", *extra, "-I", INCLUDE, str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[:4000]


def test_create_model_offline_compiles():
    _syntax(os.path.join(ROOT, "examples", "create_model_offline.cpp"))


def test_transform_and_result_cloud_compile(tmp_path):
    src = tmp_path / "plain.cpp"
    src.write_text("#include <pft/pcl_shim.hpp>\nint main() {" + USES + "  return n;\n}\n")
    _syntax(src)


@pytest.mark.parametrize("boost", [False, True])
def test_eigen_overloads_compile(tmp_path, boost):
    inc = tmp_path / "standins"
    (inc / "Eigen").mkdir(parents=True)
    (inc / "Eigen" / "Geometry").write_text(STANDIN_EIGEN)
    (inc / "boost").mkdir()
    for name in ("shared_ptr.hpp", "make_shared.hpp", "pointer_cast.hpp"):
        (inc / "boost" / name).write_text("#pragma once\n#include <memory>\nnamespace boost { using std::shared_ptr; using std::make_shared; "
                                          "using std::static_pointer_cast; using std::dynamic_pointer_cast; }\n")
    src = tmp_path / "eigen.cpp"
    src.write_text("#include <Eigen/Geometry>\n" + ("#define PFT_SHIM_USE_BOOST\n" if boost else "") + "#define PFT_SHIM_USE_EIGEN\n"
                   "#include <pft/pcl_shim.hpp>\nint main() {" + USES +
                   "  Eigen::Affine3f e = Eigen::Affine3f::Identity();\n"
                   "  pcl::transformPointCloud(*c, out, e);\n"
                   "  Eigen::Matrix4f m4 = e.matrix();\n"
                   "  pcl::transformPointCloud(*c, out, m4);\n"
                   "  pcl::transformPointCloud(out, out, m4, false);\n"
                   "  Eigen::Affine3f back = pcl::tracking::ParticleXYZRPY().toEigenMatrix();\n"
                   "  pcl::transformPointCloud(*r, out, back);\n"
                   "  return n;\n}\n")
    _syntax(src, "-I", str(inc))
