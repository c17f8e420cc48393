"""The depth-image ingest of the C++ shim (pcl::PointCloud::fromDepthImage / fromDepthImageAsync) compiles and links
with plain g++ against libpft.so.  The program below is also what tests/test_gpu_depth.py runs on the device."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# depth_ingest depth.raw bgr.raw width height depth_step bgr_step fx fy cx cy out.raw
# Converts the two images with fromDepthImage (from the files' buffers) and with fromDepthImageAsync (from pinned
# copies), prints "<points> <width> <height>" of each organised cloud and writes both clouds' 32-byte records to out.raw.
DEPTH_INGEST_CPP = r'''
#include <pft/pcl_shim.hpp>

#include <iterator>

static std::vector<unsigned char> slurp(const char* path) {
  std::ifstream f(path, std::ios::binary);
  return std::vector<unsigned char>((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
}

int main(int argc, char** argv) {
  if (argc != 12) { fprintf(stderr, "usage: %s depth.raw bgr.raw w h depth_step bgr_step fx fy cx cy out.raw\n", argv[0]); return 2; }
  const std::vector<unsigned char> depth = slurp(argv[1]), bgr = slurp(argv[2]);
  const uint32_t w = (uint32_t)atoi(argv[3]), h = (uint32_t)atoi(argv[4]), ds = (uint32_t)atoi(argv[5]), cs = (uint32_t)atoi(argv[6]);
  const double fx = atof(argv[7]), fy = atof(argv[8]), cx = atof(argv[9]), cy = atof(argv[10]);
  try {
    typedef pcl::PointXYZRGBA P;
    pcl::PointCloud<P>::Ptr a(new pcl::PointCloud<P>()), b(new pcl::PointCloud<P>());
    a->fromDepthImage(reinterpret_cast<const uint16_t*>(depth.data()), ds, bgr.data(), cs, w, h, fx, fy, cx, cy);
    void* pd = nullptr;
    void* pc = nullptr;
    pft::check(pft_host_alloc(&pd, depth.size()));
    pft::check(pft_host_alloc(&pc, bgr.size()));
    memcpy(pd, depth.data(), depth.size());
    memcpy(pc, bgr.data(), bgr.size());
    b->fromDepthImageAsync(static_cast<const uint16_t*>(pd), ds, static_cast<const uint8_t*>(pc), cs, w, h, fx, fy, cx, cy);
    std::ofstream out(argv[11], std::ios::binary);
    for (auto& c : {a, b}) {
      const uint32_t cw = c->width, ch = c->height;
      c->download();
      printf("%zu %u %u\n", c->points.size(), cw, ch);
      out.write(reinterpret_cast<const char*>(c->points.data()), (std::streamsize)(c->points.size() * sizeof(P)));
    }
    pft_host_free(pd);
    pft_host_free(pc);
  } catch (const std::exception& e) {
    fprintf(stderr, "%s\n", e.what());
    return 3;
  }
  return 0;
}
'''


def build_depth_ingest(tmp_path):
    src = tmp_path / "depth_ingest.cpp"
    src.write_text(DEPTH_INGEST_CPP)
    exe = tmp_path / "depth_ingest"
    lib_dir = os.path.join(ROOT, "pcl_tracking_b200", "lib")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src),
                           "-L", lib_dir, "-lpft", "-Wl,-rpath," + lib_dir])
    return str(exe)


def test_depth_ingest_program_builds_and_fails_loudly_without_gpu(tmp_path):
    exe = build_depth_ingest(tmp_path)
    from pcl_tracking_b200 import _capi
    if _capi.load().pft_device_count() > 0:
        return  # tests/test_gpu_depth.py runs it
    (tmp_path / "d.raw").write_bytes(b"\0" * 8)
    (tmp_path / "c.raw").write_bytes(b"\0" * 12)
    r = subprocess.run([exe, str(tmp_path / "d.raw"), str(tmp_path / "c.raw"), "2", "2", "4", "6", "365", "365", "1", "1", str(tmp_path / "o.raw")],
                       capture_output=True, text=True)
    assert r.returncode == 3
    assert "no CPU fallback" in r.stderr
