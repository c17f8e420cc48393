"""The fused depth-image ingest of the C++ shim (pcl::PointCloud::fromDepthImages / fromDepthImagesAsync with
pft::DepthCamera) compiles and links with plain g++ against libpft.so.  The program below is also what
tests/test_gpu_depth_cameras.py runs on the device."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# depth_cameras out.raw [depth.raw bgr.raw width height depth_step bgr_step fx fy cx cy pose.raw|-] ...
# Fuses the cameras (11 arguments each; pose.raw holds 12 float32, the 3x4 row-major matrix, "-" for none) with
# fromDepthImages (from the files' buffers) and with fromDepthImagesAsync (from pinned copies), prints
# "<points> <width> <height>" of each cloud and writes both clouds' 32-byte records to out.raw.
DEPTH_CAMERAS_CPP = r'''
#include <pft/pcl_shim.hpp>

#include <iterator>

static std::vector<unsigned char> slurp(const char* path) {
  std::ifstream f(path, std::ios::binary);
  return std::vector<unsigned char>((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
}

int main(int argc, char** argv) {
  if (argc < 13 || (argc - 2) % 11) {
    fprintf(stderr, "usage: %s out.raw [depth.raw bgr.raw w h depth_step bgr_step fx fy cx cy pose.raw|-] ...\n", argv[0]);
    return 2;
  }
  const int n = (argc - 2) / 11;
  std::vector<std::vector<unsigned char>> depth(n), bgr(n);
  std::vector<pft::DepthCamera> cams(n);
  for (int k = 0; k < n; ++k) {
    char** a = argv + 2 + 11 * k;
    depth[k] = slurp(a[0]);
    bgr[k] = slurp(a[1]);
    pft::DepthCamera& c = cams[k];
    c.width = (uint32_t)atoi(a[2]); c.height = (uint32_t)atoi(a[3]);
    c.depth_step = (uint32_t)atoi(a[4]); c.bgr_step = (uint32_t)atoi(a[5]);
    c.fx = atof(a[6]); c.fy = atof(a[7]); c.cx = atof(a[8]); c.cy = atof(a[9]);
    if (strcmp(a[10], "-") != 0) {
      const std::vector<unsigned char> m = slurp(a[10]);
      pft::Affine3f t;
      for (int r = 0; r < 3; ++r) for (int col = 0; col < 4; ++col) memcpy(&t(r, col), m.data() + 4 * (r * 4 + col), 4);
      c.setPose(t);
    }
  }
  try {
    typedef pcl::PointXYZRGBA P;
    pcl::PointCloud<P>::Ptr a(new pcl::PointCloud<P>()), b(new pcl::PointCloud<P>());
    for (int k = 0; k < n; ++k) {
      cams[k].depth = reinterpret_cast<const uint16_t*>(depth[k].data());
      cams[k].bgr = bgr[k].data();
    }
    a->fromDepthImages(cams);
    std::vector<void*> pinned;
    for (int k = 0; k < n; ++k) {
      void* pd = nullptr;
      void* pc = nullptr;
      pft::check(pft_host_alloc(&pd, depth[k].size()));
      pft::check(pft_host_alloc(&pc, bgr[k].size()));
      memcpy(pd, depth[k].data(), depth[k].size());
      memcpy(pc, bgr[k].data(), bgr[k].size());
      cams[k].depth = static_cast<const uint16_t*>(pd);
      cams[k].bgr = static_cast<const uint8_t*>(pc);
      pinned.push_back(pd);
      pinned.push_back(pc);
    }
    b->fromDepthImagesAsync(cams);
    std::ofstream out(argv[1], std::ios::binary);
    for (auto& c : {a, b}) {
      const uint32_t cw = c->width, ch = c->height;
      c->download();
      printf("%zu %u %u\n", c->points.size(), cw, ch);
      out.write(reinterpret_cast<const char*>(c->points.data()), (std::streamsize)(c->points.size() * sizeof(P)));
    }
    for (void* p : pinned) pft_host_free(p);
  } catch (const std::exception& e) {
    fprintf(stderr, "%s\n", e.what());
    return 3;
  }
  return 0;
}
'''


def build_depth_cameras(tmp_path):
    src = tmp_path / "depth_cameras.cpp"
    src.write_text(DEPTH_CAMERAS_CPP)
    exe = tmp_path / "depth_cameras"
    lib_dir = os.path.join(ROOT, "pcl_tracking_b200", "lib")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src),
                           "-L", lib_dir, "-lpft", "-Wl,-rpath," + lib_dir])
    return str(exe)


def test_depth_cameras_program_builds_and_fails_loudly_without_gpu(tmp_path):
    exe = build_depth_cameras(tmp_path)
    from pcl_tracking_b200 import _capi
    if _capi.load().pft_device_count() > 0:
        return  # tests/test_gpu_depth_cameras.py runs it
    (tmp_path / "d.raw").write_bytes(b"\0" * 8)
    (tmp_path / "c.raw").write_bytes(b"\0" * 12)
    (tmp_path / "m.raw").write_bytes(b"\0" * 48)
    cam = [str(tmp_path / "d.raw"), str(tmp_path / "c.raw"), "2", "2", "4", "6", "365", "365", "1", "1"]
    r = subprocess.run([exe, str(tmp_path / "o.raw")] + cam + ["-"] + cam + [str(tmp_path / "m.raw")], capture_output=True, text=True)
    assert r.returncode == 3
    assert "no CPU fallback" in r.stderr
