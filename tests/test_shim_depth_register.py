"""The registration fields of the C++ shim's pft::DepthCamera (setDepthToColour, the depth camera's size and intrinsics,
fill_upsampling) compile and link with plain g++ against libpft.so.  tests/test_gpu_depth_register.py runs the program
on the device."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# depth_register out.raw [camera] ...
# camera = depth.raw denc depth_w depth_h depth_step colour.raw cenc w h colour_step fx fy cx cy pose.raw|- then
#          "-" (already registered: depth_w x depth_h = w x h) or depth_to_colour.raw (12 float64) depth_fx depth_fy
#          depth_cx depth_cy depth_Tx depth_Ty colour_Tx colour_Ty fill_upsampling
# Fuses the cameras with fromDepthImages (from the files' buffers) and fromDepthImagesAsync (from pinned copies), prints
# "<points> <width> <height>" of each cloud and writes the clouds' 32-byte records to out.raw in that order.
DEPTH_REGISTER_CPP = r'''
#include <pft/pcl_shim.hpp>

#include <iterator>

static std::vector<unsigned char> slurp(const char* path) {
  std::ifstream f(path, std::ios::binary);
  return std::vector<unsigned char>((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
}

// any affine type with operator()(row, col) holding doubles, standing in for Eigen::Affine3d
struct Affine3d {
  double m[3][4];
  double operator()(int r, int c) const { return m[r][c]; }
};

int main(int argc, char** argv) {
  if (argc < 3) { fprintf(stderr, "usage: %s out.raw camera...\n", argv[0]); return 2; }
  std::vector<std::vector<unsigned char>> depth, colour;
  std::vector<pft::DepthCamera> cams;
  for (int i = 2; i < argc;) {
    if (argc - i < 16) { fprintf(stderr, "short camera\n"); return 2; }
    char** a = argv + i;
    pft::DepthCamera c;
    depth.push_back(slurp(a[0]));
    c.depth_encoding = a[1];
    const uint32_t dw = (uint32_t)atoi(a[2]), dh = (uint32_t)atoi(a[3]);
    c.depth_step = (uint32_t)atoi(a[4]);
    colour.push_back(slurp(a[5]));
    c.colour_encoding = a[6];
    c.width = (uint32_t)atoi(a[7]); c.height = (uint32_t)atoi(a[8]);
    c.bgr_step = (uint32_t)atoi(a[9]);
    c.fx = atof(a[10]); c.fy = atof(a[11]); c.cx = atof(a[12]); c.cy = atof(a[13]);
    if (strcmp(a[14], "-") != 0) {
      const std::vector<unsigned char> m = slurp(a[14]);
      pft::Affine3f t;
      for (int r = 0; r < 3; ++r) for (int col = 0; col < 4; ++col) memcpy(&t(r, col), m.data() + 4 * (r * 4 + col), 4);
      c.setPose(t);
    }
    if (strcmp(a[15], "-") == 0) {
      i += 16;
    } else {
      if (argc - i < 25) { fprintf(stderr, "short registration\n"); return 2; }
      const std::vector<unsigned char> m = slurp(a[15]);
      Affine3d t;
      memcpy(t.m, m.data(), sizeof(t.m));
      c.setDepthToColour(t);
      c.depth_width = dw; c.depth_height = dh;
      c.depth_fx = atof(a[16]); c.depth_fy = atof(a[17]); c.depth_cx = atof(a[18]); c.depth_cy = atof(a[19]);
      c.depth_tx = atof(a[20]); c.depth_ty = atof(a[21]); c.colour_tx = atof(a[22]); c.colour_ty = atof(a[23]);
      c.fill_upsampling = atoi(a[24]) != 0;
      i += 25;
    }
    cams.push_back(c);
  }
  const size_t n = cams.size();
  try {
    typedef pcl::PointXYZRGBA P;
    pcl::PointCloud<P> a, b;
    for (size_t k = 0; k < n; ++k) { cams[k].depth = depth[k].data(); cams[k].bgr = colour[k].data(); }
    a.fromDepthImages(cams);
    std::vector<void*> pinned;
    for (size_t k = 0; k < n; ++k) {
      void* pd = nullptr;
      void* pc = nullptr;
      pft::check(pft_host_alloc(&pd, depth[k].size()));
      pft::check(pft_host_alloc(&pc, colour[k].size()));
      memcpy(pd, depth[k].data(), depth[k].size());
      memcpy(pc, colour[k].data(), colour[k].size());
      cams[k].depth = pd;
      cams[k].bgr = static_cast<const uint8_t*>(pc);
      pinned.push_back(pd);
      pinned.push_back(pc);
    }
    b.fromDepthImagesAsync(cams);
    std::ofstream out(argv[1], std::ios::binary);
    for (pcl::PointCloud<P>* c : {&a, &b}) {
      const uint32_t cw = c->width, ch = c->height;
      c->download();
      printf("%zu %u %u\n", c->points.size(), cw, ch);
      out.write(reinterpret_cast<const char*>(c->points.data()), (std::streamsize)(c->points.size() * sizeof(P)));
    }
    for (void* p : pinned) pft_host_free(p);
  } catch (const pft::Error& e) {
    fprintf(stderr, "%s\n", e.what());
    return e.code == PFT_ERR_INVALID ? 4 : 3;
  }
  return 0;
}
'''


def build_depth_register(tmp_path):
    src = tmp_path / "depth_register.cpp"
    src.write_text(DEPTH_REGISTER_CPP)
    exe = tmp_path / "depth_register"
    lib_dir = os.path.join(ROOT, "pcl_tracking_b200", "lib")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src),
                           "-L", lib_dir, "-lpft", "-Wl,-rpath," + lib_dir])
    return str(exe)


def test_depth_register_program_builds_and_fails_loudly_without_gpu(tmp_path):
    exe = build_depth_register(tmp_path)
    from pcl_tracking_b200 import _capi
    if _capi.load().pft_device_count() > 0:
        return  # tests/test_gpu_depth_register.py runs it
    (tmp_path / "d.raw").write_bytes(b"\0" * 8)
    (tmp_path / "c.raw").write_bytes(b"\0" * 12)
    (tmp_path / "m.raw").write_bytes(b"\0" * 96)
    cam = [str(tmp_path / "d.raw"), "16UC1", "2", "2", "4", str(tmp_path / "c.raw"), "bgr8", "2", "2", "6", "365", "365", "1", "1", "-",
           str(tmp_path / "m.raw"), "365", "365", "1", "1", "0", "0", "0.052", "0", "1"]
    r = subprocess.run([exe, str(tmp_path / "o.raw")] + cam, capture_output=True, text=True)
    assert r.returncode == 3 and "no CPU fallback" in r.stderr, r.stderr
