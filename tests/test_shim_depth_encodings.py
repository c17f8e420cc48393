"""The depth-image ingest of the C++ shim in every encoding (the sensor_msgs/Image::encoding overloads of
pcl::PointCloud::fromDepthImage / fromDepthImageAsync, and pft::DepthCamera's depth_encoding / colour_encoding for
fromDepthImages) compiles and links with plain g++ against libpft.so.  tests/test_gpu_depth_encodings.py runs the
program on the device."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# depth_encodings out.raw [depth.raw depth_enc colour.raw|- colour_enc width height depth_step colour_step fx fy cx cy pose.raw|-] ...
# Fuses the cameras (13 arguments each; colour "-": no file, a null pointer; pose.raw holds 12 float32, "-" for none)
# with fromDepthImages (from the files' buffers) and fromDepthImagesAsync (from pinned copies).  With one camera it
# also converts it with the encoding overloads fromDepthImage (files' buffers) and fromDepthImageAsync (pinned).
# Prints "<points> <width> <height>" of each cloud and writes the clouds' 32-byte records to out.raw in that order.
DEPTH_ENCODINGS_CPP = r'''
#include <pft/pcl_shim.hpp>

#include <iterator>

static std::vector<unsigned char> slurp(const char* path) {
  std::ifstream f(path, std::ios::binary);
  return std::vector<unsigned char>((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
}

int main(int argc, char** argv) {
  if (argc < 15 || (argc - 2) % 13) {
    fprintf(stderr, "usage: %s out.raw [depth.raw denc colour.raw|- cenc w h depth_step colour_step fx fy cx cy pose.raw|-] ...\n", argv[0]);
    return 2;
  }
  const int n = (argc - 2) / 13;
  std::vector<std::vector<unsigned char>> depth(n), colour(n);
  std::vector<pft::DepthCamera> cams(n);
  std::vector<bool> has_colour(n);
  for (int k = 0; k < n; ++k) {
    char** a = argv + 2 + 13 * k;
    depth[k] = slurp(a[0]);
    has_colour[k] = strcmp(a[2], "-") != 0;
    if (has_colour[k]) colour[k] = slurp(a[2]);
    pft::DepthCamera& c = cams[k];
    c.depth_encoding = a[1];
    c.colour_encoding = a[3];
    c.width = (uint32_t)atoi(a[4]); c.height = (uint32_t)atoi(a[5]);
    c.depth_step = (uint32_t)atoi(a[6]); c.bgr_step = (uint32_t)atoi(a[7]);
    c.fx = atof(a[8]); c.fy = atof(a[9]); c.cx = atof(a[10]); c.cy = atof(a[11]);
    if (strcmp(a[12], "-") != 0) {
      const std::vector<unsigned char> m = slurp(a[12]);
      pft::Affine3f t;
      for (int r = 0; r < 3; ++r) for (int col = 0; col < 4; ++col) memcpy(&t(r, col), m.data() + 4 * (r * 4 + col), 4);
      c.setPose(t);
    }
  }
  try {
    typedef pcl::PointXYZRGBA P;
    std::vector<pcl::PointCloud<P>::Ptr> clouds;
    for (int k = 0; k < 4; ++k) clouds.emplace_back(new pcl::PointCloud<P>());
    for (int k = 0; k < n; ++k) {
      cams[k].depth = depth[k].data();
      cams[k].bgr = has_colour[k] ? colour[k].data() : nullptr;
    }
    clouds[0]->fromDepthImages(cams);
    if (n == 1) {
      const pft::DepthCamera& c = cams[0];
      clouds[2]->fromDepthImage(c.depth, c.depth_step, c.depth_encoding, c.bgr, c.bgr_step, c.colour_encoding, c.width, c.height, c.fx, c.fy, c.cx, c.cy);
    }
    std::vector<void*> pinned;
    for (int k = 0; k < n; ++k) {
      void* pd = nullptr;
      pft::check(pft_host_alloc(&pd, depth[k].size()));
      memcpy(pd, depth[k].data(), depth[k].size());
      cams[k].depth = pd;
      pinned.push_back(pd);
      if (has_colour[k]) {
        void* pc = nullptr;
        pft::check(pft_host_alloc(&pc, colour[k].size()));
        memcpy(pc, colour[k].data(), colour[k].size());
        cams[k].bgr = static_cast<const uint8_t*>(pc);
        pinned.push_back(pc);
      }
    }
    clouds[1]->fromDepthImagesAsync(cams);
    if (n == 1) {
      const pft::DepthCamera& c = cams[0];
      clouds[3]->fromDepthImageAsync(c.depth, c.depth_step, c.depth_encoding, c.bgr, c.bgr_step, c.colour_encoding, c.width, c.height, c.fx, c.fy, c.cx,
                                     c.cy);
    }
    std::ofstream out(argv[1], std::ios::binary);
    for (int k = 0; k < (n == 1 ? 4 : 2); ++k) {
      pcl::PointCloud<P>& c = *clouds[k];
      const uint32_t cw = c.width, ch = c.height;
      c.download();
      printf("%zu %u %u\n", c.points.size(), cw, ch);
      out.write(reinterpret_cast<const char*>(c.points.data()), (std::streamsize)(c.points.size() * sizeof(P)));
    }
    for (void* p : pinned) pft_host_free(p);
  } catch (const pft::Error& e) {
    fprintf(stderr, "%s\n", e.what());
    return e.code == PFT_ERR_INVALID ? 4 : 3;
  }
  return 0;
}
'''


def build_depth_encodings(tmp_path):
    src = tmp_path / "depth_encodings.cpp"
    src.write_text(DEPTH_ENCODINGS_CPP)
    exe = tmp_path / "depth_encodings"
    lib_dir = os.path.join(ROOT, "pcl_tracking_b200", "lib")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src),
                           "-L", lib_dir, "-lpft", "-Wl,-rpath," + lib_dir])
    return str(exe)


def run_depth_encodings(exe, tmp_path, denc, cenc):
    """The program on one 2x2 camera of zero bytes in the given encodings (steps of 8 bytes fit every encoding)."""
    (tmp_path / "d.raw").write_bytes(b"\0" * 16)
    (tmp_path / "c.raw").write_bytes(b"\0" * 16)
    cam = [str(tmp_path / "d.raw"), denc, str(tmp_path / "c.raw"), cenc, "2", "2", "8", "8", "365", "365", "1", "1", "-"]
    return subprocess.run([exe, str(tmp_path / "o.raw")] + cam, capture_output=True, text=True)


def test_depth_encodings_program_builds_and_fails_loudly_without_gpu(tmp_path):
    exe = build_depth_encodings(tmp_path)
    from pcl_tracking_b200 import _capi
    if _capi.load().pft_device_count() > 0:
        return  # tests/test_gpu_depth_encodings.py runs it
    for denc, cenc in (("16UC1", "bgr8"), ("mono16", "none"), ("32FC1", "rgba8"), ("32FC1", "mono8")):
        r = run_depth_encodings(exe, tmp_path, denc, cenc)
        assert r.returncode == 3 and "no CPU fallback" in r.stderr, (denc, cenc, r.stderr)
