// create_model_offline.cpp -- the reference's model builder without ROS, on one recorded frame.
//
// The object-cloud service of ref: src/create_model.cpp, written against include/pft/pcl_shim.hpp (PCL class names over
// the C ABI): the frame is cleaned of zero and NaN points (removeZeroPoints, ref :59-77), moved into the robot base
// frame (pcl_ros::transformPointCloud, ref :107-123), cropped to the segm_limits box of params.yaml by three
// PassThroughs (ref :148-162), split by EuclideanClusterExtraction(0.02, 500, 25000) (ref :169-179), and every cluster
// is moved back to the camera frame (ref :184-204) and written as one PCD file (ref :209-230).  The ROS service, tf
// and the parameter server are out of scope: the frame comes from a .pcd file or a raw file of 32-byte
// pcl::PointXYZRGBA records, the transform and the limits from the command line.
//
// usage: create_model_offline <frame.pcd|raw> <base_from_camera: 12 numbers> <xmin xmax ymin ymax zmin zmax> <out_dir>
// base_from_camera is the 3x4 row-major [R|t] that tf's lookupTransform(base, kinect2_link) gives, in double.  The
// forward transform rounds each entry to float, as pcl_ros does; the back transform camera_from_base is the inverse
// computed in double, (R^T, -R^T t) with each row of R^T t summed left to right, then rounded to float, as tf looks up
// the inverse in double rather than inverting the float matrix.  Writes <out_dir>/<j>.pcd (ASCII) for the clusters in
// rank order (largest first) and prints one line per cluster: its index and its number of points.  The files are the
// models auto_tracking_offline takes.
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "pft/pcl_shim.hpp"

typedef pcl::PointXYZRGBA RefPointType;
typedef pcl::PointCloud<RefPointType> Cloud;

static Cloud::Ptr load_raw(const char* path) {
  const std::string p(path);
  if (p.size() > 4 && p.compare(p.size() - 4, 4, ".pcd") == 0) {
    Cloud::Ptr c(new Cloud());
    if (pcl::io::loadPCDFile(p, *c) != 0) { std::fprintf(stderr, "cannot read %s as a PCD file\n", path); std::exit(2); }
    return c;
  }
  FILE* f = std::fopen(path, "rb");
  if (!f) { std::fprintf(stderr, "cannot open %s\n", path); std::exit(2); }
  std::fseek(f, 0, SEEK_END);
  const long bytes = std::ftell(f);
  std::fseek(f, 0, SEEK_SET);
  Cloud::Ptr c(new Cloud());
  c->points.resize((size_t)bytes / sizeof(RefPointType));
  if (std::fread(c->points.data(), sizeof(RefPointType), c->points.size(), f) != c->points.size()) { std::fprintf(stderr, "short read\n"); std::exit(2); }
  std::fclose(f);
  c->width = (uint32_t)c->points.size();
  c->touch();
  return c;
}

static double number(const char* s) {
  char* end = nullptr;
  const double v = std::strtod(s, &end);
  if (end == s || *end) { std::fprintf(stderr, "not a number: %s\n", s); std::exit(2); }
  return v;
}

// removeZeroPoints (ref :59-77), on the device: drops non-finite points and those with |x|, |y|, |z| all < 0.01
static void removeZeroPoints(const Cloud::ConstPtr& in, Cloud& out) {
  auto& ctx = pft::Context::Default();
  pft::check(pft_remove_zero_points(ctx->get(), in->device(ctx), out.device(ctx)));
  out.mark_device_written();
}

int main(int argc, char** argv) {
  if (argc != 21) {
    std::fprintf(stderr, "usage: %s frame.pcd|frame.raw <base_from_camera: 12 numbers, 3x4 row-major> xmin xmax ymin ymax zmin zmax out_dir\n", argv[0]);
    return 2;
  }
  double bc[12];
  for (int k = 0; k < 12; ++k) bc[k] = number(argv[2 + k]);
  float limits[6];
  for (int k = 0; k < 6; ++k) limits[k] = (float)number(argv[14 + k]);
  const std::string out_dir = argv[20];
  // the two Eigen::Affine3f pcl_ros builds from the double tf transforms
  pft::Affine3f base_from_camera, camera_from_base;
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 3; ++c) {
      base_from_camera(r, c) = (float)bc[r * 4 + c];
      camera_from_base(r, c) = (float)bc[c * 4 + r];
    }
    base_from_camera(r, 3) = (float)bc[r * 4 + 3];
    camera_from_base(r, 3) = (float)-((bc[0 * 4 + r] * bc[3] + bc[1 * 4 + r] * bc[7]) + bc[2 * 4 + r] * bc[11]);
  }
  try {
    Cloud::Ptr frame = load_raw(argv[1]);
    Cloud::Ptr nonzero(new Cloud()), base(new Cloud()), crop_x(new Cloud()), crop_xy(new Cloud()), crop(new Cloud());
    removeZeroPoints(frame, *nonzero);                                // ref :59-77
    pcl::transformPointCloud(*nonzero, *base, base_from_camera);     // ref :107-123
    pcl::PassThrough<RefPointType> pass;                              // ref :148-162 (segm_limits)
    pass.setInputCloud(base);
    pass.setFilterFieldName("x"); pass.setFilterLimits(limits[0], limits[1]); pass.filter(*crop_x);
    pass.setInputCloud(crop_x);
    pass.setFilterFieldName("y"); pass.setFilterLimits(limits[2], limits[3]); pass.filter(*crop_xy);
    pass.setInputCloud(crop_xy);
    pass.setFilterFieldName("z"); pass.setFilterLimits(limits[4], limits[5]); pass.filter(*crop);
    pcl::EuclideanClusterExtraction<RefPointType> ec;                 // ref :169-179
    ec.setClusterTolerance(0.02);
    ec.setMinClusterSize(500);
    ec.setMaxClusterSize(25000);
    ec.setInputCloud(crop);
    std::vector<pcl::PointIndices> cluster_indices;
    ec.extract(cluster_indices);
    pcl::PCDWriter writer;
    for (size_t j = 0; j < cluster_indices.size(); ++j) {
      Cloud cluster, cluster_camera;
      ec.clusterCloud((int)j, cluster);
      pcl::transformPointCloud(cluster, cluster_camera, camera_from_base);  // ref :184-204
      const std::string path = out_dir + "/" + std::to_string(j) + ".pcd";
      if (writer.write(path, cluster_camera, false) != 0) { std::fprintf(stderr, "cannot write %s\n", path.c_str()); return 2; }  // ref :209-230
      std::printf("%zu %zu\n", j, cluster_indices[j].indices.size());
    }
  } catch (const pft::Error& e) {
    std::fprintf(stderr, "%s\n", e.what());
    return e.code == PFT_ERR_CUDA ? 3 : 1;
  }
  return 0;
}
