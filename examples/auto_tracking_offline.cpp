// auto_tracking_offline.cpp -- the reference's tracking node without ROS, on recorded frames.
//
// initialize_trackers() and cloud_cb() of ref: src/auto_tracking.cpp:181-259, :597-727, written against
// include/pft/pcl_shim.hpp (PCL class names over the C ABI).  The ROS subscriber / service / visualiser
// parts of that file are out of scope; frames and the object model come from .pcd files (ASCII or binary, as the
// model builder writes them, ref: src/create_model.cpp:209-230) or from raw files of 32-byte pcl::PointXYZRGBA records.
//
// usage: auto_tracking_offline <model.pcd|raw>[,<model2> ...] <seed> <frame0.pcd|raw> [frame1 ...]
// One tracker per model, like the reference's tracker_vector_ (ref :198-258, :688-697); tracker k is seeded with seed + k.
// Prints one line per frame and object, objects in the order given: frame index, particle count, result x y z roll
// pitch yaw.  With PFT_OBJECT_DEVICES=0,1,... the trackers are spread over those GPUs (pcl_shim.hpp).
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "pft/pcl_shim.hpp"

typedef pcl::PointXYZRGBA RefPointType;
typedef pcl::tracking::ParticleXYZRPY ParticleT;
typedef pcl::PointCloud<RefPointType> Cloud;
typedef pcl::tracking::KLDAdaptiveParticleFilterOMPTracker<RefPointType, ParticleT> Tracker;

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

int main(int argc, char** argv) {
  if (argc < 4) { std::fprintf(stderr, "usage: %s model.raw[,model2.raw ...] seed frame0.raw [frame1.raw ...]\n", argv[0]); return 2; }
  std::vector<std::string> model_files;
  for (std::string rest = argv[1];;) {
    const size_t comma = rest.find(',');
    model_files.push_back(rest.substr(0, comma));
    if (comma == std::string::npos) break;
    rest = rest.substr(comma + 1);
  }
  try {
    // ---- initialize_trackers (ref :181-259): same literals
    std::vector<double> default_step_covariance(6, 0.015 * 0.015);
    default_step_covariance[3] *= 40.0; default_step_covariance[4] *= 40.0; default_step_covariance[5] *= 40.0;
    std::vector<double> initial_noise_covariance(6, 0.00001), default_initial_mean(6, 0.0);
    std::vector<std::shared_ptr<Tracker>> trackers;
    for (size_t k = 0; k < model_files.size(); ++k) {
      std::shared_ptr<Tracker> tracker(new Tracker(16));
      ParticleT bin_size;
      bin_size.x = bin_size.y = bin_size.z = bin_size.roll = bin_size.pitch = bin_size.yaw = 0.1f;
      tracker->setMaximumParticleNum(500);
      tracker->setDelta(0.99);
      tracker->setEpsilon(0.2);
      tracker->setBinSize(bin_size);
      tracker->setTrans(pft::Affine3f::Identity());
      tracker->setStepNoiseCovariance(default_step_covariance);
      tracker->setInitialNoiseCovariance(initial_noise_covariance);
      tracker->setInitialNoiseMean(default_initial_mean);
      tracker->setIterationNum(2);
      tracker->setParticleNum(400);
      tracker->setResampleLikelihoodThr(0.00);
      tracker->setUseNormal(false);
      auto coherence = std::make_shared<pcl::tracking::ApproxNearestPairPointCloudCoherence<RefPointType>>();
      coherence->addPointCoherence(std::make_shared<pcl::tracking::DistanceCoherence<RefPointType>>());
      auto color_coherence = std::make_shared<pcl::tracking::HSVColorCoherence<RefPointType>>();
      color_coherence->setWeight(0.1);
      coherence->addPointCoherence(color_coherence);
      coherence->setSearchMethod(std::make_shared<pcl::search::Octree<RefPointType>>(0.01));
      coherence->setMaximumDistance(0.1);
      tracker->setCloudCoherence(coherence);
      pft::check(pft_tracker_seed(tracker->handle(), (uint64_t)std::strtoull(argv[2], nullptr, 10) + k));  // upstream: time(0)

      // ---- frame 2 of cloud_cb (ref :643-679): model -> centroid frame -> VoxelGrid -> setReferenceCloud; setTrans(centroid)
      Cloud::Ptr raw_model = load_raw(model_files[k].c_str());
      Cloud::Ptr model(new Cloud());
      float c[3];
      pft::check(pft_prepare_model(pft::Context::Default()->get(), raw_model->device(), model->device(), 0.01f, c));
      model->mark_device_written();
      pft::Affine3f trans = pft::Affine3f::Identity();
      trans.translation(c[0], c[1], c[2]);
      tracker->setReferenceCloud(model);
      tracker->setTrans(trans);
      tracker->setMinIndices((int)model->size() / 2);
      trackers.push_back(tracker);
    }

    // ---- frames > 2 (ref :637, :683, :688-697)
    pcl::PassThrough<RefPointType> pass;
    pass.setFilterFieldName("z");
    pass.setFilterLimits(0.0, 10.0);
    pass.setKeepOrganized(false);
    pcl::ApproximateVoxelGrid<RefPointType> grid;
    grid.setLeafSize(0.01f, 0.01f, 0.01f);
    for (int f = 3; f < argc; ++f) {
      Cloud::Ptr cloud = load_raw(argv[f]);
      Cloud::Ptr cloud_pass(new Cloud()), cloud_pass_downsampled(new Cloud());
      pass.setInputCloud(cloud);
      pass.filter(*cloud_pass);
      grid.setInputCloud(cloud_pass);
      grid.filter(*cloud_pass_downsampled);
      for (auto& tracker : trackers) {  // compute() does not block: the trackers of several GPUs run at once
        tracker->setInputCloud(cloud_pass_downsampled);
        tracker->compute();
      }
      for (auto& tracker : trackers) {
        const ParticleT r = tracker->getResult();
        const size_t n = tracker->getParticles()->points.size();
        const pft::Affine3f T = r.toEigenMatrix();
        std::printf("%d %zu %.9g %.9g %.9g %.9g %.9g %.9g  T03=%.9g\n", f - 3, n, r.x, r.y, r.z, r.roll, r.pitch, r.yaw, T(0, 3));
      }
    }
  } catch (const pft::Error& e) {
    std::fprintf(stderr, "%s\n", e.what());
    return e.code == PFT_ERR_CUDA ? 3 : 1;
  }
  return 0;
}
