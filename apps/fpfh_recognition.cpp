// fpfh_recognition.cpp — the FPFH variant of the reference's recognition callback
// (FPFH_demo.cpp:405-585) through the PCL-style adapters: normals on the keypoint clouds by radius
// (FPFH_demo.cpp:416-420, 486-492), FPFHEstimation with input = surface = keypoints
// (FPFH_demo.cpp:422-428, 505-510), KdTreeFLANN<FPFHSignature33> k = 2 with the ratio test
// (FPFH_demo.cpp:516-538), then grouping.  By default GeometricConsistencyGrouping (the north-star grouping, which
// FPFH_demo itself does not have); with --hough the reference's own grouping block (FPFH_demo.cpp:548-585):
// NormalEstimationOMP with k = 50 on the two dense clouds (FPFH_demo.cpp:405-409), BOARD frames of the keypoints over
// the dense clouds and their normals (FPFH_demo.cpp:556-568: find_holes, rf_rad_ 0.02; the model's frames, then the
// scene's, from one rand() stream), Hough3DGrouping with bin cg_size and threshold cg_thresh (0.02 / 2).
//
// usage: fpfh_recognition [--hough <model.f32> <scene.f32>] <model_kp.f32> <scene_kp.f32> <out_prefix> [radius=0.05]
//                         [cg_size=0.02] [cg_thresh=2]
// writes <out_prefix>.desc (scene FPFH33), .normals (scene keypoint normals), .corr (b200_corr records), .T (instances
//        x 16 float); with --hough also .rf (model then scene BOARD frames, 9 float each)
#include <pcl_b200/pcl_b200.h>

#include <cmath>
#include <cstdlib>
#include <iostream>
#include <string>

namespace pcl = pcl_b200;

typedef pcl::PointXYZRGBA PointType;
typedef pcl::Normal NormalType;
typedef pcl::FPFHSignature33 DescriptorType;

static bool load_cloud(const char *path, pcl::PointCloud<PointType> &cloud) {
  FILE *f = fopen(path, "rb");
  if (!f) return false;
  float xyz[3];
  while (fread(xyz, sizeof(float), 3, f) == 3) {
    PointType p;
    p.x = xyz[0], p.y = xyz[1], p.z = xyz[2];
    cloud.push_back(p);
  }
  fclose(f);
  return true;
}

int main(int argc, char **argv) {
  const bool use_hough = argc > 3 && std::string(argv[1]) == "--hough";
  const char *model_path = use_hough ? argv[2] : nullptr, *scene_path = use_hough ? argv[3] : nullptr;
  if (use_hough) {  // the dense clouds come first; the remaining arguments are those of the GC invocation
    argc -= 3;
    argv += 3;
  }
  if (argc < 4) {
    std::cerr << "usage: fpfh_recognition [--hough model.f32 scene.f32] model_kp.f32 scene_kp.f32 out_prefix "
              << "[radius cg_size cg_thresh]" << std::endl;
    return 2;
  }
  const double radius = argc > 4 ? atof(argv[4]) : 0.05;
  const float cg_size_ = argc > 5 ? (float)atof(argv[5]) : 0.02f;
  const float cg_thresh_ = argc > 6 ? (float)atof(argv[6]) : 2.0f;
  const float rf_rad_ = 0.02f;
  pcl::PointCloud<PointType>::Ptr model_keypoints(new pcl::PointCloud<PointType>()),
      scene_keypoints(new pcl::PointCloud<PointType>());
  pcl::PointCloud<NormalType>::Ptr model_normals(new pcl::PointCloud<NormalType>()),
      scene_normals(new pcl::PointCloud<NormalType>());
  pcl::PointCloud<DescriptorType>::Ptr model_descriptors(new pcl::PointCloud<DescriptorType>()),
      scene_descriptors(new pcl::PointCloud<DescriptorType>());
  if (!load_cloud(argv[1], *model_keypoints) || !load_cloud(argv[2], *scene_keypoints)) return 1;
  pcl::PointCloud<PointType>::Ptr model(new pcl::PointCloud<PointType>()), scene(new pcl::PointCloud<PointType>());
  pcl::PointCloud<NormalType>::Ptr model_cloud_normals(new pcl::PointCloud<NormalType>()),
      scene_cloud_normals(new pcl::PointCloud<NormalType>());
  if (use_hough) {
    if (!load_cloud(model_path, *model) || !load_cloud(scene_path, *scene)) return 1;
    // FPFH_demo.cpp:405-409: normals of the dense clouds, k = 50
    pcl::NormalEstimationOMP<PointType, NormalType> cloud_norm_est;
    cloud_norm_est.setKSearch(50);
    cloud_norm_est.setInputCloud(scene);
    cloud_norm_est.compute(*scene_cloud_normals);
    cloud_norm_est.setInputCloud(model);
    cloud_norm_est.compute(*model_cloud_normals);
  }

  pcl::search::KdTree<PointType>::Ptr kdtree(new pcl::search::KdTree<PointType>());
  pcl::NormalEstimationOMP<PointType, NormalType> norm_est;
  norm_est.setSearchMethod(kdtree);
  norm_est.setRadiusSearch(radius);
  norm_est.setInputCloud(scene_keypoints);
  norm_est.compute(*scene_normals);
  norm_est.setInputCloud(model_keypoints);
  norm_est.compute(*model_normals);

  pcl::FPFHEstimation<PointType, NormalType, DescriptorType> fpfh;
  fpfh.setSearchMethod(kdtree);
  fpfh.setRadiusSearch(radius);
  fpfh.setInputCloud(scene_keypoints);
  fpfh.setInputNormals(scene_normals);
  fpfh.compute(*scene_descriptors);
  fpfh.setInputCloud(model_keypoints);
  fpfh.setInputNormals(model_normals);
  fpfh.compute(*model_descriptors);

  pcl::CorrespondencesPtr model_scene_corrs(new pcl::Correspondences());
  pcl::KdTreeFLANN<DescriptorType> match_search;
  match_search.setInputCloud(model_descriptors);
  for (size_t i = 0; i < scene_descriptors->size(); ++i) {
    std::vector<int> neigh_indices(2);
    std::vector<float> neigh_sqr_dists(2);
    if (!std::isfinite(scene_descriptors->at(i).histogram[0])) continue;
    const int found_neighs = match_search.nearestKSearch(scene_descriptors->at(i), 2, neigh_indices, neigh_sqr_dists);
    if (found_neighs < 1) continue;
    const double tau = found_neighs > 1 ? (double)neigh_sqr_dists[0] / neigh_sqr_dists[1] : 0.0;
    if (tau <= 1) model_scene_corrs->push_back(pcl::Correspondence(neigh_indices[0], static_cast<int>(i), neigh_sqr_dists[0]));
  }
  std::cout << "Correspondences found: " << model_scene_corrs->size() << std::endl;

  std::vector<pcl::Matrix4f> rototranslations;
  std::vector<pcl::Correspondences> clustered_corrs;
  const std::string prefix = argv[3];
  if (use_hough) {
    // FPFH_demo.cpp:548-585
    pcl::PointCloud<pcl::ReferenceFrame>::Ptr model_rf(new pcl::PointCloud<pcl::ReferenceFrame>()),
        scene_rf(new pcl::PointCloud<pcl::ReferenceFrame>());
    pcl::BOARDLocalReferenceFrameEstimation<PointType, NormalType, pcl::ReferenceFrame> rf_est;
    rf_est.setFindHoles(true);
    rf_est.setRadiusSearch(rf_rad_);

    rf_est.setInputCloud(model_keypoints);
    rf_est.setInputNormals(model_cloud_normals);
    rf_est.setSearchSurface(model);
    rf_est.compute(*model_rf);

    rf_est.setInputCloud(scene_keypoints);
    rf_est.setInputNormals(scene_cloud_normals);
    rf_est.setSearchSurface(scene);
    rf_est.compute(*scene_rf);

    pcl::Hough3DGrouping<PointType, PointType, pcl::ReferenceFrame, pcl::ReferenceFrame> clusterer;
    clusterer.setHoughBinSize(cg_size_);
    clusterer.setHoughThreshold(cg_thresh_);
    clusterer.setUseInterpolation(false);
    clusterer.setUseDistanceWeight(true);
    clusterer.setInputCloud(model_keypoints);
    clusterer.setInputRf(model_rf);
    clusterer.setSceneCloud(scene_keypoints);
    clusterer.setSceneRf(scene_rf);
    clusterer.setModelSceneCorrespondences(model_scene_corrs);
    clusterer.recognize(rototranslations, clustered_corrs);

    FILE *frf = fopen((prefix + ".rf").c_str(), "wb");
    for (int side = 0; side < 2; ++side)
      for (const pcl::ReferenceFrame &r : (side ? *scene_rf : *model_rf).points) {
        fwrite(r.x_axis, sizeof(float), 3, frf);
        fwrite(r.y_axis, sizeof(float), 3, frf);
        fwrite(r.z_axis, sizeof(float), 3, frf);
      }
    fclose(frf);
  } else {
    pcl::GeometricConsistencyGrouping<PointType, PointType> gc_clusterer;
    gc_clusterer.setGCSize(cg_size_);
    gc_clusterer.setGCThreshold(cg_thresh_);
    gc_clusterer.setInputCloud(model_keypoints);
    gc_clusterer.setSceneCloud(scene_keypoints);
    gc_clusterer.setModelSceneCorrespondences(model_scene_corrs);
    gc_clusterer.recognize(rototranslations, clustered_corrs);
  }
  std::cout << "Model instances found: " << rototranslations.size() << std::endl;

  FILE *f = fopen((prefix + ".desc").c_str(), "wb");
  for (size_t i = 0; i < scene_descriptors->size(); ++i) fwrite(scene_descriptors->at(i).histogram, sizeof(float), 33, f);
  fclose(f);
  // the normals the descriptors were computed from (stage-by-stage parity checks start from identical inputs)
  f = fopen((prefix + ".normals").c_str(), "wb");
  for (size_t i = 0; i < scene_normals->size(); ++i) {
    const float n4[4] = {scene_normals->at(i).normal_x, scene_normals->at(i).normal_y, scene_normals->at(i).normal_z,
                         scene_normals->at(i).curvature};
    fwrite(n4, sizeof(float), 4, f);
  }
  fclose(f);
  f = fopen((prefix + ".corr").c_str(), "wb");
  if (!model_scene_corrs->empty()) fwrite(model_scene_corrs->data(), sizeof(pcl::Correspondence), model_scene_corrs->size(), f);
  fclose(f);
  f = fopen((prefix + ".T").c_str(), "wb");
  for (size_t i = 0; i < rototranslations.size(); ++i) fwrite(rototranslations[i].m, sizeof(float), 16, f);
  fclose(f);
  return 0;
}
