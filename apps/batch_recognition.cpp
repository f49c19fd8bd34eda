// batch_recognition.cpp — a batch of scenes against one model with several scenes in flight on the GPU
// (BASELINE config 5, the per-GPU part): the C++ host side of the lanes, straight over the C ABI
// (b200_model_create_shot + b200_register_scene_batch_shot).  Parameters as SHOT_scenes.cpp:50-55.  With --hough, the
// reference's default branch instead: b200_model_create_shot_hough + b200_register_scene_batch_shot_hough (BOARD
// frames r = 0.02 with find_holes, Hough bin 0.02, threshold 2; the rand() stream of a fresh process, srand(1)).
//
// usage: batch_recognition [--hough] <model.f32> <model_kp.f32> <out_prefix> <lanes> <scene.f32> <scene_kp.f32> [<scene.f32> <scene_kp.f32> ...]
// writes <out_prefix>.<s>.T (instances x 16 float) and <out_prefix>.<s>.corr (b200_corr records) per scene s
#include <b200reg.h>

#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

static bool load(const char *path, std::vector<float> &xyz) {
  FILE *f = fopen(path, "rb");
  if (!f) {
    fprintf(stderr, "cannot open %s\n", path);
    return false;
  }
  float v[3];
  while (fread(v, sizeof(float), 3, f) == 3) xyz.insert(xyz.end(), v, v + 3);
  fclose(f);
  return true;
}

int main(int argc, char **argv) {
  const bool hough = argc > 1 && std::string(argv[1]) == "--hough";
  if (hough) {
    --argc;
    ++argv;
  }
  if (argc < 7 || ((argc - 5) % 2) != 0) {
    fprintf(stderr, "usage: %s [--hough] model.f32 model_kp.f32 out_prefix lanes scene.f32 scene_kp.f32 [...]\n", argv[0]);
    return 2;
  }
  const std::string prefix = argv[3];
  const int lanes = atoi(argv[4]);
  const int n_scenes = (argc - 5) / 2;
  std::vector<float> model, model_kp;
  if (!load(argv[1], model) || !load(argv[2], model_kp)) return 1;
  std::vector<std::vector<float>> scenes((size_t)n_scenes), kps((size_t)n_scenes);
  for (int s = 0; s < n_scenes; ++s)
    if (!load(argv[5 + 2 * s], scenes[(size_t)s]) || !load(argv[6 + 2 * s], kps[(size_t)s])) return 1;

  b200_shot_params p;
  p.normal_k = 20;
  p.normal_radius = 0.0;
  p.descr_radius = 0.02;
  p.match_mode = 1;
  p.match_thr = 0.25f;
  p.gc_size = 0.02;
  p.gc_threshold = 2;
  p.max_instances = 4096;
  b200_hough_params h;
  h.rf_radius = 0.02;
  b200_board_params_default(&h.board);
  h.board.find_holes = 1;
  h.bin_size = 0.02;
  h.threshold = 2.0;

  b200_ctx *ctx = nullptr;
  if (b200_ctx_create(&ctx, 0, nullptr) != B200_OK) {
    fprintf(stderr, "%s\n", b200_last_error(nullptr));
    return 1;
  }
  b200_model *m = nullptr;
  const int mrc = hough ? b200_model_create_shot_hough(ctx, model.data(), (int)model.size() / 3, 3, model_kp.data(),
                                                      (int)model_kp.size() / 3, 3, &p, &h, &m)
                        : b200_model_create_shot(ctx, model.data(), (int)model.size() / 3, 3, model_kp.data(),
                                                 (int)model_kp.size() / 3, 3, &p, &m);
  if (mrc != B200_OK) {
    fprintf(stderr, "%s\n", b200_last_error(ctx));
    return 1;
  }
  std::vector<const float *> sx, sk;
  std::vector<int> npts, nkp, cap, n_inst((size_t)n_scenes), n_corr((size_t)n_scenes), status((size_t)n_scenes);
  std::vector<std::vector<float>> T((size_t)n_scenes);
  std::vector<std::vector<int>> off((size_t)n_scenes);
  std::vector<std::vector<b200_corr>> ic((size_t)n_scenes), co((size_t)n_scenes);
  std::vector<float *> pT;
  std::vector<int *> poff;
  std::vector<b200_corr *> pic, pco;
  for (int s = 0; s < n_scenes; ++s) {
    const int K = (int)kps[(size_t)s].size() / 3;
    sx.push_back(scenes[(size_t)s].data());
    sk.push_back(kps[(size_t)s].data());
    npts.push_back((int)scenes[(size_t)s].size() / 3);
    nkp.push_back(K);
    cap.push_back(K > 0 ? K : 1);
    T[(size_t)s].resize((size_t)p.max_instances * 16);
    off[(size_t)s].resize((size_t)p.max_instances + 1);
    ic[(size_t)s].resize((size_t)cap.back());
    co[(size_t)s].resize((size_t)cap.back());
    pT.push_back(T[(size_t)s].data());
    poff.push_back(off[(size_t)s].data());
    pic.push_back(ic[(size_t)s].data());
    pco.push_back(co[(size_t)s].data());
  }
  const int rc =
      hough ? b200_register_scene_batch_shot_hough(0, m, n_scenes, sx.data(), npts.data(), 3, sk.data(), nkp.data(), 3, &p,
                                                   &h, lanes, pT.data(), poff.data(), pic.data(), cap.data(), n_inst.data(),
                                                   pco.data(), n_corr.data(), status.data())
            : b200_register_scene_batch_shot(0, m, n_scenes, sx.data(), npts.data(), 3, sk.data(), nkp.data(), 3, &p, lanes,
                                             pT.data(), poff.data(), pic.data(), cap.data(), n_inst.data(), pco.data(),
                                             n_corr.data(), status.data());
  if (rc != B200_OK) {
    fprintf(stderr, "%s\n", b200_last_error(nullptr));
    return 1;
  }
  for (int s = 0; s < n_scenes; ++s) {
    printf("scene %d: %d correspondences, %d instances\n", s, n_corr[(size_t)s], n_inst[(size_t)s]);
    const int kept = n_inst[(size_t)s] < p.max_instances ? n_inst[(size_t)s] : p.max_instances;
    FILE *f = fopen((prefix + "." + std::to_string(s) + ".T").c_str(), "wb");
    fwrite(T[(size_t)s].data(), sizeof(float), (size_t)kept * 16, f);
    fclose(f);
    f = fopen((prefix + "." + std::to_string(s) + ".corr").c_str(), "wb");
    fwrite(co[(size_t)s].data(), sizeof(b200_corr), (size_t)n_corr[(size_t)s], f);
    fclose(f);
  }
  b200_model_destroy(m);
  b200_ctx_destroy(ctx);
  return 0;
}
