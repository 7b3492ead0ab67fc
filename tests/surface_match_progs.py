"""Sources of the two small programs the peb_surface_match tests build in a temporary directory: a pedantic C99 consumer of
the header and a g++ consumer of the facade.  Both pin the layout of the two new structs, and both can run the whole
find_object_in_scene chain on files written by the tests (the C++ one can also pack refined records)."""
import subprocess
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
LIB_DIR = ROOT / "pose_estimation_b200"

# offsets / sizes of peb_surface_match_params and peb_surface_match_result (x86-64 / aarch64 LP64)
LAYOUT_CHECKS = r"""
#define SM_CHECK(name, cond) typedef char name[(cond) ? 1 : -1]
SM_CHECK(smp_size, sizeof(peb_surface_match_params) == 64);
SM_CHECK(smp_k, offsetof(peb_surface_match_params, normals_k) == 0);
SM_CHECK(smp_flip, offsetof(peb_surface_match_params, flip_viewpoint) == 4);
SM_CHECK(smp_vp, offsetof(peb_surface_match_params, viewpoint) == 8);
SM_CHECK(smp_max, offsetof(peb_surface_match_params, max_icp_poses) == 20);
SM_CHECK(smp_step, offsetof(peb_surface_match_params, relative_scene_sample_step) == 24);
SM_CHECK(smp_dist, offsetof(peb_surface_match_params, relative_scene_distance) == 32);
SM_CHECK(smp_icp, offsetof(peb_surface_match_params, icp) == 40);
SM_CHECK(smp_layout, offsetof(peb_surface_match_params, reference_layout) == 56);
SM_CHECK(smr_size, sizeof(peb_surface_match_result) == 48);
SM_CHECK(smr_nres, offsetof(peb_surface_match_result, n_results) == 0);
SM_CHECK(smr_nref, offsetof(peb_surface_match_result, n_refined) == 8);
SM_CHECK(smr_best, offsetof(peb_surface_match_result, best) == 12);
SM_CHECK(smr_pose7, offsetof(peb_surface_match_result, pose7) == 16);
"""

# run: <model.f32> <n_model> <cloud.f32 (x y z 1 rows)> <n> <num_planes> <leaf> <out prefix>
C_SRC = r"""
#include <stddef.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "pe_b200.h"
""" + LAYOUT_CHECKS + r"""
static float* load(const char* path, size_t n_floats) {
  float* p = (float*)malloc(n_floats * sizeof(float) + 4);
  FILE* f = fopen(path, "rb");
  if (!p || !f || fread(p, sizeof(float), n_floats, f) != n_floats) exit(2);
  fclose(f);
  return p;
}
static void save(const char* prefix, const char* what, const void* p, size_t bytes) {
  char path[1024];
  FILE* f;
  snprintf(path, sizeof(path), "%s.%s", prefix, what);
  f = fopen(path, "wb");
  if (!f || (bytes && fwrite(p, 1, bytes, f) != bytes)) exit(2);
  fclose(f);
}
int main(int argc, char** argv) {
  size_t n_model, n, m = 0;
  float *model, *cloud, *scene;
  peb_ctx* ctx = NULL;
  peb_ppf_model* det = NULL;
  peb_ppf_params pp;
  peb_prefilter_params filter;
  peb_sac_params sac;
  peb_surface_match_params prm;
  peb_surface_match_result res;
  peb_ppf_pose refined[6];
  int rc;
  if (argc != 8) return 2;
  n_model = (size_t)atol(argv[2]);
  n = (size_t)atol(argv[4]);
  model = load(argv[1], 6 * n_model);
  cloud = load(argv[3], 4 * n);
  scene = (float*)malloc(6 * n * sizeof(float) + 4);
  if (peb_ctx_create(0, &ctx) != PEB_OK) {
    fprintf(stderr, "%s\n", peb_last_error(NULL));
    return 3;
  }
  peb_ppf_params_default(&pp);
  rc = peb_ppf_train(ctx, model, n_model, &pp, &det);
  peb_surface_match_params_default(&prm);
  peb_sac_params_default(&sac);
  sac.distance_threshold = 0.0001;
  sac.max_iterations = 100;
  memset(&filter, 0, sizeof(filter));
  filter.plane_band = 0.005f;
  if (rc == PEB_OK)
    rc = peb_surface_match(ctx, det, cloud, n, 16, &filter, atoi(argv[5]), &sac, (float)atof(argv[6]), &prm, refined, &res,
                           scene, &m);
  if (rc != PEB_OK) {
    fprintf(stderr, "%s\n", peb_last_error(ctx));
    return 4;
  }
  save(argv[7], "refined", refined, (size_t)res.n_refined * sizeof(peb_ppf_pose));
  save(argv[7], "result", &res, sizeof(res));
  save(argv[7], "scene", scene, m * 6 * sizeof(float));
  peb_ppf_model_destroy(det);
  peb_ctx_destroy(ctx);
  free(model);
  free(cloud);
  free(scene);
  return 0;
}
"""

# pack <records.bin> <count> <out.f32>           : pack_pose3d of every record, corrected then reference layout
# run  <model.f32> <n_model> <cloud.f32> <n> <num_planes> <leaf> <out prefix>  : the chain through the facade
CPP_SRC = r"""
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include "pe_b200/pcl_facade.hpp"
""" + LAYOUT_CHECKS + r"""
static std::vector<char> load(const char* path, size_t bytes) {
  std::vector<char> v(bytes + 4);
  FILE* f = std::fopen(path, "rb");
  if (!f || std::fread(v.data(), 1, bytes, f) != bytes) std::exit(2);
  std::fclose(f);
  return v;
}
static void save(const std::string& path, const void* p, size_t bytes) {
  FILE* f = std::fopen(path.c_str(), "wb");
  if (!f || (bytes && std::fwrite(p, 1, bytes, f) != bytes)) std::exit(2);
  std::fclose(f);
}
int main(int argc, char** argv) {
  if (argc == 5 && std::string(argv[1]) == "pack") {
    const size_t cnt = static_cast<size_t>(std::atol(argv[3]));
    std::vector<char> raw = load(argv[2], cnt * sizeof(peb_ppf_pose));
    std::vector<float> out(14 * cnt);
    for (size_t i = 0; i < cnt; ++i) {
      peb_ppf_pose p;
      std::memcpy(&p, raw.data() + i * sizeof(p), sizeof(p));
      pe_b200::pack_pose3d(p, &out[14 * i], false);
      pe_b200::pack_pose3d(p, &out[14 * i + 7], true);
    }
    save(argv[4], out.data(), out.size() * sizeof(float));
    return 0;
  }
  if (argc != 9 || std::string(argv[1]) != "run") return 2;
  const size_t n_model = static_cast<size_t>(std::atol(argv[3])), n = static_cast<size_t>(std::atol(argv[5]));
  std::vector<char> model = load(argv[2], n_model * 24), cloud = load(argv[4], n * 16);
  try {
    pe_b200::Context c(0);
    pe_b200::PPF3DDetector det(c, 0.03, 0.03, 40);
    det.trainModel(reinterpret_cast<const float*>(model.data()), n_model);
    peb_surface_match_params prm;
    peb_surface_match_params_default(&prm);
    std::vector<peb_ppf_pose> refined;
    std::vector<float> scene;
    float pose7[7];
    const peb_surface_match_result r = pe_b200::find_object_in_scene(c, det, cloud.data(), n, 16, nullptr, 0.0f, "", std::atoi(argv[6]),
                                                                     static_cast<float>(std::atof(argv[7])), prm, refined, pose7, &scene);
    const std::string prefix = argv[8];
    save(prefix + ".refined", refined.data(), refined.size() * sizeof(peb_ppf_pose));
    save(prefix + ".result", &r, sizeof(r));
    save(prefix + ".scene", scene.data(), scene.size() * sizeof(float));
    if (std::memcmp(pose7, r.pose7, sizeof(pose7)) != 0) return 5;
  } catch (const pe_b200::Error& e) {
    std::fprintf(stderr, "%s\n", e.what());
    return 3;
  }
  return 0;
}
"""


def build(tmp_path, which: str) -> Path:
    """Compiles the C ('c', warnings are errors) or the facade ('cpp') program into tmp_path and links it."""
    if which == "c":
        src, cc = tmp_path / "sm_check.c", ["gcc", "-x", "c", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror"]
        src.write_text(C_SRC)
    else:
        src, cc = tmp_path / "sm_check.cpp", ["g++", "-std=c++17", "-O1", "-Wall", "-Wextra"]
        src.write_text(CPP_SRC)
    exe = tmp_path / f"sm_check_{which}"
    r = subprocess.run(cc + ["-I", str(ROOT / "include"), str(src), "-o", str(exe), "-L", str(LIB_DIR), "-lpe_b200", "-lm",
                             f"-Wl,-rpath,{LIB_DIR}"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe
