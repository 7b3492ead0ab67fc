// TEST: pe_b200::GeneralizedIterativeClosestPoint (include/pe_b200/pcl_facade.hpp) builds with plain g++ and, on a GPU,
// gives the C ABI's records.  argv: source.bin target.bin guesses.bin out.bin — float32 x y z 1 records, H x 16 floats
// (column-major), and the output: the single align's record of guess 0, then the batch's H records.
#include <cstdio>
#include <vector>

#include "pe_b200/pcl_facade.hpp"

static std::vector<float> read_floats(const char* path) {
  std::vector<float> v;
  if (FILE* f = std::fopen(path, "rb")) {
    float x;
    while (std::fread(&x, sizeof(x), 1, f) == 1) v.push_back(x);
    std::fclose(f);
  }
  return v;
}

int main(int argc, char** argv) {
  if (argc != 5) return 2;
  const std::vector<float> src = read_floats(argv[1]), tgt = read_floats(argv[2]), guesses = read_floats(argv[3]);
  try {
    pe_b200::Context ctx(0);
    pe_b200::GeneralizedIterativeClosestPoint gicp(ctx);
    gicp.setInputSource(src.data(), src.size() / 4, 16);
    gicp.setInputTarget(tgt.data(), tgt.size() / 4, 16);
    gicp.setMaxCorrespondenceDistance(0.05);
    gicp.setMaximumIterations(30);
    gicp.setCorrespondenceRandomness(20);
    gicp.setMaximumOptimizerIterations(20);
    gicp.setRotationEpsilon(2e-3);
    gicp.setTransformationEpsilon(5e-4);
    std::vector<float> aligned;
    gicp.align(&aligned, guesses.data());
    std::vector<peb_icp_result> batch;
    gicp.alignBatch(guesses.data(), guesses.size() / 16, batch);
    FILE* f = std::fopen(argv[4], "wb");
    if (!f) return 3;
    std::fwrite(&gicp.result(), sizeof(peb_icp_result), 1, f);
    std::fwrite(batch.data(), sizeof(peb_icp_result), batch.size(), f);
    std::fclose(f);
    std::printf("gicp facade: %d iterations, converged %d, fitness %.6e, %zu aligned points\n", gicp.nr_iterations(),
                gicp.hasConverged() ? 1 : 0, gicp.getFitnessScore(), aligned.size() / 4);
  } catch (const pe_b200::Error& e) {
    std::printf("error %d: %s\n", e.code, e.what());
    return 1;
  }
  return 0;
}
