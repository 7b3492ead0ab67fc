// The rejector chain's ABI and the facade's chain (include/pe_b200.h : peb_rejector, pcl_facade.hpp).
// Always: the record's layout.  With a device: the facade keeps PCL's order, and bad chains are refused.
// Exit 0: all checks passed; 1: a check failed; 3: no device (after the layout checks passed).
#include <cmath>
#include <cstddef>
#include <cstdio>
#include <limits>

#include "pe_b200/pcl_facade.hpp"

#define CHECK(c)                                       \
  do {                                                 \
    if (!(c)) {                                        \
      std::printf("FAILED: %s (line %d)\n", #c, __LINE__); \
      return 1;                                        \
    }                                                  \
  } while (0)

int main() {
  CHECK(sizeof(peb_rejector) == 16);
  CHECK(offsetof(peb_rejector, kind) == 0);
  CHECK(offsetof(peb_rejector, min_correspondences) == 4);
  CHECK(offsetof(peb_rejector, value) == 8);
  CHECK(sizeof(peb_icp_params) == 72);
  CHECK(PEB_REJECTOR_DISTANCE == 0 && PEB_REJECTOR_MEDIAN_DISTANCE == 1 && PEB_REJECTOR_ONE_TO_ONE == 2 &&
        PEB_REJECTOR_TRIMMED == 3 && PEB_MAX_REJECTORS == 8);
  std::printf("layout ok\n");
  try {
    pe_b200::Context ctx(0);
    pe_b200::IterativeClosestPoint icp(ctx);
    // a distance rejector before any other one is params().rejector_max_dist; after one it joins the chain in order
    icp.addCorrespondenceRejectorDistance(0.01);
    icp.addCorrespondenceRejectorOneToOne();
    icp.addCorrespondenceRejectorDistance(0.005);
    icp.addCorrespondenceRejectorMedianDistance(2.0);
    icp.addCorrespondenceRejectorTrimmed(0.7, 5);
    CHECK(icp.params().rejector_max_dist == 0.01);
    const std::vector<peb_rejector>& c = icp.correspondenceRejectors();
    CHECK(c.size() == 4);
    CHECK(c[0].kind == PEB_REJECTOR_ONE_TO_ONE);
    CHECK(c[1].kind == PEB_REJECTOR_DISTANCE && c[1].value == 0.005);
    CHECK(c[2].kind == PEB_REJECTOR_MEDIAN_DISTANCE && c[2].value == 2.0);
    CHECK(c[3].kind == PEB_REJECTOR_TRIMMED && c[3].value == 0.7 && c[3].min_correspondences == 5);
    std::printf("facade chain ok\n");

    // bad chains: PEB_E_INVALID_ARG with a message, before anything runs
    float pts[12] = {0, 0, 0, 1, 0.01f, 0, 0, 1, 0, 0.01f, 0, 1};
    ctx.check(peb_source_set(ctx.get(), pts, 3, 16));
    ctx.check(peb_target_set(ctx.get(), pts, 3, 16, nullptr, 0));
    peb_icp_params prm;
    peb_icp_params_default(&prm);
    peb_icp_result res;
    const float eye[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
    peb_rejector bad[PEB_MAX_REJECTORS + 1];
    for (auto& r : bad) r = peb_rejector{PEB_REJECTOR_ONE_TO_ONE, 0, 0.0};
    CHECK(peb_icp_align_ex(ctx.get(), nullptr, &prm, nullptr, 1, &res, nullptr, nullptr, nullptr) == PEB_E_INVALID_ARG);
    CHECK(peb_icp_align_ex(ctx.get(), nullptr, &prm, bad, PEB_MAX_REJECTORS + 1, &res, nullptr, nullptr, nullptr) == PEB_E_INVALID_ARG);
    bad[0].kind = 7;
    CHECK(peb_icp_align_ex(ctx.get(), nullptr, &prm, bad, 1, &res, nullptr, nullptr, nullptr) == PEB_E_INVALID_ARG);
    CHECK(std::string(peb_last_error(ctx.get())).find("unknown kind") != std::string::npos);
    bad[0] = peb_rejector{PEB_REJECTOR_MEDIAN_DISTANCE, 0, std::numeric_limits<double>::quiet_NaN()};
    CHECK(peb_icp_align_batch_ex(ctx.get(), eye, 1, &prm, bad, 1, &res) == PEB_E_INVALID_ARG);
    bad[0] = peb_rejector{PEB_REJECTOR_TRIMMED, 0, std::numeric_limits<double>::infinity()};
    CHECK(peb_icp_align_batch_ex(ctx.get(), eye, 1, &prm, bad, 1, &res) == PEB_E_INVALID_ARG);
    CHECK(std::string(peb_last_error(ctx.get())).find("non-finite") != std::string::npos);
    std::printf("invalid chains refused\n");
  } catch (const pe_b200::Error& e) {
    std::fprintf(stderr, "pe_b200 error %d: %s\n", e.code, e.what());
    return 3;
  }
  return 0;
}
