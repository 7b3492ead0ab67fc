/* TEST: the GeneralizedIterativeClosestPoint part of include/pe_b200.h is plain C99 — peb_gicp_params, its defaults (PCL
 * 1.10's), the entry points' signatures — and without a GPU the library says so instead of computing anything. */
#include <float.h>
#include <stdio.h>

#include "pe_b200.h"

int main(void) {
  peb_gicp_params p;
  peb_icp_result r;
  peb_ctx* ctx = NULL;
  double cov[9];
  float guess[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
  int (*align)(peb_ctx*, const float*, const peb_gicp_params*, peb_icp_result*, float*, int32_t*, float*) = peb_gicp_align;
  int (*batch)(peb_ctx*, const float*, size_t, const peb_gicp_params*, peb_icp_result*) = peb_gicp_align_batch;
  int (*covs)(peb_ctx*, int, int, double*) = peb_gicp_covariances;
  int rc;
  if (sizeof(peb_gicp_params) != 48) {
    printf("layout %zu\n", sizeof(peb_gicp_params));
    return 1;
  }
  peb_gicp_params_default(&p);
  if (p.max_iterations != 200 || p.k_correspondences != 20 || p.max_inner_iterations != 20 || p.max_corr_dist != 5.0 ||
      p.transformation_epsilon != 5e-4 || p.rotation_epsilon != 2e-3 || p.fitness_max_range != DBL_MAX) {
    printf("PCL 1.10 defaults wrong\n");
    return 2;
  }
  rc = peb_ctx_create(0, &ctx);
  if (rc != PEB_OK) {
    printf("ctx_create %d: %s\n", rc, peb_last_error(NULL));
    return ctx == NULL ? 10 : 5;
  }
  /* no source, no target: the library's own status, nothing computed */
  if (align(ctx, guess, &p, &r, NULL, NULL, NULL) != PEB_E_NO_TARGET) return 6;
  if (batch(ctx, guess, 1, &p, &r) != PEB_E_NO_TARGET) return 7;
  if (covs(ctx, 0, 20, cov) != PEB_E_NO_TARGET) return 8;
  peb_ctx_destroy(ctx);
  printf("ctx ok\n");
  return 0;
}
