/* cv_normals_check.cpp — TEST PROGRAM for peb_cv_normals / peb_cv_normals_dev and the facade's computeNormalsPC3d.
 * Compiles as C99 (gcc -x c: the prototypes of include/pe_b200.h) and as C++17 (include/pe_b200/pcl_facade.hpp).
 *   cv_normals_check IN.f32 N K FLIP OUT.f32
 * reads N x 3 floats, writes the N x 6 rows computeNormalsPC3d returns (viewpoint 0 0 0) to OUT.f32.
 * Exit codes: 0 ok, 2 usage / io, 3 no context (the library's message on stderr), 4 the call failed. */
#include <stdio.h>
#include <stdlib.h>

#ifdef __cplusplus
#include <vector>

#include "pe_b200/pcl_facade.hpp"
#else
#include "pe_b200.h"
#endif

typedef int (*cv_normals_fn)(peb_ctx*, const void*, size_t, size_t, int, int, const float*, float*, int32_t*);
typedef int (*cv_normals_dev_fn)(peb_ctx*, const void*, size_t, int, int, const float*, void*);

int main(int argc, char** argv) {
  cv_normals_fn host = &peb_cv_normals; /* the prototypes are what the ABI says */
  cv_normals_dev_fn dev = &peb_cv_normals_dev;
  size_t n, got;
  int k, flip;
  float* in;
  float* out;
  const float vp[3] = {0.0f, 0.0f, 0.0f};
  FILE* f;
  if (argc != 6 || !host || !dev) return 2;
  n = (size_t)strtoull(argv[2], NULL, 10);
  k = atoi(argv[3]);
  flip = atoi(argv[4]);
  in = (float*)malloc(3 * n * sizeof(float) + 4);
  out = (float*)malloc(6 * n * sizeof(float) + 4);
  f = fopen(argv[1], "rb");
  if (!in || !out || !f) return 2;
  got = fread(in, sizeof(float), 3 * n, f);
  fclose(f);
  if (got != 3 * n) return 2;
#ifdef __cplusplus
  {
    pe_b200::Context* ctx = nullptr;
    try {
      ctx = new pe_b200::Context(0);
    } catch (const pe_b200::Error& e) {
      fprintf(stderr, "%s\n", e.what());
      return 3;
    }
    try {
      pe_b200::computeNormalsPC3d(*ctx, in, n, 12, k, flip != 0, vp, out);
    } catch (const pe_b200::Error& e) {
      fprintf(stderr, "pe_b200 error %d: %s\n", e.code, e.what());
      delete ctx;
      return 4;
    }
    delete ctx;
  }
#else
  {
    peb_ctx* ctx = NULL;
    int rc = peb_ctx_create(0, &ctx);
    if (rc != PEB_OK) {
      fprintf(stderr, "%s\n", peb_last_error(NULL));
      return 3;
    }
    rc = host(ctx, in, n, 12, k, flip, vp, out, NULL);
    if (rc != PEB_OK) {
      fprintf(stderr, "%s\n", peb_last_error(ctx));
      peb_ctx_destroy(ctx);
      return 4;
    }
    peb_ctx_destroy(ctx);
  }
#endif
  f = fopen(argv[5], "wb");
  if (!f) return 2;
  got = fwrite(out, sizeof(float), 6 * n, f);
  fclose(f);
  free(in);
  free(out);
  return got == 6 * n ? 0 : 2;
}
