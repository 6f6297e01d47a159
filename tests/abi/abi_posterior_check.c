/* Plain-C client of include/gpb200_posterior.h: the companion header compiles as C99 together with gpb200.h, every entry
 * point it declares resolves with dlsym, and argument validation returns the documented status codes before any CUDA
 * call.  Built and run by tests/test_abi_posterior.py; needs no GPU. */
#include <dlfcn.h>
#include <stdio.h>

#include "gpb200_posterior.h"

#define CHECK(cond)                                                     \
  do {                                                                  \
    if (!(cond)) { fprintf(stderr, "FAILED: %s (line %d)\n", #cond, __LINE__); return 1; } \
  } while (0)

typedef int (*version_fn)(void);
typedef int (*pred_gx_fn)(int, const double*, int, long, const double*, int, long, int, const double*, int,
                          const double*, const double*, int, long, const double*, long, const double*, const double*,
                          long, double*, long, void*);

int main(int argc, char** argv) {
  static const char* names[] = {"gpb_pred_gx"};
  void* lib;
  size_t i;
  version_fn version;
  pred_gx_fn pred_gx;
  double x[4] = {0.0, 1.0, 2.0, 3.0};
  double g[4] = {0.0, 0.0, 0.0, 0.0};
  CHECK(argc == 2);
  lib = dlopen(argv[1], RTLD_NOW | RTLD_LOCAL);
  if (!lib) { fprintf(stderr, "dlopen: %s\n", dlerror()); return 1; }
  for (i = 0; i < sizeof(names) / sizeof(names[0]); ++i) {
    if (!dlsym(lib, names[i])) { fprintf(stderr, "missing symbol %s\n", names[i]); return 1; }
  }
  *(void**)(&version) = dlsym(lib, "gpb_version");
  *(void**)(&pred_gx) = dlsym(lib, "gpb_pred_gx");
  CHECK(version() >= 102);
  /* argument validation happens before any CUDA call: these return without touching a device */
  CHECK(pred_gx(GPB_KERN_LINEAR, x, 1, 1, x, 1, 1, 1, x, 1, x, x, 1, 1, x, 1, x, x, 1, g, 1, NULL) == GPB_ERR_BADARG);
  CHECK(pred_gx(GPB_KERN_RBF, NULL, 1, 1, x, 1, 1, 1, x, 1, x, x, 1, 1, x, 1, x, x, 1, g, 1, NULL) == GPB_ERR_BADARG);
  CHECK(pred_gx(GPB_KERN_RBF, x, 0, 1, x, 1, 1, 1, x, 1, x, x, 1, 1, x, 1, x, x, 1, g, 1, NULL) == GPB_ERR_BADARG);
  CHECK(pred_gx(GPB_KERN_RBF, x, 1, 1, x, 2, 1, 1, x, 1, x, x, 1, 1, x, 1, x, x, 1, g, 1, NULL) == GPB_ERR_BADARG);
  CHECK(pred_gx(GPB_KERN_RBF, x, 1, 161, x, 1, 161, 161, x, 1, x, x, 1, 1, x, 1, x, x, 1, g, 161, NULL) ==
        GPB_ERR_UNSUPPORTED);
  printf("abi_posterior_check: %d symbols ok\n", (int)(sizeof(names) / sizeof(names[0])));
  dlclose(lib);
  return 0;
}
