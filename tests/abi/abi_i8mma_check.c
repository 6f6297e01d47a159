/* Plain-C client of include/gpb200_i8mma.h: the companion header compiles as C99 together with gpb200.h, every entry
 * point it declares resolves with dlsym, and the switch follows the setter convention of gpb_ozaki_config (returns the
 * previous value, a negative argument only queries).  Built and run by tests/test_abi_i8mma.py; needs no GPU (the
 * process starts without GPB_I8MMA in its environment). */
#include <dlfcn.h>
#include <stdio.h>

#include "gpb200_i8mma.h"

#define CHECK(cond)                                                     \
  do {                                                                  \
    if (!(cond)) { fprintf(stderr, "FAILED: %s (line %d)\n", #cond, __LINE__); return 1; } \
  } while (0)

typedef int (*version_fn)(void);
typedef int (*config_fn)(int);

int main(int argc, char** argv) {
  static const char* names[] = {"gpb_i8mma_config"};
  void* lib;
  size_t i;
  version_fn version;
  config_fn config;
  CHECK(argc == 2);
  lib = dlopen(argv[1], RTLD_NOW | RTLD_LOCAL);
  if (!lib) { fprintf(stderr, "dlopen: %s\n", dlerror()); return 1; }
  for (i = 0; i < sizeof(names) / sizeof(names[0]); ++i) {
    if (!dlsym(lib, names[i])) { fprintf(stderr, "missing symbol %s\n", names[i]); return 1; }
  }
  *(void**)(&version) = dlsym(lib, "gpb_version");
  *(void**)(&config) = dlsym(lib, "gpb_i8mma_config");
  CHECK(version() >= 103);
  CHECK(config(-1) == 8);        /* on by default, 8 slices */
  CHECK(config(7) == 8);         /* returns the previous value */
  CHECK(config(-1) == 7);
  CHECK(config(1) == 7);         /* 1 and values above 8 select the default */
  CHECK(config(-1) == 8);
  CHECK(config(12) == 8);
  CHECK(config(-1) == 8);
  printf("abi_i8mma_check: %d symbols ok\n", (int)(sizeof(names) / sizeof(names[0])));
  dlclose(lib);
  return 0;
}
