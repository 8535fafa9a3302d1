// gemv driver, in the style of drivers/gemm.cpp (the reference declares flash::gemv but has no driver for it):
//   <A_file> <x_file> <y_file> <A_nrows> <A_ncols> <alpha> <beta> <trans N|T> <order R|C> <lda>
// All three files are mapped; y is updated in place (its old contents are read only when beta != 0).
#include "driver_common.h"

int main(int argc, char** argv) {
  if (argc != 11)
    drv::usage_exit("gemv <A> <x> <y> <m> <n> <alpha> <beta> <trans N|T> <order R|C> <lda>");
  flash::flash_setup("/tmp/gemv_driver_temps");
  auto A = flash::map_file<FPTYPE>(argv[1], flash::Mode::READWRITE);
  auto x = flash::map_file<FPTYPE>(argv[2], flash::Mode::READWRITE);
  auto y = flash::map_file<FPTYPE>(argv[3], flash::Mode::READWRITE);
  const FBLAS_UINT m = drv::to_u(argv[4]), n = drv::to_u(argv[5]);
  drv::StopWatch sw;
  const FBLAS_INT rc = flash::gemv(argv[9][0], argv[8][0], m, n, drv::to_f(argv[6]), drv::to_f(argv[7]), A, x, y,
                                   drv::to_u(argv[10]));
  drv::report("gemv()", sw.seconds(), rc);
  flash::unmap_file(A);
  flash::unmap_file(x);
  flash::unmap_file(y);
  flash::flash_destroy();
  return rc == 0 ? 0 : 1;
}
