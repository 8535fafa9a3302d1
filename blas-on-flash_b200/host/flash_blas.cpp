// flash:: adapters over the C ABI (include/bof_b200.h): the C++ host side of the drop-in boundary.
// Each function flattens its flash_ptr arguments (mmap address of the file, include/pointers/pointer.h)
// and calls the matching bof_host_* pipeline; nothing here computes.
#include <cstdio>
#include <cstdlib>
#include <map>
#include <mutex>
#include <vector>

#include "flash_blas.h"
#include "lib_funcs.h"

namespace flash {

std::string mnt_dir = "./";
Callback dummy_std_func = [] {};

namespace {
std::mutex g_mu;
bof_ctx* g_ctx = nullptr;
bof_mgpu* g_mgpu = nullptr;   // BOF_GPUS > 1: one context per GPU in this process, g_ctx = its rank 0

// BOF_GPUS=<n> | all : spread gemm / gemv / csrmm / csrgemv / kmeans_lloyd over the GPUs of the node (default: one GPU)
int env_gpus() {
  const char* v = std::getenv("BOF_GPUS");
  if (!v) return 1;
  if (std::string(v) == "all") return 0;
  return std::max(1, std::atoi(v));
}

int env_device() {
  for (const char* name : {"BOF_DEVICE", "LOCAL_RANK"})
    if (const char* v = std::getenv(name)) return std::atoi(v);
  return 0;
}

// matrices pinned in HBM by csr_pin, keyed by the address of their value array
struct Pinned { bof_csr* h; FBLAS_UINT m, n; const void *ia, *ja; };
std::map<const void*, Pinned> g_pinned;

bof_csr* find_pinned(flash_ptr<FPTYPE> a, flash_ptr<MKL_INT> ia, flash_ptr<MKL_INT> ja, FBLAS_UINT m, FBLAS_UINT n) {
  std::lock_guard<std::mutex> lk(g_mu);
  auto it = g_pinned.find(a.ptr);
  if (it == g_pinned.end()) return nullptr;
  const Pinned& p = it->second;
  return (p.m == m && p.n == n && p.ia == ia.ptr && p.ja == ja.ptr) ? p.h : nullptr;
}

FBLAS_INT done(const char* what, int rc) {
  if (rc == 0) return 0;
  const char* msg = g_ctx ? bof_last_error(g_ctx) : bof_last_error(nullptr);
  if (g_mgpu && bof_mgpu_last_error(g_mgpu)[0]) msg = bof_mgpu_last_error(g_mgpu);
  std::fprintf(stderr, "[flash::%s] %s\n", what, msg);
  return -1;
}
bool multi() { return g_mgpu != nullptr && bof_mgpu_count(g_mgpu) > 1; }
}  // namespace

bof_ctx* flash_context() {
  std::lock_guard<std::mutex> lk(g_mu);
  if (g_ctx == nullptr && env_gpus() != 1) {
    bof_config cfg{};
    if (bof_mgpu_create(&cfg, env_gpus(), nullptr, &g_mgpu) == 0) {
      g_ctx = bof_mgpu_ctx(g_mgpu, 0);
    } else {
      std::fprintf(stderr, "[flash] cannot create the multi-GPU context (%s); falling back to one GPU\n", bof_last_error(nullptr));
      g_mgpu = nullptr;
    }
  }
  if (g_ctx == nullptr) {
    bof_config cfg{};
    cfg.device = env_device();
    if (bof_ctx_create(&cfg, &g_ctx) != 0) {
      std::fprintf(stderr, "[flash] cannot create the B200 context: %s\n", bof_last_error(nullptr));
      g_ctx = nullptr;
    }
  }
  return g_ctx;
}

void flash_setup(std::string mntdir) {
  mnt_dir = mntdir;
  if (!mnt_dir.empty() && mnt_dir.back() != '/') mnt_dir += '/';
  (void)flash_context();
}

void flash_destroy() {
  std::lock_guard<std::mutex> lk(g_mu);
  for (auto& kv : g_pinned) bof_csr_close(kv.second.h);
  g_pinned.clear();
  if (g_mgpu) bof_mgpu_destroy(g_mgpu);   // owns g_ctx
  else if (g_ctx) bof_ctx_destroy(g_ctx);
  g_mgpu = nullptr;
  g_ctx = nullptr;
}

FBLAS_INT gemm(CHAR mat_ord, CHAR trans_a, CHAR trans_b, FBLAS_UINT m, FBLAS_UINT n, FBLAS_UINT k, FPTYPE alpha,
               FPTYPE beta, flash_ptr<FPTYPE> a, flash_ptr<FPTYPE> b, flash_ptr<FPTYPE> c, FBLAS_UINT lda_a,
               FBLAS_UINT lda_b, FBLAS_UINT lda_c) {
  bof_ctx* ctx = flash_context();
  if (!ctx) return -1;
  if (multi())
    return done("gemm", bof_mgpu_gemm(g_mgpu, mat_ord, trans_a, trans_b, (int64_t)m, (int64_t)n, (int64_t)k, alpha, beta, a.ptr,
                                      b.ptr, c.ptr, (int64_t)lda_a, (int64_t)lda_b, (int64_t)lda_c));
  return done("gemm", bof_host_gemm(ctx, mat_ord, trans_a, trans_b, (int64_t)m, (int64_t)n, (int64_t)k, alpha, beta,
                                    a.ptr, b.ptr, c.ptr, (int64_t)lda_a, (int64_t)lda_b, (int64_t)lda_c));
}

FBLAS_INT gemv(CHAR mat_ord, CHAR trans_a, FBLAS_UINT m, FBLAS_UINT n, FPTYPE alpha, FPTYPE beta, flash_ptr<FPTYPE> a,
               flash_ptr<FPTYPE> b, flash_ptr<FPTYPE> c, FBLAS_UINT lda_a) {
  return gemv(mat_ord, trans_a, m, n, alpha, beta, a, b.ptr, c.ptr, lda_a);
}

FBLAS_INT gemv(CHAR mat_ord, CHAR trans_a, FBLAS_UINT m, FBLAS_UINT n, FPTYPE alpha, FPTYPE beta, flash_ptr<FPTYPE> a,
               FPTYPE* b, FPTYPE* c, FBLAS_UINT lda_a) {
  bof_ctx* ctx = flash_context();
  if (!ctx) return -1;
  if (multi())
    return done("gemv", bof_mgpu_gemv(g_mgpu, mat_ord, trans_a, (int64_t)m, (int64_t)n, alpha, beta, a.ptr, (int64_t)lda_a,
                                      b, c));
  return done("gemv", bof_host_gemv(ctx, mat_ord, trans_a, (int64_t)m, (int64_t)n, alpha, beta, a.ptr, (int64_t)lda_a, b, c));
}

FBLAS_INT kmeans(CHAR mat_ord, CHAR trans_a, CHAR trans_b, FBLAS_UINT m, FBLAS_UINT n, FBLAS_UINT k, FPTYPE alpha,
                 FPTYPE beta, flash_ptr<FPTYPE> a, flash_ptr<FPTYPE> b, flash_ptr<FPTYPE> c, FBLAS_UINT lda_a,
                 FBLAS_UINT lda_b, FBLAS_UINT lda_c, FPTYPE* c_l2sq, FPTYPE* p_l2sq, FPTYPE* /*ones*/) {
  // KMeansTask::execute (reference include/tasks/kmeans_task.h:68-80): the product, then the two rank-1 updates
  // C(i, j) += c_l2sq[i] and C(i, j) += p_l2sq[j], in that order -- applied on the device before each block
  // of C is downloaded.
  bof_ctx* ctx = flash_context();
  if (!ctx) return -1;
  return done("kmeans", bof_host_kmeans_dist(ctx, mat_ord, trans_a, trans_b, (int64_t)m, (int64_t)n, (int64_t)k, alpha,
                                            beta, a.ptr, b.ptr, c.ptr, (int64_t)lda_a, (int64_t)lda_b, (int64_t)lda_c,
                                            c_l2sq, p_l2sq));
}

FBLAS_INT csrmm(CHAR trans_a, FBLAS_UINT m, FBLAS_UINT n, FBLAS_UINT k, FPTYPE alpha, FPTYPE beta,
                flash_ptr<FPTYPE> a, flash_ptr<MKL_INT> ia, flash_ptr<MKL_INT> ja, CHAR ord_b, flash_ptr<FPTYPE> b,
                flash_ptr<FPTYPE> c) {
  return csrmm(trans_a, m, n, k, alpha, beta, a, ia, ja, ord_b, b.ptr, c.ptr);
}

FBLAS_INT csrmm(CHAR trans_a, FBLAS_UINT m, FBLAS_UINT n, FBLAS_UINT k, FPTYPE alpha, FPTYPE beta,
                flash_ptr<FPTYPE> a, flash_ptr<MKL_INT> ia, flash_ptr<MKL_INT> ja, CHAR ord_b, FPTYPE* b, FPTYPE* c) {
  bof_ctx* ctx = flash_context();
  if (!ctx) return -1;
  if (bof_csr* h = find_pinned(a, ia, ja, m, n))
    return done("csrmm", bof_csr_mm(h, trans_a, (int64_t)k, alpha, beta, ord_b, b, c));
  if (multi())
    return done("csrmm", bof_mgpu_csrmm(g_mgpu, trans_a, (int64_t)m, (int64_t)n, (int64_t)k, alpha, beta, a.ptr,
                                        reinterpret_cast<const int64_t*>(ia.ptr), reinterpret_cast<const int64_t*>(ja.ptr),
                                        ord_b, b, c));
  return done("csrmm", bof_host_csrmm(ctx, trans_a, (int64_t)m, (int64_t)n, (int64_t)k, alpha, beta, a.ptr,
                                      reinterpret_cast<const int64_t*>(ia.ptr),
                                      reinterpret_cast<const int64_t*>(ja.ptr), ord_b, b, c));
}

FBLAS_INT csrcsc(FBLAS_UINT m, FBLAS_UINT n, flash_ptr<MKL_INT> ia, flash_ptr<MKL_INT> ja, flash_ptr<FPTYPE> a,
                 flash_ptr<MKL_INT> ia_tr, flash_ptr<MKL_INT> ja_tr, flash_ptr<FPTYPE> a_tr) {
  bof_ctx* ctx = flash_context();
  if (!ctx) return -1;
  return done("csrcsc", bof_host_csrcsc(ctx, (int64_t)m, (int64_t)n, reinterpret_cast<const int64_t*>(ia.ptr),
                                        reinterpret_cast<const int64_t*>(ja.ptr), a.ptr,
                                        reinterpret_cast<int64_t*>(ia_tr.ptr), reinterpret_cast<int64_t*>(ja_tr.ptr),
                                        a_tr.ptr));
}

FBLAS_INT csrgemv(CHAR trans_a, FBLAS_UINT m, FBLAS_UINT n, flash_ptr<FPTYPE> a, flash_ptr<MKL_INT> ia,
                  flash_ptr<MKL_INT> ja, FPTYPE* b, FPTYPE* c) {
  bof_ctx* ctx = flash_context();
  if (!ctx) return -1;
  if (bof_csr* h = find_pinned(a, ia, ja, m, n)) return done("csrgemv", bof_csr_mv(h, trans_a, b, c));
  if (multi())
    return done("csrgemv", bof_mgpu_csrgemv(g_mgpu, trans_a, (int64_t)m, (int64_t)n, a.ptr, reinterpret_cast<const int64_t*>(ia.ptr),
                                            reinterpret_cast<const int64_t*>(ja.ptr), b, c));
  return done("csrgemv", bof_host_csrgemv(ctx, trans_a, (int64_t)m, (int64_t)n, a.ptr,
                                          reinterpret_cast<const int64_t*>(ia.ptr),
                                          reinterpret_cast<const int64_t*>(ja.ptr), b, c));
}

FBLAS_INT csr_pin(FBLAS_UINT m, FBLAS_UINT n, flash_ptr<FPTYPE> a, flash_ptr<MKL_INT> ia, flash_ptr<MKL_INT> ja,
                  bool with_transpose) {
  bof_ctx* ctx = flash_context();
  if (!ctx) return -1;
  csr_unpin(a);
  bof_csr* h = nullptr;
  int rc = bof_csr_open(ctx, (int64_t)m, (int64_t)n, a.ptr, reinterpret_cast<const int64_t*>(ia.ptr),
                        reinterpret_cast<const int64_t*>(ja.ptr), &h);
  if (rc == 0 && with_transpose) rc = bof_csr_build_transpose(h);
  if (rc != 0) {
    if (h) bof_csr_close(h);
    return done("csr_pin", rc);
  }
  std::lock_guard<std::mutex> lk(g_mu);
  g_pinned[a.ptr] = Pinned{h, m, n, ia.ptr, ja.ptr};
  return 0;
}

FBLAS_INT csr_unpin(flash_ptr<FPTYPE> a) {
  std::lock_guard<std::mutex> lk(g_mu);
  auto it = g_pinned.find(a.ptr);
  if (it == g_pinned.end()) return 0;
  bof_csr_close(it->second.h);
  g_pinned.erase(it);
  return 0;
}

FBLAS_INT kmeans_lloyd(flash_ptr<FPTYPE> points, flash_ptr<FPTYPE> centers, FBLAS_UINT npoints, FBLAS_UINT ndims,
                       FBLAS_UINT ncenters, FBLAS_UINT n_iters, FBLAS_UINT* closest_center,
                       kmeans_allreduce_fn allreduce, void* allreduce_user) {
  bof_ctx* ctx = flash_context();
  if (!ctx) return -1;
  static_assert(sizeof(FBLAS_UINT) == sizeof(int64_t), "assignment buffer is 64-bit");
  if (multi() && allreduce == nullptr)   // this process drives several GPUs: the library shards and allreduces itself
    return done("kmeans_lloyd", bof_mgpu_kmeans_lloyd(g_mgpu, (int64_t)npoints, (int64_t)ncenters, (int64_t)ndims, points.ptr,
                                                      centers.ptr, (int64_t)n_iters, reinterpret_cast<int64_t*>(closest_center)));
  bof_kmeans* km = nullptr;
  int rc = bof_kmeans_open(ctx, (int64_t)npoints, (int64_t)ncenters, (int64_t)ndims, points.ptr, centers.ptr, &km);
  for (FBLAS_UINT it = 0; rc == 0 && it < n_iters; ++it) {
    void* partial = nullptr;
    size_t count = 0;
    rc = bof_kmeans_local_step(km, &partial, &count);
    if (rc == 0 && allreduce != nullptr && allreduce(partial, count, bof_kmeans_stream(km), allreduce_user) != 0) {
      std::fprintf(stderr, "[flash::kmeans_lloyd] allreduce callback failed\n");
      bof_kmeans_close(km);
      return -1;
    }
    if (rc == 0) rc = bof_kmeans_update(km);
  }
  if (rc == 0) {
    rc = bof_kmeans_get(km, centers.ptr, reinterpret_cast<int64_t*>(closest_center));
  }
  if (km) bof_kmeans_close(km);
  return done("kmeans_lloyd", rc);
}

}  // namespace flash
