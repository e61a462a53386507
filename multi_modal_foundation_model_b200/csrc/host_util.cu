#include "host_util.h"
#include "../../include/mmfm_b200.h"

#include <stdarg.h>
#include <stdlib.h>

#include <mutex>

namespace mmfm {

static thread_local char g_err[1024] = {0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
const char* get_error() { return g_err; }

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    // The driver entry point is resolved at run time so the library links without libcuda (no GPU at build).
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  });
  return fn;
}

static int make_tmap_2d(CUtensorMap* out, const void* base, CUtensorMapDataType dt, uint32_t esize, uint64_t rows,
                        uint64_t cols, uint64_t ld, uint32_t box_cols, uint32_t box_rows, TmaSwizzle swz);

int make_tmap_bf16_2d(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld,
                      uint32_t box_cols, uint32_t box_rows, TmaSwizzle swz) {
  return make_tmap_2d(out, base, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, rows, cols, ld, box_cols, box_rows, swz);
}
int make_tmap_f32_2d(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_cols,
                     uint32_t box_rows, TmaSwizzle swz) {
  return make_tmap_2d(out, base, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, rows, cols, ld, box_cols, box_rows, swz);
}

static int make_tmap_2d(CUtensorMap* out, const void* base, CUtensorMapDataType dt, uint32_t esize, uint64_t rows,
                        uint64_t cols, uint64_t ld, uint32_t box_cols, uint32_t box_rows, TmaSwizzle swz) {
  EncodeTiledFn enc = get_encode();
  MMFM_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled unavailable (no CUDA driver?)");
  MMFM_REQUIRE(((uintptr_t)base & 15) == 0, "TMA base %p not 16-byte aligned", base);
  MMFM_REQUIRE((ld * esize) % 16 == 0, "TMA row pitch %llu elements is not a multiple of 16 bytes",
               (unsigned long long)ld);
  MMFM_REQUIRE(box_rows <= 256 && box_cols <= 256, "TMA box too large");
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstr[1] = {ld * esize};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUtensorMapSwizzle s = swz == TMA_SW_128  ? CU_TENSOR_MAP_SWIZZLE_128B
                         : swz == TMA_SW_64 ? CU_TENSOR_MAP_SWIZZLE_64B
                         : swz == TMA_SW_32 ? CU_TENSOR_MAP_SWIZZLE_32B
                                            : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUresult r = enc(out, dt, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, s, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  MMFM_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (%d) rows=%llu cols=%llu ld=%llu box=%ux%u", (int)r,
               (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld, box_cols, box_rows);
  return 0;
}

int make_tmap_bf16_3d(CUtensorMap* out, const void* base, uint64_t batch, uint64_t rows, uint64_t cols, uint64_t ld,
                      uint32_t box_cols, uint32_t box_rows, TmaSwizzle swz) {
  EncodeTiledFn enc = get_encode();
  MMFM_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled unavailable (no CUDA driver?)");
  MMFM_REQUIRE(((uintptr_t)base & 15) == 0, "TMA base %p not 16-byte aligned", base);
  MMFM_REQUIRE((ld * 2) % 16 == 0, "TMA row pitch %llu elements is not a multiple of 16 bytes", (unsigned long long)ld);
  MMFM_REQUIRE(box_rows <= 256 && box_cols <= 256, "TMA box too large");
  cuuint64_t gdim[3] = {cols, rows, batch};
  cuuint64_t gstr[2] = {ld * 2, rows * ld * 2};
  cuuint32_t box[3] = {box_cols, box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUtensorMapSwizzle s = swz == TMA_SW_128  ? CU_TENSOR_MAP_SWIZZLE_128B
                         : swz == TMA_SW_64 ? CU_TENSOR_MAP_SWIZZLE_64B
                         : swz == TMA_SW_32 ? CU_TENSOR_MAP_SWIZZLE_32B
                                            : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), gdim, gstr, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, s, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  MMFM_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (3-d) failed (%d) batch=%llu rows=%llu cols=%llu ld=%llu box=%ux%u",
               (int)r, (unsigned long long)batch, (unsigned long long)rows, (unsigned long long)cols,
               (unsigned long long)ld, box_cols, box_rows);
  return 0;
}

bool pdl_enabled() {
  static int on = -1;
  if (on < 0) {
    const char* e = getenv("MMFM_PDL");
    on = (e && e[0] == '1') ? 1 : 0;   // measured neutral on the default step (23 181 vs 23 319 trials/s): opt-in
  }
  return on != 0;
}

static thread_local const void* g_win_ptr = nullptr;
static thread_local size_t g_win_bytes = 0;

static int l2_persist_state() {   // -1 off, else the maximum window size in MB
  static int state = -2;
  if (state == -2) {
    const char* e = getenv("MMFM_L2_PERSIST");
    state = -1;
    if (e && e[0] == '1') {
      int dev = 0, max_persist = 0, max_win = 0;
      cudaGetDevice(&dev);
      cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, dev);
      cudaDeviceGetAttribute(&max_win, cudaDevAttrMaxAccessPolicyWindowSize, dev);
      const char* mb = getenv("MMFM_L2_PERSIST_MB");       // set-aside = largest window taken (default: the device maximum)
      if (mb && atoi(mb) > 0 && ((size_t)atoi(mb) << 20) < (size_t)max_persist) max_persist = atoi(mb) << 20;
      if (max_persist > 0 && max_win > 0 &&
          cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, (size_t)max_persist) == cudaSuccess) {
        state = max_persist >> 20;
        if (getenv("MMFM_L2_PERSIST_VERBOSE"))
          fprintf(stderr, "mmfm: persisting L2 set-aside %d MB, window limit %d MB\n", max_persist >> 20, max_win >> 20);
      }
    }
  }
  return state;
}

void set_l2_window(const void* ptr, size_t bytes) {
  g_win_ptr = ptr;
  g_win_bytes = bytes;
}

bool take_l2_window(cudaAccessPolicyWindow* w) {
  const void* ptr = g_win_ptr;
  const size_t bytes = g_win_bytes;
  g_win_ptr = nullptr;
  g_win_bytes = 0;
  const int lim = l2_persist_state();
  if (lim < 0 || ptr == nullptr || bytes == 0) return false;
  if (bytes > ((size_t)lim << 20)) return false;   // an output larger than the set-aside would only thrash it
  w->base_ptr = const_cast<void*>(ptr);
  w->num_bytes = bytes;
  w->hitRatio = 1.0f;
  w->hitProp = cudaAccessPropertyPersisting;
  w->missProp = cudaAccessPropertyStreaming;
  return true;
}

int device_sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

int det_ws_check(const void* buf, long long bytes, const unsigned int* tickets, int n_tickets, const DetNeed& need,
                 const char* who) {
  MMFM_REQUIRE(bytes >= need.bytes && n_tickets >= need.tickets,
               "%s: deterministic workspace too small (%lld bytes / %d tickets given, %lld / %d needed)", who, bytes,
               n_tickets, need.bytes, need.tickets);
  MMFM_REQUIRE(need.bytes == 0 || (buf != nullptr && (reinterpret_cast<uintptr_t>(buf) & 15) == 0),
               "%s: deterministic workspace buffer missing or not 16-byte aligned", who);
  MMFM_REQUIRE(need.tickets == 0 || tickets != nullptr, "%s: deterministic workspace has no tickets", who);
  return 0;
}

}  // namespace mmfm

extern "C" const char* mmfm_last_error(void) { return mmfm::get_error(); }
extern "C" int mmfm_abi_version(void) { return MMFM_ABI_VERSION; }
extern "C" int mmfm_sm_count(void) {
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
  return n;
}

extern "C" int mmfm_det_ws_bytes(int kind, long long d0, long long d1, long long d2, long long* bytes, int* n_tickets) {
  MMFM_REQUIRE(bytes && n_tickets, "mmfm_det_ws_bytes: null output");
  MMFM_REQUIRE(d0 > 0 && d1 > 0 && d2 >= 0, "mmfm_det_ws_bytes: bad sizes (%lld, %lld, %lld)", d0, d1, d2);
  mmfm::DetNeed need{0, 0};
  if (!mmfm::det_need_gemm(kind, d0, d1, d2, &need) && !mmfm::det_need_norm(kind, d0, d1, d2, &need) &&
      !mmfm::det_need_glue(kind, d0, d1, d2, &need)) {
    mmfm::set_error("mmfm_det_ws_bytes: unknown kind %d", kind);
    return -1;
  }
  *bytes = need.bytes;
  *n_tickets = need.tickets;
  return 0;
}
