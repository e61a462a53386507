// Host-side helpers shared by the launchers: error handling, TMA tensor-map encoding.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

namespace mmfm {

// thread-local last error string (C ABI: mmfm_last_error)
void set_error(const char* fmt, ...);
const char* get_error();

#define MMFM_CHECK_CUDA(expr)                                                              \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess) {                                                               \
      ::mmfm::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return -2;                                                                           \
    }                                                                                      \
  } while (0)

#define MMFM_REQUIRE(cond, ...)            \
  do {                                     \
    if (!(cond)) {                         \
      ::mmfm::set_error(__VA_ARGS__);      \
      return -1;                           \
    }                                      \
  } while (0)

enum TmaSwizzle { TMA_SW_NONE = 0, TMA_SW_32 = 1, TMA_SW_64 = 2, TMA_SW_128 = 3 };

// 2-D bf16 tensor map over a row-major matrix [rows, cols] with row pitch `ld` elements.
// box = box_cols x box_rows elements.  Returns 0 on success.
int make_tmap_bf16_2d(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld,
                      uint32_t box_cols, uint32_t box_rows, TmaSwizzle swz);

// Same for fp32 matrices (epilogue residual loads / output stores of the TMA-store GEMM).
int make_tmap_f32_2d(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_cols,
                     uint32_t box_rows, TmaSwizzle swz);

// 3-D bf16 tensor map over [batch][rows][cols] (row pitch `ld` elements, batch pitch rows * ld): a box never crosses a
// batch entry, so rows past `rows` are clipped on store / zero-filled on load.  box = box_cols x box_rows x 1.
int make_tmap_bf16_3d(CUtensorMap* out, const void* base, uint64_t batch, uint64_t rows, uint64_t cols, uint64_t ld,
                      uint32_t box_cols, uint32_t box_rows, TmaSwizzle swz);

int device_sm_count();

// Deterministic-mode workspace need of one *_det call (mmfm_det_ws_bytes): each source file answers for its own
// kinds (false = not its kind) from the grid arithmetic its launchers use.
struct DetNeed {
  long long bytes;
  int tickets;
};
bool det_need_gemm(int kind, long long d0, long long d1, long long d2, DetNeed* need);
bool det_need_norm(int kind, long long d0, long long d1, long long d2, DetNeed* need);
bool det_need_glue(int kind, long long d0, long long d1, long long d2, DetNeed* need);
// 0 when the workspace can hold `need`; sets the error and returns -1 otherwise
int det_ws_check(const void* buf, long long bytes, const unsigned int* tickets, int n_tickets, const DetNeed& need,
                 const char* who);

}  // namespace mmfm
