// Host-side helpers shared by the C-ABI translation units.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/aptai_b200.h"

namespace aptai {

void set_error(const char* fmt, ...);
int check_arch();                       // 0 if the current device is sm_100, else APTAI_ERR_ARCH (message set)
int num_sms();
int traversal_reverse();              // 1: the next launches walk their rows / tiles / items from the end (aptai_set_traversal)
void count_launch(int n = 1);
int after_launch(const char* what);     // cudaGetLastError -> status (+ launch counter)

// cuTensorMapEncodeTiled through cudaGetDriverEntryPoint (no link-time libcuda dependency)
int encode_tmap_bf16(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                     const uint64_t* strides_bytes /* rank-1 */, const uint32_t* box, int swizzle128);
int encode_tmap_f32(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                    const uint64_t* strides_bytes /* rank-1 */, const uint32_t* box, int swizzle128);

// aptai_gemm_wgrad_bf16 that writes only dw rows [0, out_rows): N (the dY columns the TMA reads) may be a padded width
int wgrad_bf16_rows(const void* dy, int64_t dy_ld, const void* x, int64_t x_ld, int64_t M, int N, int K, float scale,
                    float* dw, int64_t dw_ld, int out_rows, void* stream);

#define APTAI_REQUIRE(cond, ...)              \
  do {                                        \
    if (!(cond)) {                            \
      ::aptai::set_error(__VA_ARGS__);        \
      return APTAI_ERR_ARG;                   \
    }                                         \
  } while (0)

}  // namespace aptai
