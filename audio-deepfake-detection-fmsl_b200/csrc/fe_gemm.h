// Interface of the tcgen05 DFT-GEMM variant (fe_stream.cu).
#ifndef FE_GEMM_H_
#define FE_GEMM_H_
#include <cuda_runtime.h>
#include "fe_common.h"
#include "fe_kernels.h"

int32_t fe_gemm_compiled(void);                       // 1 when the tcgen05 kernel is built in
bool fe_gemm_supported(const b200fe_params* p);       // configuration handled by the variant
bool fe_gemm_preferred(const b200fe_params* p);       // AUTO picks it (from measurements, DESIGN.md)
int64_t fe_gemm_workspace_bytes(const b200fe_params* p, int64_t chunk_rows, int64_t T);
// Streaming kernel: what the call's shape must satisfy on top of fe_gemm_supported (T % 4 == 0 for the TMA boxes,
// T > n_fft/2, at least two frames).  Any row count is taken: fe_stream_launch splits the rows into launches.
bool fe_stream_supported(const b200fe_params* p, int64_t T);
// Filterbank energies (+ group maxima) of rows [row_base, row_base+rows) into fa.out, like fe_launch_fft(mode 1), in
// as many launches as the kernel's 32-bit frame and element indices need.
cudaError_t fe_stream_launch(const b200fe_params* p, const fe_fft_args& fa, int64_t row_base, int64_t rows,
                             void* gemm_ws, cudaStream_t stream);
#endif
