// h264_kernels.h — launchers of the encoder stages (each returns the number of kernels launched)
#pragma once
#include <cuda_runtime.h>
namespace b2v {
struct FrameCtx;
int launch_intra(const FrameCtx& f, cudaStream_t st);    // IDR: Intra16x16 rows (h264_intra.cu)
int launch_inter(const FrameCtx& f, cudaStream_t st);    // P: motion search + residual (h264_inter.cu)
int launch_cavlc(const FrameCtx& f, cudaStream_t st);    // per-macroblock CAVLC bit strings (h264_entropy.cu)
int launch_slice_build(const FrameCtx& f, cudaStream_t st);     // slice RBSP + emulation-prevention count; its last block runs the rate-control step
int launch_pack_cap(const FrameCtx& f, long long au_cap, cudaStream_t st);   // emulation prevention + AU assembly
}  // namespace b2v
