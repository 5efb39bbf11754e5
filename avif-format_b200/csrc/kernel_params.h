// kernel_params.h -- plain parameter blocks handed to the CUDA kernels (device pointers, block-relative).
//
// "Block" = the row block [y0, y0 + rows) one launch converts.  All pointers already point at the first row of
// the block in their buffer (for sub-sampled chroma planes: at chroma row y0 >> ys), so kernels index rows from
// zero and never see y0 -- except `yPhase`, the parity of y0 for 4:2:0 decode, where an odd first row shares its
// chroma row with the row above it (ReadHeifImage.cpp:359 uvJ = y >> yChromaShift).
#ifndef AVIF_KERNEL_PARAMS_H
#define AVIF_KERNEL_PARAMS_H

#include <stdint.h>

#include <atomic>

#include "curve_tables.h"
#include "pixel_math.cuh"

namespace avifgpu
{

#if defined(__CUDACC__)
// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device setting; `configuredDevices` (one static per kernel
// instantiation) remembers the devices it has been made on, so a process that drives several GPUs configures each.
template <typename Kernel>
inline cudaError_t AllowDynamicShared(Kernel kernel, int bytes, std::atomic<uint64_t>& configuredDevices)
{
    int device = 0;
    cudaError_t e = cudaGetDevice(&device);
    if (e != cudaSuccess)
    {
        return e;
    }
    const uint64_t bit = 1ull << (device & 63);
    if (configuredDevices.load(std::memory_order_acquire) & bit)
    {
        return cudaSuccess;
    }
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess)
    {
        configuredDevices.fetch_or(bit, std::memory_order_release);
    }
    return e;
}

// Runs a counting kernel synchronously: `launch(counter)` enqueues it on `stream` with a zeroed device counter.  Returns
// the count the kernel left there, or -1 on a CUDA error.
template <typename Launch>
inline long long RunCountingKernel(cudaStream_t stream, Launch launch)
{
    unsigned long long* counter = nullptr;
    if (cudaMalloc(&counter, sizeof(unsigned long long)) != cudaSuccess)
    {
        return -1;
    }
    cudaMemsetAsync(counter, 0, sizeof(unsigned long long), stream);
    launch(counter);
    unsigned long long count = 0;
    const bool ok = cudaMemcpyAsync(&count, counter, sizeof(count), cudaMemcpyDeviceToHost, stream) == cudaSuccess &&
                    cudaStreamSynchronize(stream) == cudaSuccess;
    cudaFree(counter);
    return ok ? static_cast<long long>(count) : -1;
}

// The 65536-entry code table of Gray16 hosts (kernels_fast_int.cu); enqueued on `stream`.
cudaError_t BuildGray16Lut(uint16_t* deviceLut, int smpte428, uint32_t maxCode, void* stream);
#endif

struct EncodeParams
{
    const void* rows;      // interleaved host pixels (formatRecord->data layout), device memory
    int64_t rowStride;     // bytes
    void* plane[4];        // REFERENCE layout: [0] interleaved or Y, [3] alpha (gray); PLANAR: Y, Cb, Cr, A
    int64_t planeStride[4];
    int32_t width;
    int32_t rowCount;      // rows in this block
    int32_t channels;      // 1..4
    int32_t hasAlpha;
    int32_t premultiply;
    int32_t imageDepth;    // 8, 10, 12
    uint32_t maxCode;
    float maxCodeFloat;
    int32_t transfer;      // avifgpu_transfer (float hosts)
    float pqMultiplier;    // peak / 10000.0f
    int32_t gray16Smpte428;
    int32_t planar;        // AVIFGPU_LAYOUT_PLANAR_YCBCR
    int32_t xs, ys;        // chroma shifts
    int32_t topLeft;       // AVIFGPU_DOWN_FILTER_TOP_LEFT
    avifpix::ForwardMatrix matrix;
    float chromaOffset;
    int32_t hlgInverseOotf; // AVIFGPU_HLG_INVERSE_OOTF_THEN_OETF: ApplyInverseHLGOOTF on the pixel before LinearToHLG
    float hlgLuma[3];
    float hlgDisplayGamma;
    float hlgPeak;
    int32_t rowMatrixEnabled; // avifgpu_encode_desc.row_matrix: the colour-profile 3x3 ahead of everything else (float colour hosts)
    float rowMatrix[9];
    // Float hosts with a transfer curve: the flat step table + band bitmap in global memory (a by-value copy of
    // *curveTable made by the generic launcher), or useCurveView = 0 -> every sample takes the exact powf.
    CurveTableView curveView;
    int32_t useCurveView;
    // Host-side extras for the launcher (ignored by the kernels):
    const CurveTableView* curveTable; // verified exact step table for `transfer`, or nullptr
    const uint16_t* gray16Lut;        // 65536-entry code table for Gray16 hosts (device memory), or nullptr
    int32_t smCount;
    int32_t verifiedPremultiply;      // 1 once the context has verified FastPremultiplyBiased for this image depth on this device
};

struct DecodeParams
{
    const void* plane[4];  // YCbCr: Y, Cb, Cr, A; mono: Y, -, -, A; planar RGB: R, G, B, A
    int64_t planeStride[4];
    void* rows;            // interleaved host pixels, device memory
    int64_t rowStride;
    int32_t width;
    int32_t rowCount;
    int32_t yPhase;        // y0 & ys
    int32_t colorspace;    // avifgpu_colorspace
    int32_t xs, ys;
    int32_t hasAlpha;
    int32_t premultiplied;
    int32_t bitDepth;
    uint32_t maxCode;
    avifpix::RangeParams range;
    avifpix::InverseMatrix matrix;
    int32_t hostDepth;     // 8, 16, 32
    int32_t transfer;      // avifgpu_transfer (host depth 32)
    float pqMultiplier;    // 10000.0f / peak
    int32_t applyOotf;
    float lumaR, lumaG, lumaB;
    float gammaMinusOne;
    float hlgPeak;
    int32_t smCount;              // host-side extra for the launcher
    int32_t verifiedHlgDivisions; // 1 once the context has verified HLGToLinearUnit's fast divisions on this device
    int32_t verifiedGreenDivision; // 1 once the context has verified the fast `/ kg` of YuvDecode.cpp:308 for this matrix, depth, range
    int32_t verifiedPqRatio;       // 1 once the context has verified the branch-free division inside PQToLinear on this device
};

// A launcher that sees a CUDA error has already consumed it (cudaGetLastError clears the slot), so it leaves the code
// here -- a thread-local slot in avifgpu_api.cu -- and returns AVIFGPU_ERR_CUDA; the API reports it from there instead
// of asking CUDA a second time (which would answer cudaSuccess and turn a failed launch into AVIFGPU_OK).
int ReportLaunchFailure(int cudaErrorCode);

// True when `p` and every row `stride` bytes after it are `alignment`-byte aligned (the tuned kernels' vector accesses).
inline bool Aligned(const void* p, int64_t stride, int alignment)
{
    return (reinterpret_cast<uintptr_t>(p) % alignment) == 0 && (stride % alignment) == 0;
}

// The SM count the persistent grids are sized for: the context's device, or a B200's for a block made without one.
constexpr int kB200SmCount = 148;
inline int SmCount(int32_t smCount) { return smCount > 0 ? smCount : kB200SmCount; }

// Launchers.  They only enqueue work on `stream` and return the number of kernels launched or a negative
// avifgpu_status.  LaunchEncode / LaunchDecode (avifgpu_api.cu) try the tuned launchers in turn, each of which returns 0
// when it does not cover the configuration, and end with the generic kernel (kernels_generic.cu), which covers all.
int LaunchEncode(const EncodeParams& params, int hostDepth, void* stream);
int LaunchDecode(const DecodeParams& params, void* stream);
int LaunchEncodeGeneric(const EncodeParams& params, int hostDepth, void* stream); // 0 for an empty block
int LaunchDecodeGeneric(const DecodeParams& params, void* stream);                // 0 for an empty block
// The generic kernel over what a tuned kernel covering [0, coveredWidth) x [0, coveredRows) left: the right strip (all
// rows), then the bottom strip (the covered columns).  The number of kernels launched, or a negative status.
int LaunchEncodeRemainder(const EncodeParams& params, int hostDepth, int coveredWidth, int coveredRows, void* stream);
int LaunchDecodeRemainder(const DecodeParams& params, int coveredWidth, int coveredRows, void* stream);
int LaunchEncodeFast(const EncodeParams& params, int hostDepth, void* stream);        // kernels_fast.cu
int LaunchEncodeFastInteger(const EncodeParams& params, int hostDepth, void* stream); // kernels_fast_int.cu
int LaunchEncodeFastGray32(const EncodeParams& params, int hostDepth, void* stream);  // kernels_fast_gray32.cu
int LaunchDecodeFast(const DecodeParams& params, void* stream);                       // kernels_fast_decode.cu
int LaunchDecodeFastInteger(const DecodeParams& params, void* stream);                // kernels_fast_decode_int.cu
int LaunchDecodeFastTable(const DecodeParams& params, void* stream);                  // kernels_fast_decode_table.cu
int LaunchTransfer(int function, float param, const float* in, float* out, size_t count, void* stream);
int LaunchHlgOotf(int inverse, const float luma[3], float displayGamma, float peak, const float* in, float* out, size_t pixels, void* stream);

// One-time exhaustive checks behind the tuned kernels' arithmetic shortcuts.  Synchronous: the number of disagreements
// (0 = verified) or -1 on a CUDA error.
long long VerifyHlgDivisions(void* stream);                              // HLGToLinearUnit's fast divisions
long long VerifyPqRatio(void* stream);                                   // PqRatioPair's division, every x the PQ decode makes
long long VerifyGreenDivision(const DecodeParams& params, void* stream); // the green division of one matrix, depth, range
long long VerifyFastPremultiply(uint32_t maxCode, void* stream);         // FastPremultiplyBiased for one bit depth

} // namespace avifgpu

#endif
