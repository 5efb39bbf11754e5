// kernels_fast_decode_table.cu -- float hosts reading images whose samples decode one plane at a time: planar RGB
// (ReadHeifImageRGBThirtyTwoBit's RGB branch, ReadHeifImage.cpp:949-1178) and monochrome
// (ReadHeifImageGrayThirtyTwoBit, ReadHeifImage.cpp:863-947 driving DecodeY16RowToGray32 / ...GrayAlpha32,
// YuvDecode.cpp:199-279), 10 / 12-bit.
//
// There the whole per-sample chain -- unorm -> float table, then PQToLinear / HLGToLinear / SMPTE428ToLinear -- is a
// function of ONE code, so every CTA evaluates it once per code with the exact (glibc-identical) device libm into a
// shared-memory table (2^depth floats: 4096 exact evaluations per CTA against ~200 000 pixels it then converts) and the
// pixel loop is loads, look-ups and stores: HBM-bound (6 + 12 bytes per pixel for RGB -> RGB32f) instead of
// 6 powf per pixel.  What cannot be tabulated stays per pixel and exact: the HLG OOTF (one powf of the pixel's luma,
// ColorTransfer.cpp:192-205) and the integer-domain un-premultiplication the reference applies BEFORE the table
// (ReadHeifImage.cpp:1049-1066, YuvDecode.cpp:247-260).
// A thread converts 8 adjacent pixels: one 128-bit load per plane, 128-bit stores.
#include "group_walk.cuh"
#include "kernel_params.h"
#include "../../include/avifgpu.h"

#include <cuda_runtime.h>

namespace avifgpu
{

using namespace avifpix;
using avifmath::LibmTables;

namespace
{

constexpr int kTableThreads = 256;

struct TableDecodeParams
{
    const uint8_t* plane[4]; // RGB: R, G, B, A;  mono: Y, -, -, A
    int64_t planeStride[4];
    uint8_t* rows;
    int64_t rowStride;
    int32_t groupsPerRow; // 8 pixels each
    int32_t rowCount;
    int32_t bitDepth;
    uint32_t maxCode;
    RangeParams range;
    int32_t transfer;
    float pqMultiplier;
    int32_t applyOotf;
    float lumaR, lumaG, lumaB;
    float gammaMinusOne;
    float hlgPeak;
    int32_t premultiplied;
};

// COLOURS 3 (planar RGB) or 1 (monochrome); ALPHA adds the alpha plane as the last host channel.
template <int COLOURS, int ALPHA>
__global__ void __launch_bounds__(kTableThreads) TableDecodeF32Kernel(const TableDecodeParams p)
{
    extern __shared__ __align__(16) uint8_t sharedBytes[];
    uint64_t* libmStorage = reinterpret_cast<uint64_t*>(sharedBytes);
    float* curve = reinterpret_cast<float*>(sharedBytes + 768); // EOTF(unorm(code))
    float* plain = curve + (1u << p.bitDepth);                  // code / max (alpha)
    const LibmTables t = avifmath::StageLibmTables(libmStorage, threadIdx.x, blockDim.x);
    __syncthreads();
    for (uint32_t code = threadIdx.x; code <= p.maxCode; code += blockDim.x)
    {
        // planar RGB: BuildUnormToFloatLookupTable (ReadHeifImage.cpp:402-415) = code / max;
        // monochrome: unormFloatTableY (YuvLookupTables.cpp:157-171, limited range remapped)
        const float v = COLOURS == 3 ? UnormToFloatPlain(code, p.range.maxChannelFloat) : UnormToFloatY(code, p.range);
        float linear;
        if (p.transfer == AVIFGPU_TRANSFER_PQ) linear = PQToLinear(v, p.pqMultiplier, t);
        else if (p.transfer == AVIFGPU_TRANSFER_HLG) linear = HLGToLinear(v, t);
        else linear = SMPTE428ToLinear(v, t);
        curve[code] = linear;
        if (ALPHA)
        {
            plain[code] = UnormToFloatPlain(code, p.range.maxChannelFloat);
        }
    }
    __syncthreads();

    constexpr int kChannels = COLOURS + ALPHA;
    const float maxCodeFloat = static_cast<float>(p.maxCode);
    for (GroupWalk walk(static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x, static_cast<long long>(gridDim.x) * blockDim.x, p.groupsPerRow, p.rowCount);
         walk.Inside(p.rowCount); walk.Advance(p.rowCount))
    {
        const long long row = walk.row;
        const long long column = static_cast<long long>(walk.column) * 8;
        uint4 raw[kChannels];
#pragma unroll
        for (int c = 0; c < kChannels; ++c)
        {
            const int planeIndex = (ALPHA && c == kChannels - 1) ? 3 : c;
            raw[c] = __ldcs(reinterpret_cast<const uint4*>(p.plane[planeIndex] + row * p.planeStride[planeIndex] + column * 2));
        }
        float out[8 * kChannels];
#pragma unroll
        for (int i = 0; i < 8; ++i)
        {
            auto sample = [&](int c) -> uint32_t
            {
                const uint32_t words[4] = { raw[c].x, raw[c].y, raw[c].z, raw[c].w };
                const uint32_t w = words[i >> 1];
                return min((i & 1) ? (w >> 16) : (w & 0xffffu), p.maxCode); // DEFINED: clamp (the reference would index past its table)
            };
            uint32_t alpha = 0;
            if (ALPHA)
            {
                alpha = sample(kChannels - 1);
            }
            float colour[COLOURS];
#pragma unroll
            for (int c = 0; c < COLOURS; ++c)
            {
                uint32_t code = sample(c);
                if (ALPHA && p.premultiplied && alpha < p.maxCode)
                {
                    // integer-domain un-premultiplication before the table, as the reference does it
                    code = (alpha == 0) ? 0u : UnpremultiplyCode(code, alpha, maxCodeFloat);
                }
                colour[c] = curve[code];
            }
            if (COLOURS == 3 && p.applyOotf)
            {
                ApplyHLGOOTF<true>(colour[0], colour[1], colour[2], p.lumaR, p.lumaG, p.lumaB, p.gammaMinusOne, p.hlgPeak, t);
            }
#pragma unroll
            for (int c = 0; c < COLOURS; ++c)
            {
                out[i * kChannels + c] = colour[c];
            }
            if (ALPHA)
            {
                out[i * kChannels + COLOURS] = plain[alpha];
            }
        }
        float4* target = reinterpret_cast<float4*>(p.rows + row * p.rowStride + column * (4 * kChannels));
#pragma unroll
        for (int q = 0; q < 2 * kChannels; ++q)
        {
            __stcs(target + q, make_float4(out[4 * q], out[4 * q + 1], out[4 * q + 2], out[4 * q + 3]));
        }
    }
}

template <int COLOURS, int ALPHA>
cudaError_t LaunchTable(const TableDecodeParams& tp, int smCount, cudaStream_t stream)
{
    const long long groups = static_cast<long long>(tp.groupsPerRow) * tp.rowCount;
    long long blocks = (groups + kTableThreads - 1) / kTableThreads;
    const size_t shared = 768 + (ALPHA ? 2 : 1) * sizeof(float) * (static_cast<size_t>(1) << tp.bitDepth);
    // each CTA pays for its own table: exactly as many as are resident at once (4 at 52 registers, 8 at 32), long-lived
    int residentPerSm = 4;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&residentPerSm, TableDecodeF32Kernel<COLOURS, ALPHA>, kTableThreads, shared) != cudaSuccess || residentPerSm < 1)
    {
        (void)cudaGetLastError();
        residentPerSm = 4;
    }
    const long long cap = static_cast<long long>(smCount) * residentPerSm;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    TableDecodeF32Kernel<COLOURS, ALPHA><<<static_cast<unsigned>(blocks), kTableThreads, shared, stream>>>(tp);
    return cudaGetLastError();
}

} // namespace

// Returns the number of kernels launched, 0 if this configuration is not covered, or a negative status.
int LaunchDecodeFastTable(const DecodeParams& p, void* streamHandle)
{
    cudaStream_t stream = static_cast<cudaStream_t>(streamHandle);
    const bool mono = p.colorspace == AVIFGPU_COLORSPACE_MONOCHROME;
    if (p.hostDepth != 32 || (!mono && p.colorspace != AVIFGPU_COLORSPACE_RGB) || p.bitDepth <= 8 || p.bitDepth > 12)
    {
        return 0;
    }
    if (mono && p.transfer != AVIFGPU_TRANSFER_PQ)
    {
        return 0; // the reference's gray float path knows PQ only (YuvDecode.cpp:214-221); anything else: the generic kernel's business
    }
    if (p.transfer != AVIFGPU_TRANSFER_PQ && p.transfer != AVIFGPU_TRANSFER_HLG && p.transfer != AVIFGPU_TRANSFER_SMPTE428)
    {
        return 0;
    }
    const int colours = mono ? 1 : 3;
    for (int c = 0; c < colours; ++c)
    {
        if (!Aligned(p.plane[c], p.planeStride[c], 16))
        {
            return 0;
        }
    }
    if ((p.hasAlpha && !Aligned(p.plane[3], p.planeStride[3], 16)) || !Aligned(p.rows, p.rowStride, 16))
    {
        return 0;
    }
    const int width8 = p.width & ~7;
    if (width8 < 8 || p.rowCount < 1)
    {
        return 0;
    }
    TableDecodeParams tp{};
    for (int k = 0; k < 4; ++k)
    {
        tp.plane[k] = static_cast<const uint8_t*>(p.plane[k]);
        tp.planeStride[k] = p.planeStride[k];
    }
    tp.rows = static_cast<uint8_t*>(p.rows);
    tp.rowStride = p.rowStride;
    tp.groupsPerRow = width8 / 8;
    tp.rowCount = p.rowCount;
    tp.bitDepth = p.bitDepth;
    tp.maxCode = p.maxCode;
    tp.range = p.range;
    tp.transfer = p.transfer;
    tp.pqMultiplier = p.pqMultiplier;
    tp.applyOotf = (!mono && p.transfer == AVIFGPU_TRANSFER_HLG && p.applyOotf) ? 1 : 0;
    tp.lumaR = p.lumaR;
    tp.lumaG = p.lumaG;
    tp.lumaB = p.lumaB;
    tp.gammaMinusOne = p.gammaMinusOne;
    tp.hlgPeak = p.hlgPeak;
    tp.premultiplied = p.premultiplied;
    const int smCount = SmCount(p.smCount);
    cudaError_t e;
    if (mono) e = p.hasAlpha ? LaunchTable<1, 1>(tp, smCount, stream) : LaunchTable<1, 0>(tp, smCount, stream);
    else e = p.hasAlpha ? LaunchTable<3, 1>(tp, smCount, stream) : LaunchTable<3, 0>(tp, smCount, stream);
    if (e != cudaSuccess)
    {
        return ReportLaunchFailure(static_cast<int>(e));
    }
    const int n = LaunchDecodeRemainder(p, width8, p.rowCount, streamHandle);
    return n < 0 ? n : 1 + n;
}

} // namespace avifgpu
