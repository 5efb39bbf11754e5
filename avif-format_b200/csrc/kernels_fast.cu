// kernels_fast.cu -- dispatch of the tuned float-RGB(A) encode kernels, and the one for "no transfer curve".
// Anything the tuned kernels do not cover falls back to kernels_generic.cu (LaunchEncodeFast returns 0 = "not
// applicable").  The arithmetic is the same pixel_math.cuh; what changes is the work decomposition and where the
// transcendental work goes:
//   curve with a verified step table (PQ, SMPTE 428)   kernels_fast_flat.cu (RGB), kernels_fast_rgba.cu (RGBA)
//   no curve (clip)                                     EncodeRgbF32ClipKernel below: warp tile = 2 rows x 128 pixels, a lane
//                                                       owns 4 adjacent pixels in both rows (two 2x2 chroma sites, the box
//                                                       filter needs no cross-lane traffic), 3 x LDG.128 per row per lane
//                                                       one tile ahead, persistent grid of 3 CTAs x 8 warps per SM.
#include "kernels_fast_common.cuh"
#include "../../include/avifgpu.h"

#include <cuda_runtime.h>

#include <cstdlib>

namespace avifgpu
{

using namespace avifpix;
using namespace fastenc;
using avifmath::LibmTables;

namespace
{

constexpr int kClipThreads = 256;
constexpr int kClipWarps = kClipThreads / 32;
constexpr int kClipBlocksPerSm = 3;

// No transfer curve (AVIFGPU_TRANSFER_CLIP): code = trunc(clamp(v * max)) per sample (WriteHeifImage.cpp:1128-1130), then
// the forward matrix.  No tables, no shared memory; the loads of tile i+1 are issued before tile i's arithmetic.
template <int XS, int YS>
__global__ void __launch_bounds__(kClipThreads, kClipBlocksPerSm) EncodeRgbF32ClipKernel(const FastEncodeParams p)
{
    const int lane = threadIdx.x & 31;
    const int warpInBlock = threadIdx.x >> 5;
    const int tilesX = (p.width + kTilePixels - 1) / kTilePixels;
    const int tileRows = (p.rowCount + 1) / 2;
    const int tileCount = tilesX * tileRows;
    const int warpCount = static_cast<int>(gridDim.x) * kClipWarps;

    // Tile coordinates advance incrementally (an integer division per tile costs ~24 instructions).
    const int firstTile = static_cast<int>(blockIdx.x) * kClipWarps + warpInBlock;
    const int stepRows = warpCount / tilesX;
    const int stepX = warpCount - stepRows * tilesX;
    int tileRow = firstTile / tilesX;
    int tileX = firstTile - tileRow * tilesX;
    uint4 raw[6];
    auto loadTile = [&](int row, int column, bool valid)
    {
        const int x = column * kTilePixels + lane * 4;
        const int y = row * 2;
        const bool active = valid && x < p.width;
        const bool second = active && (y + 1) < p.rowCount;
        const uint8_t* r0 = p.rows + static_cast<int64_t>(y) * p.rowStride + static_cast<int64_t>(x) * 12;
        const uint8_t* r1 = r0 + p.rowStride;
        const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
        for (int q = 0; q < 3; ++q)
        {
            raw[q] = active ? __ldg(reinterpret_cast<const uint4*>(r0 + 16 * q)) : zero;
        }
#pragma unroll
        for (int q = 0; q < 3; ++q)
        {
            raw[3 + q] = second ? __ldg(reinterpret_cast<const uint4*>(r1 + 16 * q)) : zero;
        }
    };
    loadTile(tileRow, tileX, firstTile < tileCount);

    for (int tile = firstTile; tile < tileCount; tile += warpCount)
    {
        const int x0 = tileX * kTilePixels + lane * 4;
        const int y0 = tileRow * 2;
        const bool laneActive = x0 < p.width;
        const bool secondRow = (y0 + 1) < p.rowCount;
        const int currentRow = tileRow;

        float codeF[kValuesPerLane]; // the codes, as the floats the forward matrix consumes
#pragma unroll
        for (int q = 0; q < 6; ++q)
        {
            codeF[4 * q + 0] = CodeToFloat(FloatToCode(__uint_as_float(raw[q].x), p.maxCodeFloat));
            codeF[4 * q + 1] = CodeToFloat(FloatToCode(__uint_as_float(raw[q].y), p.maxCodeFloat));
            codeF[4 * q + 2] = CodeToFloat(FloatToCode(__uint_as_float(raw[q].z), p.maxCodeFloat));
            codeF[4 * q + 3] = CodeToFloat(FloatToCode(__uint_as_float(raw[q].w), p.maxCodeFloat));
        }
        tileRow += stepRows;
        tileX += stepX;
        if (tileX >= tilesX)
        {
            tileX -= tilesX;
            ++tileRow;
        }
        loadTile(tileRow, tileX, tile + warpCount < tileCount);

        if (laneActive)
        {
            const int64_t chromaRow = YS ? currentRow : y0;
            const int64_t chromaColumn = static_cast<int64_t>(XS ? (x0 >> 1) : x0) * 2;
            StoreTile<XS, YS>(p, codeF, p.planeY + static_cast<int64_t>(y0) * p.strideY + static_cast<int64_t>(x0) * 2,
                              p.planeCb + chromaRow * p.strideCb + chromaColumn, p.planeCr + chromaRow * p.strideCr + chromaColumn, secondRow);
        }
    }
}

template <int XS, int YS>
cudaError_t LaunchClipKernel(const FastEncodeParams& fp, int smCount, cudaStream_t stream)
{
    const long long tiles = static_cast<long long>((fp.width + kTilePixels - 1) / kTilePixels) * ((fp.rowCount + 1) / 2);
    if (tiles > 0x7fffffffll)
    {
        return cudaErrorInvalidValue;
    }
    long long blocks = (tiles + kClipWarps - 1) / kClipWarps;
    const long long resident = static_cast<long long>(smCount) * kClipBlocksPerSm;
    if (blocks > resident)
    {
        blocks = resident;
    }
    EncodeRgbF32ClipKernel<XS, YS><<<static_cast<unsigned>(blocks), kClipThreads, 0, stream>>>(fp);
    return cudaGetLastError();
}

cudaError_t DispatchClip(const FastEncodeParams& fp, int xs, int ys, int smCount, cudaStream_t stream)
{
    if (xs == 1 && ys == 1) return LaunchClipKernel<1, 1>(fp, smCount, stream);
    if (xs == 1) return LaunchClipKernel<1, 0>(fp, smCount, stream);
    return LaunchClipKernel<0, 0>(fp, smCount, stream);
}

} // namespace

// Returns the number of kernels launched, 0 if this configuration is not covered, or a negative status.
int LaunchEncodeFast(const EncodeParams& p, int hostDepth, void* streamHandle)
{
    cudaStream_t stream = static_cast<cudaStream_t>(streamHandle);
    const bool rgba = p.channels == 4 && p.hasAlpha;
    if (p.rowMatrixEnabled)
    {
        return 0; // the colour-profile matrix is a prologue of the generic kernels only (they still use the step tables)
    }
    if (hostDepth == 32 && !p.planar && p.channels == 3 && !p.hasAlpha && p.imageDepth > 8 && !p.hlgInverseOotf &&
        (p.transfer == AVIFGPU_TRANSFER_PQ || p.transfer == AVIFGPU_TRANSFER_SMPTE428) && p.curveTable != nullptr && p.curveTable->buckets != nullptr)
    {
        // The reference's own layout: interleaved RGB codes (WriteHeifImage.cpp:1098-1130), same kernel without the matrix.
        const int width4 = p.width & ~3;
        if (width4 < 4 || p.rowCount < 1 || !Aligned(p.rows, p.rowStride, 16) || !Aligned(p.plane[0], p.planeStride[0], 8))
        {
            return 0;
        }
        FastEncodeParams fp{};
        fp.rows = static_cast<const uint8_t*>(p.rows);
        fp.rowStride = p.rowStride;
        fp.planeY = static_cast<uint8_t*>(p.plane[0]);
        fp.strideY = p.planeStride[0];
        fp.width = width4;
        fp.rowCount = p.rowCount;
        fp.pqMultiplier = p.pqMultiplier;
        fp.maxCodeFloat = p.maxCodeFloat;
        fp.maxCode = static_cast<int32_t>(p.maxCode);
        fp.table = *p.curveTable;
        if (!FlatEncodeApplies(fp))
        {
            return 0;
        }
        const int curve = p.transfer == AVIFGPU_TRANSFER_PQ ? kCurveLinearToPQ : kCurveLinearToSMPTE428;
        const cudaError_t e = LaunchFastEncodeFlatInterleaved(fp, curve, SmCount(p.smCount), stream);
        if (e != cudaSuccess)
        {
            return ReportLaunchFailure(static_cast<int>(e));
        }
        const int n = LaunchEncodeRemainder(p, hostDepth, width4, p.rowCount, streamHandle);
        return n < 0 ? n : 1 + n;
    }
    if (hostDepth != 32 || !p.planar || (p.channels != 3 && !rgba) || (p.channels == 3 && p.hasAlpha) || p.imageDepth <= 8)
    {
        return 0;
    }
    int curve;
    if (p.transfer == AVIFGPU_TRANSFER_PQ) curve = kCurveLinearToPQ;
    else if (p.transfer == AVIFGPU_TRANSFER_SMPTE428) curve = kCurveLinearToSMPTE428;
    else if (p.transfer == AVIFGPU_TRANSFER_CLIP) curve = kCurveClip;
    else return 0; // HLG save path: the generic kernel (with the context's step table when it has one)
    if (curve != kCurveClip && (p.curveTable == nullptr || p.curveTable->buckets == nullptr))
    {
        return 0; // no verified table for this curve: the generic exact kernel serves it
    }
    if (!ForwardMatrixStaysInRange(p.matrix, p.chromaOffset, static_cast<int>(p.maxCode)))
    {
        return 0; // an exotic matrix: the generic kernel clamps
    }
    if (!Aligned(p.rows, p.rowStride, 16) || !Aligned(p.plane[0], p.planeStride[0], 8) ||
        !Aligned(p.plane[1], p.planeStride[1], p.xs ? 4 : 8) || !Aligned(p.plane[2], p.planeStride[2], p.xs ? 4 : 8) ||
        (rgba && !Aligned(p.plane[3], p.planeStride[3], 8)))
    {
        return 0;
    }
    if (rgba && (curve == kCurveClip || p.curveTable->flat == nullptr || p.curveTable->bandBits == nullptr))
    {
        return 0; // the RGBA kernel is built on the flat table + band bitmap; everything else with alpha: generic
    }
    const int width4 = p.width & ~3;
    const int evenRows = p.ys ? (p.rowCount & ~1) : p.rowCount;
    if (width4 < 4 || evenRows < 1)
    {
        return 0;
    }

    FastEncodeParams fp{};
    fp.rows = static_cast<const uint8_t*>(p.rows);
    fp.rowStride = p.rowStride;
    fp.planeY = static_cast<uint8_t*>(p.plane[0]);
    fp.strideY = p.planeStride[0];
    fp.planeCb = static_cast<uint8_t*>(p.plane[1]);
    fp.strideCb = p.planeStride[1];
    fp.planeCr = static_cast<uint8_t*>(p.plane[2]);
    fp.strideCr = p.planeStride[2];
    fp.width = width4;
    fp.rowCount = evenRows;
    fp.pqMultiplier = p.pqMultiplier;
    fp.maxCodeFloat = p.maxCodeFloat;
    fp.maxCode = static_cast<int32_t>(p.maxCode);
    fp.matrix = p.matrix;
    fp.chromaOffset = p.chromaOffset;
    fp.topLeft = p.topLeft;
    if (curve != kCurveClip)
    {
        fp.table = *p.curveTable;
        static const bool wide = []() { const char* v = std::getenv("AVIFGPU_WIDE_TABLE_ENTRIES"); return v != nullptr && v[0] == '1'; }();
        fp.preferWideEntries = wide ? 1 : 0;
    }
    if (rgba)
    {
        fp.planeA = static_cast<uint8_t*>(p.plane[3]);
        fp.strideA = p.planeStride[3];
        fp.premultiply = p.premultiply;
    }

    const int smCount = SmCount(p.smCount);
    cudaError_t e;
    if (rgba)
    {
        if (!RgbaEncodeApplies(fp))
        {
            return 0;
        }
        e = LaunchFastEncodeRgba(fp, curve, p.xs, p.ys, smCount, stream);
    }
    else if (curve != kCurveClip)
    {
        if (!FlatEncodeApplies(fp))
        {
            return 0; // a table too large to sit beside the staging buffers: the generic kernel looks it up in global memory
        }
        e = LaunchFastEncodeFlat(fp, curve, p.xs, p.ys, smCount, stream);
    }
    else
    {
        e = DispatchClip(fp, p.xs, p.ys, smCount, stream);
    }
    if (e != cudaSuccess)
    {
        return ReportLaunchFailure(static_cast<int>(e));
    }
    // The right strip (width % 4 columns) and, for vertically sub-sampled chroma, an odd last row: the generic kernel.
    const int n = LaunchEncodeRemainder(p, hostDepth, width4, evenRows, streamHandle);
    return n < 0 ? n : 1 + n;
}

} // namespace avifgpu
