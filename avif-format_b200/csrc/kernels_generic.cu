// kernels_generic.cu -- the general kernels: every configuration of the path, one thread per pixel (decode,
// reference-layout encode) or per chroma site (planar YCbCr encode).  Correct for every combination the
// reference's twelve row shuttles accept; the tuned kernels in kernels_fast.cu take over for the layouts
// BASELINE.json measures and fall back to these for everything else.  Both sets share pixel_math.cuh, so
// they cannot disagree on arithmetic.
#include "kernel_params.h"
#include "curve_lookup.cuh"
#include "host_params.h"
#include "../../include/avifgpu.h"

#include <cuda_runtime.h>

namespace avifgpu
{

using namespace avifpix;
using avifmath::LibmTables;

namespace
{

constexpr int kThreads = 256;

// ---- encode -------------------------------------------------------------------------------------------------

template <typename HostT>
struct HostTraits;
template <>
struct HostTraits<uint8_t>
{
    static constexpr int depth = 8;
};
template <>
struct HostTraits<uint16_t>
{
    static constexpr int depth = 16;
};
template <>
struct HostTraits<float>
{
    static constexpr int depth = 32;
};

// One host pixel -> integer codes, following the reference's inner loops:
//   float hosts   WriteHeifImage.cpp:560-622 (gray), 1039-1135 (colour)
//   integer hosts WriteHeifImage.cpp:224-331, 389-497 (gray), 682-803, 858-985 (colour)
template <typename HostT>
__device__ __forceinline__ void HostPixelToCodes(const EncodeParams& p, const HostT* px, uint32_t codes[4],
                                                 const LibmTables& t)
{
    const int channels = p.channels;
    const int colors = (channels <= 2) ? 1 : 3;

    if constexpr (HostTraits<HostT>::depth == 32)
    {
        float color[3];
        float alpha = 0.0f;
#pragma unroll
        for (int i = 0; i < 3; ++i)
        {
            color[i] = (i < colors) ? px[i] : 0.0f;
        }
        if (p.rowMatrixEnabled && colors == 3)
        {
            // the colour-profile step (ColorProfileConversion::ConvertRow before the per-pixel loop, WriteHeifImage.cpp:1028-1031)
            const float r = color[0], g = color[1], b = color[2];
            color[0] = ((p.rowMatrix[0] * r) + (p.rowMatrix[1] * g)) + (p.rowMatrix[2] * b);
            color[1] = ((p.rowMatrix[3] * r) + (p.rowMatrix[4] * g)) + (p.rowMatrix[5] * b);
            color[2] = ((p.rowMatrix[6] * r) + (p.rowMatrix[7] * g)) + (p.rowMatrix[8] * b);
        }
        if (p.hasAlpha)
        {
            alpha = ClampF(px[colors], 0.0f, 1.0f);
            if (p.premultiply)
            {
                if (alpha < 1.0f)
                {
                    if (alpha == 0)
                    {
                        color[0] = 0;
                        color[1] = 0;
                        color[2] = 0;
                    }
                    else
                    {
#pragma unroll
                        for (int i = 0; i < 3; ++i)
                        {
                            color[i] = PremultiplyColor(ClampF(color[i], 0.0f, 1.0f), alpha, 1.0f);
                        }
                    }
                }
            }
        }
        else if (colors == 1)
        {
            color[0] = ClampF(color[0], 0.0f, 1.0f); // WriteHeifImage.cpp:602
        }
        if (p.hlgInverseOotf)
        {
            ApplyInverseHLGOOTF(color[0], color[1], color[2], p.hlgLuma[0], p.hlgLuma[1], p.hlgLuma[2], p.hlgDisplayGamma, p.hlgPeak, t);
        }
#pragma unroll
        for (int i = 0; i < 3; ++i)
        {
            if (i < colors)
            {
                // A built and verified step table (curve_tables.h) answers every finite sample from global memory: one
                // 64-bit gather, plus one bit of the band bitmap for the ~1.5 % of samples inside a fuzzy band.
                if (p.useCurveView && static_cast<int32_t>(__float_as_uint(color[i])) <= 0x7f7fffff)
                {
                    bool inBand;
                    codes[i] = LookupCurveCodeFlatResolved(__float_as_uint(color[i]), p.curveView, inBand);
                    continue;
                }
                float curved;
                switch (p.transfer)
                {
                case AVIFGPU_TRANSFER_PQ: curved = LinearToPQ(color[i], p.pqMultiplier, t); break;
                case AVIFGPU_TRANSFER_SMPTE428: curved = LinearToSMPTE428(color[i], t); break;
                case AVIFGPU_TRANSFER_HLG: curved = LinearToHLG(color[i], t); break;
                default: curved = color[i]; break;
                }
                codes[i] = FloatToCode(curved, p.maxCodeFloat);
            }
        }
        if (p.hasAlpha)
        {
            codes[colors] = FloatToCode(alpha, p.maxCodeFloat);
        }
    }
    else
    {
        constexpr int hostDepth = HostTraits<HostT>::depth;
        if (hostDepth == 16 && colors == 1 && p.gray16Smpte428)
        {
            codes[0] = FloatToCode(LinearToSMPTE428(static_cast<float>(px[0]) / 32768.0f, t), p.maxCodeFloat);
            if (p.hasAlpha)
            {
                codes[1] = DepthLutEntry(px[1], 32768.0f, p.maxCode);
            }
            return;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
        {
            if (i < channels)
            {
                if (hostDepth == 8)
                {
                    codes[i] = (p.imageDepth == 8) ? static_cast<uint32_t>(px[i]) : DepthLutEntry(px[i], 255.0f, p.maxCode);
                }
                else
                {
                    codes[i] = DepthLutEntry(px[i], 32768.0f, p.maxCode);
                }
            }
        }
        if (p.hasAlpha && p.premultiply)
        {
            const uint32_t alpha = codes[colors];
#pragma unroll
            for (int i = 0; i < 3; ++i)
            {
                if (i < colors)
                {
                    codes[i] = PremultiplyCodeGuarded(codes[i], alpha, p.maxCode);
                }
            }
        }
    }
}

__device__ __forceinline__ void StoreCode(void* plane, int64_t stride, int y, int index, bool wide, uint32_t code)
{
    uint8_t* row = static_cast<uint8_t*>(plane) + static_cast<int64_t>(y) * stride;
    if (wide)
    {
        reinterpret_cast<uint16_t*>(row)[index] = static_cast<uint16_t>(code);
    }
    else
    {
        row[index] = static_cast<uint8_t>(code);
    }
}

// Reference layout: one thread per pixel.
template <typename HostT>
__global__ void __launch_bounds__(kThreads) EncodeReferenceLayoutKernel(const EncodeParams p)
{
    __shared__ uint64_t libmStorage[96];
    const LibmTables t = avifmath::StageLibmTables(libmStorage, threadIdx.x, blockDim.x);
    __syncthreads();

    const int chunks = (p.width + kThreads - 1) / kThreads;
    const int x = static_cast<int>(blockIdx.x % chunks) * kThreads + threadIdx.x;
    const int y = static_cast<int>(blockIdx.x / chunks);
    if (x >= p.width || y >= p.rowCount)
    {
        return;
    }
    const HostT* px = reinterpret_cast<const HostT*>(static_cast<const uint8_t*>(p.rows) + static_cast<int64_t>(y) * p.rowStride) +
                      static_cast<int64_t>(x) * p.channels;
    uint32_t codes[4] = { 0, 0, 0, 0 };
    HostPixelToCodes<HostT>(p, px, codes, t);

    const bool wide = p.imageDepth > 8;
    if (p.channels <= 2)
    {
        StoreCode(p.plane[0], p.planeStride[0], y, x, wide, codes[0]);
        if (p.hasAlpha)
        {
            StoreCode(p.plane[3], p.planeStride[3], y, x, wide, codes[1]);
        }
    }
    else
    {
        for (int i = 0; i < p.channels; ++i)
        {
            StoreCode(p.plane[0], p.planeStride[0], y, x * p.channels + i, wide, codes[i]);
        }
    }
}

// Planar YCbCr layout: one thread per chroma site (1x1, 2x1 or 2x2 pixels).
template <typename HostT>
__global__ void __launch_bounds__(kThreads) EncodePlanarKernel(const EncodeParams p)
{
    __shared__ uint64_t libmStorage[96];
    const LibmTables t = avifmath::StageLibmTables(libmStorage, threadIdx.x, blockDim.x);
    __syncthreads();

    const int chunks = (((p.width + p.xs) >> p.xs) + kThreads - 1) / kThreads;
    const int cx = static_cast<int>(blockIdx.x % chunks) * kThreads + threadIdx.x;
    const int cy = static_cast<int>(blockIdx.x / chunks);
    const int x0 = cx << p.xs;
    const int y0 = cy << p.ys;
    if (x0 >= p.width || y0 >= p.rowCount)
    {
        return;
    }
    const bool wide = p.imageDepth > 8;
    const int maxCode = static_cast<int>(p.maxCode);
    float cb[2][2];
    float cr[2][2];
    bool have[2][2] = { { false, false }, { false, false } };

#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
    {
#pragma unroll
        for (int dx = 0; dx < 2; ++dx)
        {
            const int x = x0 + dx;
            const int y = y0 + dy;
            cb[dy][dx] = 0.0f;
            cr[dy][dx] = 0.0f;
            if (dx > p.xs || dy > p.ys || x >= p.width || y >= p.rowCount)
            {
                continue;
            }
            const HostT* px = reinterpret_cast<const HostT*>(static_cast<const uint8_t*>(p.rows) + static_cast<int64_t>(y) * p.rowStride) +
                              static_cast<int64_t>(x) * p.channels;
            uint32_t codes[4] = { 0, 0, 0, 0 };
            HostPixelToCodes<HostT>(p, px, codes, t);
            float yf;
            ForwardPixel(p.matrix, codes[0], codes[1], codes[2], yf, cb[dy][dx], cr[dy][dx]);
            have[dy][dx] = true;
            StoreCode(p.plane[0], p.planeStride[0], y, x, wide, QuantiseLuma(yf, maxCode));
            if (p.hasAlpha)
            {
                StoreCode(p.plane[3], p.planeStride[3], y, x, wide, codes[3]);
            }
        }
    }

    float cbv, crv;
    if (p.topLeft || (!p.xs && !p.ys))
    {
        cbv = cb[0][0];
        crv = cr[0][0];
    }
    else if (have[0][1] && have[1][0])
    {
        cbv = ((cb[0][0] + cb[0][1]) + (cb[1][0] + cb[1][1])) * 0.25f;
        crv = ((cr[0][0] + cr[0][1]) + (cr[1][0] + cr[1][1])) * 0.25f;
    }
    else if (have[0][1])
    {
        cbv = (cb[0][0] + cb[0][1]) * 0.5f;
        crv = (cr[0][0] + cr[0][1]) * 0.5f;
    }
    else if (have[1][0])
    {
        cbv = (cb[0][0] + cb[1][0]) * 0.5f;
        crv = (cr[0][0] + cr[1][0]) * 0.5f;
    }
    else
    {
        cbv = cb[0][0];
        crv = cr[0][0];
    }
    StoreCode(p.plane[1], p.planeStride[1], cy, cx, wide, QuantiseChroma(cbv, p.chromaOffset, maxCode));
    StoreCode(p.plane[2], p.planeStride[2], cy, cx, wide, QuantiseChroma(crv, p.chromaOffset, maxCode));
}

// ---- decode -------------------------------------------------------------------------------------------------

template <typename PlaneT>
__device__ __forceinline__ uint32_t LoadSample(const void* plane, int64_t stride, int x, int y)
{
    return reinterpret_cast<const PlaneT*>(static_cast<const uint8_t*>(plane) + static_cast<int64_t>(y) * stride)[x];
}

// The EOTF switch of YuvDecode.cpp:559-588 / 660-689 and ReadHeifImage.cpp:1062-1090, 1129-1157.
__device__ __forceinline__ void ApplyEotf(const DecodeParams& p, float R, float G, float B, float* out, const LibmTables& t)
{
    switch (p.transfer)
    {
    case AVIFGPU_TRANSFER_PQ:
        out[0] = PQToLinear(R, p.pqMultiplier, t);
        out[1] = PQToLinear(G, p.pqMultiplier, t);
        out[2] = PQToLinear(B, p.pqMultiplier, t);
        break;
    case AVIFGPU_TRANSFER_HLG:
    {
        float r = HLGToLinear(R, t);
        float g = HLGToLinear(G, t);
        float b = HLGToLinear(B, t);
        if (p.applyOotf)
        {
            ApplyHLGOOTF(r, g, b, p.lumaR, p.lumaG, p.lumaB, p.gammaMinusOne, p.hlgPeak, t);
        }
        out[0] = r;
        out[1] = g;
        out[2] = b;
        break;
    }
    default:
        out[0] = SMPTE428ToLinear(R, t);
        out[1] = SMPTE428ToLinear(G, t);
        out[2] = SMPTE428ToLinear(B, t);
        break;
    }
}

// PlaneT uint8_t pairs with HostT uint8_t; PlaneT uint16_t with HostT uint16_t or float.
template <typename PlaneT, typename HostT>
__global__ void __launch_bounds__(kThreads) DecodeKernel(const DecodeParams p)
{
    __shared__ uint64_t libmStorage[96];
    const LibmTables t = avifmath::StageLibmTables(libmStorage, threadIdx.x, blockDim.x);
    __syncthreads();

    const int chunks = (p.width + kThreads - 1) / kThreads;
    const int x = static_cast<int>(blockIdx.x % chunks) * kThreads + threadIdx.x;
    const int y = static_cast<int>(blockIdx.x / chunks);
    if (x >= p.width || y >= p.rowCount)
    {
        return;
    }
    constexpr bool hostIs8 = sizeof(HostT) == 1;
    constexpr bool hostIsFloat = sizeof(HostT) == 4;
    const uint32_t maxCode = p.maxCode;
    const int channels = (p.colorspace == AVIFGPU_COLORSPACE_MONOCHROME) ? (p.hasAlpha ? 2 : 1) : (p.hasAlpha ? 4 : 3);
    HostT* out = reinterpret_cast<HostT*>(static_cast<uint8_t*>(p.rows) + static_cast<int64_t>(y) * p.rowStride) +
                 static_cast<int64_t>(x) * channels;

    uint32_t unormA = p.hasAlpha ? LoadSample<PlaneT>(p.plane[3], p.planeStride[3], x, y) : 0;

    if (p.colorspace == AVIFGPU_COLORSPACE_YCBCR)
    {
        // ReadHeifImage.cpp:83-400 driving YuvDecode.cpp:281-696
        const int uvI = x >> p.xs;
        const int uvJ = (y + p.yPhase) >> p.ys;
        uint32_t unormY = LoadSample<PlaneT>(p.plane[0], p.planeStride[0], x, y);
        uint32_t unormU = LoadSample<PlaneT>(p.plane[1], p.planeStride[1], uvI, uvJ);
        uint32_t unormV = LoadSample<PlaneT>(p.plane[2], p.planeStride[2], uvI, uvJ);
        if (!hostIs8)
        {
            unormY = min(unormY, maxCode);
            unormU = min(unormU, maxCode);
            unormV = min(unormV, maxCode);
            unormA = min(unormA, maxCode);
        }
        const float Y = UnormToFloatY(unormY, p.range);
        const float Cb = UnormToFloatUV(unormU, p.range);
        const float Cr = UnormToFloatUV(unormV, p.range);
        float R, G, B;
        YuvToRgb(p.matrix, Y, Cb, Cr, R, G, B);
        float A = 0.0f;
        if (p.hasAlpha)
        {
            A = UnormToFloatPlain(unormA, p.range.maxChannelFloat);
            if (p.premultiplied && unormA < maxCode)
            {
                if (unormA == 0)
                {
                    R = 0;
                    G = 0;
                    B = 0;
                }
                else
                {
                    R = UnpremultiplyColor(R, A, 1.0f);
                    G = UnpremultiplyColor(G, A, 1.0f);
                    B = UnpremultiplyColor(B, A, 1.0f);
                }
            }
        }
        if constexpr (hostIs8)
        {
            out[0] = static_cast<uint8_t>(0.5f + (R * 255.0f));
            out[1] = static_cast<uint8_t>(0.5f + (G * 255.0f));
            out[2] = static_cast<uint8_t>(0.5f + (B * 255.0f));
            if (p.hasAlpha) out[3] = static_cast<uint8_t>(unormA);
        }
        else if constexpr (hostIsFloat)
        {
            float rgb[3];
            ApplyEotf(p, R, G, B, rgb, t);
            out[0] = rgb[0];
            out[1] = rgb[1];
            out[2] = rgb[2];
            if (p.hasAlpha) out[3] = A;
        }
        else
        {
            out[0] = static_cast<uint16_t>(0.5f + (R * 32768.0f));
            out[1] = static_cast<uint16_t>(0.5f + (G * 32768.0f));
            out[2] = static_cast<uint16_t>(0.5f + (B * 32768.0f));
            if (p.hasAlpha) out[3] = static_cast<uint16_t>(0.5f + (A * 32768.0f));
        }
    }
    else if (p.colorspace == AVIFGPU_COLORSPACE_MONOCHROME)
    {
        // ReadHeifImage.cpp:418-559, 863-947 driving YuvDecode.cpp:55-279
        uint32_t unormY = LoadSample<PlaneT>(p.plane[0], p.planeStride[0], x, y);
        if (!hostIs8)
        {
            unormY = min(unormY, maxCode);
            unormA = min(unormA, maxCode);
        }
        if constexpr (hostIsFloat)
        {
            // GrayAlpha32 un-premultiplies in the INTEGER domain (YuvDecode.cpp:247-260)
            if (p.hasAlpha && p.premultiplied && unormA < maxCode)
            {
                unormY = (unormA == 0) ? 0 : UnpremultiplyCode(unormY, unormA, static_cast<float>(maxCode));
            }
            out[0] = PQToLinear(UnormToFloatY(unormY, p.range), p.pqMultiplier, t);
            if (p.hasAlpha) out[1] = UnormToFloatPlain(unormA, p.range.maxChannelFloat);
        }
        else
        {
            float Y = UnormToFloatY(unormY, p.range);
            float A = 0.0f;
            if (p.hasAlpha)
            {
                A = UnormToFloatPlain(unormA, p.range.maxChannelFloat);
                if (p.premultiplied && unormA < maxCode)
                {
                    Y = (unormA == 0) ? 0.0f : UnpremultiplyColor(Y, A, 1.0f);
                }
            }
            if constexpr (hostIs8)
            {
                out[0] = static_cast<uint8_t>(0.5f + (Y * 255.0f));
                if (p.hasAlpha) out[1] = static_cast<uint8_t>(unormA);
            }
            else
            {
                out[0] = static_cast<uint16_t>(0.5f + (Y * 32768.0f));
                if (p.hasAlpha) out[1] = static_cast<uint16_t>(0.5f + (A * 32768.0f));
            }
        }
    }
    else
    {
        // planar RGB: ReadHeifImage.cpp:561-712 (8), 714-861 (16), 949-1178 (32)
        uint32_t c[3];
#pragma unroll
        for (int i = 0; i < 3; ++i)
        {
            c[i] = LoadSample<PlaneT>(p.plane[i], p.planeStride[i], x, y);
        }
        if constexpr (hostIsFloat)
        {
#pragma unroll
            for (int i = 0; i < 3; ++i) c[i] = min(c[i], maxCode); // DEFINED: clamp (the reference indexes out of bounds)
            unormA = min(unormA, maxCode);
        }
        else if constexpr (!hostIs8)
        {
#pragma unroll
            for (int i = 0; i < 3; ++i) c[i] &= maxCode; // ReadHeifImage.cpp:789-792
            unormA &= maxCode;
        }
        if (p.hasAlpha && p.premultiplied && unormA < maxCode)
        {
#pragma unroll
            for (int i = 0; i < 3; ++i)
            {
                c[i] = (unormA == 0) ? 0 : UnpremultiplyCode(c[i], unormA, static_cast<float>(maxCode));
            }
        }
        if constexpr (hostIsFloat)
        {
            const float maxF = p.range.maxChannelFloat;
            float rgb[3];
            ApplyEotf(p, UnormToFloatPlain(c[0], maxF), UnormToFloatPlain(c[1], maxF), UnormToFloatPlain(c[2], maxF), rgb, t);
            out[0] = rgb[0];
            out[1] = rgb[1];
            out[2] = rgb[2];
            if (p.hasAlpha) out[3] = UnormToFloatPlain(unormA, maxF);
        }
        else
        {
            out[0] = static_cast<HostT>(c[0]);
            out[1] = static_cast<HostT>(c[1]);
            out[2] = static_cast<HostT>(c[2]);
            if (p.hasAlpha) out[3] = static_cast<HostT>(unormA);
        }
    }
}

// ---- primitive sweep (parity gates on the device libm) ------------------------------------------------------

__global__ void __launch_bounds__(kThreads) TransferKernel(int function, float param, const float* __restrict__ in,
                                                           float* __restrict__ out, size_t count)
{
    __shared__ uint64_t libmStorage[96];
    const LibmTables t = avifmath::StageLibmTables(libmStorage, threadIdx.x, blockDim.x);
    __syncthreads();
    const float luminanceForward = param / 10000.0f;  // ColorTransfer.cpp:86
    const float luminanceInverse = 10000.0f / param;  // ColorTransfer.cpp:114
    for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < count;
         i += static_cast<size_t>(gridDim.x) * blockDim.x)
    {
        const float v = in[i];
        float r;
        switch (function)
        {
        case AVIFGPU_FN_LINEAR_TO_PQ: r = LinearToPQ(v, luminanceForward, t); break;
        case AVIFGPU_FN_PQ_TO_LINEAR: r = PQToLinear(v, luminanceInverse, t); break;
        case AVIFGPU_FN_LINEAR_TO_SMPTE428: r = LinearToSMPTE428(v, t); break;
        case AVIFGPU_FN_SMPTE428_TO_LINEAR: r = SMPTE428ToLinear(v, t); break;
        case AVIFGPU_FN_HLG_TO_LINEAR: r = HLGToLinear(v, t); break;
        case AVIFGPU_FN_LINEAR_TO_HLG: r = LinearToHLG(v, t); break;
        case AVIFGPU_FN_POWF: r = avifmath::Powf(v, param, t); break;
        case AVIFGPU_FN_EXPF: r = avifmath::Expf(v, t); break;
        default: r = avifmath::Logf(v, t); break;
        }
        out[i] = r;
    }
}

} // namespace

int LaunchEncodeGeneric(const EncodeParams& params, int hostDepth, void* streamHandle)
{
    cudaStream_t stream = static_cast<cudaStream_t>(streamHandle);
    if (params.width <= 0 || params.rowCount <= 0)
    {
        return 0;
    }
    EncodeParams p = params;
    p.useCurveView = 0;
    if (hostDepth == 32 && p.curveTable != nullptr && p.curveTable->flat != nullptr && p.curveTable->bandBits != nullptr &&
        (p.transfer == AVIFGPU_TRANSFER_PQ || p.transfer == AVIFGPU_TRANSFER_SMPTE428 || p.transfer == AVIFGPU_TRANSFER_HLG))
    {
        p.curveView = *p.curveTable;
        p.useCurveView = 1;
    }
    if (p.planar)
    {
        const int sitesX = (p.width + p.xs) >> p.xs;
        const int sitesY = (p.rowCount + p.ys) >> p.ys;
        const unsigned grid = static_cast<unsigned>((sitesX + kThreads - 1) / kThreads) * static_cast<unsigned>(sitesY);
        switch (hostDepth)
        {
        case 8: EncodePlanarKernel<uint8_t><<<grid, kThreads, 0, stream>>>(p); break;
        case 16: EncodePlanarKernel<uint16_t><<<grid, kThreads, 0, stream>>>(p); break;
        default: EncodePlanarKernel<float><<<grid, kThreads, 0, stream>>>(p); break;
        }
    }
    else
    {
        const unsigned grid = static_cast<unsigned>((p.width + kThreads - 1) / kThreads) * static_cast<unsigned>(p.rowCount);
        switch (hostDepth)
        {
        case 8: EncodeReferenceLayoutKernel<uint8_t><<<grid, kThreads, 0, stream>>>(p); break;
        case 16: EncodeReferenceLayoutKernel<uint16_t><<<grid, kThreads, 0, stream>>>(p); break;
        default: EncodeReferenceLayoutKernel<float><<<grid, kThreads, 0, stream>>>(p); break;
        }
    }
    const cudaError_t launchError = cudaGetLastError();
    return launchError == cudaSuccess ? 1 : ReportLaunchFailure(static_cast<int>(launchError));
}

int LaunchDecodeGeneric(const DecodeParams& p, void* streamHandle)
{
    cudaStream_t stream = static_cast<cudaStream_t>(streamHandle);
    if (p.width <= 0 || p.rowCount <= 0)
    {
        return 0;
    }
    const unsigned grid = static_cast<unsigned>((p.width + kThreads - 1) / kThreads) * static_cast<unsigned>(p.rowCount);
    switch (p.hostDepth)
    {
    case 8: DecodeKernel<uint8_t, uint8_t><<<grid, kThreads, 0, stream>>>(p); break;
    case 16: DecodeKernel<uint16_t, uint16_t><<<grid, kThreads, 0, stream>>>(p); break;
    default: DecodeKernel<uint16_t, float><<<grid, kThreads, 0, stream>>>(p); break;
    }
    const cudaError_t launchError = cudaGetLastError();
    return launchError == cudaSuccess ? 1 : ReportLaunchFailure(static_cast<int>(launchError));
}

int LaunchEncodeRemainder(const EncodeParams& p, int hostDepth, int coveredWidth, int coveredRows, void* stream)
{
    const int right = LaunchEncodeGeneric(EncodeSubRect(p, hostDepth, coveredWidth, 0, p.width - coveredWidth, p.rowCount), hostDepth, stream);
    if (right < 0)
    {
        return right;
    }
    const int bottom = LaunchEncodeGeneric(EncodeSubRect(p, hostDepth, 0, coveredRows, coveredWidth, p.rowCount - coveredRows), hostDepth, stream);
    return bottom < 0 ? bottom : right + bottom;
}

int LaunchDecodeRemainder(const DecodeParams& p, int coveredWidth, int coveredRows, void* stream)
{
    const int right = LaunchDecodeGeneric(DecodeSubRect(p, coveredWidth, 0, p.width - coveredWidth, p.rowCount), stream);
    if (right < 0)
    {
        return right;
    }
    const int bottom = LaunchDecodeGeneric(DecodeSubRect(p, 0, coveredRows, coveredWidth, p.rowCount - coveredRows), stream);
    return bottom < 0 ? bottom : right + bottom;
}

int LaunchTransfer(int function, float param, const float* in, float* out, size_t count, void* streamHandle)
{
    cudaStream_t stream = static_cast<cudaStream_t>(streamHandle);
    if (count == 0)
    {
        return 0;
    }
    size_t blocks = (count + kThreads - 1) / kThreads;
    if (blocks > 148u * 16u)
    {
        blocks = 148u * 16u;
    }
    TransferKernel<<<static_cast<unsigned>(blocks), kThreads, 0, stream>>>(function, param, in, out, count);
    const cudaError_t launchError = cudaGetLastError();
    return launchError == cudaSuccess ? 1 : ReportLaunchFailure(static_cast<int>(launchError));
}

namespace
{
// ColorTransfer.cpp:192-220 over `pixels` RGB triples.
__global__ void __launch_bounds__(kThreads) HlgOotfKernel(int inverse, float lumaR, float lumaG, float lumaB, float displayGamma, float peak,
                                                          const float* __restrict__ in, float* __restrict__ out, size_t pixels)
{
    __shared__ uint64_t libmStorage[96];
    const LibmTables t = avifmath::StageLibmTables(libmStorage, threadIdx.x, blockDim.x);
    __syncthreads();
    for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < pixels; i += static_cast<size_t>(gridDim.x) * blockDim.x)
    {
        float r = in[3 * i], g = in[3 * i + 1], b = in[3 * i + 2];
        if (inverse)
        {
            ApplyInverseHLGOOTF(r, g, b, lumaR, lumaG, lumaB, displayGamma, peak, t);
        }
        else
        {
            ApplyHLGOOTF(r, g, b, lumaR, lumaG, lumaB, displayGamma - 1.0f, peak, t);
        }
        out[3 * i] = r;
        out[3 * i + 1] = g;
        out[3 * i + 2] = b;
    }
}
} // namespace

int LaunchHlgOotf(int inverse, const float luma[3], float displayGamma, float peak, const float* in, float* out, size_t pixels, void* streamHandle)
{
    if (pixels == 0)
    {
        return 0;
    }
    size_t blocks = (pixels + kThreads - 1) / kThreads;
    if (blocks > 148 * 16)
    {
        blocks = 148 * 16;
    }
    HlgOotfKernel<<<static_cast<unsigned>(blocks), kThreads, 0, static_cast<cudaStream_t>(streamHandle)>>>(inverse, luma[0], luma[1], luma[2], displayGamma, peak, in,
                                                                                                      out, pixels);
    const cudaError_t launchError = cudaGetLastError();
    return launchError == cudaSuccess ? 1 : ReportLaunchFailure(static_cast<int>(launchError));
}

} // namespace avifgpu
