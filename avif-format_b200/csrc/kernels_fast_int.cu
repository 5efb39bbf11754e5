// kernels_fast_int.cu -- tuned kernels for the 16-bit integer hosts (BASELINE configs 4 and 5).  Both are pure
// streaming conversions (a few float operations per sample), so the design goal is simply to keep HBM busy:
// 128-bit loads and stores, several of them in flight per thread, no integer<->float conversion instructions
// (they issue on the quarter-rate pipe and would cap config 4 just below the HBM roofline).
//
//   Gray16 -> Y plane          one 65536-entry uint16 table in shared memory (128 KB), built once per
//                              configuration by evaluating the exact per-sample formula for every input; a thread
//                              converts 8 samples per 128-bit load.
//   RGB(A)16 -> planar YCbCr   the 16-bit -> N-bit mapping is evaluated arithmetically (it is four float
//                              operations), the forward matrix and the 4:2:2 / 4:2:0 down-filter are fused, a
//                              thread converts 8 pixels (x 2 rows for 4:2:0).
#include "group_walk.cuh"
#include "kernel_params.h"
#include "packed_f32x2.cuh"
#include "../../include/avifgpu.h"

#include <cuda_runtime.h>

namespace avifgpu
{

using namespace avifpix;
using avifmath::LibmTables;

namespace
{

// ---- Gray16 --------------------------------------------------------------------------------------------------------

constexpr int kLutThreads = 1024;
constexpr int kLutEntries = 65536;

// Fills lut[v] for every 16-bit host sample with the exact code of the configuration:
//   reference LUT path   clamp((int)((v / 32768f) * max + 0.5f), 0, max)                       WriteHeifImage.cpp:140-166
//   SMPTE 428 curve      (u16)clamp(LinearToSMPTE428(v / 32768f) * max, 0, max)                 DESIGN.md "Config 5"
__global__ void __launch_bounds__(256) BuildGray16LutKernel(uint16_t* __restrict__ lut, int smpte428, uint32_t maxCode)
{
    __shared__ uint64_t libmStorage[96];
    const LibmTables t = avifmath::StageLibmTables(libmStorage, threadIdx.x, blockDim.x);
    __syncthreads();
    const float maxCodeFloat = static_cast<float>(maxCode);
    for (uint32_t v = blockIdx.x * blockDim.x + threadIdx.x; v < kLutEntries; v += gridDim.x * blockDim.x)
    {
        uint32_t code;
        if (smpte428)
        {
            code = FloatToCode(LinearToSMPTE428(static_cast<float>(v) / 32768.0f, t), maxCodeFloat);
        }
        else
        {
            code = DepthLutEntry(v, 32768.0f, maxCode);
        }
        lut[v] = static_cast<uint16_t>(code);
    }
}

struct Gray16Params
{
    const uint8_t* rows;
    int64_t rowStride;
    uint8_t* planeY;
    int64_t strideY;
    int32_t chunksPerRow; // 8 samples each
    int32_t rowCount;
    const uint16_t* lut;  // 65536 entries, global memory
};

__device__ __forceinline__ uint4 LookupEight(const uint16_t* __restrict__ lut, uint4 in)
{
    uint4 out;
    out.x = lut[in.x & 0xffffu] | (static_cast<uint32_t>(lut[in.x >> 16]) << 16);
    out.y = lut[in.y & 0xffffu] | (static_cast<uint32_t>(lut[in.y >> 16]) << 16);
    out.z = lut[in.z & 0xffffu] | (static_cast<uint32_t>(lut[in.z >> 16]) << 16);
    out.w = lut[in.w & 0xffffu] | (static_cast<uint32_t>(lut[in.w >> 16]) << 16);
    return out;
}

__global__ void __launch_bounds__(kLutThreads, 1) EncodeGray16LutKernel(const Gray16Params p)
{
    extern __shared__ __align__(16) uint16_t sharedLut[];
    {
        const uint4* source = reinterpret_cast<const uint4*>(p.lut);
        uint4* target = reinterpret_cast<uint4*>(sharedLut);
        for (int i = threadIdx.x; i < kLutEntries * 2 / 16; i += blockDim.x)
        {
            target[i] = source[i];
        }
    }
    __syncthreads();

    constexpr int kUnroll = 4;
    const long long chunks = static_cast<long long>(p.chunksPerRow) * p.rowCount;
    const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
    // (measured: walking row / column incrementally, group_walk.cuh, makes THIS loop slower -- 0.86 vs 0.95 of the HBM
    // peak; the division is hidden under four loads in flight and a 16-bit look-up per sample)
    for (long long base = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; base < chunks; base += stride * kUnroll)
    {
        uint4 in[kUnroll];
        long long outOffset[kUnroll];
#pragma unroll
        for (int u = 0; u < kUnroll; ++u)
        {
            const long long chunk = base + u * stride;
            if (chunk < chunks)
            {
                const long long row = chunk / p.chunksPerRow;
                const long long column = chunk - row * p.chunksPerRow;
                in[u] = __ldcs(reinterpret_cast<const uint4*>(p.rows + row * p.rowStride + column * 16));
                outOffset[u] = row * p.strideY + column * 16;
            }
            else
            {
                in[u] = make_uint4(0u, 0u, 0u, 0u);
                outOffset[u] = -1;
            }
        }
#pragma unroll
        for (int u = 0; u < kUnroll; ++u)
        {
            if (outOffset[u] >= 0)
            {
                __stcs(reinterpret_cast<uint4*>(p.planeY + outOffset[u]), LookupEight(sharedLut, in[u]));
            }
        }
    }
}

// ---- RGB(A)16 -> planar YCbCr ---------------------------------------------------------------------------------------

constexpr int kRgbThreads = 256;
constexpr float kTwo23 = 8388608.0f;

// (float)v for v < 2^23 without the conversion instruction.
__device__ __forceinline__ float UintToFloatExact(uint32_t v) { return __uint_as_float(0x4b000000u | v) - kTwo23; }

// 2^23 + min(trunc(t), maxCode) as a float, for 0 <= t < 2^23: adding 2^23 with round-toward-zero leaves floor(t) in
// the low mantissa bits.  Bit-identical to (int)t followed by the upper clamp of the reference's LUT builder.
__device__ __forceinline__ float BiasedTrunc(float t, float biasedMax) { return fminf(__fadd_rz(t, kTwo23), biasedMax); }

struct Rgb16Params
{
    const uint8_t* rows;
    int64_t rowStride;
    uint8_t* plane[4];
    int64_t stride[4];
    int32_t groupsPerRow; // 8 pixels each
    int32_t rowCount;     // even when YS == 1
    float maxCodeFloat;
    float biasedMax;      // 2^23 + maxCode
    ForwardMatrix matrix;
    float chromaOffset;
    int32_t topLeft;
    uint32_t maxCode;
    float maxReciprocal; // RN(1 / maxCode), for the verified premultiply
};

// PremultiplyColor(uint16_t, uint16_t, maxValue) (PremultipliedAlpha.cpp:62-70) behind the callers' guard
// (WriteHeifImage.cpp:947-965: alpha == max keeps the colour, alpha == 0 clears it) in six full-rate instructions:
//     product (exact: both codes < 2^12)  ->  / max by reciprocal + one residual step  ->  + 0.5, truncate.
// The division by reciprocal is not the IEEE division and trunc(x + 0.5) is not roundf(x) for every float x, but over the
// (max + 1)^2 code pairs of a bit depth it either always agrees with the reference's own sequence or it does not:
// VerifyFastPremultiplyKernel enumerates them all, and the tuned kernel is used only for depths that passed.  No special
// cases are needed: alpha == 0 gives a zero product, alpha == max gives product / max == colour exactly.
__device__ __forceinline__ float FastPremultiplyBiased(float colour, float alpha, float maxCodeFloat, float maxReciprocal)
{
    const float product = __fmul_rn(colour, alpha);
    const float quotient = DivideByConstant(product, maxCodeFloat, maxReciprocal);
    return __fadd_rz(__fadd_rn(quotient, 0.5f), kTwo23); // 2^23 + code
}

// The same six operations on two (colour, alpha) pairs at once (packed_f32x2.cuh): lane for lane the IEEE operations of
// FastPremultiplyBiased -- fma(-q, d, x) == fma(q, -d, x) -- so VerifyFastPremultiply's enumeration covers it.
__device__ __forceinline__ avifx2::F32x2 FastPremultiplyBiasedPair(avifx2::F32x2 colour, avifx2::F32x2 alpha, float maxCodeFloat, float maxReciprocal)
{
    using namespace avifx2;
    const F32x2 product = Mul2(colour, alpha);
    const F32x2 q = Mul2(product, Splat(maxReciprocal));
    const F32x2 residual = Fma2(q, Splat(-maxCodeFloat), product);
    const F32x2 quotient = Fma2(residual, Splat(maxReciprocal), q);
    return AddRz2(Add2(quotient, Splat(0.5f)), Splat(kTwo23)); // 2^23 + code
}

__global__ void VerifyFastPremultiplyKernel(uint32_t maxCode, unsigned long long* __restrict__ counter)
{
    const float maxCodeFloat = static_cast<float>(maxCode);
    const float reciprocal = 1.0f / maxCodeFloat;
    const unsigned long long pairs = static_cast<unsigned long long>(maxCode + 1u) * (maxCode + 1u);
    unsigned long long bad = 0;
    for (unsigned long long i = static_cast<unsigned long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < pairs;
         i += static_cast<unsigned long long>(gridDim.x) * blockDim.x)
    {
        const uint32_t colour = static_cast<uint32_t>(i % (maxCode + 1u));
        const uint32_t alpha = static_cast<uint32_t>(i / (maxCode + 1u));
        const uint32_t expected = PremultiplyCodeGuarded(colour, alpha, maxCode);
        const uint32_t fast = __float_as_uint(FastPremultiplyBiased(static_cast<float>(colour), static_cast<float>(alpha), maxCodeFloat, reciprocal)) & 0x7fffffu;
        if (fast != expected)
        {
            ++bad;
        }
    }
    if (bad)
    {
        atomicAdd(counter, bad);
    }
}

// Host sample -> 2^23 + code, as a float.
//   16-bit host (0..32768, or beyond: the formula is defined to continue)  WriteHeifImage.cpp:140-166:
//       (int)((v / 32768f) * max + 0.5f), clamped -- v / 32768f is exact as a multiplication;
//   8-bit host, 8-bit image   the sample is the code                        WriteHeifImage.cpp:743-747
//   8-bit host, deeper image  (int)((v / 255f) * max + 0.5f): a true division, so the 256 results are tabulated in
//                             shared memory at kernel start (the reference builds the same table, :87-112).
template <typename HostT, typename PlaneT>
__device__ __forceinline__ float SampleToBiasedCode(uint32_t v, const Rgb16Params& p, const float* __restrict__ hostLut)
{
    if (sizeof(HostT) == 2)
    {
        const float t = ((UintToFloatExact(v) * (1.0f / 32768.0f)) * p.maxCodeFloat) + 0.5f;
        return BiasedTrunc(t, p.biasedMax);
    }
    if (sizeof(PlaneT) == 1)
    {
        return __uint_as_float(0x4b000000u | v);
    }
    return hostLut[v];
}

__device__ __forceinline__ uint32_t BiasedToCode(float biased) { return __float_as_uint(biased) & 0x7fffffu; }

// 8 (4) consecutive plane samples in one vector store.
template <typename PlaneT>
__device__ __forceinline__ void StoreEight(uint8_t* address, const uint32_t (&c)[8])
{
    if (sizeof(PlaneT) == 2)
    {
        __stcs(reinterpret_cast<uint4*>(address), make_uint4(c[0] | (c[1] << 16), c[2] | (c[3] << 16), c[4] | (c[5] << 16), c[6] | (c[7] << 16)));
    }
    else
    {
        __stcs(reinterpret_cast<uint2*>(address),
               make_uint2(c[0] | (c[1] << 8) | (c[2] << 16) | (c[3] << 24), c[4] | (c[5] << 8) | (c[6] << 16) | (c[7] << 24)));
    }
}

template <typename PlaneT>
__device__ __forceinline__ void StoreFour(uint8_t* address, const uint32_t (&c)[4])
{
    if (sizeof(PlaneT) == 2)
    {
        __stcs(reinterpret_cast<uint2*>(address), make_uint2(c[0] | (c[1] << 16), c[2] | (c[3] << 16)));
    }
    else
    {
        __stcs(reinterpret_cast<uint32_t*>(address), c[0] | (c[1] << 8) | (c[2] << 16) | (c[3] << 24));
    }
}

// HostT: uint8_t / uint16_t host samples; PlaneT: uint8_t (8-bit image) / uint16_t (10 / 12-bit image) plane samples.
// PREMULTIPLY (CHANNELS == 4 only): the colour codes are multiplied by the alpha code in the image's depth before the matrix
// (WriteHeifImage.cpp:700-718, 760-778, 877-895, 947-965), through FastPremultiplyBiased.
template <typename HostT, typename PlaneT, int CHANNELS, int XS, int YS, int PREMULTIPLY>
__global__ void __launch_bounds__(kRgbThreads) EncodeRgbIntPlanarKernel(const Rgb16Params p)
{
    constexpr int kRows = 1 + YS;
    constexpr int kWordsPerRow = CHANNELS * 2 * static_cast<int>(sizeof(HostT)); // 8 pixels x CHANNELS samples / 4 bytes
    constexpr int kVectorWords = (kWordsPerRow % 4 == 0) ? 4 : 2;                 // 128-bit loads where the row chunk allows
    constexpr int kPlaneBytes = static_cast<int>(sizeof(PlaneT));
    // (one copy: a copy per shared-memory bank makes the look-up conflict-free but costs every CTA 32 KB and 8192 table
    // entries to fill -- measured slower, 724 -> 694 Gpx/s for RGB8 -> 10-bit 4:2:0 and 1711 -> 1377 for Gray8 -> 10-bit;
    // computing the entry instead -- division by 255 through a verified reciprocal step, packed -- is slower too, 727 -> 641:
    // the look-up's shared-memory pipe is the lesser evil next to six more instructions per sample)
    __shared__ float hostLut[(sizeof(HostT) == 1 && sizeof(PlaneT) == 2) ? 256 : 1];
    if (sizeof(HostT) == 1 && sizeof(PlaneT) == 2)
    {
        for (uint32_t v = threadIdx.x; v < 256; v += blockDim.x)
        {
            hostLut[v] = __uint_as_float(0x4b000000u | DepthLutEntry(v, 255.0f, p.maxCode));
        }
        __syncthreads();
    }
    const int32_t rowPairs = (p.rowCount + YS) >> YS;
    for (GroupWalk walk(static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x, static_cast<long long>(gridDim.x) * blockDim.x, p.groupsPerRow, rowPairs);
         walk.Inside(rowPairs); walk.Advance(rowPairs))
    {
        const long long rowPair = walk.row;
        const int column = walk.column; // in units of 8 pixels
        const long long y0 = rowPair << YS;

        uint32_t words[kRows][kWordsPerRow];
#pragma unroll
        for (int r = 0; r < kRows; ++r)
        {
            const uint8_t* source = p.rows + (y0 + r) * p.rowStride + static_cast<long long>(column) * (kWordsPerRow * 4);
#pragma unroll
            for (int q = 0; q < kWordsPerRow / kVectorWords; ++q)
            {
                if (kVectorWords == 4)
                {
                    const uint4 w = __ldcs(reinterpret_cast<const uint4*>(source) + q);
                    words[r][4 * q + 0] = w.x;
                    words[r][4 * q + 1] = w.y;
                    words[r][4 * q + 2] = w.z;
                    words[r][4 * q + 3] = w.w;
                }
                else
                {
                    const uint2 w = __ldcs(reinterpret_cast<const uint2*>(source) + q);
                    words[r][2 * q + 0] = w.x;
                    words[r][2 * q + 1] = w.y;
                }
            }
        }

        // The matrix runs on pixel pairs (2j, 2j + 1) in the two-lane FP32 instructions (packed_f32x2.cuh; its rule: a product
        // is never the operand of a packed add, so the three luma products and the chroma sums are added as scalars).  The
        // operations per pixel, and their roundings, are pixel_math.cuh's ForwardPixelFloat.
        using namespace avifx2;
        const F32x2 half2 = Splat(0.5f), bias2 = Splat(kTwo23), offset2 = Splat(p.chromaOffset);
        const F32x2 kr2 = Splat(p.matrix.kr), kg2 = Splat(p.matrix.kg), kb2 = Splat(p.matrix.kb);
        const F32x2 cbScale2 = Splat(p.matrix.cbScale), crScale2 = Splat(p.matrix.crScale);
        const F32x2 hostScale2 = Splat(p.maxCodeFloat * (1.0f / 32768.0f)); // exact: max <= 4095 times a power of two
        // 2^23 + trunc(v + 0.5) for both halves: BiasedToCode of either is the code (no upper clamp here)
        const auto biasedPair = [&](F32x2 v, float& lo, float& hi) { Unpack(AddRz2(Add2(v, half2), bias2), lo, hi); };
        const auto chromaClamp = [&](float biased) -> uint32_t { return BiasedToCode(fminf(biased, p.biasedMax)); }; // H.273: 2^depth -> 2^depth - 1

        F32x2 cb[kRows][4], cr[kRows][4]; // [row][pair]
#pragma unroll
        for (int r = 0; r < kRows; ++r)
        {
            uint32_t yCodes[8];
            uint32_t aCodes[8];
#pragma unroll
            for (int j = 0; j < 4; ++j)
            {
                // sample k of the row sits in half-word (byte) k of the loaded words
                auto sample = [&](int k) -> uint32_t
                {
                    if (sizeof(HostT) == 2)
                    {
                        const uint32_t w = words[r][k >> 1];
                        return (k & 1) ? (w >> 16) : (w & 0xffffu);
                    }
                    return (words[r][k >> 2] >> (8 * (k & 3))) & 0xffu;
                };
                // channel c of pixels 2j and 2j + 1 as 2^23-biased codes in the image's depth
                const auto biasedCodes = [&](int c) -> F32x2
                {
                    const uint32_t v0 = sample((2 * j) * CHANNELS + c), v1 = sample((2 * j + 1) * CHANNELS + c);
                    if (sizeof(HostT) == 2)
                    {
                        // SampleToBiasedCode on the pair: (v / 32768f) * max is ONE rounding (the division is a scaling by 2^-15 and
                        // max * 2^-15 is exact), so the single packed multiply by that constant is the same number; + 0.5f follows a
                        // product and stays scalar
                        float t0, t1;
                        Unpack(Mul2(Sub2(Pack(__uint_as_float(0x4b000000u | v0), __uint_as_float(0x4b000000u | v1)), bias2), hostScale2), t0, t1);
                        float b0, b1;
                        Unpack(AddRz2(Pack(__fadd_rn(t0, 0.5f), __fadd_rn(t1, 0.5f)), bias2), b0, b1);
                        return Pack(fminf(b0, p.biasedMax), fminf(b1, p.biasedMax));
                    }
                    return Pack(SampleToBiasedCode<HostT, PlaneT>(v0, p, hostLut), SampleToBiasedCode<HostT, PlaneT>(v1, p, hostLut));
                };
                F32x2 red, green, blue;
                if (PREMULTIPLY)
                {
                    // colour * alpha / max per channel on the pair
                    const F32x2 alphaBiased = biasedCodes(3);
                    const F32x2 alpha = Sub2(alphaBiased, bias2);
                    red = Sub2(FastPremultiplyBiasedPair(Sub2(biasedCodes(0), bias2), alpha, p.maxCodeFloat, p.maxReciprocal), bias2);
                    green = Sub2(FastPremultiplyBiasedPair(Sub2(biasedCodes(1), bias2), alpha, p.maxCodeFloat, p.maxReciprocal), bias2);
                    blue = Sub2(FastPremultiplyBiasedPair(Sub2(biasedCodes(2), bias2), alpha, p.maxCodeFloat, p.maxReciprocal), bias2);
                    float a0, a1;
                    Unpack(alphaBiased, a0, a1);
                    aCodes[2 * j] = BiasedToCode(a0);
                    aCodes[2 * j + 1] = BiasedToCode(a1);
                }
                else if (sizeof(HostT) == 2)
                {
                    red = Sub2(biasedCodes(0), bias2);
                    green = Sub2(biasedCodes(1), bias2);
                    blue = Sub2(biasedCodes(2), bias2);
                    if (CHANNELS == 4)
                    {
                        float a0, a1;
                        Unpack(biasedCodes(3), a0, a1);
                        aCodes[2 * j] = BiasedToCode(a0);
                        aCodes[2 * j + 1] = BiasedToCode(a1);
                    }
                }
                else
                {
                    float rf[2], gf[2], bf[2];
#pragma unroll
                    for (int h = 0; h < 2; ++h)
                    {
                        const int i = 2 * j + h;
                        if (sizeof(HostT) == 1 && sizeof(PlaneT) == 1)
                        {
                            // 8-bit host into an 8-bit image: the sample is the code.  Byte -> float is one conversion instruction
                            // (it takes the byte lane as an operand modifier).
                            rf[h] = static_cast<float>(static_cast<uint8_t>(sample(i * CHANNELS + 0)));
                            gf[h] = static_cast<float>(static_cast<uint8_t>(sample(i * CHANNELS + 1)));
                            bf[h] = static_cast<float>(static_cast<uint8_t>(sample(i * CHANNELS + 2)));
                        }
                        else
                        {
                            rf[h] = SampleToBiasedCode<HostT, PlaneT>(sample(i * CHANNELS + 0), p, hostLut) - kTwo23;
                            gf[h] = SampleToBiasedCode<HostT, PlaneT>(sample(i * CHANNELS + 1), p, hostLut) - kTwo23;
                            bf[h] = SampleToBiasedCode<HostT, PlaneT>(sample(i * CHANNELS + 2), p, hostLut) - kTwo23;
                        }
                        if (CHANNELS == 4)
                        {
                            aCodes[i] = (sizeof(HostT) == 1 && sizeof(PlaneT) == 1) ? sample(i * CHANNELS + 3)
                                                                                    : BiasedToCode(SampleToBiasedCode<HostT, PlaneT>(sample(i * CHANNELS + 3), p, hostLut));
                        }
                    }
                    red = Pack(rf[0], rf[1]);
                    green = Pack(gf[0], gf[1]);
                    blue = Pack(bf[0], bf[1]);
                }
                F32x2 luma;
                if (p.matrix.identity)
                {
                    luma = green;
                    cb[r][j] = blue;
                    cr[r][j] = red;
                }
                else
                {
                    float r0, r1, g0, g1, b0, b1;
                    Unpack(Mul2(red, kr2), r0, r1);
                    Unpack(Mul2(green, kg2), g0, g1);
                    Unpack(Mul2(blue, kb2), b0, b1);
                    luma = Pack(__fadd_rn(__fadd_rn(r0, g0), b0), __fadd_rn(__fadd_rn(r1, g1), b1)); // (kr R + kg G) + kb B
                    cb[r][j] = Mul2(Sub2(blue, luma), cbScale2);
                    cr[r][j] = Mul2(Sub2(red, luma), crScale2);
                }
                float luma0, luma1;
                biasedPair(luma, luma0, luma1); // no upper clamp: ForwardMatrixStaysInRange (launcher)
                yCodes[2 * j] = BiasedToCode(luma0);
                yCodes[2 * j + 1] = BiasedToCode(luma1);
            }
            StoreEight<PlaneT>(p.plane[0] + (y0 + r) * p.stride[0] + static_cast<long long>(column) * (8 * kPlaneBytes), yCodes);
            if (CHANNELS == 4)
            {
                StoreEight<PlaneT>(p.plane[3] + (y0 + r) * p.stride[3] + static_cast<long long>(column) * (8 * kPlaneBytes), aCodes);
            }
        }

        // chroma: down-filter in float, then quantise (the offset is 0 for the identity matrix); chroma values are products
        // (or, for the identity matrix, plain samples): the offset is added to each half as a scalar, like the sums
        const auto addOffset = [&](F32x2 product) -> F32x2
        {
            float c0, c1;
            Unpack(product, c0, c1);
            return Pack(__fadd_rn(c0, p.chromaOffset), __fadd_rn(c1, p.chromaOffset));
        };
        if (XS == 0)
        {
#pragma unroll
            for (int r = 0; r < kRows; ++r)
            {
                uint32_t cbCode[8], crCode[8];
#pragma unroll
                for (int j = 0; j < 4; ++j)
                {
                    float b0, b1, r0, r1;
                    biasedPair(addOffset(cb[r][j]), b0, b1);
                    biasedPair(addOffset(cr[r][j]), r0, r1);
                    cbCode[2 * j] = chromaClamp(b0);
                    cbCode[2 * j + 1] = chromaClamp(b1);
                    crCode[2 * j] = chromaClamp(r0);
                    crCode[2 * j + 1] = chromaClamp(r1);
                }
                const long long offset = static_cast<long long>(column) * (8 * kPlaneBytes);
                StoreEight<PlaneT>(p.plane[1] + (y0 + r) * p.stride[1] + offset, cbCode);
                StoreEight<PlaneT>(p.plane[2] + (y0 + r) * p.stride[2] + offset, crCode);
            }
        }
        else
        {
            // site s = pixels 2s, 2s + 1 (of both rows for 4:2:0) = the two halves of pair s; two sites per packed value
            uint32_t cbCode[4], crCode[4];
#pragma unroll
            for (int s = 0; s < 4; s += 2)
            {
                F32x2 cbBiased, crBiased; // chroma + offset for sites s, s + 1
                if (p.topLeft)
                {
                    float b0, b1, r0, r1, unused;
                    Unpack(cb[0][s], b0, unused);
                    Unpack(cb[0][s + 1], b1, unused);
                    Unpack(cr[0][s], r0, unused);
                    Unpack(cr[0][s + 1], r1, unused);
                    cbBiased = Pack(__fadd_rn(b0, p.chromaOffset), __fadd_rn(b1, p.chromaOffset));
                    crBiased = Pack(__fadd_rn(r0, p.chromaOffset), __fadd_rn(r1, p.chromaOffset));
                }
                else
                {
                    const auto siteSum = [&](const F32x2 (&plane)[kRows][4], int site) -> float
                    {
                        float top0, top1;
                        Unpack(plane[0][site], top0, top1);
                        const float top = __fadd_rn(top0, top1);
                        if (YS == 0)
                        {
                            return top;
                        }
                        float bottom0, bottom1;
                        Unpack(plane[kRows - 1][site], bottom0, bottom1);
                        return __fadd_rn(top, __fadd_rn(bottom0, bottom1)); // (c00 + c01) + (c10 + c11)
                    };
                    // * 0.25f (0.5f) is exact, so the fused multiply-add with the offset is the two-step number
                    const F32x2 scale2 = Splat(YS == 1 ? 0.25f : 0.5f);
                    cbBiased = Fma2(Pack(siteSum(cb, s), siteSum(cb, s + 1)), scale2, offset2);
                    crBiased = Fma2(Pack(siteSum(cr, s), siteSum(cr, s + 1)), scale2, offset2);
                }
                float b0, b1, r0, r1;
                biasedPair(cbBiased, b0, b1);
                biasedPair(crBiased, r0, r1);
                cbCode[s] = chromaClamp(b0);
                cbCode[s + 1] = chromaClamp(b1);
                crCode[s] = chromaClamp(r0);
                crCode[s + 1] = chromaClamp(r1);
            }
            const long long offset = static_cast<long long>(column) * (4 * kPlaneBytes);
            const long long chromaRow = YS ? rowPair : y0;
            StoreFour<PlaneT>(p.plane[1] + chromaRow * p.stride[1] + offset, cbCode);
            StoreFour<PlaneT>(p.plane[2] + chromaRow * p.stride[2] + offset, crCode);
        }
    }
}

// ---- Gray(+A) 8/16-bit hosts -> Y (+A) planes (WriteHeifImage.cpp:169-500 without premultiplication) ------------------------
// The same depth mapping as the colour kernel, no matrix: a thread converts 8 pixels.
template <typename HostT, typename PlaneT, int CHANNELS>
__global__ void __launch_bounds__(kRgbThreads) EncodeGrayIntKernel(const Rgb16Params p)
{
    constexpr int kWordsPerRow = CHANNELS * 2 * static_cast<int>(sizeof(HostT)); // 8 pixels x CHANNELS samples / 4 bytes
    constexpr int kVectorWords = (kWordsPerRow % 4 == 0) ? 4 : 2;
    constexpr int kPlaneBytes = static_cast<int>(sizeof(PlaneT));
    __shared__ float hostLut[(sizeof(HostT) == 1 && sizeof(PlaneT) == 2) ? 256 : 1];
    if (sizeof(HostT) == 1 && sizeof(PlaneT) == 2)
    {
        for (uint32_t v = threadIdx.x; v < 256; v += blockDim.x)
        {
            hostLut[v] = __uint_as_float(0x4b000000u | DepthLutEntry(v, 255.0f, p.maxCode));
        }
        __syncthreads();
    }
    const auto loadGroup = [&](uint32_t (&words)[kWordsPerRow], long long row, long long column)
    {
        const uint8_t* source = p.rows + row * p.rowStride + column * (kWordsPerRow * 4);
#pragma unroll
        for (int q = 0; q < kWordsPerRow / kVectorWords; ++q)
        {
            if (kVectorWords == 4)
            {
                const uint4 w = __ldcs(reinterpret_cast<const uint4*>(source) + q);
                words[4 * q + 0] = w.x;
                words[4 * q + 1] = w.y;
                words[4 * q + 2] = w.z;
                words[4 * q + 3] = w.w;
            }
            else
            {
                const uint2 w = __ldcs(reinterpret_cast<const uint2*>(source) + q);
                words[2 * q + 0] = w.x;
                words[2 * q + 1] = w.y;
            }
        }
    };
    const auto convertGroup = [&](const uint32_t (&words)[kWordsPerRow], long long row, long long column)
    {
        if (sizeof(HostT) == 1 && sizeof(PlaneT) == 1 && CHANNELS == 1)
        {
            // Gray8 into an 8-bit image: the sample is the code (WriteHeifImage.cpp:224-240) -- the 8 bytes as they are
            __stcs(reinterpret_cast<uint2*>(p.plane[0] + row * p.stride[0] + column * 8), make_uint2(words[0], words[1]));
            return;
        }
        auto sample = [&](int k) -> uint32_t
        {
            if (sizeof(HostT) == 2)
            {
                const uint32_t w = words[k >> 1];
                return (k & 1) ? (w >> 16) : (w & 0xffffu);
            }
            return (words[k >> 2] >> (8 * (k & 3))) & 0xffu;
        };
        uint32_t yCodes[8], aCodes[8];
#pragma unroll
        for (int i = 0; i < 8; ++i)
        {
            yCodes[i] = BiasedToCode(SampleToBiasedCode<HostT, PlaneT>(sample(i * CHANNELS), p, hostLut));
            if (CHANNELS == 2)
            {
                aCodes[i] = BiasedToCode(SampleToBiasedCode<HostT, PlaneT>(sample(i * CHANNELS + 1), p, hostLut));
            }
        }
        StoreEight<PlaneT>(p.plane[0] + row * p.stride[0] + column * (8 * kPlaneBytes), yCodes);
        if (CHANNELS == 2)
        {
            StoreEight<PlaneT>(p.plane[3] + row * p.stride[3] + column * (8 * kPlaneBytes), aCodes);
        }
    };
    // 8-bit hosts: a group is 8 or 16 bytes -- four groups' loads in flight before the first is converted (the launch is bound
    // by memory latency otherwise: 28 % of the issue slots used, every warp on long_scoreboard); 16-bit hosts one at a time
    constexpr int kInFlight = sizeof(HostT) == 1 ? 4 : 1;
    GroupWalk walk(static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x, static_cast<long long>(gridDim.x) * blockDim.x, p.groupsPerRow, p.rowCount);
    if (kInFlight == 1)
    {
        for (; walk.Inside(p.rowCount); walk.Advance(p.rowCount))
        {
            uint32_t words[kWordsPerRow];
            loadGroup(words, walk.row, walk.column);
            convertGroup(words, walk.row, walk.column);
        }
        return;
    }
    while (walk.Inside(p.rowCount))
    {
        uint32_t wordsAll[kInFlight][kWordsPerRow];
        int rowOf[kInFlight], columnOf[kInFlight];
#pragma unroll
        for (int u = 0; u < kInFlight; ++u)
        {
            rowOf[u] = -1;
            columnOf[u] = 0;
            if (walk.Inside(p.rowCount))
            {
                rowOf[u] = walk.row;
                columnOf[u] = walk.column;
                loadGroup(wordsAll[u], walk.row, walk.column);
            }
            walk.Advance(p.rowCount);
        }
#pragma unroll
        for (int u = 0; u < kInFlight; ++u)
        {
            if (rowOf[u] >= 0)
            {
                convertGroup(wordsAll[u], rowOf[u], columnOf[u]);
            }
        }
    }
}

template <typename HostT, typename PlaneT>
cudaError_t LaunchGrayInt(const Rgb16Params& rp, int channels, int smCount, cudaStream_t stream)
{
    const long long groups = static_cast<long long>(rp.groupsPerRow) * rp.rowCount;
    long long blocks = (groups + kRgbThreads - 1) / kRgbThreads;
    const long long cap = static_cast<long long>(smCount) * 16;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    const unsigned grid = static_cast<unsigned>(blocks);
    if (channels == 2) EncodeGrayIntKernel<HostT, PlaneT, 2><<<grid, kRgbThreads, 0, stream>>>(rp);
    else EncodeGrayIntKernel<HostT, PlaneT, 1><<<grid, kRgbThreads, 0, stream>>>(rp);
    return cudaGetLastError();
}

template <typename HostT, typename PlaneT, int CHANNELS, int PREMULTIPLY>
cudaError_t LaunchRgbInt(const Rgb16Params& rp, int xs, int ys, int smCount, cudaStream_t stream)
{
    const long long groups = static_cast<long long>(rp.groupsPerRow) * ((rp.rowCount + ys) >> ys);
    long long blocks = (groups + kRgbThreads - 1) / kRgbThreads;
    const long long cap = static_cast<long long>(smCount) * 16;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    const unsigned grid = static_cast<unsigned>(blocks);
    if (xs == 1 && ys == 1) EncodeRgbIntPlanarKernel<HostT, PlaneT, CHANNELS, 1, 1, PREMULTIPLY><<<grid, kRgbThreads, 0, stream>>>(rp);
    else if (xs == 1) EncodeRgbIntPlanarKernel<HostT, PlaneT, CHANNELS, 1, 0, PREMULTIPLY><<<grid, kRgbThreads, 0, stream>>>(rp);
    else EncodeRgbIntPlanarKernel<HostT, PlaneT, CHANNELS, 0, 0, PREMULTIPLY><<<grid, kRgbThreads, 0, stream>>>(rp);
    return cudaGetLastError();
}

template <typename HostT, typename PlaneT>
cudaError_t LaunchRgbIntChannels(const Rgb16Params& rp, int channels, bool premultiply, int xs, int ys, int smCount, cudaStream_t stream)
{
    if (channels == 4 && premultiply) return LaunchRgbInt<HostT, PlaneT, 4, 1>(rp, xs, ys, smCount, stream);
    return channels == 4 ? LaunchRgbInt<HostT, PlaneT, 4, 0>(rp, xs, ys, smCount, stream) : LaunchRgbInt<HostT, PlaneT, 3, 0>(rp, xs, ys, smCount, stream);
}

} // namespace

long long VerifyFastPremultiply(uint32_t maxCode, void* streamHandle)
{
    cudaStream_t stream = static_cast<cudaStream_t>(streamHandle);
    return RunCountingKernel(stream, [&](unsigned long long* counter) { VerifyFastPremultiplyKernel<<<148 * 8, 256, 0, stream>>>(maxCode, counter); });
}

cudaError_t BuildGray16Lut(uint16_t* deviceLut, int smpte428, uint32_t maxCode, void* streamHandle)
{
    BuildGray16LutKernel<<<64, 256, 0, static_cast<cudaStream_t>(streamHandle)>>>(deviceLut, smpte428, maxCode);
    return cudaGetLastError();
}

// Returns the number of kernels launched, 0 if this configuration is not covered, or a negative status.
int LaunchEncodeFastInteger(const EncodeParams& p, int hostDepth, void* streamHandle)
{
    cudaStream_t stream = static_cast<cudaStream_t>(streamHandle);
    if (hostDepth != 16 && hostDepth != 8)
    {
        return 0;
    }
    const int smCount = SmCount(p.smCount);

    if (hostDepth == 16 && p.imageDepth > 8 && p.channels == 1 && !p.planar)
    {
        if (p.gray16Lut == nullptr || p.width < 8 || !Aligned(p.rows, p.rowStride, 16) || !Aligned(p.plane[0], p.planeStride[0], 16))
        {
            return 0;
        }
        static std::atomic<uint64_t> configuredDevices{ 0 };
        if (const cudaError_t configured = AllowDynamicShared(EncodeGray16LutKernel, kLutEntries * 2, configuredDevices))
        {
            return ReportLaunchFailure(static_cast<int>(configured));
        }
        Gray16Params gp{};
        gp.rows = static_cast<const uint8_t*>(p.rows);
        gp.rowStride = p.rowStride;
        gp.planeY = static_cast<uint8_t*>(p.plane[0]);
        gp.strideY = p.planeStride[0];
        gp.chunksPerRow = p.width / 8;
        gp.rowCount = p.rowCount;
        gp.lut = p.gray16Lut;
        EncodeGray16LutKernel<<<smCount, kLutThreads, kLutEntries * 2, stream>>>(gp);
        if (const cudaError_t launchError = cudaGetLastError())
        {
            return ReportLaunchFailure(static_cast<int>(launchError));
        }
        const int n = LaunchEncodeRemainder(p, hostDepth, gp.chunksPerRow * 8, p.rowCount, streamHandle);
        return n < 0 ? n : 1 + n;
    }

    // Gray(+A) hosts in the reference layout (Y plane [0], alpha plane [3]); premultiplication and the Gray16 SMPTE 428
    // composition stay with the generic kernel (the latter has its own table kernel above for one channel).
    if (!p.planar && (p.channels == 1 || p.channels == 2) && !p.premultiply && !p.gray16Smpte428 && p.imageDepth <= 12)
    {
        const int hostBytes = hostDepth / 8;
        const int planeBytes = p.imageDepth > 8 ? 2 : 1;
        const int rowAlign = (8 * p.channels * hostBytes) % 16 == 0 ? 16 : 8;
        if (p.width < 8 || p.rowCount < 1 || !Aligned(p.rows, p.rowStride, rowAlign) || !Aligned(p.plane[0], p.planeStride[0], 8 * planeBytes) ||
            (p.channels == 2 && !Aligned(p.plane[3], p.planeStride[3], 8 * planeBytes)))
        {
            return 0;
        }
        const int width8 = p.width & ~7;
        Rgb16Params rp{};
        rp.rows = static_cast<const uint8_t*>(p.rows);
        rp.rowStride = p.rowStride;
        for (int k = 0; k < 4; ++k)
        {
            rp.plane[k] = static_cast<uint8_t*>(p.plane[k]);
            rp.stride[k] = p.planeStride[k];
        }
        rp.groupsPerRow = width8 / 8;
        rp.rowCount = p.rowCount;
        rp.maxCodeFloat = p.maxCodeFloat;
        rp.biasedMax = 8388608.0f + p.maxCodeFloat;
        rp.maxCode = p.maxCode;
        rp.maxReciprocal = 1.0f / p.maxCodeFloat;
        cudaError_t e;
        if (hostBytes == 2)
        {
            e = planeBytes == 2 ? LaunchGrayInt<uint16_t, uint16_t>(rp, p.channels, smCount, stream) : LaunchGrayInt<uint16_t, uint8_t>(rp, p.channels, smCount, stream);
        }
        else
        {
            e = planeBytes == 2 ? LaunchGrayInt<uint8_t, uint16_t>(rp, p.channels, smCount, stream) : LaunchGrayInt<uint8_t, uint8_t>(rp, p.channels, smCount, stream);
        }
        if (e != cudaSuccess)
        {
            return ReportLaunchFailure(static_cast<int>(e));
        }
        const int n = LaunchEncodeRemainder(p, hostDepth, width8, p.rowCount, streamHandle);
        return n < 0 ? n : 1 + n;
    }

    // The biased-truncation trick needs non-negative intermediates: true for every matrix with kr, kg, kb >= 0
    // (all of H.273's); anything else takes the generic kernel.
    if (p.planar && (p.channels == 3 || p.channels == 4) && (!p.premultiply || (p.channels == 4 && p.verifiedPremultiply)) && p.imageDepth <= 12 &&
        (p.matrix.identity || (p.matrix.kr >= 0.0f && p.matrix.kg >= 0.0f && p.matrix.kb >= 0.0f && p.matrix.kr < 1.0f && p.matrix.kb < 1.0f)) &&
        ForwardMatrixStaysInRange(p.matrix, p.chromaOffset, static_cast<int>(p.maxCode)))
    {
        const int hostBytes = hostDepth / 8;
        const int planeBytes = p.imageDepth > 8 ? 2 : 1;
        const int rowAlign = (8 * p.channels * hostBytes) % 16 == 0 ? 16 : 8; // a thread's 8-pixel chunk: 128-bit or 64-bit loads
        const int lumaAlign = 8 * planeBytes;
        const int chromaAlign = (p.xs ? 4 : 8) * planeBytes;
        if (p.width < 8 || !Aligned(p.rows, p.rowStride, rowAlign) || !Aligned(p.plane[0], p.planeStride[0], lumaAlign) ||
            !Aligned(p.plane[1], p.planeStride[1], chromaAlign) || !Aligned(p.plane[2], p.planeStride[2], chromaAlign) ||
            (p.channels == 4 && !Aligned(p.plane[3], p.planeStride[3], lumaAlign)))
        {
            return 0;
        }
        const int width8 = p.width & ~7;
        const int evenRows = p.ys ? (p.rowCount & ~1) : p.rowCount;
        if (evenRows < 1)
        {
            return 0;
        }
        Rgb16Params rp{};
        rp.rows = static_cast<const uint8_t*>(p.rows);
        rp.rowStride = p.rowStride;
        for (int k = 0; k < 4; ++k)
        {
            rp.plane[k] = static_cast<uint8_t*>(p.plane[k]);
            rp.stride[k] = p.planeStride[k];
        }
        rp.groupsPerRow = width8 / 8;
        rp.rowCount = evenRows;
        rp.maxCodeFloat = p.maxCodeFloat;
        rp.biasedMax = 8388608.0f + p.maxCodeFloat;
        rp.matrix = p.matrix;
        rp.chromaOffset = p.chromaOffset;
        rp.topLeft = p.topLeft;
        rp.maxCode = p.maxCode;
        rp.maxReciprocal = 1.0f / p.maxCodeFloat;
        cudaError_t e;
        if (hostBytes == 2)
        {
            e = planeBytes == 2 ? LaunchRgbIntChannels<uint16_t, uint16_t>(rp, p.channels, p.premultiply != 0, p.xs, p.ys, smCount, stream)
                                : LaunchRgbIntChannels<uint16_t, uint8_t>(rp, p.channels, p.premultiply != 0, p.xs, p.ys, smCount, stream);
        }
        else
        {
            e = planeBytes == 2 ? LaunchRgbIntChannels<uint8_t, uint16_t>(rp, p.channels, p.premultiply != 0, p.xs, p.ys, smCount, stream)
                                : LaunchRgbIntChannels<uint8_t, uint8_t>(rp, p.channels, p.premultiply != 0, p.xs, p.ys, smCount, stream);
        }
        if (e != cudaSuccess)
        {
            return ReportLaunchFailure(static_cast<int>(e));
        }
        const int n = LaunchEncodeRemainder(p, hostDepth, width8, evenRows, streamHandle);
        return n < 0 ? n : 1 + n;
    }
    return 0;
}

} // namespace avifgpu
