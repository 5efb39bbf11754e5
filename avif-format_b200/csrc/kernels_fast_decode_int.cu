// kernels_fast_decode_int.cu -- tuned decode kernels for the integer hosts: planar YCbCr (+ alpha) -> interleaved
// RGB(A) 8-bit (YuvDecode.cpp:281-399 driven by ReadHeifImage.cpp:83-184) and 16-bit (YuvDecode.cpp:401-519 driven by
// ReadHeifImage.cpp:186-288).  No transfer curve on these paths: table look-up, matrix, clamp, round -- HBM-bound work
// (4.5 B/px for 8-bit 4:2:0) if the instruction count per pixel stays near 25.
//
//   * a warp converts units of (2 rows for 4:2:0, else 1) x 256 pixels; a lane owns 8 adjacent pixels per row: one
//     64/128-bit load of Y per row, one 32/64-bit (sub-sampled) load of Cb and of Cr, 3-4 vector stores per row;
//   * the unorm -> float tables (YuvLookupTables.cpp:115-192) sit in shared memory; for 16-bit hosts the alpha output
//     (u16)(0.5f + a * 32768f) is tabulated whole;
//   * the chroma-dependent terms of YuvDecode.cpp:306-312 are evaluated once per chroma site and reused for every luma
//     sample the site covers (both rows of a 4:2:0 site); same float expressions, same association;
//   * premultiplied alpha, odd starting rows of a 4:2:0 block, depths above 12 bits and unaligned buffers stay with the
//     generic kernel.
#include "group_walk.cuh"
#include "kernel_params.h"
#include "packed_f32x2.cuh"
#include "pixel_math.cuh"
#include "../../include/avifgpu.h"

#include <cuda_runtime.h>

namespace avifgpu
{

using namespace avifpix;

namespace
{

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kBlocksPerSm = 3;
constexpr int kUnitPixels = 256; // per row: 32 lanes x 8 pixels

struct IntDecodeParams
{
    const uint8_t* plane[4];
    int64_t planeStride[4];
    uint8_t* rows;
    int64_t rowStride;
    int32_t width;    // multiple of 8
    int32_t rowCount; // even when the chroma is vertically sub-sampled
    int32_t bitDepth;
    uint32_t maxCode;
    RangeParams range;
    InverseMatrix matrix;
    int32_t verifiedGreenDivision;
};

// Eight (four) consecutive samples of a plane as they sit in memory, and their expansion into 32-bit codes.
template <typename SampleT>
struct Raw8
{
    uint32_t w[sizeof(SampleT) == 1 ? 2 : 4];
};

template <typename SampleT>
__device__ __forceinline__ Raw8<SampleT> LoadEight(const uint8_t* address)
{
    Raw8<SampleT> raw;
    if (sizeof(SampleT) == 1)
    {
        const uint2 v = __ldg(reinterpret_cast<const uint2*>(address));
        raw.w[0] = v.x;
        raw.w[1] = v.y;
    }
    else
    {
        const uint4 v = __ldg(reinterpret_cast<const uint4*>(address));
        raw.w[0] = v.x;
        raw.w[1] = v.y;
        raw.w[sizeof(SampleT) == 1 ? 0 : 2] = v.z;
        raw.w[sizeof(SampleT) == 1 ? 1 : 3] = v.w;
    }
    return raw;
}

// The four samples of the sub-sampled chroma under eight luma samples land in the first half of a Raw8.
template <typename SampleT>
__device__ __forceinline__ Raw8<SampleT> LoadFour(const uint8_t* address)
{
    Raw8<SampleT> raw = {};
    if (sizeof(SampleT) == 1)
    {
        raw.w[0] = __ldg(reinterpret_cast<const uint32_t*>(address));
    }
    else
    {
        const uint2 v = __ldg(reinterpret_cast<const uint2*>(address));
        raw.w[0] = v.x;
        raw.w[1] = v.y;
    }
    return raw;
}

template <typename SampleT>
__device__ __forceinline__ uint32_t Sample(const Raw8<SampleT>& raw, int i)
{
    if (sizeof(SampleT) == 1)
    {
        return (raw.w[i >> 2] >> (8 * (i & 3))) & 0xffu;
    }
    return (i & 1) ? (raw.w[i >> 1] >> 16) : (raw.w[i >> 1] & 0xffffu);
}

constexpr float kTwo23 = 8388608.0f;

// 2^23 + (uint)(0.5f + (c * scale)) as a float, for c in [0, 1]: YuvDecode.cpp:314-316 / 437-439 in two instructions and
// without the conversion pipe.  The reference forms the sum with two roundings (multiply, then add); for every float c in
// [0, 1] and scale = 255 or 32768 the single-rounding fmaf(c, scale, 0.5f) truncates to the same integer -- proven by
// enumeration, tools/check_fused_quantiser.py -- so the sum is one FMA; adding 2^23 with round-toward-zero then leaves
// its integer part in the low mantissa bits, which is the truncation of the cast.
__device__ __forceinline__ uint32_t QuantiseBiased(float c, float scale) { return __float_as_uint(__fadd_rz(__fmaf_rn(c, scale, 0.5f), kTwo23)); }

template <typename SampleT, int XS, int YS, int ALPHA>
__global__ void __launch_bounds__(kThreads, kBlocksPerSm) DecodeYccToRgbIntKernel(const IntDecodeParams p)
{
    constexpr bool kHost8 = sizeof(SampleT) == 1;
    constexpr int kRows = YS ? 2 : 1;
    constexpr int kSites = XS ? 4 : 8;          // chroma sites under a lane's 8 luma samples
    constexpr int kChannels = ALPHA ? 4 : 3;
    extern __shared__ __align__(16) uint8_t sharedBytes[];
    float* tableY = reinterpret_cast<float*>(sharedBytes);
    float* tableUV = tableY + (1u << p.bitDepth);
    uint16_t* tableAlpha = reinterpret_cast<uint16_t*>(tableUV + (1u << p.bitDepth)); // 16-bit hosts with alpha only

    for (uint32_t i = threadIdx.x; i <= p.maxCode; i += blockDim.x)
    {
        tableY[i] = UnormToFloatY(i, p.range);   // YuvLookupTables.cpp:157-171
        tableUV[i] = UnormToFloatUV(i, p.range); // YuvLookupTables.cpp:173-184
        if (ALPHA && !kHost8)
        {
            // YuvLookupTables.cpp:186-190 then YuvDecode.cpp:515
            tableAlpha[i] = static_cast<uint16_t>(0.5f + (UnormToFloatPlain(i, p.range.maxChannelFloat) * 32768.0f));
        }
    }
    __syncthreads();

    // YuvDecode.cpp:306-312, the pixel-independent factors (same float expressions, evaluated once)
    const float kr = p.matrix.kr, kg = p.matrix.kg, kb = p.matrix.kb;
    const float rGain = (2 * (1 - kr));
    const float bGain = (2 * (1 - kb));
    const float gCr = kr * (1 - kr);
    const float gCb = kb * (1 - kb);
    const float kgReciprocal = 1.0f / kg;
    const float outScale = kHost8 ? 255.0f : 32768.0f;

    const int lane = threadIdx.x & 31;
    const int warpInBlock = threadIdx.x >> 5;
    const int unitsX = (p.width + kUnitPixels - 1) / kUnitPixels;
    const int unitRows = (p.rowCount + kRows - 1) / kRows;
    const long long unitCount = static_cast<long long>(unitsX) * unitRows;
    const int warpCount = static_cast<int>(gridDim.x) * kWarps;
    // unit coordinates advance incrementally (no division per unit)
    const long long firstUnit = static_cast<long long>(blockIdx.x) * kWarps + warpInBlock;
    const int stepRows = warpCount / unitsX;
    const int stepX = warpCount - stepRows * unitsX;
    int unitRow = static_cast<int>(firstUnit / unitsX);
    int unitX = static_cast<int>(firstUnit - static_cast<long long>(unitRow) * unitsX);

    // Software pipeline: the loads of unit i+1 are issued once unit i's samples have been expanded, so they are in flight
    // during its arithmetic and stores.
    Raw8<SampleT> rawY[kRows], rawA[kRows], rawCb, rawCr;
    auto loadUnit = [&](int row, int column, bool valid)
    {
        const int x = column * kUnitPixels + lane * 8;
        const int y = row * kRows;
        if (!valid || x >= p.width)
        {
            return;
        }
        const int64_t chromaRow = YS ? row : y;
        const int64_t chromaColumn = static_cast<int64_t>(XS ? (x >> 1) : x) * sizeof(SampleT);
        if (XS)
        {
            rawCb = LoadFour<SampleT>(p.plane[1] + chromaRow * p.planeStride[1] + chromaColumn);
            rawCr = LoadFour<SampleT>(p.plane[2] + chromaRow * p.planeStride[2] + chromaColumn);
        }
        else
        {
            rawCb = LoadEight<SampleT>(p.plane[1] + chromaRow * p.planeStride[1] + chromaColumn);
            rawCr = LoadEight<SampleT>(p.plane[2] + chromaRow * p.planeStride[2] + chromaColumn);
        }
#pragma unroll
        for (int r = 0; r < kRows; ++r)
        {
            if (y + r < p.rowCount)
            {
                rawY[r] = LoadEight<SampleT>(p.plane[0] + static_cast<int64_t>(y + r) * p.planeStride[0] + static_cast<int64_t>(x) * sizeof(SampleT));
                if (ALPHA)
                {
                    rawA[r] = LoadEight<SampleT>(p.plane[3] + static_cast<int64_t>(y + r) * p.planeStride[3] + static_cast<int64_t>(x) * sizeof(SampleT));
                }
            }
        }
    };
#pragma unroll
    for (int r = 0; r < kRows; ++r)
    {
        rawY[r] = {};
        rawA[r] = {};
    }
    rawCb = {};
    rawCr = {};
    loadUnit(unitRow, unitX, firstUnit < unitCount);

#pragma unroll 1
    for (long long unit = firstUnit; unit < unitCount; unit += warpCount)
    {
        const int x0 = unitX * kUnitPixels + lane * 8;
        const int y0 = unitRow * kRows;
        const bool laneActive = x0 < p.width;
        const bool secondRow = kRows == 2 && (y0 + 1) < p.rowCount;
        int nextRow = unitRow + stepRows;
        int nextX = unitX + stepX;
        if (nextX >= unitsX)
        {
            nextX -= unitsX;
            ++nextRow;
        }

        // ---- samples -> floats through the shared-memory tables; chroma terms once per site -----------------------------
        float Yf[kRows][8];
        uint32_t alphaOut[kRows][8];
#pragma unroll
        for (int r = 0; r < kRows; ++r)
        {
#pragma unroll
            for (int i = 0; i < 8; ++i)
            {
                const uint32_t code = Sample<SampleT>(rawY[r], i);
                Yf[r][i] = tableY[kHost8 ? code : min(code, p.maxCode)];
                if (ALPHA)
                {
                    const uint32_t a = Sample<SampleT>(rawA[r], i);
                    alphaOut[r][i] = kHost8 ? a : tableAlpha[min(a, p.maxCode)];
                }
            }
        }
        float rOffset[kSites], bOffset[kSites], gOffset[kSites];
#pragma unroll
        for (int s = 0; s < kSites; ++s)
        {
            const uint32_t cbCode = Sample<SampleT>(rawCb, s);
            const uint32_t crCode = Sample<SampleT>(rawCr, s);
            const float Cb = tableUV[kHost8 ? cbCode : min(cbCode, p.maxCode)];
            const float Cr = tableUV[kHost8 ? crCode : min(crCode, p.maxCode)];
            rOffset[s] = rGain * Cr;
            bOffset[s] = bGain * Cb;
            const float greenNumerator = 2 * ((gCr * Cr) + (gCb * Cb));
            gOffset[s] = p.verifiedGreenDivision ? DivideByConstant(greenNumerator, kg, kgReciprocal) : greenNumerator / kg;
        }

        loadUnit(nextRow, nextX, unit + warpCount < unitCount);
        unitRow = nextRow;
        unitX = nextX;
        if (!laneActive)
        {
            continue;
        }

        // ---- pixels ---------------------------------------------------------------------------------------------------
#pragma unroll
        for (int r = 0; r < kRows; ++r)
        {
            if (r == 1 && !secondRow)
            {
                break;
            }
            uint32_t out[8][kChannels]; // colour channels: 2^23-biased float bit patterns (the code is in the low bits)
            // Two pixels per step: the clamped sums are scalar (the saturation modifier has no packed form), the quantiser --
            // QuantiseBiased's fused multiply-add and biased truncation -- runs on the pair (packed_f32x2.cuh).
            const avifx2::F32x2 scale2 = avifx2::Splat(outScale), half2 = avifx2::Splat(0.5f), bias2 = avifx2::Splat(kTwo23);
            const auto quantisePair = [&](float c0, float c1, uint32_t& q0, uint32_t& q1)
            {
                float b0, b1;
                avifx2::Unpack(avifx2::AddRz2(avifx2::Fma2(avifx2::Pack(c0, c1), scale2, half2), bias2), b0, b1);
                q0 = __float_as_uint(b0);
                q1 = __float_as_uint(b1);
            };
            if (!kHost8)
            {
                // 16-bit hosts: one pixel at a time (the pair form measured 4 % slower there: registers)
#pragma unroll
                for (int i = 0; i < 8; ++i)
                {
                    const int s = XS ? (i >> 1) : i;
                    out[i][0] = QuantiseBiased(__saturatef(Yf[r][i] + rOffset[s]), outScale);
                    out[i][1] = QuantiseBiased(__saturatef(Yf[r][i] - gOffset[s]), outScale);
                    out[i][2] = QuantiseBiased(__saturatef(Yf[r][i] + bOffset[s]), outScale);
                    if (ALPHA)
                    {
                        out[i][3] = alphaOut[r][i];
                    }
                }
            }
#pragma unroll
            for (int i = 0; kHost8 && i < 8; i += 2)
            {
                const int s0 = XS ? (i >> 1) : i, s1 = XS ? (i >> 1) : i + 1;
                // std::clamp(v, 0, 1) as the add's saturation modifier: the table entries are finite and Y >= +0, so the
                // sums are never NaN or -0.0 and the two agree for every input.
                quantisePair(__saturatef(Yf[r][i] + rOffset[s0]), __saturatef(Yf[r][i + 1] + rOffset[s1]), out[i][0], out[i + 1][0]);
                quantisePair(__saturatef(Yf[r][i] - gOffset[s0]), __saturatef(Yf[r][i + 1] - gOffset[s1]), out[i][1], out[i + 1][1]);
                quantisePair(__saturatef(Yf[r][i] + bOffset[s0]), __saturatef(Yf[r][i + 1] + bOffset[s1]), out[i][2], out[i + 1][2]);
                if (ALPHA)
                {
                    out[i][3] = alphaOut[r][i];
                    out[i + 1][3] = alphaOut[r][i + 1];
                }
            }
            uint8_t* target = p.rows + static_cast<int64_t>(y0 + r) * p.rowStride + static_cast<int64_t>(x0) * (kChannels * sizeof(SampleT));
            if (kHost8)
            {
                // 8 pixels x kChannels bytes: byte 0 of every value, four to a word
                uint32_t words[2 * kChannels];
#pragma unroll
                for (int w = 0; w < 2 * kChannels; ++w)
                {
                    uint32_t v[4];
#pragma unroll
                    for (int b = 0; b < 4; ++b)
                    {
                        const int byteIndex = 4 * w + b;
                        v[b] = out[byteIndex / kChannels][byteIndex % kChannels];
                    }
                    words[w] = __byte_perm(__byte_perm(v[0], v[1], 0x0040), __byte_perm(v[2], v[3], 0x0040), 0x5410);
                }
                if (ALPHA)
                {
                    __stcs(reinterpret_cast<uint4*>(target), make_uint4(words[0], words[1], words[2], words[3]));
                    __stcs(reinterpret_cast<uint4*>(target) + 1, make_uint4(words[4], words[5], words[6], words[7]));
                }
                else
                {
#pragma unroll
                    for (int q = 0; q < 3; ++q)
                    {
                        __stcs(reinterpret_cast<uint2*>(target) + q, make_uint2(words[2 * q], words[2 * q + 1]));
                    }
                }
            }
            else
            {
                // 8 pixels x kChannels 16-bit samples: the low half of every value, two to a word
                uint32_t words[4 * kChannels];
#pragma unroll
                for (int w = 0; w < 4 * kChannels; ++w)
                {
                    const int first = 2 * w;
                    words[w] = __byte_perm(out[first / kChannels][first % kChannels], out[(first + 1) / kChannels][(first + 1) % kChannels], 0x5410);
                }
#pragma unroll
                for (int q = 0; q < kChannels; ++q)
                {
                    __stcs(reinterpret_cast<uint4*>(target) + q, make_uint4(words[4 * q], words[4 * q + 1], words[4 * q + 2], words[4 * q + 3]));
                }
            }
        }
    }
}

template <typename SampleT, int XS, int YS, int ALPHA>
cudaError_t LaunchOne(const IntDecodeParams& fp, int smCount, cudaStream_t stream)
{
    const size_t entries = static_cast<size_t>(1) << fp.bitDepth;
    const size_t shared = 2 * sizeof(float) * entries + ((ALPHA && sizeof(SampleT) == 2) ? sizeof(uint16_t) * entries : 0);
    static std::atomic<uint64_t> configuredDevices{ 0 }; // per instantiation
    {
        const cudaError_t e = AllowDynamicShared(DecodeYccToRgbIntKernel<SampleT, XS, YS, ALPHA>, 64 * 1024, configuredDevices);
        if (e != cudaSuccess)
        {
            return e;
        }
    }
    constexpr int rowsPerUnit = YS ? 2 : 1;
    const long long units = static_cast<long long>((fp.width + kUnitPixels - 1) / kUnitPixels) * ((fp.rowCount + rowsPerUnit - 1) / rowsPerUnit);
    long long blocks = (units + kWarps - 1) / kWarps;
    const long long resident = static_cast<long long>(smCount) * kBlocksPerSm;
    if (blocks > resident)
    {
        blocks = resident;
    }
    DecodeYccToRgbIntKernel<SampleT, XS, YS, ALPHA><<<static_cast<unsigned>(blocks), kThreads, shared, stream>>>(fp);
    return cudaGetLastError();
}

template <typename SampleT, int ALPHA>
cudaError_t DispatchChroma(const IntDecodeParams& fp, int xs, int ys, int smCount, cudaStream_t stream)
{
    if (xs == 1 && ys == 1) return LaunchOne<SampleT, 1, 1, ALPHA>(fp, smCount, stream);
    if (xs == 1) return LaunchOne<SampleT, 1, 0, ALPHA>(fp, smCount, stream);
    return LaunchOne<SampleT, 0, 0, ALPHA>(fp, smCount, stream);
}

// ---- monochrome and planar-RGB images: pure streaming ------------------------------------------------------------------
//
// Monochrome (ReadHeifImage.cpp:418-559 driving YuvDecode.cpp:55-203): out = round(table[Y]) -- no matrix, so the whole
// per-sample result is tabulated in shared memory; alpha is copied (8-bit) or tabulated (16-bit).
// Planar RGB (ReadHeifImage.cpp:561-861): the samples are interleaved as they are; 16-bit hosts mask them with the
// image's maximum (:789-792).  A thread moves 8 pixels: one vector load per plane, CH * 8 samples stored as 64/128-bit words.
struct StreamDecodeParams
{
    const uint8_t* plane[4];
    int64_t planeStride[4];
    uint8_t* rows;
    int64_t rowStride;
    int32_t groupsPerRow; // 8 pixels each
    int32_t rowCount;
    int32_t bitDepth;
    uint32_t maxCode;
    RangeParams range;
};

constexpr int kStreamThreads = 256;

template <typename SampleT, int CHANNELS, bool MONO>
__global__ void __launch_bounds__(kStreamThreads) StreamDecodeKernel(const StreamDecodeParams p)
{
    constexpr bool kHost8 = sizeof(SampleT) == 1;
    extern __shared__ __align__(16) uint8_t sharedBytes[];
    uint16_t* lutY = reinterpret_cast<uint16_t*>(sharedBytes);
    uint16_t* lutA = lutY + (1u << p.bitDepth);
    if (MONO)
    {
        for (uint32_t i = threadIdx.x; i <= p.maxCode; i += blockDim.x)
        {
            const float y = UnormToFloatY(i, p.range); // YuvLookupTables.cpp:157-171
            lutY[i] = static_cast<uint16_t>(0.5f + (y * (kHost8 ? 255.0f : 32768.0f))); // YuvDecode.cpp:76, 150
            lutA[i] = static_cast<uint16_t>(0.5f + (UnormToFloatPlain(i, p.range.maxChannelFloat) * 32768.0f)); // YuvDecode.cpp:197
        }
        __syncthreads();
    }
    // An 8-bit full-range monochrome image read by an 8-bit host: the table maps every code to itself (checked, not
    // assumed) and the kernel is a strided copy -- eight shared-memory look-ups per 8 bytes otherwise bound it.
    bool identityLuma = false;
    if (MONO && kHost8)
    {
        bool mine = true;
        for (uint32_t i = threadIdx.x; i <= p.maxCode; i += blockDim.x)
        {
            mine = mine && lutY[i] == i;
        }
        identityLuma = __syncthreads_and(mine ? 1 : 0) != 0;
    }
    // source planes: mono -> Y (, A at index 3); RGB -> R, G, B (, A)
    constexpr int kColours = MONO ? 1 : 3;
    constexpr bool kAlpha = CHANNELS > kColours;
    // A group is 8 samples per plane -- 8 bytes for an 8-bit image: there a thread keeps several groups' loads in flight
    // before it converts the first (ncu: 2048 threads x 8 bytes per SM in flight is too little; planar RGB8 +4 %).  With
    // 16-byte groups one at a time is better (two in flight cost registers and occupancy: planar RGB 10-bit -12 %).
    constexpr int kInFlight = kHost8 ? 4 : 1;
    // one group: 8 samples per plane -> 8 host pixels at `target`
    const auto convertGroup = [&](const Raw8<SampleT>(&raw)[CHANNELS], uint8_t* target)
    {
        if (MONO && kHost8 && CHANNELS == 1)
        {
            if (identityLuma)
            {
                // the 8 bytes as they are: unpacking and repacking them made this path instruction-bound (76 % of the issue slots)
                __stcs(reinterpret_cast<uint2*>(target), make_uint2(raw[0].w[0], raw[0].w[1]));
                return;
            }
        }
        uint32_t samples[8 * CHANNELS];
#pragma unroll
        for (int i = 0; i < 8; ++i)
        {
#pragma unroll
            for (int c = 0; c < CHANNELS; ++c)
            {
                uint32_t v = Sample<SampleT>(raw[c], i);
                if (MONO)
                {
                    const bool isAlpha = kAlpha && c == CHANNELS - 1;
                    if (!isAlpha)
                    {
                        if (!(kHost8 && identityLuma))
                        {
                            v = lutY[kHost8 ? v : min(v, p.maxCode)];
                        }
                    }
                    else if (!kHost8)
                    {
                        v = lutA[min(v, p.maxCode)];
                    }
                }
                else if (!kHost8)
                {
                    v &= p.maxCode;
                }
                samples[i * CHANNELS + c] = v;
            }
        }
        constexpr int kWords = 8 * CHANNELS * static_cast<int>(sizeof(SampleT)) / 4;
        uint32_t words[kWords];
#pragma unroll
        for (int w = 0; w < kWords; ++w)
        {
            if (kHost8)
            {
                words[w] = samples[4 * w] | (samples[4 * w + 1] << 8) | (samples[4 * w + 2] << 16) | (samples[4 * w + 3] << 24);
            }
            else
            {
                words[w] = samples[2 * w] | (samples[2 * w + 1] << 16);
            }
        }
        if (kWords % 4 == 0)
        {
#pragma unroll
            for (int q = 0; q < kWords / 4; ++q)
            {
                __stcs(reinterpret_cast<uint4*>(target) + q, make_uint4(words[4 * q], words[4 * q + 1], words[4 * q + 2], words[4 * q + 3]));
            }
        }
        else
        {
#pragma unroll
            for (int q = 0; q < kWords / 2; ++q)
            {
                __stcs(reinterpret_cast<uint2*>(target) + q, make_uint2(words[2 * q], words[2 * q + 1]));
            }
        }
    };
    const auto loadGroup = [&](Raw8<SampleT>(&raw)[CHANNELS], long long row, long long column)
    {
#pragma unroll
        for (int c = 0; c < CHANNELS; ++c)
        {
            const int planeIndex = (kAlpha && c == CHANNELS - 1) ? 3 : c;
            raw[c] = LoadEight<SampleT>(p.plane[planeIndex] + row * p.planeStride[planeIndex] + column * static_cast<long long>(sizeof(SampleT)));
        }
    };
    GroupWalk walk(static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x, static_cast<long long>(gridDim.x) * blockDim.x, p.groupsPerRow, p.rowCount);
    if (kInFlight == 1)
    {
        for (; walk.Inside(p.rowCount); walk.Advance(p.rowCount))
        {
            const long long row = walk.row;
            const long long column = static_cast<long long>(walk.column) * 8;
            Raw8<SampleT> raw[CHANNELS];
            loadGroup(raw, row, column);
            convertGroup(raw, p.rows + row * p.rowStride + column * static_cast<long long>(CHANNELS * sizeof(SampleT)));
        }
        return;
    }
    while (walk.Inside(p.rowCount))
    {
        Raw8<SampleT> rawAll[kInFlight][CHANNELS];
        long long targetOffset[kInFlight];
#pragma unroll
        for (int u = 0; u < kInFlight; ++u)
        {
            targetOffset[u] = -1;
            if (walk.Inside(p.rowCount))
            {
                const long long row = walk.row;
                const long long column = static_cast<long long>(walk.column) * 8;
                loadGroup(rawAll[u], row, column);
                targetOffset[u] = row * p.rowStride + column * static_cast<long long>(CHANNELS * sizeof(SampleT));
            }
            walk.Advance(p.rowCount);
        }
#pragma unroll
        for (int u = 0; u < kInFlight; ++u)
        {
            if (targetOffset[u] >= 0)
            {
                convertGroup(rawAll[u], p.rows + targetOffset[u]);
            }
        }
    }
}

template <typename SampleT, int CHANNELS, bool MONO>
cudaError_t LaunchStream(const StreamDecodeParams& sp, int smCount, cudaStream_t stream)
{
    const long long groups = static_cast<long long>(sp.groupsPerRow) * sp.rowCount;
    long long blocks = (groups + kStreamThreads - 1) / kStreamThreads;
    const long long cap = static_cast<long long>(smCount) * 16;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    const size_t shared = MONO ? 2 * sizeof(uint16_t) * (static_cast<size_t>(1) << sp.bitDepth) : 0;
    StreamDecodeKernel<SampleT, CHANNELS, MONO><<<static_cast<unsigned>(blocks), kStreamThreads, shared, stream>>>(sp);
    return cudaGetLastError();
}

} // namespace

// Monochrome and planar-RGB images for the integer hosts (no premultiplied alpha, depth <= 12: checked by the caller).
static int LaunchDecodeStream(const DecodeParams& p, void* streamHandle)
{
    cudaStream_t stream = static_cast<cudaStream_t>(streamHandle);
    const int sampleBytes = p.hostDepth == 8 ? 1 : 2;
    if ((sampleBytes == 1) != (p.bitDepth <= 8))
    {
        return 0;
    }
    const bool mono = p.colorspace == AVIFGPU_COLORSPACE_MONOCHROME;
    const int colours = mono ? 1 : 3;
    const int channels = colours + (p.hasAlpha ? 1 : 0);
    const int planeAlign = 8 * sampleBytes;
    const int rowAlign = (8 * channels * sampleBytes) % 16 == 0 ? 16 : 8;
    for (int c = 0; c < colours; ++c)
    {
        if (!Aligned(p.plane[c], p.planeStride[c], planeAlign))
        {
            return 0;
        }
    }
    if ((p.hasAlpha && !Aligned(p.plane[3], p.planeStride[3], planeAlign)) || !Aligned(p.rows, p.rowStride, rowAlign))
    {
        return 0;
    }
    const int width8 = p.width & ~7;
    if (width8 < 8 || p.rowCount < 1)
    {
        return 0;
    }
    StreamDecodeParams sp{};
    for (int k = 0; k < 4; ++k)
    {
        sp.plane[k] = static_cast<const uint8_t*>(p.plane[k]);
        sp.planeStride[k] = p.planeStride[k];
    }
    sp.rows = static_cast<uint8_t*>(p.rows);
    sp.rowStride = p.rowStride;
    sp.groupsPerRow = width8 / 8;
    sp.rowCount = p.rowCount;
    sp.bitDepth = p.bitDepth;
    sp.maxCode = p.maxCode;
    sp.range = p.range;
    const int smCount = SmCount(p.smCount);
    cudaError_t e;
    if (sampleBytes == 1)
    {
        if (mono) e = p.hasAlpha ? LaunchStream<uint8_t, 2, true>(sp, smCount, stream) : LaunchStream<uint8_t, 1, true>(sp, smCount, stream);
        else e = p.hasAlpha ? LaunchStream<uint8_t, 4, false>(sp, smCount, stream) : LaunchStream<uint8_t, 3, false>(sp, smCount, stream);
    }
    else
    {
        if (mono) e = p.hasAlpha ? LaunchStream<uint16_t, 2, true>(sp, smCount, stream) : LaunchStream<uint16_t, 1, true>(sp, smCount, stream);
        else e = p.hasAlpha ? LaunchStream<uint16_t, 4, false>(sp, smCount, stream) : LaunchStream<uint16_t, 3, false>(sp, smCount, stream);
    }
    if (e != cudaSuccess)
    {
        return ReportLaunchFailure(static_cast<int>(e));
    }
    const int n = LaunchDecodeRemainder(p, width8, p.rowCount, streamHandle);
    return n < 0 ? n : 1 + n;
}

// Returns the number of kernels launched, 0 if this configuration is not covered, or a negative status.
int LaunchDecodeFastInteger(const DecodeParams& p, void* streamHandle)
{
    cudaStream_t stream = static_cast<cudaStream_t>(streamHandle);
    if ((p.hostDepth != 8 && p.hostDepth != 16) || p.bitDepth > 12 || (p.hasAlpha && p.premultiplied))
    {
        return 0;
    }
    if (p.colorspace != AVIFGPU_COLORSPACE_YCBCR)
    {
        return LaunchDecodeStream(p, streamHandle);
    }
    if (p.yPhase != 0)
    {
        return 0;
    }
    const int sampleBytes = p.hostDepth == 8 ? 1 : 2;
    if ((sampleBytes == 1) != (p.bitDepth <= 8))
    {
        return 0; // 8-bit hosts read 8-bit planes, 16-bit hosts read 16-bit planes (ReadHeifImage.cpp:83, 186)
    }
    const int channels = p.hasAlpha ? 4 : 3;
    const int lumaAlign = 8 * sampleBytes;
    const int chromaAlign = (p.xs ? 4 : 8) * sampleBytes;
    const int rowAlign = channels == 4 ? 16 : 8 * sampleBytes; // RGB8: 64-bit stores, everything else 128-bit
    if (!Aligned(p.plane[0], p.planeStride[0], lumaAlign) || !Aligned(p.plane[1], p.planeStride[1], chromaAlign) ||
        !Aligned(p.plane[2], p.planeStride[2], chromaAlign) || (p.hasAlpha && !Aligned(p.plane[3], p.planeStride[3], lumaAlign)) ||
        !Aligned(p.rows, p.rowStride, rowAlign))
    {
        return 0;
    }
    const int width8 = p.width & ~7;
    const int evenRows = p.ys ? (p.rowCount & ~1) : p.rowCount;
    if (width8 < 8 || evenRows < 1)
    {
        return 0;
    }
    IntDecodeParams fp{};
    for (int k = 0; k < 4; ++k)
    {
        fp.plane[k] = static_cast<const uint8_t*>(p.plane[k]);
        fp.planeStride[k] = p.planeStride[k];
    }
    fp.rows = static_cast<uint8_t*>(p.rows);
    fp.rowStride = p.rowStride;
    fp.width = width8;
    fp.rowCount = evenRows;
    fp.bitDepth = p.bitDepth;
    fp.maxCode = p.maxCode;
    fp.range = p.range;
    fp.matrix = p.matrix;
    fp.verifiedGreenDivision = p.verifiedGreenDivision;

    const int smCount = SmCount(p.smCount);
    cudaError_t e;
    if (sampleBytes == 1)
    {
        e = p.hasAlpha ? DispatchChroma<uint8_t, 1>(fp, p.xs, p.ys, smCount, stream) : DispatchChroma<uint8_t, 0>(fp, p.xs, p.ys, smCount, stream);
    }
    else
    {
        e = p.hasAlpha ? DispatchChroma<uint16_t, 1>(fp, p.xs, p.ys, smCount, stream) : DispatchChroma<uint16_t, 0>(fp, p.xs, p.ys, smCount, stream);
    }
    if (e != cudaSuccess)
    {
        return ReportLaunchFailure(static_cast<int>(e));
    }
    // The right strip (width % 8 columns) and, for vertically sub-sampled chroma, an odd last row: the generic kernel.
    const int n = LaunchDecodeRemainder(p, width8, evenRows, streamHandle);
    return n < 0 ? n : 1 + n;
}

} // namespace avifgpu
