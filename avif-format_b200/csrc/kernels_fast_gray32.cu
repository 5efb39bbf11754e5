// kernels_fast_gray32.cu -- Gray(+A) float hosts -> Y (+ Alpha) planes: CreateHeifImageGrayThirtyTwoBit
// (WriteHeifImage.cpp:502-627; gray knows the PQ and clip transfers only, :578-588).
//
// One sample per pixel goes through the curve, so this is a streaming kernel: a thread converts 4 adjacent pixels
// (one or two 128-bit loads, 64-bit stores), the PQ code comes from the compact step table in shared memory
// (curve_tables.h; flagged samples are resolved from first_k and the band bitmap on the spot, +inf / NaN take the exact
// evaluation), the clip transfer is the quantiser alone.  4 + 2 (or 8 + 4) bytes per pixel: HBM-bound.
#include "group_walk.cuh"
#include "kernels_fast_common.cuh"
#include "table_staging.cuh"
#include "../../include/avifgpu.h"

namespace avifgpu
{

using namespace avifpix;
using avifmath::LibmTables;

namespace
{

constexpr int kGrayTableThreads = 1024; // PQ: one CTA per SM stages the table once and keeps 32 warps on it
constexpr int kGrayClipThreads = 256;   // clip: no table, many small CTAs
constexpr int kGroupsInFlight = 2;      // groups (4 pixels each) a thread loads before it converts the first

struct Gray32Params
{
    const uint8_t* rows;
    int64_t rowStride;
    uint8_t* planeY;
    int64_t strideY;
    uint8_t* planeA;
    int64_t strideA;
    int32_t groupsPerRow; // 4 pixels each
    int32_t rowCount;
    int32_t premultiply;
    float pqMultiplier;
    float maxCodeFloat;
    int32_t maxCode;
    CurveTableView table;
};

// CHANNELS 1 (Gray) or 2 (Gray + alpha); PQ = 1: LinearToPQ through the compact table, 0: clip.
template <int CHANNELS, int PQ>
__global__ void __launch_bounds__(PQ ? kGrayTableThreads : kGrayClipThreads) EncodeGrayF32Kernel(const Gray32Params p)
{
    extern __shared__ __align__(16) uint8_t sharedBytes[];
    uint64_t* libmStorage = reinterpret_cast<uint64_t*>(sharedBytes);
    uint64_t* tableBarrierStorage = reinterpret_cast<uint64_t*>(sharedBytes + 768);
    uint32_t* compactEntries = reinterpret_cast<uint32_t*>(sharedBytes + 768 + 16);
    const uint32_t* firstBits = compactEntries + ((p.table.flatCount + 3) & ~3);
    if (PQ && threadIdx.x == 0)
    {
        staging::BeginTableImageCopy(p.table, compactEntries, tableBarrierStorage); // table_staging.cuh
    }
    const LibmTables t = avifmath::StageLibmTables(libmStorage, threadIdx.x, blockDim.x);
    __syncthreads();
    if (PQ)
    {
        staging::WaitTableImage(tableBarrierStorage);
    }

    const uint32_t shift = p.table.flatShift;
    const int32_t negativeLow = -static_cast<int32_t>(p.table.flatLow);
    const int32_t span = static_cast<int32_t>(p.table.flatHigh - p.table.flatLow);
    const uint32_t topShift = 32u - shift;

    GroupWalk walk(static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x, static_cast<long long>(gridDim.x) * blockDim.x, p.groupsPerRow, p.rowCount);
    while (walk.Inside(p.rowCount))
    {
        float4 loaded[kGroupsInFlight][CHANNELS];
        long long planeOffsetY[kGroupsInFlight], planeOffsetA[kGroupsInFlight];
#pragma unroll
        for (int u = 0; u < kGroupsInFlight; ++u)
        {
            planeOffsetY[u] = -1;
            planeOffsetA[u] = 0;
#pragma unroll
            for (int c = 0; c < CHANNELS; ++c)
            {
                loaded[u][c] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            }
            if (walk.Inside(p.rowCount))
            {
                const long long row = walk.row;
                const long long column = static_cast<long long>(walk.column) * 4;
                const float4* source = reinterpret_cast<const float4*>(p.rows + row * p.rowStride + column * (4 * CHANNELS));
#pragma unroll
                for (int c = 0; c < CHANNELS; ++c)
                {
                    loaded[u][c] = __ldcs(source + c);
                }
                planeOffsetY[u] = row * p.strideY + column * 2;
                planeOffsetA[u] = row * p.strideA + column * 2;
            }
            walk.Advance(p.rowCount);
        }
        // ---- the values the curve sees, the alpha codes ---------------------------------------------------------------
        constexpr int kSamples = 4 * kGroupsInFlight;
        float value[kSamples];
        uint32_t aCode[kSamples];
#pragma unroll
        for (int u = 0; u < kGroupsInFlight; ++u)
        {
            float gray[4], alpha[4];
            if (CHANNELS == 1)
            {
                const float4 v = loaded[u][0];
                gray[0] = v.x; gray[1] = v.y; gray[2] = v.z; gray[3] = v.w;
            }
            else
            {
                const float4 a = loaded[u][0], b = loaded[u][CHANNELS - 1];
                gray[0] = a.x; alpha[0] = a.y; gray[1] = a.z; alpha[1] = a.w;
                gray[2] = b.x; alpha[2] = b.y; gray[3] = b.z; alpha[3] = b.w;
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
            {
                float v = gray[i];
                if (CHANNELS == 2)
                {
                    // WriteHeifImage.cpp:556-575
                    const float a = ClampF(alpha[i], 0.0f, 1.0f);
                    if (p.premultiply && a < 1.0f)
                    {
                        v = (a == 0) ? 0.0f : PremultiplyColor(ClampF(v, 0.0f, 1.0f), a, 1.0f);
                    }
                    aCode[4 * u + i] = FloatToCode(a, p.maxCodeFloat);
                }
                else
                {
                    v = ClampF(v, 0.0f, 1.0f); // WriteHeifImage.cpp:602
                }
                value[4 * u + i] = v; // a group past the image was loaded as zeros
            }
        }

        // ---- float -> code: all look-ups first, then the few flagged samples, then +inf / NaN ------------------------------
        uint32_t yCode[kSamples];
        if (!PQ)
        {
#pragma unroll
            for (int j = 0; j < kSamples; ++j)
            {
                yCode[j] = FloatToCode(value[j], p.maxCodeFloat);
            }
        }
        else
        {
            uint32_t flagged = 0;
            int32_t largest = 0;
#pragma unroll
            for (int j = 0; j < kSamples; ++j)
            {
                const uint32_t bits = __float_as_uint(value[j]);
                bool inBand;
                uint32_t entry;
                yCode[j] = static_cast<uint32_t>(LookupCurveCompact<0>(bits, compactEntries, shift, negativeLow, span, topShift, p.table.compactCodeMask,
                                                                       p.table.compactMagic, inBand, entry));
                flagged |= inBand ? (1u << j) : 0u;
                largest = max(largest, static_cast<int32_t>(bits));
            }
            uint32_t lower = 0; // samples whose exact code is one below the table's
            while (flagged != 0)
            {
                const int j = __ffs(static_cast<int>(flagged)) - 1;
                flagged &= flagged - 1;
                uint32_t bits = __float_as_uint(value[0]);
#pragma unroll
                for (int k = 1; k < kSamples; ++k)
                {
                    bits = (j == k) ? __float_as_uint(value[k]) : bits;
                }
                // the sample's step and its distance from first_k, then one bit of the band bitmap (curve_lookup.cuh ResolveCompactInBand)
                const int32_t bucket = __viaddmin_s32_relu(static_cast<int32_t>(bits) >> shift, negativeLow, span);
                const uint32_t entry = compactEntries[bucket];
                const uint32_t step = ((entry & p.table.compactCodeMask) >> kCompactLenBits) + ((entry >> topShift) != 0 ? 1u : 0u);
                const uint32_t distance = bits - firstBits[step];
                if (step != 0 && distance < (1u << p.table.bandStrideLog2))
                {
                    const uint32_t index = (step << p.table.bandStrideLog2) + distance;
                    const uint32_t word = __ldg(p.table.bandBits + (index >> 5));
                    // step or step - 1; the table said field + carry, which is `step` whenever bits >= first_k
                    lower |= ((word >> (index & 31u)) & 1u) ? 0u : (1u << j);
                }
            }
#pragma unroll
            for (int j = 0; j < kSamples; ++j)
            {
                yCode[j] -= (lower >> j) & 1u;
            }
            if (largest > 0x7f7fffff)
            {
#pragma unroll
                for (int j = 0; j < kSamples; ++j)
                {
                    if (static_cast<int32_t>(__float_as_uint(value[j])) > 0x7f7fffff)
                    {
                        yCode[j] = ExactCurveCode<kCurveLinearToPQ>(value[j], p.pqMultiplier, p.maxCodeFloat, t); // +inf / NaN
                    }
                }
            }
        }

#pragma unroll
        for (int u = 0; u < kGroupsInFlight; ++u)
        {
            if (planeOffsetY[u] < 0)
            {
                continue;
            }
            __stcs(reinterpret_cast<uint2*>(p.planeY + planeOffsetY[u]),
                   make_uint2(yCode[4 * u] | (yCode[4 * u + 1] << 16), yCode[4 * u + 2] | (yCode[4 * u + 3] << 16)));
            if (CHANNELS == 2)
            {
                __stcs(reinterpret_cast<uint2*>(p.planeA + planeOffsetA[u]),
                       make_uint2(aCode[4 * u] | (aCode[4 * u + 1] << 16), aCode[4 * u + 2] | (aCode[4 * u + 3] << 16)));
            }
        }
    }
}

template <int CHANNELS, int PQ>
cudaError_t LaunchGray32(const Gray32Params& gp, size_t shared, int smCount, cudaStream_t stream)
{
    static std::atomic<uint64_t> configuredDevices{ 0 };
    {
        const cudaError_t e = AllowDynamicShared(EncodeGrayF32Kernel<CHANNELS, PQ>, 100 * 1024, configuredDevices);
        if (e != cudaSuccess)
        {
            return e;
        }
    }
    constexpr int kThreads = PQ ? kGrayTableThreads : kGrayClipThreads;
    const long long groups = static_cast<long long>(gp.groupsPerRow) * gp.rowCount;
    long long blocks = (groups + kThreads - 1) / kThreads;
    const long long cap = PQ ? static_cast<long long>(smCount) : static_cast<long long>(smCount) * 8; // a table per CTA: one long-lived CTA per SM
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    EncodeGrayF32Kernel<CHANNELS, PQ><<<static_cast<unsigned>(blocks), kThreads, shared, stream>>>(gp);
    return cudaGetLastError();
}

} // namespace

// Returns the number of kernels launched, 0 if this configuration is not covered, or a negative status.
int LaunchEncodeFastGray32(const EncodeParams& p, int hostDepth, void* streamHandle)
{
    cudaStream_t stream = static_cast<cudaStream_t>(streamHandle);
    if (hostDepth != 32 || p.planar || p.channels > 2 || p.imageDepth <= 8 || p.hlgInverseOotf || p.rowMatrixEnabled)
    {
        return 0;
    }
    const bool pq = p.transfer == AVIFGPU_TRANSFER_PQ;
    if (!pq && p.transfer != AVIFGPU_TRANSFER_CLIP)
    {
        return 0; // the reference rejects anything else for gray (WriteHeifImage.cpp:586-587): the generic kernel's business
    }
    if (pq && (p.curveTable == nullptr || p.curveTable->compact == nullptr || p.curveTable->firstBits == nullptr || p.curveTable->bandBits == nullptr))
    {
        return 0; // no verified compact table: the generic exact kernel serves it
    }
    const int width4 = p.width & ~3;
    if (width4 < 4 || p.rowCount < 1 || !Aligned(p.rows, p.rowStride, 16) || !Aligned(p.plane[0], p.planeStride[0], 8) ||
        (p.channels == 2 && !Aligned(p.plane[3], p.planeStride[3], 8)))
    {
        return 0;
    }
    Gray32Params gp{};
    gp.rows = static_cast<const uint8_t*>(p.rows);
    gp.rowStride = p.rowStride;
    gp.planeY = static_cast<uint8_t*>(p.plane[0]);
    gp.strideY = p.planeStride[0];
    gp.planeA = static_cast<uint8_t*>(p.plane[3]);
    gp.strideA = p.planeStride[3];
    gp.groupsPerRow = width4 / 4;
    gp.rowCount = p.rowCount;
    gp.premultiply = p.premultiply;
    gp.pqMultiplier = p.pqMultiplier;
    gp.maxCodeFloat = p.maxCodeFloat;
    gp.maxCode = static_cast<int32_t>(p.maxCode);
    size_t shared = 768 + 16;
    if (pq)
    {
        gp.table = *p.curveTable;
        shared += gp.table.compactImageBytes;
        if (shared > 100 * 1024)
        {
            return 0;
        }
    }
    const int smCount = SmCount(p.smCount);
    cudaError_t e;
    if (p.channels == 2) e = pq ? LaunchGray32<2, 1>(gp, shared, smCount, stream) : LaunchGray32<2, 0>(gp, shared, smCount, stream);
    else e = pq ? LaunchGray32<1, 1>(gp, shared, smCount, stream) : LaunchGray32<1, 0>(gp, shared, smCount, stream);
    if (e != cudaSuccess)
    {
        return ReportLaunchFailure(static_cast<int>(e));
    }
    const int n = LaunchEncodeRemainder(p, hostDepth, width4, p.rowCount, streamHandle);
    return n < 0 ? n : 1 + n;
}

} // namespace avifgpu
