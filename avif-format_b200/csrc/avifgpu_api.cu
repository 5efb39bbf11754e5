// avifgpu_api.cu -- the extern "C" surface declared in include/avifgpu.h: context, validation, PCIe staging for
// the host-pointer entry points, and dispatch to the kernels.  No CPU fallback anywhere: every entry point that
// converts pixels launches a CUDA kernel or fails.
#include "../../include/avifgpu.h"

#include "curve_tables.h"
#include "host_params.h"
#include "kernel_params.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>


namespace avifgpu
{

namespace
{
    thread_local int g_launchFailure = 0; // cudaError_t of the last failed launch on this thread, 0 = none
}

int ReportLaunchFailure(int cudaErrorCode)
{
    g_launchFailure = cudaErrorCode;
    return AVIFGPU_ERR_CUDA;
}

static int TakeLaunchFailure()
{
    const int code = g_launchFailure;
    g_launchFailure = 0;
    return code;
}

int LaunchEncode(const EncodeParams& params, int hostDepth, void* stream)
{
    int fast = LaunchEncodeFast(params, hostDepth, stream);
    if (fast != 0)
    {
        return fast;
    }
    fast = LaunchEncodeFastInteger(params, hostDepth, stream);
    if (fast != 0)
    {
        return fast;
    }
    fast = LaunchEncodeFastGray32(params, hostDepth, stream);
    if (fast != 0)
    {
        return fast;
    }
    return LaunchEncodeGeneric(params, hostDepth, stream);
}

int LaunchDecode(const DecodeParams& params, void* stream)
{
    int fast = LaunchDecodeFast(params, stream);
    if (fast != 0)
    {
        return fast;
    }
    fast = LaunchDecodeFastInteger(params, stream);
    if (fast != 0)
    {
        return fast;
    }
    fast = LaunchDecodeFastTable(params, stream);
    if (fast != 0)
    {
        return fast;
    }
    return LaunchDecodeGeneric(params, stream);
}
} // namespace avifgpu

using namespace avifgpu;

namespace
{
    thread_local std::string g_creationError;

    // A host-pointer call is cut into row-block slices that rotate through this many pipeline slots (stream + staging
    // buffers each), so that the H2D copy of slice i+1, the kernel of slice i and the D2H copy of slice i-1 overlap.
    // Two slots keep both copy engines busy; the third lets the host thread fill / drain a pinned bounce buffer
    // (pageable caller memory) while the other two are on the wire.
    constexpr int kPipelineStreams = 3;
}

struct avifgpu_context
{
    int device = -1;
    cudaStream_t streams[kPipelineStreams] = {};
    cudaEvent_t sliceDone[kPipelineStreams] = {};
    cudaEvent_t rowsConsumed[kPipelineStreams] = {}; // encode: the slot's H2D of caller rows has finished
    cudaEvent_t callRowsConsumed[2] = {};            // the last H2D of an asynchronous encode call (calls alternate between the two)
    int64_t asyncEncodeCalls = 0;
    bool previousCallRowsPending = false;            // callRowsConsumed[(asyncEncodeCalls - 1) & 1] guards caller memory still on the wire

    // Work a slot still owes the caller once its stream has drained: copies from a pinned bounce buffer into pageable
    // caller memory (libheif's planes on the encode side, pageable host rows on the decode side).
    struct HostCopy
    {
        uint8_t* target;
        int64_t targetStride;
        const uint8_t* source;
        int64_t sourceStride;
        int64_t payload;
        int rows;
    };
    struct SlotState
    {
        bool busy = false;
        int64_t ticket = 0;
        std::vector<HostCopy> owed;
    };
    SlotState slots[kPipelineStreams];
    int nextSlot = 0;
    int64_t lastTicket = 0;       // ticket of the most recent host-pointer call
    std::string lastError;
    int64_t launches = 0;
    int smCount = 0;

    // Device staging for the host-pointer entry points (grow-only).
    struct Buffer
    {
        void* ptr = nullptr;
        size_t bytes = 0;
    };
    Buffer deviceRows[kPipelineStreams];
    Buffer devicePlanes[kPipelineStreams][AVIFGPU_MAX_PLANES];
    // Pinned bounce buffers for pageable caller memory (grow-only).
    Buffer pinnedRows[kPipelineStreams];
    Buffer pinnedPlanes[kPipelineStreams][AVIFGPU_MAX_PLANES];
    Buffer transferScratch[2];
    std::vector<CurveTable*> curveTables; // exact step tables, built per (curve, param, depth): explicitly or once they pay off
    struct PendingTable
    {
        int curve, param, depth;
        int64_t pixels; // converted with the exact kernel so far
    };
    std::vector<PendingTable> pendingTables;
    int64_t tableAutoBuildPixels = AVIFGPU_TABLE_AUTOBUILD_DEFAULT;
    struct Gray16Lut
    {
        int depth = 0;
        int smpte428 = 0;
        uint16_t* device = nullptr;
    };
    std::vector<Gray16Lut> gray16Luts;
    int premultiplyState[3] = { -1, -1, -1 }; // image depth 8 / 10 / 12: -1 not checked yet, 0 keep the reference sequence, 1 fast form verified
    // The tuned integer encode kernel premultiplies with a 6-instruction form, but only after it has been compared with
    // PremultiplyColor's own sequence for every (colour, alpha) code pair of the depth, on this device.
    int VerifiedPremultiply(const avifgpu_encode_desc& d)
    {
        if (d.alpha_state != AVIFGPU_ALPHA_PREMULTIPLIED || d.host_depth == 32 || d.host_channels != 4 || d.layout != AVIFGPU_LAYOUT_PLANAR_YCBCR)
        {
            return 0;
        }
        const int slot = d.image_bit_depth == 8 ? 0 : d.image_bit_depth == 10 ? 1 : 2;
        if (premultiplyState[slot] < 0)
        {
            premultiplyState[slot] = VerifyFastPremultiply((1u << d.image_bit_depth) - 1u, streams[0]) == 0 ? 1 : 0;
            launches += 1;
        }
        return premultiplyState[slot];
    }
    int hlgDivisionState = -1; // -1 not checked yet, 0 keep IEEE divisions, 1 fast divisions verified exact

    // HLG decode replaces two constant divisions by a 3-instruction form, but only after comparing it with the
    // IEEE division over every numerator the call sites can produce, on this device.
    int VerifiedHlgDivisions()
    {
        if (hlgDivisionState < 0)
        {
            const long long disagreements = VerifyHlgDivisions(streams[0]);
            hlgDivisionState = disagreements == 0 ? 1 : 0;
            launches += 1;
        }
        return hlgDivisionState;
    }

    // The quotient inside PQToLinear (ColorTransfer.cpp:110-112): the tuned float decode kernel uses a branch-free division
    // once it has been compared with the IEEE one for every value the quotient's operands can take, on this device.
    int pqRatioState = -1;
    int VerifiedPqRatio()
    {
        if (pqRatioState < 0)
        {
            const long long disagreements = VerifyPqRatio(streams[0]);
            pqRatioState = disagreements == 0 ? 1 : 0;
            launches += 1;
        }
        return pqRatioState;
    }

    // YuvDecode.cpp:308 divides by the per-image constant kg; the tuned decode kernels use a 3-instruction form after
    // it has been compared with the IEEE division for every (Cb, Cr) code pair of the configuration, on this device.
    struct GreenDivision
    {
        avifpix::InverseMatrix matrix;
        avifpix::RangeParams range;
        uint32_t maxCode;
        int state;
    };
    std::vector<GreenDivision> greenDivisions;
    int VerifiedGreenDivision(const DecodeParams& p)
    {
        if (p.colorspace != AVIFGPU_COLORSPACE_YCBCR || p.bitDepth > 12)
        {
            return 0;
        }
        for (const GreenDivision& g : greenDivisions)
        {
            if (std::memcmp(&g.matrix, &p.matrix, sizeof(g.matrix)) == 0 && std::memcmp(&g.range, &p.range, sizeof(g.range)) == 0 && g.maxCode == p.maxCode)
            {
                return g.state;
            }
        }
        GreenDivision g{};
        g.matrix = p.matrix;
        g.range = p.range;
        g.maxCode = p.maxCode;
        g.state = VerifyGreenDivision(p, streams[0]) == 0 ? 1 : 0;
        launches += 1;
        greenDivisions.push_back(g);
        return g.state;
    }

    // The 65536-entry code table of a Gray16 host configuration (built on the device on first use), or nullptr.
    const uint16_t* Gray16LutFor(const avifgpu_encode_desc& d)
    {
        if (d.host_depth != 16 || d.host_channels != 1 || d.layout != AVIFGPU_LAYOUT_REFERENCE || d.image_bit_depth <= 8)
        {
            return nullptr;
        }
        const int smpte428 = d.gray16_curve == AVIFGPU_GRAY16_SMPTE428 ? 1 : 0;
        for (const Gray16Lut& l : gray16Luts)
        {
            if (l.depth == d.image_bit_depth && l.smpte428 == smpte428)
            {
                return l.device;
            }
        }
        Gray16Lut lut;
        lut.depth = d.image_bit_depth;
        lut.smpte428 = smpte428;
        if (cudaMalloc(&lut.device, 65536 * sizeof(uint16_t)) != cudaSuccess)
        {
            cudaGetLastError();
            return nullptr;
        }
        if (BuildGray16Lut(lut.device, smpte428, (1u << d.image_bit_depth) - 1u, streams[0]) != cudaSuccess ||
            cudaStreamSynchronize(streams[0]) != cudaSuccess)
        {
            cudaGetLastError();
            cudaFree(lut.device);
            return nullptr;
        }
        launches += 1;
        gray16Luts.push_back(lut);
        return lut.device;
    }

    // The verified step table for a float-host encode description, or nullptr when the description does not use
    // one / the table could not be verified / building it has not paid off yet (then the generic exact kernel serves
    // the call).  `pixels` = the size of the call that asks; `force` = avifgpu_prepare_encode.
    CurveTable* CurveTableFor(const avifgpu_encode_desc& d, int64_t pixels, bool force)
    {
        if (d.host_depth != 32 || d.image_bit_depth > 12)
        {
            return nullptr;
        }
        int curve;
        int param = 0;
        if (d.transfer == AVIFGPU_TRANSFER_PQ)
        {
            curve = kCurveLinearToPQ;
            param = d.pq_peak_nits;
        }
        else if (d.transfer == AVIFGPU_TRANSFER_SMPTE428)
        {
            curve = kCurveLinearToSMPTE428;
        }
        else if (d.transfer == AVIFGPU_TRANSFER_HLG)
        {
            curve = kCurveLinearToHLG;
        }
        else
        {
            return nullptr;
        }
        for (CurveTable* t : curveTables)
        {
            if (t->curve == curve && t->param == param && t->depth == d.image_bit_depth)
            {
                return t;
            }
        }
        if (!force)
        {
            // ~40 ms of sweeps buy a ~7x faster kernel: worth it once a configuration has seen enough pixels
            PendingTable* pending = nullptr;
            for (PendingTable& candidate : pendingTables)
            {
                if (candidate.curve == curve && candidate.param == param && candidate.depth == d.image_bit_depth)
                {
                    pending = &candidate;
                }
            }
            if (pending == nullptr)
            {
                pendingTables.push_back(PendingTable{ curve, param, d.image_bit_depth, 0 });
                pending = &pendingTables.back();
            }
            pending->pixels += pixels;
            if (tableAutoBuildPixels < 0 || pending->pixels <= tableAutoBuildPixels)
            {
                return nullptr;
            }
        }
        CurveTable* t = new (std::nothrow) CurveTable();
        if (t == nullptr)
        {
            return nullptr;
        }
        BuildCurveTable(curve, param, d.image_bit_depth, streams[0], t);
        launches += t->stats.sweptInputs ? (t->stats.bandBitmapBytes ? 3 : 2) : 0; // sweep, (band bitmap,) verify
        curveTables.push_back(t);
        return t;
    }

    int Fail(int status, const std::string& message)
    {
        lastError = message;
        return status;
    }

    // A launcher returned a negative status: report the CUDA error it recorded (it has already cleared CUDA's own
    // slot), after draining the pipeline streams so that no copy of an earlier slice is still writing into caller memory
    // when the entry point returns.
    int LaunchFailed(int status, const char* what)
    {
        const int code = TakeLaunchFailure();
        for (cudaStream_t stream : streams)
        {
            if (stream)
            {
                cudaStreamSynchronize(stream);
            }
        }
        cudaGetLastError();
        lastError = std::string(what) + " failed: " + (code != 0 ? cudaGetErrorString(static_cast<cudaError_t>(code)) : avifgpu_status_string(status));
        return status;
    }

    // Any failure in the middle of a host-pointer call: same draining, then the status.
    int Abandon(int status)
    {
        for (cudaStream_t stream : streams)
        {
            if (stream)
            {
                cudaStreamSynchronize(stream);
            }
        }
        cudaGetLastError();
        return status;
    }

    int Cuda(cudaError_t e, const char* what)
    {
        if (e == cudaSuccess)
        {
            return AVIFGPU_OK;
        }
        lastError = std::string(what) + ": " + cudaGetErrorString(e);
        return (e == cudaErrorMemoryAllocation) ? AVIFGPU_ERR_OOM : AVIFGPU_ERR_CUDA;
    }

    int EnsureDevice(Buffer& b, size_t bytes)
    {
        if (b.bytes >= bytes)
        {
            return AVIFGPU_OK;
        }
        if (b.ptr)
        {
            cudaFree(b.ptr);
            b.ptr = nullptr;
            b.bytes = 0;
        }
        const size_t rounded = ((bytes + (1u << 20) - 1) >> 20) << 20;
        const int status = Cuda(cudaMalloc(&b.ptr, rounded), "cudaMalloc");
        if (status == AVIFGPU_OK)
        {
            b.bytes = rounded;
        }
        return status;
    }

    int EnsurePinned(Buffer& b, size_t bytes)
    {
        if (b.bytes >= bytes)
        {
            return AVIFGPU_OK;
        }
        if (b.ptr)
        {
            cudaFreeHost(b.ptr);
            b.ptr = nullptr;
            b.bytes = 0;
        }
        const size_t rounded = ((bytes + (1u << 20) - 1) >> 20) << 20;
        const int status = Cuda(cudaHostAlloc(&b.ptr, rounded, cudaHostAllocDefault), "cudaHostAlloc");
        if (status == AVIFGPU_OK)
        {
            b.bytes = rounded;
        }
        return status;
    }
};

static int RetireThrough(avifgpu_context* ctx, int64_t ticket);

namespace
{
    bool IsPinned(const void* p)
    {
        cudaPointerAttributes attr{};
        if (cudaPointerGetAttributes(&attr, p) != cudaSuccess)
        {
            cudaGetLastError();
            return false;
        }
        return attr.type == cudaMemoryTypeHost;
    }

    struct DeviceGuard
    {
        int previous = -1;
        explicit DeviceGuard(int device)
        {
            cudaGetDevice(&previous);
            if (previous != device)
            {
                cudaSetDevice(device);
            }
            else
            {
                previous = -1;
            }
        }
        ~DeviceGuard()
        {
            if (previous >= 0)
            {
                cudaSetDevice(previous);
            }
        }
    };

    int CheckBlock(avifgpu_context* ctx, int height, int ys, int y0, int nrows)
    {
        if (y0 < 0 || nrows < 0 || y0 > height || nrows > height - y0)
        {
            return ctx->Fail(AVIFGPU_ERR_BAD_PARAM, "row block outside the image");
        }
        if (ys && (y0 & 1))
        {
            return ctx->Fail(AVIFGPU_ERR_BAD_PARAM, "4:2:0 row blocks must start on an even row");
        }
        if (ys && (nrows & 1) && y0 + nrows != height)
        {
            return ctx->Fail(AVIFGPU_ERR_BAD_PARAM, "4:2:0 row blocks must have an even height unless they end the image");
        }
        return AVIFGPU_OK;
    }
}

// ---- context ------------------------------------------------------------------------------------------------

extern "C" {

AVIFGPU_EXPORT int avifgpu_api_version(void) { return AVIFGPU_API_VERSION; }

AVIFGPU_EXPORT const char* avifgpu_status_string(int status)
{
    switch (status)
    {
    case AVIFGPU_OK: return "ok";
    case AVIFGPU_ERR_BAD_PARAM: return "bad parameter";
    case AVIFGPU_ERR_UNSUPPORTED: return "unsupported";
    case AVIFGPU_ERR_NO_DEVICE: return "no usable CUDA device";
    case AVIFGPU_ERR_CUDA: return "CUDA error";
    case AVIFGPU_ERR_OOM: return "out of memory";
    case AVIFGPU_ERR_CANCELED: return "canceled";
    default: return "unknown status";
    }
}

AVIFGPU_EXPORT int avifgpu_create(int device_ordinal, avifgpu_context** out_ctx)
{
    if (out_ctx == nullptr)
    {
        g_creationError = "out_ctx is NULL";
        return AVIFGPU_ERR_BAD_PARAM;
    }
    *out_ctx = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count <= 0)
    {
        cudaGetLastError();
        g_creationError = std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
                          " (this library has no CPU fallback)";
        return AVIFGPU_ERR_NO_DEVICE;
    }
    if (device_ordinal < 0 || device_ordinal >= count)
    {
        g_creationError = "device ordinal out of range";
        return AVIFGPU_ERR_BAD_PARAM;
    }
    cudaDeviceProp prop{};
    e = cudaGetDeviceProperties(&prop, device_ordinal);
    if (e != cudaSuccess)
    {
        g_creationError = std::string("cudaGetDeviceProperties: ") + cudaGetErrorString(e);
        return AVIFGPU_ERR_NO_DEVICE;
    }
    if (prop.major != 10)
    {
        char text[160];
        std::snprintf(text, sizeof(text), "device %d is sm_%d%d; this library ships sm_100a code only", device_ordinal, prop.major, prop.minor);
        g_creationError = text;
        return AVIFGPU_ERR_NO_DEVICE;
    }
    avifgpu_context* ctx = new (std::nothrow) avifgpu_context();
    if (ctx == nullptr)
    {
        g_creationError = "out of host memory";
        return AVIFGPU_ERR_OOM;
    }
    ctx->device = device_ordinal;
    ctx->smCount = prop.multiProcessorCount;
    DeviceGuard guard(device_ordinal);
    for (int i = 0; i < kPipelineStreams; ++i)
    {
        if (cudaStreamCreateWithFlags(&ctx->streams[i], cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&ctx->sliceDone[i], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&ctx->rowsConsumed[i], cudaEventDisableTiming) != cudaSuccess ||
            (i < 2 && cudaEventCreateWithFlags(&ctx->callRowsConsumed[i], cudaEventDisableTiming) != cudaSuccess))
        {
            g_creationError = std::string("stream/event creation failed: ") + cudaGetErrorString(cudaGetLastError());
            avifgpu_destroy(ctx);
            return AVIFGPU_ERR_CUDA;
        }
    }
    *out_ctx = ctx;
    return AVIFGPU_OK;
}

AVIFGPU_EXPORT void avifgpu_destroy(avifgpu_context* ctx)
{
    if (ctx == nullptr)
    {
        return;
    }
    DeviceGuard guard(ctx->device);
    cudaDeviceSynchronize();
    for (int i = 0; i < kPipelineStreams; ++i)
    {
        if (ctx->streams[i]) cudaStreamDestroy(ctx->streams[i]);
        if (ctx->sliceDone[i]) cudaEventDestroy(ctx->sliceDone[i]);
        if (ctx->rowsConsumed[i]) cudaEventDestroy(ctx->rowsConsumed[i]);
        if (i < 2 && ctx->callRowsConsumed[i]) cudaEventDestroy(ctx->callRowsConsumed[i]);
        if (ctx->deviceRows[i].ptr) cudaFree(ctx->deviceRows[i].ptr);
        if (ctx->pinnedRows[i].ptr) cudaFreeHost(ctx->pinnedRows[i].ptr);
        for (int k = 0; k < AVIFGPU_MAX_PLANES; ++k)
        {
            if (ctx->devicePlanes[i][k].ptr) cudaFree(ctx->devicePlanes[i][k].ptr);
            if (ctx->pinnedPlanes[i][k].ptr) cudaFreeHost(ctx->pinnedPlanes[i][k].ptr);
        }
    }
    for (auto& b : ctx->transferScratch)
    {
        if (b.ptr) cudaFree(b.ptr);
    }
    for (CurveTable* t : ctx->curveTables)
    {
        FreeCurveTable(t);
        delete t;
    }
    for (auto& l : ctx->gray16Luts)
    {
        cudaFree(l.device);
    }
    delete ctx;
}

AVIFGPU_EXPORT const char* avifgpu_last_error(const avifgpu_context* ctx)
{
    return ctx ? ctx->lastError.c_str() : g_creationError.c_str();
}

AVIFGPU_EXPORT int64_t avifgpu_launch_count(const avifgpu_context* ctx) { return ctx ? ctx->launches : 0; }

AVIFGPU_EXPORT int avifgpu_synchronize(avifgpu_context* ctx)
{
    if (ctx == nullptr)
    {
        return AVIFGPU_ERR_BAD_PARAM;
    }
    DeviceGuard guard(ctx->device);
    const int status = ctx->Cuda(cudaDeviceSynchronize(), "cudaDeviceSynchronize");
    const int retired = RetireThrough(ctx, ctx->lastTicket); // pays the bounce copies asynchronous calls still owe
    ctx->previousCallRowsPending = false;
    return status != AVIFGPU_OK ? status : retired;
}

AVIFGPU_EXPORT int avifgpu_host_alloc(avifgpu_context* ctx, size_t bytes, void** out_ptr)
{
    if (ctx == nullptr || out_ptr == nullptr)
    {
        return AVIFGPU_ERR_BAD_PARAM;
    }
    DeviceGuard guard(ctx->device);
    *out_ptr = nullptr;
    return ctx->Cuda(cudaHostAlloc(out_ptr, bytes ? bytes : 1, cudaHostAllocDefault), "cudaHostAlloc");
}

AVIFGPU_EXPORT int avifgpu_host_free(avifgpu_context* ctx, void* ptr)
{
    if (ctx == nullptr)
    {
        return AVIFGPU_ERR_BAD_PARAM;
    }
    DeviceGuard guard(ctx->device);
    return ctx->Cuda(cudaFreeHost(ptr), "cudaFreeHost");
}

// ---- geometry and parameter derivation (no device needed) -----------------------------------------------------

AVIFGPU_EXPORT int avifgpu_encode_host_col_bytes(const avifgpu_encode_desc* desc)
{
    return ValidateEncodeDesc(desc, nullptr) == AVIFGPU_OK ? EncodeHostColBytes(*desc) : AVIFGPU_ERR_BAD_PARAM;
}

AVIFGPU_EXPORT int avifgpu_decode_host_col_bytes(const avifgpu_decode_desc* desc)
{
    int32_t transfer;
    return ValidateDecodeDesc(desc, &transfer, nullptr) == AVIFGPU_OK ? DecodeHostColBytes(*desc) : AVIFGPU_ERR_BAD_PARAM;
}

static int ReportGeometry(const PlaneGeometry& g, int32_t* w, int32_t* h, int32_t* b)
{
    if (w) *w = g.present ? g.widthSamples : 0;
    if (h) *h = g.present ? g.height : 0;
    if (b) *b = g.present ? g.bytesPerSample : 0;
    return g.present ? 1 : 0;
}

AVIFGPU_EXPORT int avifgpu_encode_plane_geometry(const avifgpu_encode_desc* desc, int index, int32_t* w, int32_t* h, int32_t* b)
{
    const int status = ValidateEncodeDesc(desc, nullptr);
    if (status != AVIFGPU_OK || index < 0 || index >= AVIFGPU_MAX_PLANES)
    {
        ReportGeometry(PlaneGeometry(), w, h, b);
        return status != AVIFGPU_OK ? status : AVIFGPU_ERR_BAD_PARAM;
    }
    return ReportGeometry(EncodePlaneGeometry(*desc, index), w, h, b);
}

AVIFGPU_EXPORT int avifgpu_decode_plane_geometry(const avifgpu_decode_desc* desc, int index, int32_t* w, int32_t* h, int32_t* b)
{
    int32_t transfer;
    const int status = ValidateDecodeDesc(desc, &transfer, nullptr);
    if (status != AVIFGPU_OK || index < 0 || index >= AVIFGPU_MAX_PLANES)
    {
        ReportGeometry(PlaneGeometry(), w, h, b);
        return status != AVIFGPU_OK ? status : AVIFGPU_ERR_BAD_PARAM;
    }
    return ReportGeometry(DecodePlaneGeometry(*desc, index), w, h, b);
}

AVIFGPU_EXPORT int avifgpu_get_yuv_coefficients(const avifgpu_nclx* nclx, float* out)
{
    if (out == nullptr)
    {
        return AVIFGPU_ERR_BAD_PARAM;
    }
    GetYuvCoefficients(nclx, out);
    return AVIFGPU_OK;
}

AVIFGPU_EXPORT int avifgpu_get_hlg_luma_coefficients(int32_t color_primaries, float* out)
{
    if (out == nullptr)
    {
        return AVIFGPU_ERR_BAD_PARAM;
    }
    return GetHlgLumaCoefficients(color_primaries, out) ? AVIFGPU_OK : AVIFGPU_ERR_UNSUPPORTED;
}

AVIFGPU_EXPORT int avifgpu_build_yuv_tables(const avifgpu_nclx* nclx, int32_t bit_depth, int32_t monochrome, float* out_y,
                                            float* out_uv, float* out_alpha)
{
    if (bit_depth != 8 && bit_depth != 10 && bit_depth != 12 && bit_depth != 16)
    {
        return AVIFGPU_ERR_UNSUPPORTED;
    }
    const avifpix::RangeParams range = MakeRangeParams(nclx, bit_depth, monochrome != 0);
    const uint32_t count = 1u << bit_depth;
    for (uint32_t i = 0; i < count; ++i)
    {
        if (out_y) out_y[i] = avifpix::UnormToFloatY(i, range);
        if (out_uv && !monochrome) out_uv[i] = avifpix::UnormToFloatUV(i, range);
        if (out_alpha) out_alpha[i] = avifpix::UnormToFloatPlain(i, range.maxChannelFloat);
    }
    return AVIFGPU_OK;
}

// ---- device-pointer entry points -------------------------------------------------------------------------------

AVIFGPU_EXPORT int avifgpu_encode_rows_device(avifgpu_context* ctx, const avifgpu_encode_desc* desc, const void* device_rows,
                                              int64_t row_stride_bytes, int32_t y0, int32_t nrows,
                                              const avifgpu_planes* device_dst, void* cuda_stream)
{
    if (ctx == nullptr)
    {
        return AVIFGPU_ERR_BAD_PARAM;
    }
    std::string error;
    int status = ValidateEncodeDesc(desc, &error);
    if (status != AVIFGPU_OK)
    {
        return ctx->Fail(status, error);
    }
    if (device_dst == nullptr || (device_rows == nullptr && nrows > 0 && desc->width > 0))
    {
        return ctx->Fail(AVIFGPU_ERR_BAD_PARAM, "NULL buffer");
    }
    EncodeParams p;
    FillEncodeParams(*desc, &p);
    status = CheckBlock(ctx, desc->height, p.ys, y0, nrows);
    if (status != AVIFGPU_OK)
    {
        return status;
    }
    if (nrows == 0 || desc->width == 0)
    {
        return AVIFGPU_OK;
    }
    p.rows = device_rows;
    p.rowStride = row_stride_bytes;
    p.rowCount = nrows;
    for (int k = 0; k < AVIFGPU_MAX_PLANES; ++k)
    {
        const PlaneGeometry g = EncodePlaneGeometry(*desc, k);
        if (!g.present)
        {
            continue;
        }
        if (device_dst->data[k] == nullptr)
        {
            return ctx->Fail(AVIFGPU_ERR_BAD_PARAM, "missing destination plane");
        }
        p.plane[k] = static_cast<uint8_t*>(device_dst->data[k]) + static_cast<int64_t>(y0 >> g.ys) * device_dst->stride[k];
        p.planeStride[k] = device_dst->stride[k];
    }
    DeviceGuard guard(ctx->device);
    p.smCount = ctx->smCount;
    if (CurveTable* table = ctx->CurveTableFor(*desc, static_cast<int64_t>(desc->width) * nrows, false))
    {
        p.curveTable = table->valid ? &table->view : nullptr;
    }
    p.gray16Lut = ctx->Gray16LutFor(*desc);
    p.verifiedPremultiply = ctx->VerifiedPremultiply(*desc);
    const int launched = LaunchEncode(p, desc->host_depth, cuda_stream);
    if (launched < 0)
    {
        return ctx->LaunchFailed(launched, "encode kernel launch");
    }
    ctx->launches += launched;
    return AVIFGPU_OK;
}

AVIFGPU_EXPORT int avifgpu_decode_rows_device(avifgpu_context* ctx, const avifgpu_decode_desc* desc,
                                              const avifgpu_planes* device_src, int32_t y0, int32_t nrows, void* device_rows,
                                              int64_t row_stride_bytes, void* cuda_stream)
{
    if (ctx == nullptr)
    {
        return AVIFGPU_ERR_BAD_PARAM;
    }
    std::string error;
    int32_t transfer;
    int status = ValidateDecodeDesc(desc, &transfer, &error);
    if (status != AVIFGPU_OK)
    {
        return ctx->Fail(status, error);
    }
    if (device_src == nullptr || (device_rows == nullptr && nrows > 0 && desc->width > 0))
    {
        return ctx->Fail(AVIFGPU_ERR_BAD_PARAM, "NULL buffer");
    }
    DecodeParams p;
    if (!FillDecodeParams(*desc, transfer, &p, &error))
    {
        return ctx->Fail(AVIFGPU_ERR_UNSUPPORTED, error);
    }
    if (y0 < 0 || nrows < 0 || y0 > desc->height || nrows > desc->height - y0)
    {
        return ctx->Fail(AVIFGPU_ERR_BAD_PARAM, "row block outside the image");
    }
    if (nrows == 0 || desc->width == 0)
    {
        return AVIFGPU_OK;
    }
    p.rows = device_rows;
    p.rowStride = row_stride_bytes;
    p.rowCount = nrows;
    p.yPhase = y0 & p.ys;
    p.smCount = ctx->smCount;
    DeviceGuard deviceGuardForTables(ctx->device);
    p.verifiedHlgDivisions = (desc->host_depth == 32 && transfer == AVIFGPU_TRANSFER_HLG) ? ctx->VerifiedHlgDivisions() : 0;
    p.verifiedGreenDivision = ctx->VerifiedGreenDivision(p);
    p.verifiedPqRatio = (desc->host_depth == 32 && transfer == AVIFGPU_TRANSFER_PQ && desc->colorspace == AVIFGPU_COLORSPACE_YCBCR) ? ctx->VerifiedPqRatio() : 0;
    for (int k = 0; k < AVIFGPU_MAX_PLANES; ++k)
    {
        const PlaneGeometry g = DecodePlaneGeometry(*desc, k);
        if (!g.present)
        {
            continue;
        }
        if (device_src->data[k] == nullptr)
        {
            return ctx->Fail(AVIFGPU_ERR_BAD_PARAM, "missing source plane");
        }
        p.plane[k] = static_cast<const uint8_t*>(device_src->data[k]) + static_cast<int64_t>(y0 >> g.ys) * device_src->stride[k];
        p.planeStride[k] = device_src->stride[k];
    }
    DeviceGuard guard(ctx->device);
    const int launched = LaunchDecode(p, cuda_stream);
    if (launched < 0)
    {
        return ctx->LaunchFailed(launched, "decode kernel launch");
    }
    ctx->launches += launched;
    return AVIFGPU_OK;
}

} // extern "C"

// ---- host-pointer entry points (PCIe inside) ---------------------------------------------------------------------
//
// A call is cut into row-block slices; slice i uses pipeline slot i mod kPipelineStreams (a stream, device staging,
// pinned bounce buffers).  Caller memory that is not page-locked is bounced through the slot's pinned buffers on BOTH
// sides -- a copy to or from pageable memory would make the driver stage it synchronously and serialise the pipeline --
// and the bounce -> pageable copies a slot still owes are made when the slot is retired (before it is reused, when a
// call or a ticket is waited for).  Slots retire in issue order, so "everything up to ticket t" is a prefix.

// Rows per pipeline slice: big enough to amortise launch + copy latency, small enough that the slots overlap.
static int SliceRows(int nrows, int64_t bytesPerRow)
{
    const int64_t target = 32ll << 20; // ~32 MiB of host rows per slice
    int64_t rows = bytesPerRow > 0 ? target / bytesPerRow : nrows;
    rows = std::max<int64_t>(rows, 2);
    rows &= ~1ll; // keep 4:2:0 row pairs together
    return static_cast<int>(std::min<int64_t>(rows, nrows));
}

static void CopyRowsSerial(uint8_t* target, int64_t targetStride, const uint8_t* source, int64_t sourceStride, int64_t payload, int rows)
{
    if (targetStride == payload && sourceStride == payload)
    {
        std::memcpy(target, source, static_cast<size_t>(payload) * rows);
        return;
    }
    for (int r = 0; r < rows; ++r)
    {
        std::memcpy(target + static_cast<int64_t>(r) * targetStride, source + static_cast<int64_t>(r) * sourceStride, static_cast<size_t>(payload));
    }
}

// Bounce copies between pageable caller memory and the pinned slot buffers.  One core moves ~10 GB/s, a fifth of what
// the PCIe link next to it carries, and an 8K frame owes 100 MB of plane copies: a small pool of parked threads (created
// at the first bounce, process-wide, joined at exit) shares every batch of copies above a megabyte, cut into chunks of
// rows that the threads -- and the caller -- pull from a common counter.
namespace
{
    struct RowCopy
    {
        uint8_t* target;
        int64_t targetStride;
        const uint8_t* source;
        int64_t sourceStride;
        int64_t payload;
        int rows;
    };

    class CopyPool
    {
    public:
        static CopyPool& Instance()
        {
            static CopyPool pool;
            return pool;
        }

        void Copy(const RowCopy* copies, int count)
        {
            int64_t bytes = 0;
            for (int i = 0; i < count; ++i)
            {
                bytes += copies[i].payload * copies[i].rows;
            }
            if (bytes < (1ll << 20) || workers.empty())
            {
                for (int i = 0; i < count; ++i)
                {
                    CopyRowsSerial(copies[i].target, copies[i].targetStride, copies[i].source, copies[i].sourceStride, copies[i].payload, copies[i].rows);
                }
                return;
            }
            std::unique_lock<std::mutex> callers(callerMutex); // one batch at a time (contexts on several threads share the pool)
            {
                std::lock_guard<std::mutex> lock(mutex);
                chunks.clear();
                for (int i = 0; i < count; ++i)
                {
                    const RowCopy& c = copies[i];
                    const int rowsPerChunk = static_cast<int>(std::max<int64_t>((256ll << 10) / std::max<int64_t>(c.payload, 1), 1));
                    for (int begin = 0; begin < c.rows; begin += rowsPerChunk)
                    {
                        chunks.push_back(RowCopy{ c.target + static_cast<int64_t>(begin) * c.targetStride, c.targetStride,
                                                  c.source + static_cast<int64_t>(begin) * c.sourceStride, c.sourceStride, c.payload,
                                                  std::min(rowsPerChunk, c.rows - begin) });
                    }
                }
                next.store(0, std::memory_order_relaxed);
                remaining = static_cast<int>(chunks.size());
                ++generation;
            }
            wake.notify_all();
            Drain();
            std::unique_lock<std::mutex> lock(mutex);
            done.wait(lock, [&] { return remaining == 0; });
        }

    private:
        CopyPool()
        {
            const unsigned cores = std::thread::hardware_concurrency();
            // 8 copying threads with the caller.  More is worse, measured (profiles/r2_shuttle_pipeline.md): with 16 an 8K frame
            // with pageable planes took 10.1 ms against 7.9 ms with 8 or 4 -- the copies then disturb the DMA they run beside --
            // while fewer than 4 cannot keep up with config 4's 1.6 GB of planes or with first-touch page faults.
            const int count = static_cast<int>(std::min<unsigned>(cores > 1 ? cores - 1 : 0, 7));
            for (int i = 0; i < count; ++i)
            {
                workers.emplace_back([this] { Run(); });
            }
        }

        ~CopyPool()
        {
            {
                std::lock_guard<std::mutex> lock(mutex);
                stopping = true;
            }
            wake.notify_all();
            for (std::thread& t : workers)
            {
                t.join();
            }
        }

        // Pulls chunks until none is left; returns how many this thread copied.
        void Drain()
        {
            int copied = 0;
            const int total = static_cast<int>(chunks.size());
            for (;;)
            {
                const int i = next.fetch_add(1, std::memory_order_relaxed);
                if (i >= total)
                {
                    break;
                }
                const RowCopy& c = chunks[i];
                CopyRowsSerial(c.target, c.targetStride, c.source, c.sourceStride, c.payload, c.rows);
                ++copied;
            }
            if (copied)
            {
                std::lock_guard<std::mutex> lock(mutex);
                remaining -= copied;
                if (remaining == 0)
                {
                    done.notify_all();
                }
            }
        }

        void Run()
        {
            uint64_t seen = 0;
            for (;;)
            {
                {
                    std::unique_lock<std::mutex> lock(mutex);
                    wake.wait(lock, [&] { return stopping || generation != seen; });
                    if (stopping)
                    {
                        return;
                    }
                    seen = generation;
                }
                Drain(); // `chunks` is stable until the caller has seen remaining == 0, which needs every pulled chunk finished
            }
        }

        std::vector<std::thread> workers;
        std::mutex mutex, callerMutex;
        std::condition_variable wake, done;
        std::vector<RowCopy> chunks;
        std::atomic<int> next{ 0 };
        int remaining = 0;
        uint64_t generation = 0;
        bool stopping = false;
    };
}

static void CopyRows(uint8_t* target, int64_t targetStride, const uint8_t* source, int64_t sourceStride, int64_t payload, int rows)
{
    const RowCopy one{ target, targetStride, source, sourceStride, payload, rows };
    CopyPool::Instance().Copy(&one, 1);
}

// Waits for the slot's stream work (its device buffers are free again after this); what it owes the caller stays owed.
static int WaitSlot(avifgpu_context* ctx, int slot)
{
    avifgpu_context::SlotState& state = ctx->slots[slot];
    if (!state.busy)
    {
        return AVIFGPU_OK;
    }
    const int status = ctx->Cuda(cudaEventSynchronize(ctx->sliceDone[slot]), "cudaEventSynchronize");
    if (status != AVIFGPU_OK)
    {
        state.owed.clear();
    }
    state.busy = false;
    return status;
}

// Pays what a waited-for slot owes the caller: the copies out of its pinned bounce buffers.
static void PayOwed(avifgpu_context* ctx, int slot)
{
    avifgpu_context::SlotState& state = ctx->slots[slot];
    if (!state.owed.empty())
    {
        RowCopy batch[AVIFGPU_MAX_PLANES + 1];
        int count = 0;
        for (const avifgpu_context::HostCopy& c : state.owed)
        {
            if (count == AVIFGPU_MAX_PLANES + 1)
            {
                CopyPool::Instance().Copy(batch, count);
                count = 0;
            }
            batch[count++] = RowCopy{ c.target, c.targetStride, c.source, c.sourceStride, c.payload, c.rows };
        }
        CopyPool::Instance().Copy(batch, count); // all planes of the slice share the pool's threads
    }
    state.owed.clear();
}

static int RetireSlot(avifgpu_context* ctx, int slot)
{
    const int status = WaitSlot(ctx, slot);
    if (status == AVIFGPU_OK)
    {
        PayOwed(ctx, slot);
    }
    return status;
}

// Retires, oldest first, every slot issued by a call with ticket <= `ticket`.
static int RetireThrough(avifgpu_context* ctx, int64_t ticket)
{
    int result = AVIFGPU_OK;
    for (int i = 0; i < kPipelineStreams; ++i)
    {
        const int slot = (ctx->nextSlot + i) % kPipelineStreams; // nextSlot is the oldest
        if ((ctx->slots[slot].busy || !ctx->slots[slot].owed.empty()) && ctx->slots[slot].ticket <= ticket)
        {
            const int status = RetireSlot(ctx, slot);
            if (result == AVIFGPU_OK) result = status;
        }
    }
    return result;
}

// A failure in the middle of a call: nothing of this context may still be writing into caller memory on return.
static int AbandonCall(avifgpu_context* ctx, int status)
{
    for (int i = 0; i < kPipelineStreams; ++i)
    {
        cudaStreamSynchronize(ctx->streams[i]);
        ctx->slots[i].owed.clear();
        ctx->slots[i].busy = false;
    }
    cudaGetLastError();
    return status;
}

static int EncodeRowsHost(avifgpu_context* ctx, const avifgpu_encode_desc* desc, const void* host_rows, int64_t row_stride_bytes, int32_t y0,
                          int32_t nrows, const avifgpu_planes* dst, bool wait, int64_t* out_ticket)
{
    if (ctx == nullptr)
    {
        return AVIFGPU_ERR_BAD_PARAM;
    }
    std::string error;
    int status = ValidateEncodeDesc(desc, &error);
    if (status != AVIFGPU_OK)
    {
        return ctx->Fail(status, error);
    }
    if (dst == nullptr || (host_rows == nullptr && nrows > 0 && desc->width > 0))
    {
        return ctx->Fail(AVIFGPU_ERR_BAD_PARAM, "NULL buffer");
    }
    EncodeParams base;
    FillEncodeParams(*desc, &base);
    status = CheckBlock(ctx, desc->height, base.ys, y0, nrows);
    if (status != AVIFGPU_OK)
    {
        return status;
    }
    const int64_t ticket = ++ctx->lastTicket;
    if (out_ticket != nullptr)
    {
        *out_ticket = ticket;
    }
    DeviceGuard guard(ctx->device);
    if (nrows == 0 || desc->width == 0)
    {
        return wait ? RetireThrough(ctx, ticket) : AVIFGPU_OK;
    }
    PlaneGeometry geometry[AVIFGPU_MAX_PLANES];
    bool planePinned[AVIFGPU_MAX_PLANES] = {};
    for (int k = 0; k < AVIFGPU_MAX_PLANES; ++k)
    {
        geometry[k] = EncodePlaneGeometry(*desc, k);
        if (geometry[k].present && dst->data[k] == nullptr)
        {
            return ctx->Fail(AVIFGPU_ERR_BAD_PARAM, "missing destination plane");
        }
        planePinned[k] = geometry[k].present && IsPinned(dst->data[k]);
    }

    base.smCount = ctx->smCount;
    if (CurveTable* table = ctx->CurveTableFor(*desc, static_cast<int64_t>(desc->width) * nrows, false))
    {
        base.curveTable = table->valid ? &table->view : nullptr;
    }
    base.gray16Lut = ctx->Gray16LutFor(*desc);
    base.verifiedPremultiply = ctx->VerifiedPremultiply(*desc);
    const int64_t rowPayload = static_cast<int64_t>(desc->width) * EncodeHostColBytes(*desc);
    const int64_t deviceRowStride = (rowPayload + 255) & ~255ll;
    const bool rowsPinned = IsPinned(host_rows);
    const int sliceRows = SliceRows(nrows, rowPayload);

    // The rows handed to the PREVIOUS asynchronous call may be overwritten once this call returns.  Their last H2D is
    // waited for at the END of this call, after this call's own copies are queued behind it, so the link never idles
    // at a call boundary.
    const bool waitForPreviousRows = ctx->previousCallRowsPending;
    const int previousRowsEvent = static_cast<int>((ctx->asyncEncodeCalls - 1) & 1);
    ctx->previousCallRowsPending = false;
    bool recordedCallRows = false;

    for (int begin = 0; begin < nrows; begin += sliceRows)
    {
        const int rows = std::min(sliceRows, nrows - begin);
        const int slot = ctx->nextSlot;
        cudaStream_t stream = ctx->streams[slot];
        // The slot's previous slice: wait for the GPU, but pay its bounce copies only after this slice's H2D and kernel are
        // queued -- the host then copies while the link and the SMs work (its D2H, which reuses the bounce buffers, comes last).
        if ((status = WaitSlot(ctx, slot)) != AVIFGPU_OK) return AbandonCall(ctx, status);
        ctx->nextSlot = (slot + 1) % kPipelineStreams;

        if ((status = ctx->EnsureDevice(ctx->deviceRows[slot], static_cast<size_t>(deviceRowStride) * rows)) != AVIFGPU_OK) return AbandonCall(ctx, status);
        const uint8_t* source = static_cast<const uint8_t*>(host_rows) + static_cast<int64_t>(begin) * row_stride_bytes;
        int64_t sourceStride = row_stride_bytes;
        if (!rowsPinned)
        {
            if ((status = ctx->EnsurePinned(ctx->pinnedRows[slot], static_cast<size_t>(rowPayload) * rows)) != AVIFGPU_OK) return AbandonCall(ctx, status);
            uint8_t* bounce = static_cast<uint8_t*>(ctx->pinnedRows[slot].ptr);
            CopyRows(bounce, rowPayload, source, row_stride_bytes, rowPayload, rows);
            source = bounce;
            sourceStride = rowPayload;
        }
        if ((status = ctx->Cuda(cudaMemcpy2DAsync(ctx->deviceRows[slot].ptr, static_cast<size_t>(deviceRowStride), source,
                                                  static_cast<size_t>(sourceStride), static_cast<size_t>(rowPayload),
                                                  static_cast<size_t>(rows), cudaMemcpyHostToDevice, stream),
                                "H2D rows")) != AVIFGPU_OK) return AbandonCall(ctx, status);
        if ((status = ctx->Cuda(cudaEventRecord(ctx->rowsConsumed[slot], stream), "cudaEventRecord")) != AVIFGPU_OK) return AbandonCall(ctx, status);
        if (!wait && rowsPinned && begin + sliceRows >= nrows)
        {
            // the caller's own memory is on the wire until this H2D, the last of the call: the NEXT call waits for it before it returns
            if ((status = ctx->Cuda(cudaEventRecord(ctx->callRowsConsumed[ctx->asyncEncodeCalls & 1], stream), "cudaEventRecord")) != AVIFGPU_OK) return AbandonCall(ctx, status);
            recordedCallRows = true;
        }

        EncodeParams p = base;
        p.rows = ctx->deviceRows[slot].ptr;
        p.rowStride = deviceRowStride;
        p.rowCount = rows;
        int64_t planeStride[AVIFGPU_MAX_PLANES] = {};
        int planeRows[AVIFGPU_MAX_PLANES] = {};
        int64_t planePayload[AVIFGPU_MAX_PLANES] = {};
        for (int k = 0; k < AVIFGPU_MAX_PLANES; ++k)
        {
            const PlaneGeometry& g = geometry[k];
            if (!g.present)
            {
                continue;
            }
            planePayload[k] = static_cast<int64_t>(g.widthSamples) * g.bytesPerSample;
            planeStride[k] = (planePayload[k] + 255) & ~255ll;
            planeRows[k] = (rows + g.ys) >> g.ys;
            if ((status = ctx->EnsureDevice(ctx->devicePlanes[slot][k], static_cast<size_t>(planeStride[k]) * planeRows[k])) != AVIFGPU_OK) return AbandonCall(ctx, status);
            p.plane[k] = ctx->devicePlanes[slot][k].ptr;
            p.planeStride[k] = planeStride[k];
        }
        const int launched = LaunchEncode(p, desc->host_depth, stream);
        if (launched < 0)
        {
            return AbandonCall(ctx, ctx->LaunchFailed(launched, "encode kernel launch"));
        }
        ctx->launches += launched;

        PayOwed(ctx, slot); // the previous slice's planes leave the bounce buffers now
        avifgpu_context::SlotState& state = ctx->slots[slot];
        for (int k = 0; k < AVIFGPU_MAX_PLANES; ++k)
        {
            const PlaneGeometry& g = geometry[k];
            if (!g.present)
            {
                continue;
            }
            uint8_t* target = static_cast<uint8_t*>(dst->data[k]) + static_cast<int64_t>((y0 + begin) >> g.ys) * dst->stride[k];
            int64_t targetStride = dst->stride[k];
            if (!planePinned[k])
            {
                // pageable plane (libheif's): land in pinned memory now, copy across when the slot retires
                if ((status = ctx->EnsurePinned(ctx->pinnedPlanes[slot][k], static_cast<size_t>(planePayload[k]) * planeRows[k])) != AVIFGPU_OK) return AbandonCall(ctx, status);
                uint8_t* bounce = static_cast<uint8_t*>(ctx->pinnedPlanes[slot][k].ptr);
                state.owed.push_back(avifgpu_context::HostCopy{ target, dst->stride[k], bounce, planePayload[k], planePayload[k], planeRows[k] });
                target = bounce;
                targetStride = planePayload[k];
            }
            if ((status = ctx->Cuda(cudaMemcpy2DAsync(target, static_cast<size_t>(targetStride), p.plane[k],
                                                      static_cast<size_t>(planeStride[k]), static_cast<size_t>(planePayload[k]),
                                                      static_cast<size_t>(planeRows[k]), cudaMemcpyDeviceToHost, stream),
                                    "D2H plane")) != AVIFGPU_OK) return AbandonCall(ctx, status);
        }
        if ((status = ctx->Cuda(cudaEventRecord(ctx->sliceDone[slot], stream), "cudaEventRecord")) != AVIFGPU_OK) return AbandonCall(ctx, status);
        state.busy = true;
        state.ticket = ticket;
    }
    if (waitForPreviousRows)
    {
        if ((status = ctx->Cuda(cudaEventSynchronize(ctx->callRowsConsumed[previousRowsEvent]), "cudaEventSynchronize")) != AVIFGPU_OK) return AbandonCall(ctx, status);
    }
    if (wait)
    {
        status = RetireThrough(ctx, ticket);
        return status == AVIFGPU_OK ? AVIFGPU_OK : AbandonCall(ctx, status);
    }
    if (recordedCallRows)
    {
        ctx->asyncEncodeCalls += 1;
        ctx->previousCallRowsPending = true;
    }
    return AVIFGPU_OK;
}

static int DecodeRowsHost(avifgpu_context* ctx, const avifgpu_decode_desc* desc, const avifgpu_planes* src, int32_t y0, int32_t nrows,
                          void* host_rows, int64_t row_stride_bytes, bool wait, int64_t* out_ticket)
{
    if (ctx == nullptr)
    {
        return AVIFGPU_ERR_BAD_PARAM;
    }
    std::string error;
    int32_t transfer;
    int status = ValidateDecodeDesc(desc, &transfer, &error);
    if (status != AVIFGPU_OK)
    {
        return ctx->Fail(status, error);
    }
    if (src == nullptr || (host_rows == nullptr && nrows > 0 && desc->width > 0))
    {
        return ctx->Fail(AVIFGPU_ERR_BAD_PARAM, "NULL buffer");
    }
    DecodeParams base;
    if (!FillDecodeParams(*desc, transfer, &base, &error))
    {
        return ctx->Fail(AVIFGPU_ERR_UNSUPPORTED, error);
    }
    if (y0 < 0 || nrows < 0 || y0 > desc->height || nrows > desc->height - y0)
    {
        return ctx->Fail(AVIFGPU_ERR_BAD_PARAM, "row block outside the image");
    }
    const int64_t ticket = ++ctx->lastTicket;
    if (out_ticket != nullptr)
    {
        *out_ticket = ticket;
    }
    DeviceGuard guard(ctx->device);
    if (nrows == 0 || desc->width == 0)
    {
        return wait ? RetireThrough(ctx, ticket) : AVIFGPU_OK;
    }
    PlaneGeometry geometry[AVIFGPU_MAX_PLANES];
    bool planePinned[AVIFGPU_MAX_PLANES] = {};
    for (int k = 0; k < AVIFGPU_MAX_PLANES; ++k)
    {
        geometry[k] = DecodePlaneGeometry(*desc, k);
        if (geometry[k].present && src->data[k] == nullptr)
        {
            return ctx->Fail(AVIFGPU_ERR_BAD_PARAM, "missing source plane");
        }
        planePinned[k] = geometry[k].present && IsPinned(src->data[k]);
    }

    base.verifiedHlgDivisions = (desc->host_depth == 32 && transfer == AVIFGPU_TRANSFER_HLG) ? ctx->VerifiedHlgDivisions() : 0;
    base.verifiedGreenDivision = ctx->VerifiedGreenDivision(base);
    base.verifiedPqRatio = (desc->host_depth == 32 && transfer == AVIFGPU_TRANSFER_PQ && desc->colorspace == AVIFGPU_COLORSPACE_YCBCR) ? ctx->VerifiedPqRatio() : 0;
    const int64_t rowPayload = static_cast<int64_t>(desc->width) * DecodeHostColBytes(*desc);
    const int64_t deviceRowStride = (rowPayload + 255) & ~255ll;
    const int sliceRows = SliceRows(nrows, rowPayload);
    const bool rowsPinned = IsPinned(host_rows);

    for (int begin = 0; begin < nrows; begin += sliceRows)
    {
        const int rows = std::min(sliceRows, nrows - begin);
        const int slot = ctx->nextSlot;
        cudaStream_t stream = ctx->streams[slot];
        if ((status = RetireSlot(ctx, slot)) != AVIFGPU_OK) return AbandonCall(ctx, status);
        ctx->nextSlot = (slot + 1) % kPipelineStreams;

        const int yFirst = y0 + begin;
        DecodeParams p = base;
        p.rowCount = rows;
        p.yPhase = yFirst & p.ys;
        p.smCount = ctx->smCount;
        // pageable planes (libheif's) go through the slot's pinned buffers: every plane of the slice in ONE batch for the copy
        // pool (three separate batches cost three wake-ups and waits per slice, ~0.5 ms, ahead of anything the GPU could do)
        struct PlaneStage
        {
            const uint8_t* source;
            int64_t sourceStride, payload, stride;
            int planeRows;
        } stage[AVIFGPU_MAX_PLANES] = {};
        RowCopy bounceBatch[AVIFGPU_MAX_PLANES];
        int bounceCount = 0;
        for (int k = 0; k < AVIFGPU_MAX_PLANES; ++k)
        {
            const PlaneGeometry& g = geometry[k];
            if (!g.present)
            {
                continue;
            }
            const int firstRow = yFirst >> g.ys;
            const int lastRow = (yFirst + rows - 1) >> g.ys;
            PlaneStage& st = stage[k];
            st.planeRows = lastRow - firstRow + 1;
            st.payload = static_cast<int64_t>(g.widthSamples) * g.bytesPerSample;
            st.stride = (st.payload + 255) & ~255ll;
            if ((status = ctx->EnsureDevice(ctx->devicePlanes[slot][k], static_cast<size_t>(st.stride) * st.planeRows)) != AVIFGPU_OK) return AbandonCall(ctx, status);
            st.source = static_cast<const uint8_t*>(src->data[k]) + static_cast<int64_t>(firstRow) * src->stride[k];
            st.sourceStride = src->stride[k];
            if (!planePinned[k])
            {
                if ((status = ctx->EnsurePinned(ctx->pinnedPlanes[slot][k], static_cast<size_t>(st.payload) * st.planeRows)) != AVIFGPU_OK) return AbandonCall(ctx, status);
                uint8_t* bounce = static_cast<uint8_t*>(ctx->pinnedPlanes[slot][k].ptr);
                bounceBatch[bounceCount++] = RowCopy{ bounce, st.payload, st.source, st.sourceStride, st.payload, st.planeRows };
                st.source = bounce;
                st.sourceStride = st.payload;
            }
        }
        if (bounceCount > 0)
        {
            CopyPool::Instance().Copy(bounceBatch, bounceCount);
        }
        for (int k = 0; k < AVIFGPU_MAX_PLANES; ++k)
        {
            if (!geometry[k].present)
            {
                continue;
            }
            const PlaneStage& st = stage[k];
            if ((status = ctx->Cuda(cudaMemcpy2DAsync(ctx->devicePlanes[slot][k].ptr, static_cast<size_t>(st.stride), st.source,
                                                      static_cast<size_t>(st.sourceStride), static_cast<size_t>(st.payload),
                                                      static_cast<size_t>(st.planeRows), cudaMemcpyHostToDevice, stream),
                                    "H2D plane")) != AVIFGPU_OK) return AbandonCall(ctx, status);
            p.plane[k] = ctx->devicePlanes[slot][k].ptr;
            p.planeStride[k] = st.stride;
        }
        if ((status = ctx->EnsureDevice(ctx->deviceRows[slot], static_cast<size_t>(deviceRowStride) * rows)) != AVIFGPU_OK) return AbandonCall(ctx, status);
        p.rows = ctx->deviceRows[slot].ptr;
        p.rowStride = deviceRowStride;
        const int launched = LaunchDecode(p, stream);
        if (launched < 0)
        {
            return AbandonCall(ctx, ctx->LaunchFailed(launched, "decode kernel launch"));
        }
        ctx->launches += launched;

        avifgpu_context::SlotState& state = ctx->slots[slot];
        uint8_t* target = static_cast<uint8_t*>(host_rows) + static_cast<int64_t>(begin) * row_stride_bytes;
        int64_t targetStride = row_stride_bytes;
        if (!rowsPinned)
        {
            if ((status = ctx->EnsurePinned(ctx->pinnedRows[slot], static_cast<size_t>(rowPayload) * rows)) != AVIFGPU_OK) return AbandonCall(ctx, status);
            uint8_t* bounce = static_cast<uint8_t*>(ctx->pinnedRows[slot].ptr);
            state.owed.push_back(avifgpu_context::HostCopy{ target, row_stride_bytes, bounce, rowPayload, rowPayload, rows });
            target = bounce;
            targetStride = rowPayload;
        }
        if ((status = ctx->Cuda(cudaMemcpy2DAsync(target, static_cast<size_t>(targetStride), ctx->deviceRows[slot].ptr,
                                                  static_cast<size_t>(deviceRowStride), static_cast<size_t>(rowPayload),
                                                  static_cast<size_t>(rows), cudaMemcpyDeviceToHost, stream),
                                "D2H rows")) != AVIFGPU_OK) return AbandonCall(ctx, status);
        if ((status = ctx->Cuda(cudaEventRecord(ctx->sliceDone[slot], stream), "cudaEventRecord")) != AVIFGPU_OK) return AbandonCall(ctx, status);
        state.busy = true;
        state.ticket = ticket;
    }
    if (wait)
    {
        status = RetireThrough(ctx, ticket);
        return status == AVIFGPU_OK ? AVIFGPU_OK : AbandonCall(ctx, status);
    }
    return AVIFGPU_OK;
}

extern "C" {

AVIFGPU_EXPORT int avifgpu_encode_rows(avifgpu_context* ctx, const avifgpu_encode_desc* desc, const void* host_rows,
                                       int64_t row_stride_bytes, int32_t y0, int32_t nrows, const avifgpu_planes* dst)
{
    return EncodeRowsHost(ctx, desc, host_rows, row_stride_bytes, y0, nrows, dst, true, nullptr);
}

AVIFGPU_EXPORT int avifgpu_decode_rows(avifgpu_context* ctx, const avifgpu_decode_desc* desc, const avifgpu_planes* src,
                                       int32_t y0, int32_t nrows, void* host_rows, int64_t row_stride_bytes)
{
    return DecodeRowsHost(ctx, desc, src, y0, nrows, host_rows, row_stride_bytes, true, nullptr);
}

AVIFGPU_EXPORT int avifgpu_encode_rows_async(avifgpu_context* ctx, const avifgpu_encode_desc* desc, const void* host_rows,
                                             int64_t row_stride_bytes, int32_t y0, int32_t nrows, const avifgpu_planes* dst,
                                             int64_t* out_ticket)
{
    return EncodeRowsHost(ctx, desc, host_rows, row_stride_bytes, y0, nrows, dst, false, out_ticket);
}

AVIFGPU_EXPORT int avifgpu_decode_rows_async(avifgpu_context* ctx, const avifgpu_decode_desc* desc, const avifgpu_planes* src,
                                             int32_t y0, int32_t nrows, void* host_rows, int64_t row_stride_bytes, int64_t* out_ticket)
{
    return DecodeRowsHost(ctx, desc, src, y0, nrows, host_rows, row_stride_bytes, false, out_ticket);
}

AVIFGPU_EXPORT int avifgpu_wait(avifgpu_context* ctx, int64_t ticket)
{
    if (ctx == nullptr)
    {
        return AVIFGPU_ERR_BAD_PARAM;
    }
    DeviceGuard guard(ctx->device);
    if (ticket <= 0 || ticket >= ctx->lastTicket)
    {
        ticket = ctx->lastTicket;
        ctx->previousCallRowsPending = false; // everything is about to be drained
    }
    const int status = RetireThrough(ctx, ticket);
    return status == AVIFGPU_OK ? AVIFGPU_OK : AbandonCall(ctx, status);
}

// ---- several GPUs of one box -----------------------------------------------------------------------------------------

} // extern "C"

struct avifgpu_shard_group
{
    std::vector<avifgpu_context*> members;
    std::vector<int> devices;
    std::vector<uint8_t> peer; // peer[from * n + to]
    std::string lastError;

    int Fail(int status, const std::string& message)
    {
        lastError = message;
        return status;
    }

    // Runs work(r) for every member on its own host thread (each drives its own device and PCIe link); returns the
    // first failure and keeps its message.
    template <typename Work>
    int ForEachMember(Work work)
    {
        const int n = static_cast<int>(members.size());
        std::vector<int> status(n, AVIFGPU_OK);
        std::vector<std::thread> threads;
        threads.reserve(n > 0 ? n - 1 : 0);
        for (int r = 1; r < n; ++r)
        {
            threads.emplace_back([&, r] { status[r] = work(r); });
        }
        if (n > 0)
        {
            status[0] = work(0);
        }
        for (std::thread& t : threads)
        {
            t.join();
        }
        for (int r = 0; r < n; ++r)
        {
            if (status[r] != AVIFGPU_OK)
            {
                return Fail(status[r], "member " + std::to_string(r) + " (device " + std::to_string(devices[r]) + "): " + members[r]->lastError);
            }
        }
        return AVIFGPU_OK;
    }
};

static void RowBlocks(int y0, int nrows, int parts, int32_t* outY0, int32_t* outRows)
{
    // inner boundaries at even image rows: a 2x2 chroma site never straddles two blocks (4:2:0), and the same split
    // serves every other layout
    int previous = y0;
    for (int i = 0; i < parts; ++i)
    {
        int end = (i == parts - 1) ? y0 + nrows : y0 + static_cast<int>((static_cast<int64_t>(nrows) * (i + 1)) / parts);
        if (i != parts - 1)
        {
            end &= ~1;
        }
        end = std::min(std::max(end, previous), y0 + nrows);
        outY0[i] = previous;
        outRows[i] = end - previous;
        previous = end;
    }
}

extern "C" {

AVIFGPU_EXPORT int avifgpu_shard_row_blocks(int32_t y0, int32_t nrows, int32_t parts, int32_t* out_y0, int32_t* out_nrows)
{
    if (parts <= 0 || nrows < 0 || y0 < 0 || out_y0 == nullptr || out_nrows == nullptr)
    {
        return AVIFGPU_ERR_BAD_PARAM;
    }
    RowBlocks(y0, nrows, parts, out_y0, out_nrows);
    return AVIFGPU_OK;
}

AVIFGPU_EXPORT int avifgpu_shard_group_create(const int32_t* device_ordinals, int32_t count, avifgpu_shard_group** out_group)
{
    if (out_group == nullptr)
    {
        g_creationError = "out_group is NULL";
        return AVIFGPU_ERR_BAD_PARAM;
    }
    *out_group = nullptr;
    if (device_ordinals == nullptr || count <= 0 || count > 64)
    {
        g_creationError = "a shard group needs 1..64 device ordinals";
        return AVIFGPU_ERR_BAD_PARAM;
    }
    for (int i = 0; i < count; ++i)
    {
        for (int j = 0; j < i; ++j)
        {
            if (device_ordinals[i] == device_ordinals[j])
            {
                g_creationError = "device ordinals of a shard group must be distinct";
                return AVIFGPU_ERR_BAD_PARAM;
            }
        }
    }
    avifgpu_shard_group* group = new (std::nothrow) avifgpu_shard_group();
    if (group == nullptr)
    {
        g_creationError = "out of host memory";
        return AVIFGPU_ERR_OOM;
    }
    for (int i = 0; i < count; ++i)
    {
        avifgpu_context* ctx = nullptr;
        const int status = avifgpu_create(device_ordinals[i], &ctx);
        if (status != AVIFGPU_OK)
        {
            avifgpu_shard_group_destroy(group);
            return status; // g_creationError set by avifgpu_create
        }
        group->members.push_back(ctx);
        group->devices.push_back(device_ordinals[i]);
    }
    group->peer.assign(static_cast<size_t>(count) * count, 0);
    for (int from = 0; from < count; ++from)
    {
        DeviceGuard guard(group->devices[from]);
        for (int to = 0; to < count; ++to)
        {
            if (from == to)
            {
                group->peer[from * count + to] = 1;
                continue;
            }
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, group->devices[from], group->devices[to]) != cudaSuccess || !can)
            {
                cudaGetLastError();
                continue;
            }
            const cudaError_t e = cudaDeviceEnablePeerAccess(group->devices[to], 0);
            if (e == cudaSuccess || e == cudaErrorPeerAccessAlreadyEnabled)
            {
                group->peer[from * count + to] = 1;
            }
            cudaGetLastError();
        }
    }
    *out_group = group;
    return AVIFGPU_OK;
}

AVIFGPU_EXPORT void avifgpu_shard_group_destroy(avifgpu_shard_group* group)
{
    if (group == nullptr)
    {
        return;
    }
    for (avifgpu_context* ctx : group->members)
    {
        avifgpu_destroy(ctx);
    }
    delete group;
}

AVIFGPU_EXPORT int32_t avifgpu_shard_group_size(const avifgpu_shard_group* group) { return group ? static_cast<int32_t>(group->members.size()) : 0; }

AVIFGPU_EXPORT avifgpu_context* avifgpu_shard_group_context(avifgpu_shard_group* group, int32_t index)
{
    return (group != nullptr && index >= 0 && index < static_cast<int32_t>(group->members.size())) ? group->members[index] : nullptr;
}

AVIFGPU_EXPORT int avifgpu_shard_group_peer_access(const avifgpu_shard_group* group, int32_t from, int32_t to)
{
    const int n = group ? static_cast<int>(group->members.size()) : 0;
    return (from >= 0 && to >= 0 && from < n && to < n) ? group->peer[from * n + to] : 0;
}

AVIFGPU_EXPORT const char* avifgpu_shard_group_last_error(const avifgpu_shard_group* group)
{
    return group ? group->lastError.c_str() : g_creationError.c_str();
}

AVIFGPU_EXPORT int avifgpu_shard_group_prepare_encode(avifgpu_shard_group* group, const avifgpu_encode_desc* desc)
{
    if (group == nullptr)
    {
        return AVIFGPU_ERR_BAD_PARAM;
    }
    return group->ForEachMember([&](int r) { return avifgpu_prepare_encode(group->members[r], desc, nullptr); });
}

AVIFGPU_EXPORT int avifgpu_shard_group_synchronize(avifgpu_shard_group* group)
{
    if (group == nullptr)
    {
        return AVIFGPU_ERR_BAD_PARAM;
    }
    int result = AVIFGPU_OK;
    for (size_t r = 0; r < group->members.size(); ++r)
    {
        const int status = avifgpu_synchronize(group->members[r]);
        if (status != AVIFGPU_OK && result == AVIFGPU_OK)
        {
            result = group->Fail(status, "member " + std::to_string(r) + ": " + group->members[r]->lastError);
        }
    }
    return result;
}

AVIFGPU_EXPORT int avifgpu_encode_rows_sharded(avifgpu_shard_group* group, const avifgpu_encode_desc* desc, const void* host_rows,
                                               int64_t row_stride_bytes, int32_t y0, int32_t nrows, const avifgpu_planes* dst)
{
    if (group == nullptr)
    {
        return AVIFGPU_ERR_BAD_PARAM;
    }
    const int n = static_cast<int>(group->members.size());
    if (nrows < 0 || y0 < 0)
    {
        return group->Fail(AVIFGPU_ERR_BAD_PARAM, "row block outside the image");
    }
    std::vector<int32_t> blockY0(n), blockRows(n);
    RowBlocks(y0, nrows, n, blockY0.data(), blockRows.data());
    return group->ForEachMember([&](int r) -> int
    {
        if (blockRows[r] == 0 && !(r == 0 && nrows == 0))
        {
            return AVIFGPU_OK;
        }
        const uint8_t* rows = host_rows ? static_cast<const uint8_t*>(host_rows) + static_cast<int64_t>(blockY0[r] - y0) * row_stride_bytes : nullptr;
        return avifgpu_encode_rows(group->members[r], desc, rows, row_stride_bytes, blockY0[r], blockRows[r], dst);
    });
}

AVIFGPU_EXPORT int avifgpu_decode_rows_sharded(avifgpu_shard_group* group, const avifgpu_decode_desc* desc, const avifgpu_planes* src,
                                               int32_t y0, int32_t nrows, void* host_rows, int64_t row_stride_bytes)
{
    if (group == nullptr)
    {
        return AVIFGPU_ERR_BAD_PARAM;
    }
    const int n = static_cast<int>(group->members.size());
    if (nrows < 0 || y0 < 0)
    {
        return group->Fail(AVIFGPU_ERR_BAD_PARAM, "row block outside the image");
    }
    std::vector<int32_t> blockY0(n), blockRows(n);
    RowBlocks(y0, nrows, n, blockY0.data(), blockRows.data());
    return group->ForEachMember([&](int r) -> int
    {
        if (blockRows[r] == 0 && !(r == 0 && nrows == 0))
        {
            return AVIFGPU_OK;
        }
        uint8_t* rows = host_rows ? static_cast<uint8_t*>(host_rows) + static_cast<int64_t>(blockY0[r] - y0) * row_stride_bytes : nullptr;
        return avifgpu_decode_rows(group->members[r], desc, src, blockY0[r], blockRows[r], rows, row_stride_bytes);
    });
}

AVIFGPU_EXPORT int avifgpu_encode_rows_sharded_device(avifgpu_shard_group* group, const avifgpu_encode_desc* desc,
                                                      const void* const* device_rows, const int64_t* row_stride_bytes,
                                                      const avifgpu_planes* owner_planes, int32_t owner)
{
    if (group == nullptr)
    {
        return AVIFGPU_ERR_BAD_PARAM;
    }
    const int n = static_cast<int>(group->members.size());
    if (desc == nullptr || device_rows == nullptr || row_stride_bytes == nullptr || owner_planes == nullptr || owner < 0 || owner >= n)
    {
        return group->Fail(AVIFGPU_ERR_BAD_PARAM, "NULL argument or owner outside the group");
    }
    std::vector<int32_t> blockY0(n), blockRows(n);
    RowBlocks(0, desc->height, n, blockY0.data(), blockRows.data());
    for (int r = 0; r < n; ++r)
    {
        if (blockRows[r] > 0 && !group->peer[r * n + owner])
        {
            return group->Fail(AVIFGPU_ERR_UNSUPPORTED, "member " + std::to_string(r) + " has no peer access to the owner's memory");
        }
    }
    // Launches are asynchronous: a plain loop enqueues all of them in microseconds, each on its member's own stream.
    for (int r = 0; r < n; ++r)
    {
        if (blockRows[r] == 0)
        {
            continue;
        }
        avifgpu_context* ctx = group->members[r];
        const int status = avifgpu_encode_rows_device(ctx, desc, device_rows[r], row_stride_bytes[r], blockY0[r], blockRows[r], owner_planes,
                                                      ctx->streams[0]);
        if (status != AVIFGPU_OK)
        {
            return group->Fail(status, "member " + std::to_string(r) + ": " + ctx->lastError);
        }
    }
    return AVIFGPU_OK;
}

// ---- preparation ------------------------------------------------------------------------------------------------

AVIFGPU_EXPORT int avifgpu_prepare_encode(avifgpu_context* ctx, const avifgpu_encode_desc* desc, avifgpu_curve_stats* out_stats)
{
    if (ctx == nullptr)
    {
        return AVIFGPU_ERR_BAD_PARAM;
    }
    std::string error;
    const int status = ValidateEncodeDesc(desc, &error);
    if (status != AVIFGPU_OK)
    {
        return ctx->Fail(status, error);
    }
    DeviceGuard guard(ctx->device);
    CurveTable* table = ctx->CurveTableFor(*desc, 0, true);
    ctx->Gray16LutFor(*desc);
    if (out_stats != nullptr)
    {
        std::memset(out_stats, 0, sizeof(*out_stats));
        if (table != nullptr)
        {
            out_stats->applicable = 1;
            out_stats->valid = table->valid ? 1 : 0;
            out_stats->steps = table->stats.steps;
            out_stats->bands = table->stats.bands;
            out_stats->widest_band_ulps = table->stats.widestBand;
            out_stats->bucket_count = table->view.bucketCount;
            out_stats->swept_inputs = table->stats.sweptInputs;
            out_stats->in_band_inputs = table->stats.inBandInputs;
            out_stats->verify_mismatches = table->stats.verifyMismatches;
            out_stats->build_ms = table->stats.buildMilliseconds;
        }
    }
    if (table != nullptr && !table->valid)
    {
        ctx->lastError = "step table not used (generic exact kernel serves this configuration): " + table->error;
    }
    return AVIFGPU_OK;
}

AVIFGPU_EXPORT int avifgpu_set_table_autobuild(avifgpu_context* ctx, int64_t pixels)
{
    if (ctx == nullptr)
    {
        return AVIFGPU_ERR_BAD_PARAM;
    }
    ctx->tableAutoBuildPixels = pixels;
    return AVIFGPU_OK;
}

// ---- primitives -------------------------------------------------------------------------------------------------

AVIFGPU_EXPORT int avifgpu_transfer_f32(avifgpu_context* ctx, int32_t function, float param, const float* in, float* out, size_t n)
{
    if (ctx == nullptr)
    {
        return AVIFGPU_ERR_BAD_PARAM;
    }
    if (function < AVIFGPU_FN_LINEAR_TO_PQ || function > AVIFGPU_FN_LOGF)
    {
        return ctx->Fail(AVIFGPU_ERR_BAD_PARAM, "unknown function");
    }
    if (n == 0)
    {
        return AVIFGPU_OK;
    }
    if (in == nullptr || out == nullptr)
    {
        return ctx->Fail(AVIFGPU_ERR_BAD_PARAM, "NULL buffer");
    }
    DeviceGuard guard(ctx->device);
    int status;
    const size_t bytes = n * sizeof(float);
    if ((status = ctx->EnsureDevice(ctx->transferScratch[0], bytes)) != AVIFGPU_OK) return status;
    if ((status = ctx->EnsureDevice(ctx->transferScratch[1], bytes)) != AVIFGPU_OK) return status;
    cudaStream_t stream = ctx->streams[0];
    if ((status = ctx->Cuda(cudaMemcpyAsync(ctx->transferScratch[0].ptr, in, bytes, cudaMemcpyHostToDevice, stream), "H2D")) != AVIFGPU_OK) return status;
    const int launched = LaunchTransfer(function, param, static_cast<const float*>(ctx->transferScratch[0].ptr),
                                        static_cast<float*>(ctx->transferScratch[1].ptr), n, stream);
    if (launched < 0)
    {
        return ctx->LaunchFailed(launched, "transfer kernel launch");
    }
    ctx->launches += launched;
    if ((status = ctx->Cuda(cudaMemcpyAsync(out, ctx->transferScratch[1].ptr, bytes, cudaMemcpyDeviceToHost, stream), "D2H")) != AVIFGPU_OK) return status;
    return ctx->Cuda(cudaStreamSynchronize(stream), "cudaStreamSynchronize");
}

AVIFGPU_EXPORT int avifgpu_hlg_ootf_f32(avifgpu_context* ctx, int32_t inverse, int32_t color_primaries, float display_gamma,
                                        float nominal_peak_nits, const float* rgb_in, float* rgb_out, size_t pixels)
{
    if (ctx == nullptr)
    {
        return AVIFGPU_ERR_BAD_PARAM;
    }
    float luma[3];
    if (!GetHlgLumaCoefficients(color_primaries, luma))
    {
        return ctx->Fail(AVIFGPU_ERR_UNSUPPORTED, "no HLG luma coefficients for these colour primaries");
    }
    if (pixels == 0)
    {
        return AVIFGPU_OK;
    }
    if (rgb_in == nullptr || rgb_out == nullptr)
    {
        return ctx->Fail(AVIFGPU_ERR_BAD_PARAM, "NULL buffer");
    }
    DeviceGuard guard(ctx->device);
    int status;
    const size_t bytes = pixels * 3 * sizeof(float);
    if ((status = ctx->EnsureDevice(ctx->transferScratch[0], bytes)) != AVIFGPU_OK) return status;
    if ((status = ctx->EnsureDevice(ctx->transferScratch[1], bytes)) != AVIFGPU_OK) return status;
    cudaStream_t stream = ctx->streams[0];
    if ((status = ctx->Cuda(cudaMemcpyAsync(ctx->transferScratch[0].ptr, rgb_in, bytes, cudaMemcpyHostToDevice, stream), "H2D")) != AVIFGPU_OK) return status;
    const int launched = LaunchHlgOotf(inverse != 0, luma, display_gamma, nominal_peak_nits, static_cast<const float*>(ctx->transferScratch[0].ptr),
                                       static_cast<float*>(ctx->transferScratch[1].ptr), pixels, stream);
    if (launched < 0)
    {
        return ctx->LaunchFailed(launched, "OOTF kernel launch");
    }
    ctx->launches += launched;
    if ((status = ctx->Cuda(cudaMemcpyAsync(rgb_out, ctx->transferScratch[1].ptr, bytes, cudaMemcpyDeviceToHost, stream), "D2H")) != AVIFGPU_OK) return status;
    return ctx->Cuda(cudaStreamSynchronize(stream), "cudaStreamSynchronize");
}

} // extern "C"
