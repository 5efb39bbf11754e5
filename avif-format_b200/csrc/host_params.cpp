// host_params.cpp -- see host_params.h.  Compiled by the host compiler with -ffp-contract=off: the few float
// expressions here (matrix coefficients, luminance multipliers) feed the kernels and must round exactly as the
// reference's do.
#include "host_params.h"

#include <cassert>
#include <cstring>
#include <type_traits>

namespace avifgpu
{

namespace
{
    struct PrimariesRow
    {
        int32_t code;
        float v[8]; // rX rY gX gY bX bY wX wY
    };

    // Chromaticities per H.273 colour-primaries code point as the reference tabulates them
    // (YUVCoefficiants.cpp:56-68; values are the H.273 / libavif ones, kept digit for digit because the
    // chromaticity-derived matrix is computed from them in float).
    const PrimariesRow kPrimaries[] = {
        { 1, { 0.64f, 0.33f, 0.3f, 0.6f, 0.15f, 0.06f, 0.3127f, 0.329f } },
        { 4, { 0.67f, 0.33f, 0.21f, 0.71f, 0.14f, 0.08f, 0.310f, 0.316f } },
        { 5, { 0.64f, 0.33f, 0.29f, 0.60f, 0.15f, 0.06f, 0.3127f, 0.3290f } },
        { 6, { 0.630f, 0.340f, 0.310f, 0.595f, 0.155f, 0.070f, 0.3127f, 0.3290f } },
        { 7, { 0.630f, 0.340f, 0.310f, 0.595f, 0.155f, 0.070f, 0.3127f, 0.3290f } },
        { 8, { 0.681f, 0.319f, 0.243f, 0.692f, 0.145f, 0.049f, 0.310f, 0.316f } },
        { 9, { 0.708f, 0.292f, 0.170f, 0.797f, 0.131f, 0.046f, 0.3127f, 0.3290f } },
        { 10, { 1.0f, 0.0f, 0.0f, 1.0f, 0.0f, 0.0f, 0.3333f, 0.3333f } },
        { 11, { 0.680f, 0.320f, 0.265f, 0.690f, 0.150f, 0.060f, 0.314f, 0.351f } },
        { 12, { 0.680f, 0.320f, 0.265f, 0.690f, 0.150f, 0.060f, 0.3127f, 0.3290f } },
        { 22, { 0.630f, 0.340f, 0.295f, 0.605f, 0.155f, 0.077f, 0.3127f, 0.3290f } },
    };

    struct MatrixRow
    {
        int32_t code;
        float kr;
        float kb;
    };

    // YUVCoefficiants.cpp:94-106
    const MatrixRow kMatrices[] = {
        { 1, 0.2126f, 0.0722f }, { 4, 0.30f, 0.11f },     { 5, 0.299f, 0.114f },
        { 6, 0.299f, 0.114f },   { 7, 0.212f, 0.087f },   { 9, 0.2627f, 0.0593f },
    };

    const float* LookupPrimaries(int32_t code)
    {
        for (const PrimariesRow& row : kPrimaries)
        {
            if (row.code == code)
            {
                return row.v;
            }
        }
        return kPrimaries[0].v; // YUVCoefficiants.cpp:81-82
    }

    int Fail(std::string* error, int status, const char* message)
    {
        if (error)
        {
            *error = message;
        }
        return status;
    }
}

void GetYuvCoefficients(const avifgpu_nclx* nclx, float out[3])
{
    // YUVCoefficiants.cpp:171-174: BT.601 unless the CICP says otherwise
    float kr = 0.299f;
    float kb = 0.114f;
    float kg = 1.0f - kr - kb;

    if (nclx != nullptr && nclx->present)
    {
        if (nclx->matrix_coefficients == 12)
        {
            // YUVCoefficiants.cpp:110-137 (H.273 equations 32-37), float arithmetic in the reference's association
            const float* p = LookupPrimaries(nclx->color_primaries);
            const float rX = p[0], rY = p[1], gX = p[2], gY = p[3], bX = p[4], bY = p[5], wX = p[6], wY = p[7];
            const float rZ = 1.0f - (rX + rY);
            const float gZ = 1.0f - (gX + gY);
            const float bZ = 1.0f - (bX + bY);
            const float wZ = 1.0f - (wX + wY);
            kr = (rY * (wX * (gY * bZ - bY * gZ) + wY * (bX * gZ - gX * bZ) + wZ * (gX * bY - bX * gY))) /
                 (wY * (rX * (gY * bZ - bY * gZ) + gX * (bY * rZ - rY * bZ) + bX * (rY * gZ - gY * rZ)));
            kb = (bY * (wX * (rY * gZ - gY * rZ) + wY * (gX * rZ - rX * gZ) + wZ * (rX * gY - gX * rY))) /
                 (wY * (rX * (gY * bZ - bY * gZ) + gX * (bY * rZ - rY * bZ) + bX * (rY * gZ - gY * rZ)));
            kg = 1.0f - kr - kb;
        }
        else
        {
            for (const MatrixRow& row : kMatrices)
            {
                if (row.code == nclx->matrix_coefficients)
                {
                    kr = row.kr;
                    kb = row.kb;
                    kg = 1.0f - kr - kb;
                    break;
                }
            }
        }
    }
    out[0] = kr;
    out[1] = kg;
    out[2] = kb;
}

bool GetHlgLumaCoefficients(int32_t colorPrimaries, float out[3])
{
    switch (colorPrimaries)
    {
    case 1:
        out[0] = 0.2126f; out[1] = 0.7152f; out[2] = 0.0722f;
        return true;
    case 5:
    case 6:
        out[0] = 0.299f; out[1] = 0.587f; out[2] = 0.114f;
        return true;
    case 9:
        out[0] = 0.2627f; out[1] = 0.6780f; out[2] = 0.0593f;
        return true;
    default:
        return false;
    }
}

bool TransferFromNclx(int32_t transferCharacteristics, int32_t* outTransfer)
{
    switch (transferCharacteristics)
    {
    case 16: *outTransfer = AVIFGPU_TRANSFER_PQ; return true;
    case 18: *outTransfer = AVIFGPU_TRANSFER_HLG; return true;
    case 17: *outTransfer = AVIFGPU_TRANSFER_SMPTE428; return true;
    default: return false;
    }
}

avifpix::RangeParams MakeRangeParams(const avifgpu_nclx* nclx, int bitDepth, bool monochrome)
{
    avifpix::RangeParams r{};
    const bool hasNclx = nclx != nullptr && nclx->present;
    // YuvLookupTables.cpp:143-144: full range and BT.601 when there is no nclx
    r.fullRange = hasNclx ? (nclx->full_range_flag != 0) : 1;
    const int matrix = hasNclx ? nclx->matrix_coefficients : 6;
    r.identityMatrix = (!monochrome && matrix == 0) ? 1 : 0;
    r.maxChannel = (1 << bitDepth) - 1;
    r.maxChannelFloat = static_cast<float>(r.maxChannel);
    switch (bitDepth)
    {
    case 8: r.yLo = 16; r.yHi = 235; r.uvLo = 16; r.uvHi = 240; break;
    case 10: r.yLo = 64; r.yHi = 940; r.uvLo = 64; r.uvHi = 960; break;
    case 12: r.yLo = 256; r.yHi = 3760; r.uvLo = 256; r.uvHi = 3840; break;
    default: r.yLo = 1024; r.yHi = 60160; r.uvLo = 1024; r.uvHi = 61440; break;
    }
    return r;
}

int ValidateEncodeDesc(const avifgpu_encode_desc* d, std::string* error)
{
    if (d == nullptr || d->struct_size != sizeof(avifgpu_encode_desc)) return Fail(error, AVIFGPU_ERR_BAD_PARAM, "bad encode desc size");
    if (d->width < 0 || d->height < 0) return Fail(error, AVIFGPU_ERR_BAD_PARAM, "negative image size");
    if (d->host_depth != 8 && d->host_depth != 16 && d->host_depth != 32) return Fail(error, AVIFGPU_ERR_BAD_PARAM, "host depth must be 8, 16 or 32");
    if (d->host_channels < 1 || d->host_channels > 4) return Fail(error, AVIFGPU_ERR_BAD_PARAM, "host channels must be 1..4");
    if (d->image_bit_depth != 8 && d->image_bit_depth != 10 && d->image_bit_depth != 12) return Fail(error, AVIFGPU_ERR_BAD_PARAM, "image bit depth must be 8, 10 or 12");
    const bool expectsAlpha = d->host_channels == 2 || d->host_channels == 4;
    const bool hasAlpha = d->alpha_state != AVIFGPU_ALPHA_NONE;
    if (d->alpha_state < AVIFGPU_ALPHA_NONE || d->alpha_state > AVIFGPU_ALPHA_PREMULTIPLIED || expectsAlpha != hasAlpha)
    {
        return Fail(error, AVIFGPU_ERR_BAD_PARAM, "alpha state does not match the channel count");
    }
    if (d->host_depth == 32)
    {
        if (d->image_bit_depth == 8) return Fail(error, AVIFGPU_ERR_UNSUPPORTED, "32-bit hosts require a 10- or 12-bit image");
        // WriteHeifImage.cpp:578-588 (gray: PQ, Clip), :1079-1091 (colour: PQ, SMPTE428, Clip)
        const bool gray = d->host_channels <= 2;
        // plus, only on request, the HLG save path the reference has the functions for but never calls (avifgpu.h)
        const bool hlg = !gray && d->transfer == AVIFGPU_TRANSFER_HLG &&
                         (d->hlg_extension == AVIFGPU_HLG_OETF || d->hlg_extension == AVIFGPU_HLG_INVERSE_OOTF_THEN_OETF);
        const bool ok = d->transfer == AVIFGPU_TRANSFER_PQ || d->transfer == AVIFGPU_TRANSFER_CLIP ||
                        (!gray && d->transfer == AVIFGPU_TRANSFER_SMPTE428) || hlg;
        if (!ok) return Fail(error, AVIFGPU_ERR_UNSUPPORTED, "Unsupported color transfer function.");
        if (hlg && d->hlg_extension == AVIFGPU_HLG_INVERSE_OOTF_THEN_OETF)
        {
            float luma[3];
            if (!d->nclx.present || !GetHlgLumaCoefficients(d->nclx.color_primaries, luma))
            {
                return Fail(error, AVIFGPU_ERR_UNSUPPORTED, "the inverse HLG OOTF needs nclx colour primaries with known luma coefficients");
            }
            if (!(d->hlg_display_gamma > 0.0f) || d->hlg_peak_nits <= 0)
            {
                return Fail(error, AVIFGPU_ERR_BAD_PARAM, "bad HLG display gamma / peak brightness");
            }
        }
    }
    if (d->layout == AVIFGPU_LAYOUT_PLANAR_YCBCR)
    {
        if (d->host_channels <= 2) return Fail(error, AVIFGPU_ERR_BAD_PARAM, "planar YCbCr needs a colour host");
        if (d->chroma != AVIFGPU_CHROMA_420 && d->chroma != AVIFGPU_CHROMA_422 && d->chroma != AVIFGPU_CHROMA_444) return Fail(error, AVIFGPU_ERR_BAD_PARAM, "bad chroma");
        if (d->nclx.present && !d->nclx.full_range_flag) return Fail(error, AVIFGPU_ERR_UNSUPPORTED, "the encode path is full range only");
        if (d->nclx.present && d->nclx.matrix_coefficients == 0 && d->chroma != AVIFGPU_CHROMA_444) return Fail(error, AVIFGPU_ERR_UNSUPPORTED, "identity (GBR) matrix requires 4:4:4");
    }
    else if (d->layout != AVIFGPU_LAYOUT_REFERENCE)
    {
        return Fail(error, AVIFGPU_ERR_BAD_PARAM, "bad layout");
    }
    return AVIFGPU_OK;
}

int ValidateDecodeDesc(const avifgpu_decode_desc* d, int32_t* outTransfer, std::string* error)
{
    *outTransfer = AVIFGPU_TRANSFER_CLIP;
    if (d == nullptr || d->struct_size != sizeof(avifgpu_decode_desc)) return Fail(error, AVIFGPU_ERR_BAD_PARAM, "bad decode desc size");
    if (d->width < 0 || d->height < 0) return Fail(error, AVIFGPU_ERR_BAD_PARAM, "negative image size");
    if (d->host_depth != 8 && d->host_depth != 16 && d->host_depth != 32) return Fail(error, AVIFGPU_ERR_BAD_PARAM, "host depth must be 8, 16 or 32");
    if (d->bit_depth != 8 && d->bit_depth != 10 && d->bit_depth != 12 && d->bit_depth != 16) return Fail(error, AVIFGPU_ERR_UNSUPPORTED, "The image has an unsupported bit depth, must be 8, 10, 12 or 16.");
    if (d->colorspace != AVIFGPU_COLORSPACE_YCBCR && d->colorspace != AVIFGPU_COLORSPACE_RGB && d->colorspace != AVIFGPU_COLORSPACE_MONOCHROME) return Fail(error, AVIFGPU_ERR_UNSUPPORTED, "Unsupported image color space, expected RGB.");
    if (d->alpha_state < AVIFGPU_ALPHA_NONE || d->alpha_state > AVIFGPU_ALPHA_PREMULTIPLIED) return Fail(error, AVIFGPU_ERR_BAD_PARAM, "bad alpha state");
    if ((d->host_depth == 8) != (d->bit_depth == 8)) return Fail(error, AVIFGPU_ERR_UNSUPPORTED, "host depth 8 pairs with 8-bit planes only");
    if (d->colorspace == AVIFGPU_COLORSPACE_YCBCR && d->chroma != AVIFGPU_CHROMA_420 && d->chroma != AVIFGPU_CHROMA_422 && d->chroma != AVIFGPU_CHROMA_444) return Fail(error, AVIFGPU_ERR_BAD_PARAM, "bad chroma");
    if (d->host_depth == 32)
    {
        if (!d->nclx.present) return Fail(error, AVIFGPU_ERR_UNSUPPORTED, "The nclxProfile is null.");
        if (!TransferFromNclx(d->nclx.transfer_characteristics, outTransfer)) return Fail(error, AVIFGPU_ERR_UNSUPPORTED, "Unsupported NCLX transfer characteristic.");
        if (d->colorspace == AVIFGPU_COLORSPACE_MONOCHROME && *outTransfer != AVIFGPU_TRANSFER_PQ) return Fail(error, AVIFGPU_ERR_UNSUPPORTED, "Unsupported color transfer function.");
    }
    return AVIFGPU_OK;
}

static void ChromaShifts(int chroma, int* xs, int* ys)
{
    // ReadHeifImage.cpp:52-81
    *xs = (chroma == AVIFGPU_CHROMA_420 || chroma == AVIFGPU_CHROMA_422) ? 1 : 0;
    *ys = (chroma == AVIFGPU_CHROMA_420) ? 1 : 0;
}

PlaneGeometry EncodePlaneGeometry(const avifgpu_encode_desc& d, int index)
{
    PlaneGeometry g;
    const bool hasAlpha = d.alpha_state != AVIFGPU_ALPHA_NONE;
    g.bytesPerSample = d.image_bit_depth > 8 ? 2 : 1;
    if (d.layout == AVIFGPU_LAYOUT_REFERENCE)
    {
        const bool gray = d.host_channels <= 2;
        if (index == 0)
        {
            g.present = true;
            g.widthSamples = gray ? d.width : d.width * d.host_channels;
            g.height = d.height;
        }
        else if (index == 3 && gray && hasAlpha)
        {
            g.present = true;
            g.widthSamples = d.width;
            g.height = d.height;
        }
    }
    else
    {
        int xs, ys;
        ChromaShifts(d.chroma, &xs, &ys);
        if (index == 0 || (index == 3 && hasAlpha))
        {
            g.present = true;
            g.widthSamples = d.width;
            g.height = d.height;
        }
        else if (index == 1 || index == 2)
        {
            g.present = true;
            g.xs = xs;
            g.ys = ys;
            g.widthSamples = (d.width + xs) >> xs;
            g.height = (d.height + ys) >> ys;
        }
    }
    if (!g.present)
    {
        g.bytesPerSample = 0;
    }
    return g;
}

PlaneGeometry DecodePlaneGeometry(const avifgpu_decode_desc& d, int index)
{
    PlaneGeometry g;
    const bool hasAlpha = d.alpha_state != AVIFGPU_ALPHA_NONE;
    g.bytesPerSample = d.bit_depth > 8 ? 2 : 1;
    if (index == 0 || (index == 3 && hasAlpha))
    {
        g.present = true;
        g.widthSamples = d.width;
        g.height = d.height;
    }
    else if ((index == 1 || index == 2) && d.colorspace == AVIFGPU_COLORSPACE_YCBCR)
    {
        int xs, ys;
        ChromaShifts(d.chroma, &xs, &ys);
        g.present = true;
        g.xs = xs;
        g.ys = ys;
        g.widthSamples = (d.width + xs) >> xs;
        g.height = (d.height + ys) >> ys;
    }
    else if ((index == 1 || index == 2) && d.colorspace == AVIFGPU_COLORSPACE_RGB)
    {
        g.present = true;
        g.widthSamples = d.width;
        g.height = d.height;
    }
    if (!g.present)
    {
        g.bytesPerSample = 0;
    }
    return g;
}

int EncodeHostColBytes(const avifgpu_encode_desc& d) { return d.host_channels * ((d.host_depth + 7) / 8); }

int DecodeHostChannels(const avifgpu_decode_desc& d)
{
    const bool hasAlpha = d.alpha_state != AVIFGPU_ALPHA_NONE;
    if (d.colorspace == AVIFGPU_COLORSPACE_MONOCHROME)
    {
        return hasAlpha ? 2 : 1;
    }
    return hasAlpha ? 4 : 3;
}

int DecodeHostColBytes(const avifgpu_decode_desc& d) { return DecodeHostChannels(d) * ((d.host_depth + 7) / 8); }

// Sample (column, row) of a buffer whose rows are `stride` bytes apart and whose samples are `bytes` wide.
template <typename Void>
static Void* SampleAt(Void* base, int64_t stride, int column, int row, int bytes)
{
    using Byte = typename std::conditional<std::is_const<Void>::value, const uint8_t, uint8_t>::type;
    return static_cast<Byte*>(base) + static_cast<int64_t>(row) * stride + static_cast<int64_t>(column) * bytes;
}

EncodeParams EncodeSubRect(const EncodeParams& p, int hostDepth, int x, int y, int width, int rows)
{
    assert((x & p.xs) == 0 && (y & p.ys) == 0);
    const int sample = p.imageDepth > 8 ? 2 : 1;
    const bool gray = p.channels <= 2;
    EncodeParams s = p;
    s.rows = SampleAt(p.rows, p.rowStride, x, y, p.channels * (hostDepth / 8));
    // Planar: Y, Cb, Cr, A.  Reference layout: [0] holds all channels of a colour pixel or gray's Y; [3] gray's alpha.
    s.plane[0] = SampleAt(p.plane[0], p.planeStride[0], x, y, (p.planar || gray ? 1 : p.channels) * sample);
    if (p.planar)
    {
        s.plane[1] = SampleAt(p.plane[1], p.planeStride[1], x >> p.xs, y >> p.ys, sample);
        s.plane[2] = SampleAt(p.plane[2], p.planeStride[2], x >> p.xs, y >> p.ys, sample);
    }
    if (p.hasAlpha && (p.planar || gray))
    {
        s.plane[3] = SampleAt(p.plane[3], p.planeStride[3], x, y, sample);
    }
    s.width = width;
    s.rowCount = rows;
    return s;
}

DecodeParams DecodeSubRect(const DecodeParams& p, int x, int y, int width, int rows)
{
    assert((x & p.xs) == 0);
    const int sample = p.bitDepth > 8 ? 2 : 1;
    const bool mono = p.colorspace == AVIFGPU_COLORSPACE_MONOCHROME;
    const int hostChannels = (mono ? 1 : 3) + (p.hasAlpha ? 1 : 0);
    DecodeParams s = p;
    s.rows = SampleAt(p.rows, p.rowStride, x, y, hostChannels * (p.hostDepth / 8));
    s.plane[0] = SampleAt(p.plane[0], p.planeStride[0], x, y, sample);
    if (!mono)
    {
        // YCbCr chroma, or planar G and B (xs = ys = yPhase = 0)
        const int chromaRow = (p.yPhase + y) >> p.ys;
        s.plane[1] = SampleAt(p.plane[1], p.planeStride[1], x >> p.xs, chromaRow, sample);
        s.plane[2] = SampleAt(p.plane[2], p.planeStride[2], x >> p.xs, chromaRow, sample);
    }
    if (p.hasAlpha)
    {
        s.plane[3] = SampleAt(p.plane[3], p.planeStride[3], x, y, sample);
    }
    s.width = width;
    s.rowCount = rows;
    s.yPhase = (p.yPhase + y) & p.ys;
    return s;
}

void FillEncodeParams(const avifgpu_encode_desc& d, EncodeParams* p)
{
    std::memset(p, 0, sizeof(*p));
    p->width = d.width;
    p->channels = d.host_channels;
    p->hasAlpha = d.alpha_state != AVIFGPU_ALPHA_NONE;
    p->premultiply = d.alpha_state == AVIFGPU_ALPHA_PREMULTIPLIED;
    p->imageDepth = d.image_bit_depth;
    p->maxCode = (1u << d.image_bit_depth) - 1u;
    p->maxCodeFloat = static_cast<float>(p->maxCode);
    p->transfer = d.transfer;
    p->pqMultiplier = static_cast<float>(d.pq_peak_nits) / 10000.0f; // ColorTransfer.cpp:86
    p->gray16Smpte428 = (d.host_depth == 16 && d.host_channels <= 2 && d.gray16_curve == AVIFGPU_GRAY16_SMPTE428) ? 1 : 0;
    if (d.host_depth == 32 && d.transfer == AVIFGPU_TRANSFER_HLG && d.hlg_extension == AVIFGPU_HLG_INVERSE_OOTF_THEN_OETF)
    {
        p->hlgInverseOotf = 1;
        GetHlgLumaCoefficients(d.nclx.color_primaries, p->hlgLuma);
        p->hlgDisplayGamma = d.hlg_display_gamma;
        p->hlgPeak = static_cast<float>(d.hlg_peak_nits);
    }
    p->rowMatrixEnabled = (d.row_matrix_enabled && d.host_depth == 32 && d.host_channels >= 3) ? 1 : 0;
    for (int i = 0; i < 9; ++i)
    {
        p->rowMatrix[i] = d.row_matrix[i];
    }
    p->planar = d.layout == AVIFGPU_LAYOUT_PLANAR_YCBCR;
    if (p->planar)
    {
        int xs, ys;
        ChromaShifts(d.chroma, &xs, &ys);
        p->xs = xs;
        p->ys = ys;
        p->topLeft = d.down_filter == AVIFGPU_DOWN_FILTER_TOP_LEFT;
        float k[3];
        GetYuvCoefficients(&d.nclx, k);
        p->matrix.kr = k[0];
        p->matrix.kg = k[1];
        p->matrix.kb = k[2];
        p->matrix.cbScale = 0.5f / (1.0f - k[2]);
        p->matrix.crScale = 0.5f / (1.0f - k[0]);
        p->matrix.identity = (d.nclx.present && d.nclx.matrix_coefficients == 0) ? 1 : 0;
        // H.273 full range (and libheif's RGB->YCbCr): Ccode = Clip(Round(C) + 2^(depth-1)); neutral grey sits on 2^(depth-1).
        // (The reference DEcoder's chroma zero is max/2, YuvLookupTables.cpp:183: half a code lower -- its own business.)
        p->chromaOffset = p->matrix.identity ? 0.0f : static_cast<float>(1u << (d.image_bit_depth - 1));
    }
}

bool FillDecodeParams(const avifgpu_decode_desc& d, int32_t transfer, DecodeParams* p, std::string* error)
{
    std::memset(p, 0, sizeof(*p));
    p->width = d.width;
    p->colorspace = d.colorspace;
    if (d.colorspace == AVIFGPU_COLORSPACE_YCBCR)
    {
        int xs, ys;
        ChromaShifts(d.chroma, &xs, &ys);
        p->xs = xs;
        p->ys = ys;
    }
    p->hasAlpha = d.alpha_state != AVIFGPU_ALPHA_NONE;
    p->premultiplied = d.alpha_state == AVIFGPU_ALPHA_PREMULTIPLIED;
    p->bitDepth = d.bit_depth;
    p->maxCode = (1u << d.bit_depth) - 1u;
    p->range = MakeRangeParams(&d.nclx, d.bit_depth, d.colorspace == AVIFGPU_COLORSPACE_MONOCHROME);
    if (d.colorspace == AVIFGPU_COLORSPACE_RGB)
    {
        p->range.fullRange = 1; // ReadHeifImage.cpp:402-415: plain i / max table
        p->range.identityMatrix = 0;
    }
    float k[3];
    GetYuvCoefficients(&d.nclx, k);
    p->matrix.kr = k[0];
    p->matrix.kg = k[1];
    p->matrix.kb = k[2];
    p->hostDepth = d.host_depth;
    p->transfer = transfer;
    p->pqMultiplier = 10000.0f / static_cast<float>(d.pq_peak_nits); // ColorTransfer.cpp:114
    p->applyOotf = d.hlg_apply_ootf != 0;
    p->gammaMinusOne = d.hlg_display_gamma - 1.0f; // ColorTransfer.cpp:201
    p->hlgPeak = static_cast<float>(d.hlg_peak_nits);
    if (d.host_depth == 32 && transfer == AVIFGPU_TRANSFER_HLG && d.hlg_apply_ootf && d.colorspace != AVIFGPU_COLORSPACE_MONOCHROME)
    {
        float luma[3];
        if (!GetHlgLumaCoefficients(d.nclx.color_primaries, luma))
        {
            if (error)
            {
                *error = "Unsupported color primaries for the HLG Luma Coefficients ";
            }
            return false;
        }
        p->lumaR = luma[0];
        p->lumaG = luma[1];
        p->lumaB = luma[2];
    }
    return true;
}

} // namespace avifgpu
