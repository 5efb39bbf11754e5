// The sub-rectangle rule of host_params.cpp (EncodeSubRect / DecodeSubRect) on the CPU: for every valid description
// and the edge splits the tuned launchers make (LaunchEncodeRemainder / LaunchDecodeRemainder), each pixel of a
// sub-rectangle must address the same host-row bytes and plane samples as that pixel of the whole block, and the tuned
// interior plus the two strips must cover each pixel exactly once.  The addressing below restates the generic kernels'
// own indexing (kernels_generic.cu); the pointers are made-up addresses that are compared, never dereferenced.
#include "host_params.h"

#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

using namespace avifgpu;

namespace
{

long long g_checks = 0;
long long g_failures = 0;

void Expect(bool ok, const std::string& what)
{
    ++g_checks;
    if (!ok && ++g_failures <= 20)
    {
        std::printf("FAIL %s\n", what.c_str());
    }
}

uintptr_t At(const void* base, int64_t stride, int row, int64_t index, int bytes)
{
    return reinterpret_cast<uintptr_t>(base) + static_cast<uintptr_t>(row * stride + index * bytes);
}

const void* FakePointer(uintptr_t address) { return reinterpret_cast<const void*>(address); }

// Every address the generic encode kernels touch for pixel (x, y) of block `p`: its host pixel, then the plane samples
// it writes (EncodeReferenceLayoutKernel) or writes / contributes to (EncodePlanarKernel, chroma site (x >> xs, y >> ys)).
std::vector<uintptr_t> EncodeAddresses(const EncodeParams& p, int hostDepth, int x, int y)
{
    const int sample = p.imageDepth > 8 ? 2 : 1;
    std::vector<uintptr_t> a{ At(p.rows, p.rowStride, y, static_cast<int64_t>(x) * p.channels, hostDepth / 8) };
    if (p.planar)
    {
        a.push_back(At(p.plane[0], p.planeStride[0], y, x, sample));
        a.push_back(At(p.plane[1], p.planeStride[1], y >> p.ys, x >> p.xs, sample));
        a.push_back(At(p.plane[2], p.planeStride[2], y >> p.ys, x >> p.xs, sample));
        if (p.hasAlpha) a.push_back(At(p.plane[3], p.planeStride[3], y, x, sample));
    }
    else if (p.channels <= 2)
    {
        a.push_back(At(p.plane[0], p.planeStride[0], y, x, sample));
        if (p.hasAlpha) a.push_back(At(p.plane[3], p.planeStride[3], y, x, sample));
    }
    else
    {
        for (int i = 0; i < p.channels; ++i) a.push_back(At(p.plane[0], p.planeStride[0], y, static_cast<int64_t>(x) * p.channels + i, sample));
    }
    return a;
}

// The same for DecodeKernel<PlaneT, HostT>: PlaneT is 8-bit for 8-bit hosts and 16-bit otherwise.
std::vector<uintptr_t> DecodeAddresses(const DecodeParams& p, int x, int y)
{
    const int sample = p.hostDepth == 8 ? 1 : 2;
    const int channels = (p.colorspace == AVIFGPU_COLORSPACE_MONOCHROME) ? (p.hasAlpha ? 2 : 1) : (p.hasAlpha ? 4 : 3);
    std::vector<uintptr_t> a{ At(p.rows, p.rowStride, y, static_cast<int64_t>(x) * channels, p.hostDepth / 8),
                              At(p.plane[0], p.planeStride[0], y, x, sample) };
    if (p.hasAlpha) a.push_back(At(p.plane[3], p.planeStride[3], y, x, sample));
    if (p.colorspace == AVIFGPU_COLORSPACE_YCBCR)
    {
        a.push_back(At(p.plane[1], p.planeStride[1], (y + p.yPhase) >> p.ys, x >> p.xs, sample));
        a.push_back(At(p.plane[2], p.planeStride[2], (y + p.yPhase) >> p.ys, x >> p.xs, sample));
    }
    else if (p.colorspace == AVIFGPU_COLORSPACE_RGB)
    {
        a.push_back(At(p.plane[1], p.planeStride[1], y, x, sample));
        a.push_back(At(p.plane[2], p.planeStride[2], y, x, sample));
    }
    return a;
}

// Everything but the pointers, the size and yPhase must be the whole block's.
template <typename Params>
bool SameOtherwise(Params sub, const Params& whole)
{
    sub.rows = whole.rows;
    std::memcpy(sub.plane, whole.plane, sizeof(sub.plane));
    sub.width = whole.width;
    sub.rowCount = whole.rowCount;
    return std::memcmp(&sub, &whole, sizeof(sub)) == 0;
}

// Sub-rectangle [x, x + width) x [y, y + rows) of `whole`, checked pixel by pixel; marks the pixels it covers.
template <typename Params, typename Make, typename Addresses>
void CheckSubRect(const Params& whole, int x, int y, int width, int rows, const std::string& what, Make make, Addresses addresses,
                  std::vector<int>& covered)
{
    const Params sub = make(x, y, width, rows);
    Expect(sub.width == width && sub.rowCount == rows, what + " size");
    for (int k = 0; k < 4; ++k)
    {
        if (whole.plane[k] == nullptr || (reinterpret_cast<uintptr_t>(whole.plane[k]) >> 60) == 0xa)
        {
            Expect(sub.plane[k] == whole.plane[k], what + " absent plane " + std::to_string(k) + " moved");
        }
    }
    for (int j = 0; j < rows; ++j)
    {
        for (int i = 0; i < width; ++i)
        {
            ++covered[static_cast<size_t>(y + j) * whole.width + (x + i)];
            Expect(addresses(sub, i, j) == addresses(whole, x + i, y + j),
                   what + " pixel (" + std::to_string(x + i) + ", " + std::to_string(y + j) + ")");
        }
    }
}

// The split of LaunchEncodeRemainder / LaunchDecodeRemainder after a tuned kernel over [0, coveredWidth) x [0, coveredRows).
template <typename Params, typename Make, typename Addresses>
void CheckSplit(const Params& whole, int coveredWidth, int coveredRows, const std::string& what, Make make, Addresses addresses)
{
    std::vector<int> covered(static_cast<size_t>(whole.width) * whole.rowCount, 0);
    for (int j = 0; j < coveredRows; ++j)
    {
        for (int i = 0; i < coveredWidth; ++i) ++covered[static_cast<size_t>(j) * whole.width + i];
    }
    CheckSubRect(whole, coveredWidth, 0, whole.width - coveredWidth, whole.rowCount, what + " right strip", make, addresses, covered);
    CheckSubRect(whole, 0, coveredRows, coveredWidth, whole.rowCount - coveredRows, what + " bottom strip", make, addresses, covered);
    bool once = true;
    for (int c : covered) once = once && c == 1;
    Expect(once, what + ": interior and strips do not cover each pixel exactly once");
}

const int kWidths[] = { 1, 2, 3, 4, 5, 7, 8, 9, 12, 13, 17, 37, 131 };
const int kHeights[] = { 1, 2, 3, 4, 5, 7, 23 };

// Made-up device addresses: host rows and each plane in a region of their own, strides padded past the row's bytes.
// Absent planes get a recognisable non-null address, so that "left unchanged" is visible.
void PlaceBuffers(const void** rows, int64_t* rowStride, int64_t rowBytes, const void* plane[4], int64_t planeStride[4],
                  const PlaneGeometry (&g)[4])
{
    *rows = FakePointer(0x100000000ull + 256);
    *rowStride = rowBytes + 48;
    for (int k = 0; k < 4; ++k)
    {
        if (g[k].present)
        {
            plane[k] = FakePointer(0x1000000000ull * (k + 2) + 64 * k);
            planeStride[k] = static_cast<int64_t>(g[k].widthSamples) * g[k].bytesPerSample + 16 * (k + 1);
        }
        else
        {
            plane[k] = FakePointer(0xa000000000000000ull + 0x1000 * k);
            planeStride[k] = 0;
        }
    }
}

void CheckEncode()
{
    avifgpu_nclx nclx{ 1, 9, 16, 9, 1 };
    for (int layout : { AVIFGPU_LAYOUT_REFERENCE, AVIFGPU_LAYOUT_PLANAR_YCBCR })
    for (int hostDepth : { 8, 16, 32 })
    for (int channels = 1; channels <= 4; ++channels)
    for (int alpha : { AVIFGPU_ALPHA_NONE, AVIFGPU_ALPHA_STRAIGHT, AVIFGPU_ALPHA_PREMULTIPLIED })
    for (int depth : { 8, 10, 12 })
    for (int chroma : { AVIFGPU_CHROMA_420, AVIFGPU_CHROMA_422, AVIFGPU_CHROMA_444 })
    for (int w : kWidths)
    for (int h : kHeights)
    {
        if (layout == AVIFGPU_LAYOUT_REFERENCE && chroma != AVIFGPU_CHROMA_420)
        {
            continue; // chroma is a planar setting only
        }
        avifgpu_encode_desc d{};
        d.struct_size = sizeof(d);
        d.width = w;
        d.height = h;
        d.host_depth = hostDepth;
        d.host_channels = channels;
        d.alpha_state = alpha;
        d.image_bit_depth = depth;
        d.transfer = AVIFGPU_TRANSFER_PQ;
        d.pq_peak_nits = 80;
        d.layout = layout;
        d.chroma = chroma;
        d.nclx = nclx;
        if (ValidateEncodeDesc(&d, nullptr) != AVIFGPU_OK)
        {
            continue;
        }
        EncodeParams p;
        FillEncodeParams(d, &p);
        p.rowCount = h;
        PlaneGeometry g[4];
        for (int k = 0; k < 4; ++k) g[k] = EncodePlaneGeometry(d, k);
        const void* planes[4];
        PlaceBuffers(&p.rows, &p.rowStride, static_cast<int64_t>(w) * EncodeHostColBytes(d), planes, p.planeStride, g);
        for (int k = 0; k < 4; ++k) p.plane[k] = const_cast<void*>(planes[k]);

        const std::string what = "encode layout " + std::to_string(layout) + " host " + std::to_string(hostDepth) + "x" + std::to_string(channels) +
                                 " alpha " + std::to_string(alpha) + " depth " + std::to_string(depth) + " chroma " + std::to_string(chroma) + " " +
                                 std::to_string(w) + "x" + std::to_string(h);
        const auto make = [&](int x, int y, int width, int rows) { return EncodeSubRect(p, hostDepth, x, y, width, rows); };
        const auto addresses = [&](const EncodeParams& q, int x, int y) { return EncodeAddresses(q, hostDepth, x, y); };
        for (int coveredWidth : { w & ~3, w & ~7 })
        {
            for (int coveredRows : { h, h & ~1 })
            {
                if ((coveredRows & p.ys) == 0)
                {
                    CheckSplit(p, coveredWidth, coveredRows, what + " covered " + std::to_string(coveredWidth) + "x" + std::to_string(coveredRows), make, addresses);
                }
            }
        }
        Expect(SameOtherwise(make(w & ~3, h & ~1, w - (w & ~3), h - (h & ~1)), p), what + ": a field other than pointers and size changed");
    }
}

void CheckDecode()
{
    for (int colorspace : { AVIFGPU_COLORSPACE_YCBCR, AVIFGPU_COLORSPACE_MONOCHROME, AVIFGPU_COLORSPACE_RGB })
    for (int chroma : { AVIFGPU_CHROMA_420, AVIFGPU_CHROMA_422, AVIFGPU_CHROMA_444 })
    for (int bitDepth : { 8, 10, 12, 16 })
    for (int hostDepth : { 8, 16, 32 })
    for (int alpha : { AVIFGPU_ALPHA_NONE, AVIFGPU_ALPHA_STRAIGHT, AVIFGPU_ALPHA_PREMULTIPLIED })
    for (int w : kWidths)
    for (int h : kHeights)
    {
        if (colorspace != AVIFGPU_COLORSPACE_YCBCR && chroma != AVIFGPU_CHROMA_420)
        {
            continue; // chroma only shapes YCbCr planes
        }
        avifgpu_decode_desc d{};
        d.struct_size = sizeof(d);
        d.width = w;
        d.height = h;
        d.colorspace = colorspace;
        d.chroma = chroma;
        d.bit_depth = bitDepth;
        d.alpha_state = alpha;
        d.host_depth = hostDepth;
        d.nclx = avifgpu_nclx{ 1, 9, 16, 9, 1 };
        d.hlg_display_gamma = 1.2f;
        d.hlg_peak_nits = 1000;
        d.pq_peak_nits = 10000;
        int32_t transfer = 0;
        if (ValidateDecodeDesc(&d, &transfer, nullptr) != AVIFGPU_OK)
        {
            continue;
        }
        DecodeParams whole;
        if (!FillDecodeParams(d, transfer, &whole, nullptr))
        {
            Expect(false, "FillDecodeParams rejected a valid description");
            continue;
        }
        PlaneGeometry g[4];
        for (int k = 0; k < 4; ++k) g[k] = DecodePlaneGeometry(d, k);
        const void* rows;
        PlaceBuffers(&rows, &whole.rowStride, static_cast<int64_t>(w) * DecodeHostColBytes(d), whole.plane, whole.planeStride, g);
        whole.rows = const_cast<void*>(rows);

        // A block of the image starting on row y0 (yPhase = y0 & ys); 4:2:0 chroma of an odd first row is the row above's.
        for (int yPhase = 0; yPhase <= whole.ys; ++yPhase)
        {
            DecodeParams p = whole;
            p.yPhase = yPhase;
            p.rowCount = h;
            const std::string what = "decode colorspace " + std::to_string(colorspace) + " chroma " + std::to_string(chroma) + " depth " +
                                     std::to_string(bitDepth) + " host " + std::to_string(hostDepth) + " alpha " + std::to_string(alpha) + " " +
                                     std::to_string(w) + "x" + std::to_string(h) + " yPhase " + std::to_string(yPhase);
            const auto make = [&](int x, int y, int width, int rows) { return DecodeSubRect(p, x, y, width, rows); };
            const auto addresses = [](const DecodeParams& q, int x, int y) { return DecodeAddresses(q, x, y); };
            for (int coveredWidth : { w & ~3, w & ~7 })
            {
                for (int coveredRows = 0; coveredRows <= h; ++coveredRows) // odd first rows of the bottom strip included
                {
                    CheckSplit(p, coveredWidth, coveredRows, what + " covered " + std::to_string(coveredWidth) + "x" + std::to_string(coveredRows), make, addresses);
                }
            }
            for (int y = 0; y <= h; ++y)
            {
                const DecodeParams sub = make(w & ~3, y, w - (w & ~3), h - y);
                Expect(sub.yPhase == ((yPhase + y) & p.ys), what + " yPhase of a block at row " + std::to_string(y));
                DecodeParams rest = sub;
                rest.yPhase = p.yPhase;
                Expect(SameOtherwise(rest, p), what + ": a field other than pointers, size and yPhase changed");
            }
        }
    }
}

} // namespace

int main()
{
    CheckEncode();
    const long long encodeChecks = g_checks;
    CheckDecode();
    std::printf("%lld encode checks, %lld decode checks, %lld failures\n", encodeChecks, g_checks - encodeChecks, g_failures);
    if (g_failures == 0)
    {
        std::printf("ALL PASSED\n");
    }
    return g_failures == 0 ? 0 : 1;
}
