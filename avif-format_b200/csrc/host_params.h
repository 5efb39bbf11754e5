// host_params.h -- host-side derivation of everything the kernels need from the reference's parameter blocks:
// description validation (same acceptance rules and messages as the reference's throws), matrix coefficients
// (YUVCoefficiants.cpp), range / table parameters (YuvLookupTables.cpp), transfer selection
// (ColorTransfer.cpp:31-67) and plane geometry.  Pure C++ -- no CUDA -- so it is unit-tested without a GPU.
#ifndef AVIF_HOST_PARAMS_H
#define AVIF_HOST_PARAMS_H

#include <string>

#include "../../include/avifgpu.h"
#include "kernel_params.h"

namespace avifgpu
{

// GetYUVCoefficiants, YUVCoefficiants.cpp:154-188.
void GetYuvCoefficients(const avifgpu_nclx* nclx, float out[3]);

// GetHLGLumaCoefficients, ColorTransfer.cpp:31-45; false for unsupported primaries.
bool GetHlgLumaCoefficients(int32_t colorPrimaries, float out[3]);

// GetTransferFunctionFromNclx, ColorTransfer.cpp:47-67; false for unsupported characteristics.
bool TransferFromNclx(int32_t transferCharacteristics, int32_t* outTransfer);

// Range parameters of YUVLookupTables (YuvLookupTables.cpp:115-192) for the arithmetic table evaluation.
avifpix::RangeParams MakeRangeParams(const avifgpu_nclx* nclx, int bitDepth, bool monochrome);

// Validation: 0 or a negative avifgpu_status with `error` filled in.
int ValidateEncodeDesc(const avifgpu_encode_desc* desc, std::string* error);
int ValidateDecodeDesc(const avifgpu_decode_desc* desc, int32_t* outTransfer, std::string* error);

struct PlaneGeometry
{
    int32_t widthSamples = 0; // samples per row (interleaved: width * channels)
    int32_t height = 0;
    int32_t bytesPerSample = 0;
    int32_t xs = 0;           // sub-sampling shifts relative to the image
    int32_t ys = 0;
    bool present = false;
};

PlaneGeometry EncodePlaneGeometry(const avifgpu_encode_desc& desc, int index);
PlaneGeometry DecodePlaneGeometry(const avifgpu_decode_desc& desc, int index);
int EncodeHostColBytes(const avifgpu_encode_desc& desc);
int DecodeHostChannels(const avifgpu_decode_desc& desc);
int DecodeHostColBytes(const avifgpu_decode_desc& desc);

// The block's pixels [x, x + width) x [y, y + rows) as a block of their own: every pointer moved to that origin.
// Encode needs x even when chroma is sub-sampled horizontally and y even when vertically; decode needs x even likewise
// and takes any y (the result's yPhase says where its first row sits in its chroma row).
EncodeParams EncodeSubRect(const EncodeParams& p, int hostDepth, int x, int y, int width, int rows);
DecodeParams DecodeSubRect(const DecodeParams& p, int x, int y, int width, int rows);

// Fills the kernel parameter blocks (pointers and row counts are set by the caller).
void FillEncodeParams(const avifgpu_encode_desc& desc, EncodeParams* params);
bool FillDecodeParams(const avifgpu_decode_desc& desc, int32_t transfer, DecodeParams* params, std::string* error);

} // namespace avifgpu

#endif
