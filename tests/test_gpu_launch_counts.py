"""Kernels started by one call of each tuned launcher whose interior leaves edge strips: the tuned kernel, then the
generic kernel once per non-empty strip (the right strip, then an odd last row under 4:2:0).  The widths leave a
right strip for interiors of width & ~3 and width & ~7 alike; the 4:2:0 shapes have an odd row count.  The context
is warmed by a first call, so step tables, the Gray16 code table and the one-time exactness checks are not counted."""
import numpy as np
import pytest

import cases
from avifgpu import abi

pytestmark = pytest.mark.gpu

ENCODES = [  # (tuned launcher, description, kernels per call)
    ("LaunchEncodeFast interleaved RGB32f", abi.EncodeDesc(37, 23, 32, 3, abi.ALPHA_NONE, 12, abi.TRANSFER_PQ, 80, abi.LAYOUT_REFERENCE,
                                                           nclx=cases.NCLX_2020_PQ()), 2),
    ("LaunchEncodeFast planar RGB32f 4:2:0", abi.EncodeDesc(131, 5, 32, 3, abi.ALPHA_NONE, 12, abi.TRANSFER_PQ, 80, abi.LAYOUT_PLANAR_YCBCR,
                                                            abi.CHROMA_420, nclx=cases.NCLX_2020_PQ()), 3),
    ("LaunchEncodeFastInteger Gray16 code table", abi.EncodeDesc(37, 23, 16, 1, abi.ALPHA_NONE, 10), 2),
    ("LaunchEncodeFastInteger Gray8+A", abi.EncodeDesc(37, 23, 8, 2, abi.ALPHA_STRAIGHT, 10), 2),
    ("LaunchEncodeFastInteger planar RGB16 4:2:0", abi.EncodeDesc(131, 5, 16, 3, abi.ALPHA_NONE, 10, abi.TRANSFER_CLIP, 80, abi.LAYOUT_PLANAR_YCBCR,
                                                                  abi.CHROMA_420), 3),
    ("LaunchEncodeFastGray32", abi.EncodeDesc(37, 23, 32, 1, abi.ALPHA_NONE, 12, abi.TRANSFER_CLIP), 2),
]

DECODES = [
    ("LaunchDecodeFast YCbCr 4:2:0 to RGB32f", abi.DecodeDesc(131, 5, abi.COLORSPACE_YCBCR, abi.CHROMA_420, 10, abi.ALPHA_NONE, 32,
                                                              cases.NCLX_2020_PQ(1)), 3),
    ("LaunchDecodeFastInteger planar RGB to RGB16", abi.DecodeDesc(37, 23, abi.COLORSPACE_RGB, abi.CHROMA_444, 10, abi.ALPHA_NONE, 16,
                                                                   cases.NCLX_601(1)), 2),
    ("LaunchDecodeFastInteger YCbCr 4:2:0 to RGB8", abi.DecodeDesc(131, 5, abi.COLORSPACE_YCBCR, abi.CHROMA_420, 8, abi.ALPHA_NONE, 8,
                                                                   cases.NCLX_601(1)), 3),
    ("LaunchDecodeFastTable planar RGB to RGB32f", abi.DecodeDesc(37, 23, abi.COLORSPACE_RGB, abi.CHROMA_444, 10, abi.ALPHA_NONE, 32,
                                                                  cases.NCLX_2020_PQ(1)), 2),
]


def launches_of_second_call(ctx, call):
    call()
    before = ctx.launch_count()
    call()
    return ctx.launch_count() - before


@pytest.mark.parametrize("desc,expected", [case[1:] for case in ENCODES], ids=[case[0] for case in ENCODES])
def test_encode_edge_strips(gpu, desc, expected):
    rng = np.random.default_rng(desc.width * 100 + desc.host_channels)
    if desc.host_depth == 32:
        rows = cases.float_host_rows(rng, desc.height, desc.width, desc.host_channels)
    else:
        rows = cases.int_host_rows(rng, desc.height, desc.width, desc.host_channels, desc.host_depth)
    assert launches_of_second_call(gpu, lambda: gpu.encode(desc, rows)) == expected


@pytest.mark.parametrize("desc,expected", [case[1:] for case in DECODES], ids=[case[0] for case in DECODES])
def test_decode_edge_strips(gpu, desc, expected):
    planes = cases.code_planes(np.random.default_rng(desc.width * 100 + desc.colorspace), desc)
    assert launches_of_second_call(gpu, lambda: gpu.decode(desc, planes)) == expected
