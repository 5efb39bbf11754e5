"""Pins the C restatement (oracle/avif_oracle.c) to the reference itself: the UNMODIFIED reference translation
units compiled in place (oracle/_ref/libavifref.so) must agree with it bit for bit -- scalars exhaustively where
the domain is small, images over the whole case matrix, and the known-answer values recorded in SURVEY.md 4.
Where oracle/_ref is not built, `ref` holds the restatement to the reference's recorded results (conftest.py)."""
import numpy as np
import pytest

import cases
from avifgpu import abi


def bits(values):
    return [hex(int(v)) for v in np.asarray(values, np.float32).view(np.uint32)]


def test_known_answers_from_survey(ref, port):
    for c in (ref, port):
        assert bits(c.transfer(abi.FN_LINEAR_TO_PQ, [1.0, 0.18, 0.0, 125.0], 80.0)) == ["0x3ef8c243", "0x3ea88c61", "0x354436e8", "0x3f800000"]
        codes = np.clip(c.transfer(abi.FN_LINEAR_TO_PQ, [1.0, 0.18, 0.0, 125.0], 80.0) * 4095, 0, 4095).astype(np.uint16)
        assert codes.tolist() == [1989, 1348, 0, 4095]
        s428 = np.clip(c.transfer(abi.FN_LINEAR_TO_SMPTE428, [0.18, 1.0, 2.0]) * np.float32(4095), 0, 4095).astype(np.uint16)
        assert s428.tolist() == [2047, 3960, 4095]
        assert bits(c.transfer(abi.FN_PQ_TO_LINEAR, [0.5, 1.0], 80.0)) == ["0x3f939704", "0x42fa0000"]
        assert bits(c.transfer(abi.FN_HLG_TO_LINEAR, [0.5, 0.75, 1.0])) == ["0x3daaaaab", "0x3e87a92d", "0x3f800001"]
        assert c._premultiply_u8(200, 128) == 100
        assert c._premultiply_u16(1000, 512, 1023) == 500
        assert c._unpremultiply_u8(100, 128) == 199
        assert c._unpremultiply_u16(300, 512, 1023) == 599
        assert c._unpremultiply_u8(200, 100) == 255
        k2020 = c.yuv_coefficients(abi.Nclx(1, 9, 16, 9, 1))
        assert [float(v).hex() for v in k2020] == ["0x1.0d013a0000000p-2", "0x1.5b22d20000000p-1", "0x1.e5c91e0000000p-5"]
        k601 = c.yuv_coefficients(None)
        assert [float(v).hex() for v in k601] == ["0x1.322d0e0000000p-2", "0x1.2c8b420000000p-1", "0x1.d2f1aa0000000p-4"]
        y, uv, _ = c.yuv_tables(abi.Nclx(1, 9, 16, 9, 0), 10, False)
        assert y[64] == 0 and y[940] == 1 and uv[64] == -0.5 and uv[960] == 0.5
        _, uv_full, _ = c.yuv_tables(abi.Nclx(1, 9, 16, 9, 1), 10, False)
        assert float(uv_full[512]).hex() == "0x1.0040000000000p-11"


def test_known_answer_pixels(ref, port):
    hlg = abi.DecodeDesc(2, 2, abi.COLORSPACE_YCBCR, abi.CHROMA_420, 10, abi.ALPHA_NONE, 32, cases.NCLX_2020_HLG())
    for c in (ref, port):
        planes = [np.full((2, 2), 512, np.uint16), np.full((1, 1), 512, np.uint16), np.full((1, 1), 512, np.uint16), None]
        assert bits(c.decode(hlg, planes)[0, :3]) == ["0x424bda35", "0x424af8ed", "0x424c03cd"]
        planes = [np.full((2, 2), 940, np.uint16), np.full((1, 1), 700, np.uint16), np.full((1, 1), 300, np.uint16), None]
        assert bits(c.decode(hlg, planes)[0, :3]) == ["0x4301a461", "0x446d762c", "0x446d762c"]
        bt601 = abi.DecodeDesc(1, 1, abi.COLORSPACE_YCBCR, abi.CHROMA_444, 8, abi.ALPHA_NONE, 8, None)
        px = lambda y, cb, cr: [np.full((1, 1), v, np.uint8) for v in (y, cb, cr)] + [None]  # noqa: E731
        assert c.decode(bt601, px(81, 90, 240))[0].tolist() == [239, 14, 15]
        assert c.decode(bt601, px(145, 90, 240))[0].tolist() == [255, 78, 79]


@pytest.mark.parametrize("function,param,lo,hi", [
    (abi.FN_LINEAR_TO_PQ, 80.0, -1.0, 130.0), (abi.FN_LINEAR_TO_PQ, 10000.0, 0.0, 1.5), (abi.FN_PQ_TO_LINEAR, 80.0, -0.1, 1.1),
    (abi.FN_LINEAR_TO_SMPTE428, 0.0, -0.5, 2.0), (abi.FN_SMPTE428_TO_LINEAR, 0.0, -0.1, 1.2), (abi.FN_HLG_TO_LINEAR, 0.0, -0.1, 1.2),
    (abi.FN_LINEAR_TO_HLG, 0.0, -0.1, 1.2)])
def test_transfer_functions_match(ref, port, function, param, lo, hi):
    rng = np.random.default_rng(function * 7 + 1)
    x = rng.uniform(lo, hi, 200_000).astype(np.float32)
    assert cases.same_bits(ref.transfer(function, x, param), port.transfer(function, x, param))


@pytest.mark.parametrize("primaries", [abi.PRIMARIES_BT709, abi.PRIMARIES_BT2020])
def test_hlg_ootfs_match(ref, port, primaries):
    """ApplyHLGOOTF and the (uncalled) ApplyInverseHLGOOTF, ColorTransfer.cpp:192-220."""
    rng = np.random.default_rng(primaries)
    rgb = np.concatenate([rng.uniform(0.0, 1.0, (20000, 3)), np.exp(rng.uniform(np.log(1e-9), np.log(1000.0), (20000, 3))),
                          [[0.0, 0.0, 0.0], [1.0, 1.0, 1.0], [np.inf, 0.1, 0.2], [np.nan, 0.3, 0.3], [-0.1, 0.2, 0.3]]]).astype(np.float32)
    for gamma, peak in ((1.2, 1000.0), (1.0, 400.0), (1.5, 4000.0)):
        assert cases.same_bits(ref.hlg_ootf(rgb, primaries, gamma, peak), port.hlg_ootf(rgb, primaries, gamma, peak))
        assert cases.same_bits(ref.hlg_inverse_ootf(rgb, primaries, gamma, peak), port.hlg_inverse_ootf(rgb, primaries, gamma, peak))


def test_premultiply_tables_exhaustive(ref, port):
    for max_value in (255, 1023):
        for un in (False, True):
            assert np.array_equal(ref.premultiply_table(max_value, un), port.premultiply_table(max_value, un))


def test_premultiply_12bit_sampled(ref, port):
    rng = np.random.default_rng(5)
    c = rng.integers(0, 4096, 20000)
    a = rng.integers(1, 4096, 20000)
    for un in (False, True):
        assert np.array_equal(ref.premultiply_samples(c, a, 4095, un), port.premultiply_samples(c, a, 4095, un))


def test_coefficients_and_tables_match(ref, port):
    for matrix in (0, 1, 2, 4, 5, 6, 7, 9, 10, 12, 14):
        for primaries in (1, 2, 4, 5, 6, 7, 8, 9, 10, 11, 12, 22):
            n = abi.Nclx(1, primaries, 13, matrix, 1)
            assert cases.same_bits(ref.yuv_coefficients(n), port.yuv_coefficients(n)), (matrix, primaries)
    assert cases.same_bits(ref.yuv_coefficients(None), port.yuv_coefficients(None))
    for primaries in (1, 5, 6, 9):
        assert cases.same_bits(ref.hlg_luma_coefficients(primaries), port.hlg_luma_coefficients(primaries))
    for depth in (8, 10, 12, 16):
        for full in (0, 1):
            if depth == 16 and not full:
                continue  # int overflow in the reference's LIMITED_TO_FULL at 16 bit (undefined behaviour)
            for matrix in (0, 6, 9):
                for mono in (False, True):
                    n = abi.Nclx(1, 9, 16, matrix, full)
                    a, b = ref.yuv_tables(n, depth, mono), port.yuv_tables(n, depth, mono)
                    for ta, tb in zip(a, b):
                        assert (ta is None) == (tb is None)
                        if ta is not None:
                            assert cases.same_bits(ta, tb), (depth, full, matrix, mono)


def test_depth_luts_match_reference_encode(ref, port):
    # The reference's LUT builders are file-local; observe them through a 1-row image holding every input.
    for host_depth, count in ((8, 256), (16, 32769)):
        for depth in (8, 10, 12):
            dtype = np.uint8 if host_depth == 8 else np.uint16
            rows = np.arange(count, dtype=np.uint32).astype(dtype).reshape(1, count)
            desc = abi.EncodeDesc(count, 1, host_depth, 1, abi.ALPHA_NONE, depth)
            got = ref.encode(desc, rows)[0][0].astype(np.uint16)
            if host_depth == 8 and depth == 8:
                assert np.array_equal(got, rows[0])
            else:
                assert np.array_equal(got, port.depth_lut(host_depth, depth))


ENCODE_CASES = [c for c in cases.encode_cases(cases.SIZES, full=True) if c[3]]
DECODE_CASES = [c for c in cases.decode_cases(cases.SIZES, full=True) if c[3]]


@pytest.mark.parametrize("case", ENCODE_CASES, ids=[c[0] for c in ENCODE_CASES])
def test_encode_images_match(ref, port, case):
    _, desc, rows, _ = case
    assert cases.same_planes(ref.encode(desc, rows, pad=3), port.encode(desc, rows, pad=5))


@pytest.mark.parametrize("case", DECODE_CASES, ids=[c[0] for c in DECODE_CASES])
def test_decode_images_match(ref, port, case):
    _, desc, planes, _ = case
    assert cases.same_bits(ref.decode(desc, planes), port.decode(desc, planes))


def test_multithreaded_drivers_equal_single_thread(ref, port):
    for c in (ref, port):
        name, desc, rows, _ = next(x for x in cases.encode_cases([(64, 16)], full=False) if "h32_c3" in x[0])
        assert cases.same_planes(c.encode(desc, rows, threads=1), c.encode(desc, rows, threads=5))
        name, desc, planes, _ = next(x for x in cases.decode_cases([(37, 23)], full=False) if "ch1" in x[0] and "ycc32" in x[0])
        assert cases.same_bits(c.decode(desc, planes, threads=1), c.decode(desc, planes, threads=4))


def test_error_behaviour_matches(ref, port):
    import oracle
    bad = [
        abi.DecodeDesc(4, 4, abi.COLORSPACE_YCBCR, abi.CHROMA_420, 10, abi.ALPHA_NONE, 32, None),            # nclx null
        abi.DecodeDesc(4, 4, abi.COLORSPACE_YCBCR, abi.CHROMA_420, 10, abi.ALPHA_NONE, 32, cases.NCLX_709()),  # sRGB transfer
        abi.DecodeDesc(4, 4, abi.COLORSPACE_MONOCHROME, abi.CHROMA_MONOCHROME, 10, abi.ALPHA_NONE, 32, cases.NCLX_2020_HLG()),
    ]
    for desc in bad:
        planes = cases.code_planes(np.random.default_rng(0), desc)
        messages = []
        for c in (ref, port):
            with pytest.raises(oracle.OracleError) as info:
                c.decode(desc, planes)
            assert info.value.status == abi.ERR_UNSUPPORTED
            messages.append(str(info.value))
        assert messages[0] == messages[1]
    hlg_odd = abi.DecodeDesc(4, 4, abi.COLORSPACE_YCBCR, abi.CHROMA_420, 10, abi.ALPHA_NONE, 32,
                             abi.Nclx(1, abi.PRIMARIES_BT709 + 3, abi.TRANSFER_CHAR_HLG, abi.MATRIX_BT709, 1))
    planes = cases.code_planes(np.random.default_rng(0), hlg_odd)
    for c in (ref, port):
        with pytest.raises(oracle.OracleError):
            c.decode(hlg_odd, planes)
    gray_428 = abi.EncodeDesc(4, 4, 32, 1, abi.ALPHA_NONE, 12, abi.TRANSFER_SMPTE428)
    for c in (ref, port):
        with pytest.raises(oracle.OracleError):
            c.encode(gray_428, np.zeros((4, 4), np.float32))
