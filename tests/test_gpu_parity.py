"""The parity tests proper (B200): every configuration of the path through the C ABI of libavifgpu.so against the
CPU checker -- the compiled reference where the reference has that path, the C restatement otherwise.
Integer outputs AND float outputs are compared bit for bit (the device libm reproduces glibc's results, so the
float transfer curves are held to 0 ULP, tighter than the 1 ULP north_star allows)."""
import ctypes as C
import os

import numpy as np
import pytest

import cases
from avifgpu import abi

pytestmark = pytest.mark.gpu

ENCODE_CASES = list(cases.encode_cases(cases.SIZES, full=True))
DECODE_CASES = list(cases.decode_cases(cases.SIZES, full=True))


def pick(checker_ref, checker_port, reference_ok):
    """The compiled reference (or, where oracle/_ref is not built, the restatement held to the reference's recorded
    results) for every case the reference has a path for; the restatement alone only where it has none.  Having neither
    is an error here, not a quiet downgrade: "bit-identical to the compiled reference" must not turn green against the
    restatement alone (AVIFGPU_ALLOW_RESTATEMENT=1 opts out explicitly)."""
    if reference_ok and checker_ref is None:
        if os.environ.get("AVIFGPU_ALLOW_RESTATEMENT") == "1":
            return checker_port
        pytest.fail("neither oracle/_ref/libavifref.so nor reference results recorded with this libm: build oracle/_ref where the "
                    "reference's sources are at hand (make -C oracle), or set AVIFGPU_ALLOW_RESTATEMENT=1 to compare against the restatement")
    return checker_ref if reference_ok else checker_port


@pytest.fixture(scope="module")
def checkers():
    import oracle
    return oracle.load_reference() or oracle.load_recorded_reference(), oracle.load_restatement()


@pytest.mark.parametrize("case", ENCODE_CASES, ids=[c[0] for c in ENCODE_CASES])
def test_encode_matches_checker(gpu, gpu_exact, checkers, case):
    _, desc, rows, reference_ok = case
    expected = pick(*checkers, reference_ok).encode(desc, rows, pad=2)
    # `gpu` builds step tables at first use (float hosts then go through table look-ups in every kernel), `gpu_exact`
    # never does (exact powf per sample): both must reproduce the checker.
    contexts = (gpu, gpu_exact) if desc.host_depth == 32 else (gpu,)
    for ctx in contexts:
        got = ctx.encode(desc, rows, pad=7)
        for k, (e, g) in enumerate(zip(expected, got)):
            assert (e is None) == (g is None)
            if e is not None:
                assert np.array_equal(e, g), f"plane {k}: {int((e != g).sum())} of {e.size} samples differ"
                assert (g.base[:, g.shape[1]:] == 0xCD).all(), "wrote into the row padding"


@pytest.mark.parametrize("case", DECODE_CASES, ids=[c[0] for c in DECODE_CASES])
def test_decode_matches_checker(gpu, checkers, case):
    _, desc, planes, reference_ok = case
    expected = pick(*checkers, reference_ok).decode(desc, planes)
    got = gpu.decode(desc, planes)
    if not cases.same_bits(expected, got):
        bad = np.flatnonzero(expected.view(np.uint32 if expected.dtype == np.float32 else expected.dtype).ravel() !=
                             got.view(np.uint32 if got.dtype == np.float32 else got.dtype).ravel())
        raise AssertionError(f"{bad.size} of {expected.size} samples differ; first at {bad[0]}: "
                             f"expected {expected.ravel()[bad[0]]!r} got {got.ravel()[bad[0]]!r}")


def test_row_blocks_equal_whole_image(gpu, checkers):
    """The FormatRecord drop-in converts theRect row blocks: any even-aligned partition must give the same planes."""
    port = checkers[1]
    w, h = 53, 31
    desc = abi.EncodeDesc(w, h, 32, 4, abi.ALPHA_STRAIGHT, 12, abi.TRANSFER_PQ, 80, abi.LAYOUT_PLANAR_YCBCR, abi.CHROMA_420,
                          abi.DOWN_FILTER_BOX, abi.GRAY16_LUT, cases.NCLX_2020_PQ())
    rows = cases.float_host_rows(np.random.default_rng(3), h, w, 4)
    expected = port.encode(desc, rows)
    planes = None
    for y0, n in ((0, 2), (2, 10), (12, 18), (30, 1)):
        planes = gpu.encode(desc, rows[y0:y0 + n], y0=y0, nrows=n, planes=planes)
    assert cases.same_planes(expected, planes)

    ddesc = abi.DecodeDesc(w, h, abi.COLORSPACE_YCBCR, abi.CHROMA_420, 10, abi.ALPHA_PREMULTIPLIED, 32, cases.NCLX_2020_HLG())
    src = cases.code_planes(np.random.default_rng(4), ddesc)
    expected = port.decode(ddesc, src)
    out = np.zeros_like(expected)
    for y0, n in ((0, 1), (1, 4), (5, 7), (12, 19)):  # decode blocks may start on odd rows
        gpu.decode(ddesc, src, y0=y0, nrows=n, out=out[y0:y0 + n])
    assert cases.same_bits(expected, out)


def test_bad_blocks_and_descriptions_are_rejected(gpu):
    import avifgpu
    desc = abi.EncodeDesc(8, 8, 8, 3, abi.ALPHA_NONE, 8, layout=abi.LAYOUT_PLANAR_YCBCR, chroma=abi.CHROMA_420)
    rows = np.zeros((8, 24), np.uint8)
    for y0, n in ((1, 2), (0, 3), (6, 4), (-1, 2)):
        with pytest.raises(avifgpu.AvifGpuError) as info:
            gpu.encode(desc, rows[:max(n, 1)], y0=y0, nrows=n)
        assert info.value.status == abi.ERR_BAD_PARAM
    bad = desc.copy(host_channels=4)  # alpha state NONE with 4 channels
    with pytest.raises(avifgpu.AvifGpuError):
        gpu.encode(bad, np.zeros((8, 32), np.uint8))
    gray_428 = abi.EncodeDesc(4, 4, 32, 1, abi.ALPHA_NONE, 12, abi.TRANSFER_SMPTE428)
    with pytest.raises(avifgpu.AvifGpuError) as info:
        gpu.encode(gray_428, np.zeros((4, 4), np.float32))
    assert info.value.status == abi.ERR_UNSUPPORTED and "Unsupported color transfer function." in info.value.message
    no_nclx = abi.DecodeDesc(4, 4, abi.COLORSPACE_YCBCR, abi.CHROMA_420, 10, abi.ALPHA_NONE, 32, None)
    with pytest.raises(avifgpu.AvifGpuError) as info:
        gpu.decode(no_nclx, cases.code_planes(np.random.default_rng(0), no_nclx))
    assert "The nclxProfile is null." in info.value.message


def test_empty_images(gpu):
    for w, h in ((0, 0), (0, 5), (5, 0)):
        desc = abi.EncodeDesc(w, h, 16, 3, abi.ALPHA_NONE, 10, layout=abi.LAYOUT_PLANAR_YCBCR, chroma=abi.CHROMA_420)
        gpu.encode(desc, np.zeros((h, w * 3), np.uint16))
        ddesc = abi.DecodeDesc(w, h, abi.COLORSPACE_YCBCR, abi.CHROMA_420, 10, abi.ALPHA_NONE, 16, None)
        out = gpu.decode(ddesc, [np.zeros(s, np.uint16) if s else None for s in abi.decode_plane_shapes(ddesc)])
        assert out.shape == (h, w * 3)


def test_device_pointer_entry_points(gpu, checkers):
    """avifgpu_*_rows_device on torch-owned HBM, on a non-default stream, with padded strides."""
    import torch
    import avifgpu
    port = checkers[1]
    dev = torch.device("cuda", gpu.device)
    w, h = 101, 46
    desc = abi.EncodeDesc(w, h, 32, 3, abi.ALPHA_NONE, 12, abi.TRANSFER_PQ, 80, abi.LAYOUT_PLANAR_YCBCR, abi.CHROMA_420,
                          abi.DOWN_FILTER_BOX, abi.GRAY16_LUT, cases.NCLX_2020_PQ())
    rows = cases.float_host_rows(np.random.default_rng(9), h, w, 3)
    expected = port.encode(desc, rows)
    stream = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(stream):
        d_rows = torch.zeros((h, w * 3 + 5), dtype=torch.float32, device=dev)
        d_rows[:, :w * 3] = torch.from_numpy(rows).to(dev)
        shapes = abi.encode_plane_shapes(desc)
        d_planes = [None if s is None else torch.full((s[0], s[1] + 3), 0x7777, dtype=torch.int16, device=dev) for s in shapes]
        views = [None if t is None else t[:, :s[1]] for t, s in zip(d_planes, shapes)]
        pl = avifgpu.planes_from_tensors(views)
        before = gpu.launch_count()
        gpu.encode_device(desc, d_rows.data_ptr(), d_rows.stride(0) * 4, pl, stream=stream.cuda_stream)
        assert gpu.launch_count() > before
    stream.synchronize()
    for e, t, s in zip(expected, d_planes, shapes):
        if e is not None:
            got = t.cpu().numpy().view(np.uint16)
            assert np.array_equal(got[:, :s[1]], e)
            assert (got[:, s[1]:] == 0x7777).all()

    ddesc = abi.DecodeDesc(w, h, abi.COLORSPACE_YCBCR, abi.CHROMA_420, 10, abi.ALPHA_NONE, 32, cases.NCLX_2020_HLG())
    src = cases.code_planes(np.random.default_rng(10), ddesc)
    expected = port.decode(ddesc, src)
    with torch.cuda.stream(stream):
        d_src = [None if p is None else torch.from_numpy(p.view(np.int16)).to(dev) for p in src]
        d_out = torch.zeros((h, w * 3), dtype=torch.float32, device=dev)
        gpu.decode_device(ddesc, avifgpu.planes_from_tensors(d_src), d_out.data_ptr(), d_out.stride(0) * 4, stream=stream.cuda_stream)
    stream.synchronize()
    assert cases.same_bits(expected, d_out.cpu().numpy())
