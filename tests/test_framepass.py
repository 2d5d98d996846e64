"""The frame-level pass: CPU checks of the reference arm (ref_framepass.c) and the GPU-vs-reference blob parity."""
import numpy as np
import pytest

import _cases as cs


def synth_frame(width, height, seed=1234, frame_idx=0):
    """Deterministic I420 frame: diagonal ramp + drifting low-frequency sinusoid + +-4 noise (SURVEY.md 8d)."""
    r = np.random.default_rng(seed + frame_idx)
    y, x = np.mgrid[0:height, 0:width]
    luma = (x + y) * 0.11 + 60 * np.sin((x + 3 * frame_idx) / 37.0) * np.cos(y / 29.0) + 128 + r.integers(-4, 5, (height, width))
    cy, cx = np.mgrid[0:height // 2, 0:width // 2]
    u = 128 + 40 * np.sin(cx / 23.0 + frame_idx * 0.1) + r.integers(-2, 3, cx.shape)
    v = 128 + 40 * np.cos(cy / 19.0) + r.integers(-2, 3, cx.shape)
    return np.concatenate([np.clip(p, 0, 255).astype(np.uint8).ravel() for p in (luma, u, v)])


def test_layout_needs_no_gpu():
    import kvazaar_b200 as kb
    lay = kb.fp_layout_for(1920, 1080)
    assert list(lay.nblk) == [60 * 33, 120 * 67, 240 * 135, 480 * 270]
    assert lay.nctu == 30 * 17
    assert lay.host_bytes > 1920 * 1080 * 3 // 2


def test_expand_compact_host_helper():
    """kvz_cuda_fp_expand_compact is plain host code: bitmap + packed chunks -> dense region (no GPU needed)."""
    import ctypes as C
    from kvazaar_b200 import api, lib
    lay = api.fp_layout_for(128, 64)
    n = int(lay.n_chunks)
    rng = np.random.default_rng(9)
    region = np.zeros((n, 32), np.uint8)
    nz = rng.random(n) < 0.07
    region[nz] = rng.integers(1, 256, (int(nz.sum()), 32), dtype=np.uint8)
    hdr = int(lay.compact_header_bytes)
    compact = np.zeros(hdr + 32 * int(nz.sum()), np.uint8)
    compact[:8].view(np.uint32)[:] = (int(nz.sum()), n)
    bits = np.packbits(nz, bitorder="little")
    compact[256:256 + bits.size] = bits
    compact[hdr:] = region[nz].ravel()
    out = np.full(n * 32, 0xAA, np.uint8)
    rc = lib().kvz_cuda_fp_expand_compact(C.byref(lay), C.c_void_p(compact.ctypes.data), C.c_size_t(compact.size), C.c_void_p(out.ctypes.data))
    assert rc == 0 and np.array_equal(out, region.ravel())
    # truncated buffer is refused
    assert lib().kvz_cuda_fp_expand_compact(C.byref(lay), C.c_void_p(compact.ctypes.data), C.c_size_t(compact.size - 32), C.c_void_p(out.ctypes.data)) != 0
    # the numpy expansion used by the GPU tests agrees
    small = np.zeros(int(lay.coeff_begin), np.uint8)
    assert np.array_equal(api.fp_expand_compact(lay, small, compact)[int(lay.coeff_begin):], region.ravel())


def test_reference_frame_pass_is_self_consistent(ref, orc):
    """The CPU arm against independent oracle computations on a small frame."""
    import kvazaar_b200 as kb
    W, H, qp = 136, 72, 27
    src = synth_frame(W, H)
    lay = kb.fp_layout_for(W, H, qp)
    blob = __import__("_oracle").ref_frame_pass(ref, src, W, H, qp, lay, nthreads=4)
    sec = kb.fp_sections(lay, W, H)
    g = lambda n: kb.fp_section(blob, sec, n)  # noqa: E731
    luma = cs.al(src[: W * H])
    # depth 2 (8x8): recompute block (3, 2) with the oracle only
    d, w, bx, by = 2, 8, 3, 2
    b = by * (W // w) + bx
    top, left = orc.intra_build_reference(3, 0, bx * w, by * w, W, H, luma, W)
    blk = cs.al(np.ascontiguousarray(luma.reshape(H, W)[by * w:(by + 1) * w, bx * w:(bx + 1) * w]).ravel())
    costs = [orc.satd_nxn(w, cs.al(orc.intra_predict(3, m, 0, top, left, 1)), blk) for m in range(35)]
    assert g("mode_y2")[b] == int(np.argmin(costs)) and g("cost_y2")[b] == min(costs)
    mode = int(g("mode_y2")[b])
    pred = cs.al(orc.intra_predict(3, mode, 0, top, left, 1))
    scan = 2 if 6 <= mode <= 14 else (1 if 22 <= mode <= 30 else 0)
    has, rec, coeff = orc.quantize_residual(qp, w, 0, scan, 0, 1, w, blk, pred)
    assert g("has_y2")[b] == has
    assert np.array_equal(g("coeff_y2")[b * 64:(b + 1) * 64], coeff)
    assert g("ssd_y2")[b] == orc.pixels_calc_ssd(blk, rec, w, w, w)
    # checksum section == oracle checksum of the SAO-filtered planes
    sao_rec = g("sao_rec")
    for c, (off, pw, ph) in enumerate([(0, W, H), (W * H, W // 2, H // 2), (W * H * 5 // 4, W // 2, H // 2)]):
        assert np.array_equal(g("checksum")[4 * c: 4 * c + 4], orc.array_checksum(cs.al(sao_rec[off: off + pw * ph]), ph, pw, pw))
    # threads do not change the result
    blob1 = __import__("_oracle").ref_frame_pass(ref, src, W, H, qp, lay, nthreads=1)
    assert np.array_equal(blob, blob1)


PARITY_CASES = [((136, 72), 27, 0, 0), ((200, 136), 27, 0, 0), ((320, 192), 27, 0, 0),
                ((200, 136), 22, 1, 0), ((136, 72), 37, 1, 0), ((320, 192), 17, 1, 0),
                ((200, 136), 27, 0, 1), ((320, 192), 22, 1, 1), ((136, 72), 32, 0, 1),
                ((320, 192), 22, 1, 3), ((200, 136), 27, 0, 2), ((136, 72), 17, 1, 3)]
# the BASELINE configs[1] and configs[2] shapes at their full sizes: (dims, qp, signhide, rdoq, trskip, frame_idx)
FULL_SIZE_CASES = {"1080p_medium": ((1920, 1080), 27, 0, 1, 0, 5), "2160p_veryslow": ((3840, 2160), 22, 1, 1, 1, 7)}


def parity_frame(W, H, qp, trskip):
    """the source of a PARITY_CASES case"""
    src = synth_frame(W, H, frame_idx=W + qp)
    if trskip:                                              # text-like content in a corner so that transform skip wins somewhere
        y = src[:W * H].reshape(H, W)
        y[:64, :64] = np.where((np.add.outer(np.arange(64), np.arange(64)) // 3) % 2, 40, 220).astype(np.uint8)
    return src


@pytest.mark.parametrize("dims,qp,signhide,rdoq", PARITY_CASES)
def test_reference_frame_pass_matches_golden(ref, dims, qp, signhide, rdoq):
    """the digests the GPU tests compare with are those of the reference's own pass"""
    import kvazaar_b200 as kb
    from _golden import assert_matches_reference, fp_case
    from _oracle import ref_frame_pass
    W, H = dims
    trskip, rdoq = rdoq >> 1, rdoq & 1
    lay = kb.fp_layout_for(W, H, qp, signhide)
    want = ref_frame_pass(ref, parity_frame(W, H, qp, trskip), W, H, qp, lay, nthreads=4, signhide=signhide, rdoq=rdoq, trskip=trskip)
    assert_matches_reference(want, kb.fp_sections(lay, W, H), fp_case(W, H, qp, signhide, rdoq, trskip))


@pytest.mark.gpu
@pytest.mark.parametrize("dims,qp,signhide,rdoq", PARITY_CASES)
def test_cuda_frame_pass_matches_reference(cuda_lib, dims, qp, signhide, rdoq):
    """Byte-identical result blob: CUDA frame pass vs the reference's own strategy functions (medium-like:
    signhide off; veryslow-like: QP 22 with sign-bit hiding; rdoq = 1: kvz_rdoq instead of kvz_quant, as medium and
    veryslow configure it), through the digests of the reference's blob (tests/_golden.py)."""
    import torch
    from _golden import assert_matches_reference, fp_case
    kb = cuda_lib
    W, H = dims
    trskip, rdoq = rdoq >> 1, rdoq & 1                     # bit 1 of the parameter: also try transform skip on 4x4 luma (veryslow)
    case = fp_case(W, H, qp, signhide, rdoq, trskip)
    src = parity_frame(W, H, qp, trskip)
    fp = kb.FramePass(W, H, qp, signhide, rdoq, 0.0, trskip)
    fp.run_dev(kb.to_dev(src))
    got = fp.result_host()
    sec = kb.fp_sections(fp.layout, W, H)
    assert_matches_reference(got, sec, case)
    if trskip:
        flags = kb.fp_section(got, sec, "trskip_y")
        assert 0 < int(flags.sum()) < flags.size, "transform skip never (or always) chosen: the case does not exercise the choice"
    # host-buffer entry point gives the same blob
    src_pin = torch.from_numpy(src.copy()).pin_memory()
    res_pin = torch.empty(fp.host_bytes, dtype=torch.uint8).pin_memory()
    fp.run_host(src_pin, res_pin)
    torch.cuda.synchronize()
    assert_matches_reference(res_pin.numpy(), sec, case)
    # compact result (bitmap + non-zero coefficient chunks) expands to the same blob
    L = fp.layout
    assert int(L.coeff_begin) + 32 * int(L.n_chunks) == fp.host_bytes
    small = torch.zeros(int(L.coeff_begin), dtype=torch.uint8).pin_memory()
    compact = torch.zeros(int(L.compact_header_bytes) + 32 * int(L.n_chunks), dtype=torch.uint8).pin_memory()
    fp.run_host_compact(src_pin, small, compact, int(L.n_chunks))
    torch.cuda.synchronize()
    full = kb.fp_expand_compact(L, small.numpy(), compact.numpy())
    assert np.array_equal(full, res_pin.numpy()), "compact result does not expand to the full blob"
    nonzero = int(compact.numpy()[:4].view(np.uint32)[0])
    assert 0 < nonzero < int(L.n_chunks)                      # dense at low QP on tiny frames, ~5 % at 1080p QP27
    fp.close()


@pytest.mark.gpu
def test_cuda_frame_pass_full_size_1080p_medium(cuda_lib):
    """BASELINE configs[1] at its full size (1920x1080, QP27, RDOQ + deblocking + SAO): every section of the result blob
    equals the pass through the reference's strategy functions (its digests, tests/_golden.py); the compact result expands
    to the same bytes."""
    import torch
    from _golden import assert_matches_reference, fp_case
    kb = cuda_lib
    (W, H), qp, signhide, rdoq, trskip, idx = FULL_SIZE_CASES["1080p_medium"]
    src = synth_frame(W, H, frame_idx=idx)
    fp = kb.FramePass(W, H, qp, signhide, rdoq, 0.0, trskip)
    src_pin = torch.from_numpy(src.copy()).pin_memory()
    res_pin = torch.empty(fp.host_bytes, dtype=torch.uint8).pin_memory()
    fp.run_host(src_pin, res_pin)
    torch.cuda.synchronize()
    assert_matches_reference(res_pin.numpy(), kb.fp_sections(fp.layout, W, H), fp_case(W, H, qp, signhide, rdoq, trskip))
    L = fp.layout
    small = torch.zeros(int(L.coeff_begin), dtype=torch.uint8).pin_memory()
    compact = torch.zeros(int(L.compact_header_bytes) + 32 * (int(L.n_chunks) // 8), dtype=torch.uint8).pin_memory()
    fp.run_host_compact(src_pin, small, compact, int(L.n_chunks) // 8)
    torch.cuda.synchronize()
    assert np.array_equal(kb.fp_expand_compact(L, small.numpy(), compact.numpy()), res_pin.numpy())
    fp.close()


@pytest.mark.gpu
def test_cuda_frame_pass_full_size_2160p_veryslow_shape(cuda_lib):
    """The configs[2] shape at its full size (3840x2160, QP22, RDOQ + sign hiding + transform-skip choice + deblocking +
    SAO): one frame, every section of the result blob equals the pass through the reference's strategy functions (its
    digests, tests/_golden.py)."""
    import torch
    from _golden import assert_matches_reference, fp_case
    kb = cuda_lib
    (W, H), qp, signhide, rdoq, trskip, idx = FULL_SIZE_CASES["2160p_veryslow"]
    src = synth_frame(W, H, frame_idx=idx)
    fp = kb.FramePass(W, H, qp, signhide, rdoq, 0.0, trskip)
    src_pin = torch.from_numpy(src.copy()).pin_memory()
    res_pin = torch.empty(fp.host_bytes, dtype=torch.uint8).pin_memory()
    fp.run_host(src_pin, res_pin)
    torch.cuda.synchronize()
    assert_matches_reference(res_pin.numpy(), kb.fp_sections(fp.layout, W, H), fp_case(W, H, qp, signhide, rdoq, trskip))
    fp.close()
