"""10-bit (kvz_pixel = uint16_t) coverage: the oracle's 10-bit build pinned against the reference's 10-bit build (CPU),
and the CUDA kernels' 16-bit instantiations against the oracle (GPU).  The reference's own unit suites are compiled
out at 10 bits (tests/tests_main.c:38-44), so the differential test against generic C is the pin here."""
import numpy as np
import pytest

import _cases as cs

U16 = np.uint16


def rp(r, n, kind="uniform"):
    return cs.rand_pix(r, n, U16, kind)


# ------------------------------------------------------------------------------------------------ CPU: oracle vs reference
def test_oracle10_picture_vs_reference(orc10, ref10):
    r = cs.rng(1)
    assert orc10.bitdepth == 10
    for n in (4, 8, 16, 32, 64):
        for kind in cs.KINDS:
            a, b = rp(r, n * n, kind), rp(r, n * n)
            assert orc10.sad_nxn(n, a, b) == ref10.nxn("sad", n, a, b)
            assert orc10.satd_nxn(n, a, b) == ref10.nxn("satd", n, a, b)
    a, b = rp(r, 96 * 64), rp(r, 80 * 64, "smooth")
    for (w, h) in [(8, 8), (16, 12), (12, 16), (64, 64), (24, 32), (4, 8)]:
        assert orc10.reg_sad(a, b, w, h, 96, 80) == ref10.reg_sad(a, b, w, h, 96, 80)
        assert orc10.satd_any_size(w, h, a, 96, b, 80) == ref10.satd_any_size(w, h, a, 96, b, 80)
    for width in (4, 8, 16, 32, 64):
        assert orc10.pixels_calc_ssd(a, b, 96, 80, width) == ref10.pixels_calc_ssd(a, b, 96, 80, width)
    data = rp(r, 520 * 300)
    assert np.array_equal(orc10.array_checksum(data, 300, 520, 520), ref10.array_checksum(data, 300, 520, 520))


def test_oracle10_intra_ipol_sao_quant_vs_reference(orc10, ref10):
    r = cs.rng(2)
    for log2w in (2, 3, 4, 5):
        top, left = cs.rand_refs(r, log2w, U16)
        for mode in range(35):
            for color in (0, 1):
                assert np.array_equal(orc10.intra_predict(log2w, mode, color, top, left, 1),
                                      ref10.intra_predict(log2w, mode, color, top, left, 1)), (log2w, mode, color)
    stride = 40
    src = rp(r, stride * 40)
    src[: stride * 12] = rp(r, stride * 12, "extreme")
    org = 8 * stride + 8
    for (w, h) in [(8, 8), (16, 12), (4, 4)]:
        for mvx in range(4):
            for mvy in range(4):
                for k in ("luma", "luma_hi", "chroma", "chroma_hi"):
                    assert np.array_equal(orc10.sample(k, src, org, stride, w, h, mvx * 2, mvy * 2 + 1),
                                          ref10.sample(k, src, org, stride, w, h, mvx * 2, mvy * 2 + 1)), (k, w, h, mvx, mvy)
    for (bw, bh) in [(64, 64), (32, 32), (24, 40)]:
        orig = rp(r, bw * bh)
        rec = np.clip(orig.astype(int) + r.integers(-9, 10, bw * bh), 0, 1023).astype(U16)
        rec = cs.al(rec)
        for eo in range(4):
            assert np.array_equal(orc10.calc_sao_edge_dir(10, orig, rec, eo, bw, bh), ref10.calc_sao_edge_dir(orig, rec, eo, bw, bh))
            offs = r.integers(-7, 8, 5).astype(np.int32)
            assert orc10.sao_edge_ddistortion(10, orig, rec, bw, bh, eo, offs) == ref10.sao_edge_ddistortion(orig, rec, bw, bh, eo, offs)
        bands = r.integers(-7, 8, 4).astype(np.int32)
        assert orc10.sao_band_ddistortion(10, orig, rec, bw, bh, 11, bands) == ref10.sao_band_ddistortion(orig, rec, bw, bh, 11, bands)
    for n in (4, 8, 16, 32):
        s2 = rp(r, n * 64)
        pred = np.clip(s2.astype(int) + r.integers(-60, 61, s2.size), 0, 1023).astype(U16)
        pred = cs.al(pred)
        for color in ((0, 1) if n < 32 else (0,)):
            for signhide in (0, 1):
                o = orc10.quantize_residual(30, n, color, 0, 0, 1, 64, s2, pred, 1, signhide)
                g = ref10.quantize_residual(30, n, color, 0, 0, 1, 64, s2, pred, 1, signhide)
                assert o[0] == g[0] and np.array_equal(o[2], g[2])
                assert np.array_equal(o[1].reshape(n, 64)[:, :n], g[1].reshape(n, 64)[:, :n])


# ------------------------------------------------------------------------------------------------ GPU: CUDA vs oracle
def dev16(kb, a):
    return kb.to_dev(np.ascontiguousarray(a))          # uint16 travels as int16


@pytest.mark.gpu
def test_cuda10_picture(cuda_lib, orc10):
    kb = cuda_lib
    r = cs.rng(3)
    for n in (4, 8, 16, 32, 64):
        count = 65
        a = np.concatenate([rp(r, n * n, cs.KINDS[i % 3]) for i in range(count)])
        b = np.concatenate([rp(r, n * n) for _ in range(count)])
        sad = kb.sad_nxn_batch(n, dev16(kb, a), dev16(kb, b), count).cpu().numpy()
        satd = kb.satd_nxn_batch(n, dev16(kb, a), dev16(kb, b), count).cpu().numpy()
        for i in range(count):
            ai, bi = cs.al(a[i * n * n:(i + 1) * n * n]), cs.al(b[i * n * n:(i + 1) * n * n])
            assert sad[i] == orc10.sad_nxn(n, ai, bi) and satd[i] == orc10.satd_nxn(n, ai, bi), (n, i)
    sa, sb, rows = 208, 176, 100
    a, b = rp(r, sa * rows), rp(r, sb * rows, "smooth")
    shapes = [(w, h) for w in (4, 8, 12, 16, 32, 64) for h in (4, 8, 12, 16, 32, 64)]
    descs = np.zeros(len(shapes), kb.BLK)
    for i, (w, h) in enumerate(shapes):
        descs[i] = (int(r.integers(0, rows - 64)) * sa + int(r.integers(0, sa - 64)), int(r.integers(0, rows - 64)) * sb + int(r.integers(0, sb - 64)), w, h, 0, 0)
    sad = kb.block_cost_batch(kb.OP_REG_SAD, dev16(kb, a), sa, dev16(kb, b), sb, descs).cpu().numpy()
    satd = kb.block_cost_batch(kb.OP_SATD_ANY, dev16(kb, a), sa, dev16(kb, b), sb, descs).cpu().numpy()
    for i, d in enumerate(descs):
        w, h = int(d["w"]), int(d["h"])
        assert sad[i] == orc10.reg_sad(a[d["off_a"]:], b[d["off_b"]:], w, h, sa, sb)
        assert satd[i] == orc10.satd_any_size(w, h, a[d["off_a"]:], sa, b[d["off_b"]:], sb)
    data = rp(r, 520 * 300)
    assert np.array_equal(kb.array_checksum(dev16(kb, data), 300, 520, 520).cpu().numpy(), orc10.array_checksum(data, 300, 520, 520))


@pytest.mark.gpu
def test_cuda10_intra_rough_search_and_quant(cuda_lib, orc10):
    import torch
    kb = cuda_lib
    r = cs.rng(4)
    pic_w, pic_h = 72, 40
    src = rp(r, pic_w * pic_h, "smooth")
    rec = cs.al(np.clip(src.astype(int) + r.integers(-20, 21, src.size), 0, 1023).astype(U16))
    for log2w in (2, 3, 4, 5):
        w = 1 << log2w
        costs = kb.intra_rough_search_frame(log2w, dev16(kb, src), dev16(kb, rec), pic_w, pic_w, pic_h).cpu().numpy()
        bx, by = pic_w // w, pic_h // w
        for j in range(by):
            for i in range(bx):
                top, left = orc10.intra_build_reference(log2w, 0, i * w, j * w, pic_w, pic_h, rec, pic_w)
                blk = cs.al(np.ascontiguousarray(src.reshape(pic_h, pic_w)[j * w:(j + 1) * w, i * w:(i + 1) * w]).ravel())
                for mode in (0, 1, 2, 9, 10, 11, 18, 25, 26, 27, 34):
                    pred = cs.al(orc10.intra_predict(log2w, mode, 0, top, left, 1))
                    assert costs[j * bx + i, mode] == orc10.satd_nxn(w, pred, blk), (log2w, i, j, mode)
    stride = 64
    for n in (4, 8, 16, 32):
        s2 = rp(r, n * stride)
        pred = cs.al(np.clip(s2.astype(int) + r.integers(-60, 61, s2.size), 0, 1023).astype(U16))
        tus = np.zeros(1, kb.TU)
        tus[0] = (0, 0, 0, 0, n, 0, 0, 0, 1, 0, 0, 0)
        rec_t = torch.zeros(n * stride, dtype=torch.int16, device="cuda")
        coeff = torch.zeros(n * n, dtype=torch.int16, device="cuda")
        for signhide in (0, 1):
            has = kb.quantize_residual_batch(kb.quant_params(30, 10, 1, signhide), dev16(kb, s2), dev16(kb, pred), stride, rec_t, stride, coeff, tus)
            o = orc10.quantize_residual(30, n, 0, 0, 0, 1, stride, s2, pred, 1, signhide)
            assert int(has[0]) == o[0] and np.array_equal(coeff.cpu().numpy(), o[2]), (n, signhide)
            got = rec_t.cpu().numpy().view(U16).reshape(n, stride)[:, :n]
            assert np.array_equal(got, o[1].reshape(n, stride)[:, :n])


@pytest.mark.gpu
def test_cuda10_ipol_sao(cuda_lib, orc10):
    import torch
    kb = cuda_lib
    r = cs.rng(5)
    stride, rows = 96, 80
    src = rp(r, stride * rows)
    src[: stride * 30] = rp(r, stride * 30, "extreme")
    for kind, name in ((kb.IPOL_LUMA, "luma"), (kb.IPOL_LUMA_HI, "luma_hi"), (kb.IPOL_CHROMA, "chroma"), (kb.IPOL_CHROMA_HI, "chroma_hi")):
        descs = []
        w, h = 16, 12
        for k in range(12):
            y, x = int(r.integers(8, rows - 8 - h)), int(r.integers(8, stride - 8 - w))
            descs.append((y * stride + x, k * w * h, w, h, int(r.integers(0, 8)), int(r.integers(0, 8))))
        d = np.array(descs, kb.IPOL)
        dst = torch.zeros(12 * w * h, dtype=torch.int16, device="cuda")
        kb.sample_batch(kind, dev16(kb, src), stride, dst, w, d)
        out = dst.cpu().numpy()
        for t in d:
            want = orc10.sample(name, src, int(t["off_src"]), stride, w, h, int(t["mvx"]), int(t["mvy"]))
            got = out[t["off_dst"]: t["off_dst"] + w * h]
            assert np.array_equal(got.view(U16) if not name.endswith("_hi") else got, want.view(U16) if not name.endswith("_hi") else want), name
    bw, bh = 64, 48
    orig = rp(r, bw * bh)
    rec = cs.al(np.clip(orig.astype(int) + r.integers(-9, 10, bw * bh), 0, 1023).astype(U16))
    blks = np.array([(0, 0, bw, bh, 0, 0)], kb.SAO_BLK)
    stats = kb.sao_edge_stats_batch(10, dev16(kb, orig), dev16(kb, rec), blks).cpu().numpy()
    for eo in range(4):
        assert np.array_equal(stats[0, eo].ravel(), orc10.calc_sao_edge_dir(10, orig, rec, eo, bw, bh))
    offs = r.integers(-7, 8, (1, 5)).astype(np.int32)
    assert int(kb.sao_edge_ddistortion_batch(10, dev16(kb, orig), dev16(kb, rec), blks, [2], offs)[0]) == \
        orc10.sao_edge_ddistortion(10, orig, rec, bw, bh, 2, offs[0])
    bands = r.integers(-7, 8, (1, 4)).astype(np.int32)
    assert int(kb.sao_band_ddistortion_batch(10, dev16(kb, orig), dev16(kb, rec), blks, [11], bands)[0]) == \
        orc10.sao_band_ddistortion(10, orig, rec, bw, bh, 11, bands[0])


def test_oracle10_rdoq_vs_reference(orc10, ref10):
    """orc_rdoq with bitdepth 10 == kvz_rdoq of the 10-bit reference build (transform_shift, q_bits, error scale and the
    sign-hiding rd_factor all depend on the bit depth)."""
    from test_rdoq import synth_coeffs, lambda_for
    rng = np.random.default_rng(15)
    for n, count in ((4, 60), (8, 40), (16, 16), (32, 6)):
        for qp in (22, 34):
            coef = synth_coeffs(rng, n, count, energy=24.0 * 2.0 ** ((qp - 4) / 6.0))
            for signhide in (0, 1):
                for type_ in (0, 2):
                    if n == 32 and type_ == 2:
                        continue
                    cabac = ref10.init_contexts(qp, 2)
                    lam = lambda_for(qp) * float(rng.uniform(0.5, 2.0))
                    nz = 0
                    for i in range(count):
                        scan = int(rng.integers(0, 3)) if n <= 8 else 0
                        want = ref10.rdoq(coef[i].ravel(), n, qp, lam, cabac, type_, scan, 1, 0, signhide)
                        got = orc10.rdoq(coef[i].ravel(), n, qp, lam, cabac, type_, scan, 1, 0, signhide, bitdepth=10)
                        assert np.array_equal(want, got), (n, qp, signhide, type_, i)
                        nz += int(np.count_nonzero(want))
                    assert nz > 0


@pytest.mark.gpu
def test_cuda10_rdoq(cuda_lib, ref10):
    """kvz_cuda_rdoq_batch with bitdepth 10 == kvz_rdoq of the 10-bit reference build."""
    from kvazaar_b200 import api
    from test_rdoq import synth_coeffs, lambda_for
    rng = np.random.default_rng(16)
    for n, count in ((4, 120), (8, 80), (16, 40), (32, 12)):
        for qp, signhide in ((24, 0), (33, 1)):
            coef = synth_coeffs(rng, n, count, energy=24.0 * 2.0 ** ((qp - 4) / 6.0))
            tus = np.zeros(count, api.RDOQ_TU)
            tus["off_coef"] = tus["off_dest"] = np.arange(count) * n * n
            tus["scan_idx"] = rng.integers(0, 3, count) if n <= 8 else 0
            tus["block_type"] = 1
            cabac = ref10.init_contexts(qp, 2)
            lam = lambda_for(qp)
            got = api.rdoq_batch(api.to_dev(coef.ravel()), n, tus, cabac, qp, lam, 10, signhide).cpu().numpy().reshape(count, n * n)
            for i in range(count):
                want = ref10.rdoq(coef[i].ravel(), n, qp, lam, cabac, 0, int(tus["scan_idx"][i]), 1, 0, signhide)
                assert np.array_equal(want, got[i]), (n, qp, signhide, i)


def synth_frame10(W, H, idx):
    """10-bit I420 test frame: the 8-bit synthetic frame scaled by 4 plus two fresh low bits."""
    from test_framepass import synth_frame
    f8 = synth_frame(W, H, frame_idx=idx).astype(np.uint16)
    low = np.random.default_rng(idx).integers(0, 4, f8.size).astype(np.uint16)
    return (f8 * 4 + low).astype(np.uint16)


def test_reference_frame_pass_10bit_runs(ref10):
    """The CPU arm (oracle/ref_framepass.c in the KVZ_BIT_DEPTH=10 build) is deterministic and thread-count independent."""
    from _oracle import ref_frame_pass
    from kvazaar_b200 import api
    W, H, qp = 136, 72, 30
    src = synth_frame10(W, H, 2)
    lay = api.fp_layout_for(W, H, qp, 0, 10)
    a = ref_frame_pass(ref10, src, W, H, qp, lay, nthreads=1, rdoq=1)
    b = ref_frame_pass(ref10, src, W, H, qp, lay, nthreads=4, rdoq=1)
    assert np.array_equal(a, b)
    sec = api.fp_sections(lay, W, H, 10)
    assert api.fp_section(a, sec, "sao_rec").max() > 255 and api.fp_section(a, sec, "checksum").any()


PARITY10_CASES = [((136, 72), 30, 0, 0, 0), ((200, 136), 27, 1, 1, 0), ((320, 192), 34, 1, 1, 1)]
# the configs[4] shape at its full size: (dims, qp, signhide, rdoq, trskip, frame index)
FULL_SIZE10_CASE = ((7680, 4320), 22, 0, 1, 0, 3)


@pytest.mark.parametrize("dims,qp,signhide,rdoq,trskip", PARITY10_CASES)
def test_reference_frame_pass_10bit_matches_golden(ref10, dims, qp, signhide, rdoq, trskip):
    """the digests the GPU tests compare with are those of the 10-bit reference build's own pass"""
    from _golden import assert_matches_reference, fp_case
    from _oracle import ref_frame_pass
    from kvazaar_b200 import api
    W, H = dims
    lay = api.fp_layout_for(W, H, qp, signhide, 10)
    want = ref_frame_pass(ref10, synth_frame10(W, H, W + qp), W, H, qp, lay, nthreads=4, signhide=signhide, rdoq=rdoq, trskip=trskip)
    assert_matches_reference(want, api.fp_sections(lay, W, H, 10), fp_case(W, H, qp, signhide, rdoq, trskip, 10))


@pytest.mark.gpu
@pytest.mark.parametrize("dims,qp,signhide,rdoq,trskip", PARITY10_CASES)
def test_cuda10_frame_pass_matches_reference(cuda_lib, dims, qp, signhide, rdoq, trskip):
    """The whole frame-level pass on 10-bit samples (config-5 bit depth): blob identical to the pass through the 10-bit
    reference build's strategy functions (its digests, tests/_golden.py)."""
    from _golden import assert_matches_reference, fp_case
    kb = cuda_lib
    W, H = dims
    src = synth_frame10(W, H, W + qp)
    fp = kb.FramePass(W, H, qp, signhide, rdoq, 0.0, trskip, 10)
    fp.run_dev(kb.to_dev(src))
    got = fp.result_host()
    assert_matches_reference(got, kb.fp_sections(fp.layout, W, H, 10), fp_case(W, H, qp, signhide, rdoq, trskip, 10))
    fp.close()


@pytest.mark.gpu
def test_cuda10_frame_pass_full_size_4320p(cuda_lib):
    """The configs[4] shape at its full size (7680x4320 10-bit, QP22, RDOQ + deblocking + SAO): one frame, every section of
    the result blob equals the pass through the 10-bit reference build's strategy functions (its digests, tests/_golden.py)."""
    from _golden import assert_matches_reference, fp_case
    kb = cuda_lib
    (W, H), qp, signhide, rdoq, trskip, idx = FULL_SIZE10_CASE
    src = synth_frame10(W, H, idx)
    fp = kb.FramePass(W, H, qp, signhide, rdoq, 0.0, trskip, 10)
    fp.run_dev(kb.to_dev(src))
    got = fp.result_host()
    assert_matches_reference(got, kb.fp_sections(fp.layout, W, H, 10), fp_case(W, H, qp, signhide, rdoq, trskip, 10))
    fp.close()
