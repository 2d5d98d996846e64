"""ctypes access to the parity checkers (TEST INFRASTRUCTURE ONLY).

* ``Oracle``  -- oracle/libkvz_oracle.so, our plain-C restatement of the reference's
  generic strategies (oracle/kvz_oracle.c).
* ``Ref``     -- oracle/_ref/libkvzref_shim.so, the UNMODIFIED reference compiled from
  /root/reference (oracle/Makefile `ref` target) behind oracle/ref_shim.c.

Nothing in kvazaar_b200/ imports this module.
"""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
REF_DIR = os.path.join(ORACLE_DIR, "_ref")


def aligned(n, dtype, align=64, pad=64, fill=0):
    """`align`-byte aligned array with `pad` readable slack bytes behind it: the reference's SIMD
    strategies use aligned loads / over-reads (MALLOC_SIMD_PADDED, SIMD_ALIGNMENT,
    src/global.h:244-268)."""
    item = np.dtype(dtype).itemsize
    raw = np.zeros(n * item + align + pad, np.uint8)
    off = (-raw.ctypes.data) % align
    out = raw[off:off + n * item].view(dtype)
    if fill:
        out[:] = fill
    return out


def al(a, dtype=None):
    a = np.asarray(a)
    out = aligned(a.size, dtype or a.dtype)
    out[:] = a.ravel()
    return out


def P(a):
    """numpy array -> void* (keeps no reference; caller holds the array)."""
    if a is None:
        return C.c_void_p(0)
    assert a.flags["C_CONTIGUOUS"] or a.ndim <= 1 or a.strides[-1] == a.itemsize
    return C.c_void_p(a.ctypes.data)


def build_oracle(bitdepth=8):
    so = os.path.join(ORACLE_DIR, "libkvz_oracle.so" if bitdepth == 8 else "libkvz_oracle_10b.so")
    src = os.path.join(ORACLE_DIR, "kvz_oracle.c")
    if not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.check_call(["make", "-s", "-C", ORACLE_DIR, "oracle"])
    return so


def build_ref(bitdepth=8):
    """The compiled reference shim that __graft_entry__.build() made under oracle/_ref (when the reference sources were
    there to build it from), or None; tests never compile the reference themselves."""
    so = os.path.join(REF_DIR, "libkvzref_shim.so" if bitdepth == 8 else "libkvzref_shim_10b.so")
    return so if os.path.exists(so) else None


class DbkParams(C.Structure):
    """orc_dbk_params / kvz_cuda_dbk_params (same field order)."""
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("qp", C.c_int32), ("beta_offset_div2", C.c_int32),
                ("tc_offset_div2", C.c_int32), ("slice_is_b", C.c_int32), ("per_cu_qp", C.c_int32),
                ("cu_stride_scu", C.c_int32), ("ref_LX", C.c_uint8 * 32)]


def make_cu_records(type_, depth, part_size, tr_depth, cbf, qp, mv_dir, mv, mv_ref):
    """Pack per-SCU field arrays into 20-byte records (the reference's cu_info_t layout on x86-64,
    src/cu.h:126-165; pinned against the compiled reference by tests/test_deblock.py)."""
    shape = np.shape(type_)
    r = np.zeros(shape + (20,), np.uint8)
    r[..., 0] = (np.asarray(type_) & 3) | ((np.asarray(depth) & 7) << 2) | ((np.asarray(part_size) & 7) << 5)
    r[..., 1] = np.asarray(tr_depth) & 7
    cbf = np.asarray(cbf).astype(np.uint16)
    r[..., 4] = cbf & 0xff
    r[..., 5] = cbf >> 8
    r[..., 6] = qp
    inter = np.asarray(type_) != 1
    mvb = np.ascontiguousarray(np.asarray(mv, np.int16)).view(np.uint8).reshape(shape + (8,))
    r[..., 8:16] = np.where(inter[..., None], mvb, 0)
    r[..., 16] = np.where(inter, np.asarray(mv_ref)[..., 0], 0)
    r[..., 17] = np.where(inter, np.asarray(mv_ref)[..., 1], 0)
    r[..., 18] = np.where(inter, (np.asarray(mv_dir) & 3) << 6, 0)
    return r


def random_cu_grid(rng, width, height, intra_only=False, p_split=(0.7, 0.6, 0.5), max_mv=24):
    """Random CU/TU quadtree per 64x64 LCU -> [rows_scu, stride_scu, 20] records (stride padded to whole LCUs,
    like kvz_cu_array_alloc, cu.c:113-131)."""
    ws, hs = (width + 63) // 64 * 16, (height + 63) // 64 * 16
    f = {k: np.zeros((hs, ws), np.int32) for k in ("type", "depth", "part", "trd", "cbf", "qp", "dir")}
    mv = np.zeros((hs, ws, 4), np.int16)
    mref = np.zeros((hs, ws, 2), np.uint8)

    def leaf(x, y, d):
        w = 16 >> d                                      # in SCUs
        intra = intra_only or rng.random() < 0.4
        if intra:
            part = 3 if (d == 3 and rng.random() < 0.5) else 0
        else:
            part = int(rng.integers(0, 8)) if d < 3 else int(rng.integers(0, 3))
            if d == 0 and part > 3:
                part = int(rng.integers(0, 3))
        trd = max(d, 1)
        if part == 3:
            trd = 4
        elif rng.random() < 0.5 and trd < 3:
            trd += 1
        sl = (slice(y, y + w), slice(x, x + w))
        f["type"][sl] = 1 if intra else 2
        f["depth"][sl] = d
        f["part"][sl] = part
        f["trd"][sl] = trd
        f["qp"][sl] = int(rng.integers(20, 40))
        # per-TU cbf bits for luma (bit 0x10 >> tr_depth) so cbf_is_set(cbf, tr_depth, Y) varies between TUs
        tw = max(16 >> trd, 1)
        for ty in range(y, y + w, tw):
            for tx in range(x, x + w, tw):
                f["cbf"][ty:ty + tw, tx:tx + tw] = (0x10 >> trd) if rng.random() < 0.5 else 0
        if not intra:
            # one motion per PU: approximate with per-half randomness so PU edges separate different motion
            for hy in range(2):
                for hx in range(2):
                    sub = (slice(y + hy * w // 2, y + (hy + 1) * w // 2 if w > 1 else y + 1),
                           slice(x + hx * w // 2, x + (hx + 1) * w // 2 if w > 1 else x + 1))
                    if w == 1 and (hx or hy):
                        continue
                    same = rng.random() < 0.5
                    base = rng.integers(-max_mv, max_mv + 1, 4)
                    f["dir"][sub] = int(rng.integers(1, 4))
                    mv[sub] = base if not same else np.array([4, -4, 8, 0])
                    mref[sub] = rng.integers(0, 2, 2)

    def rec(x, y, d):
        if d < 3 and rng.random() < p_split[d]:
            h = 8 >> d
            for dy in (0, h):
                for dx in (0, h):
                    rec(x + dx, y + dy, d + 1)
        else:
            leaf(x, y, d)

    for ly in range(0, hs, 16):
        for lx in range(0, ws, 16):
            rec(lx, ly, 0)
    return make_cu_records(f["type"], f["depth"], f["part"], f["trd"], f["cbf"], f["qp"], f["dir"], mv.reshape(hs, ws, 2, 2), mref)


class Oracle:
    def __init__(self, bitdepth=8):
        self.lib = C.CDLL(build_oracle(bitdepth))
        L = self.lib
        for name in ("orc_reg_sad", "orc_sad_nxn", "orc_satd_nxn", "orc_satd_any_size", "orc_pixels_calc_ssd",
                     "orc_ver_sad", "orc_hor_sad", "orc_coeff_abs_sum"):
            getattr(L, name).restype = C.c_uint32
        L.orc_pixel_var.restype = C.c_double
        L.orc_fast_coeff_cost.restype = C.c_double
        L.orc_fast_coeff_cost.argtypes = [C.c_void_p, C.c_int32, C.c_uint64]
        L.orc_coeff_abs_sum.argtypes = [C.c_void_p, C.c_size_t]
        L.orc_scan_table.restype = C.POINTER(C.c_uint32)
        self.bitdepth = L.orc_bitdepth()
        self.pix = np.uint8 if self.bitdepth == 8 else np.uint16

    # picture
    def reg_sad(self, a, b, w, h, s1, s2):
        return self.lib.orc_reg_sad(P(a), P(b), w, h, s1, s2)

    def sad_nxn(self, n, a, b):
        return self.lib.orc_sad_nxn(n, P(a), P(b))

    def satd_nxn(self, n, a, b):
        return self.lib.orc_satd_nxn(n, P(a), P(b))

    def _dual(self, fn, n, preds, orig):
        costs = np.zeros(2, np.uint32)
        fn(n, P(preds), P(orig), P(costs))
        return costs

    def sad_nxn_dual(self, n, preds, orig):
        return self._dual(self.lib.orc_sad_nxn_dual, n, preds, orig)

    def satd_nxn_dual(self, n, preds, orig):
        return self._dual(self.lib.orc_satd_nxn_dual, n, preds, orig)

    def satd_any_size(self, w, h, b1, s1, b2, s2):
        return self.lib.orc_satd_any_size(w, h, P(b1), s1, P(b2), s2)

    def satd_any_size_quad(self, w, h, preds4, stride, orig, orig_stride):
        ptrs = (C.c_void_p * 4)(*[p.ctypes.data for p in preds4])
        costs = np.zeros(4, np.uint32)
        valid = np.ones(4, np.int8)
        self.lib.orc_satd_any_size_quad(w, h, ptrs, stride, P(orig), orig_stride, 4, P(costs), P(valid))
        return costs

    def pixels_calc_ssd(self, ref, rec, rs, cs, width):
        return self.lib.orc_pixels_calc_ssd(P(ref), P(rec), rs, cs, width)

    def ver_sad(self, pic, ref, w, h, ps):
        return self.lib.orc_ver_sad(P(pic), P(ref), w, h, ps)

    def hor_sad(self, pic, ref, w, h, ps, rs, left, right):
        return self.lib.orc_hor_sad(P(pic), P(ref), w, h, ps, rs, left, right)

    def bipred_average_plane(self, l0, l1, l0_im, l1_im, w, h, dst_stride):
        dst = np.zeros(h * dst_stride, self.pix)
        self.lib.orc_bipred_average_plane(P(dst), dst_stride, P(l0), P(l1), int(l0_im), int(l1_im), w, h)
        return dst

    def pixel_var(self, buf):
        return self.lib.orc_pixel_var(P(buf), buf.size)

    # dct
    def _tr(self, fn, n, bitdepth, inp):
        out = np.zeros(n * n, np.int16)
        inp = np.ascontiguousarray(inp, np.int16)
        if n is None:
            fn(bitdepth, P(inp), P(out))
        else:
            fn(n, bitdepth, P(inp), P(out))
        return out

    def dct(self, n, bitdepth, inp):
        return self._tr(self.lib.orc_dct_nxn, n, bitdepth, inp)

    def idct(self, n, bitdepth, inp):
        return self._tr(self.lib.orc_idct_nxn, n, bitdepth, inp)

    def dst4(self, bitdepth, inp):
        out = np.zeros(16, np.int16)
        self.lib.orc_dst_4x4(bitdepth, P(np.ascontiguousarray(inp, np.int16)), P(out))
        return out

    def idst4(self, bitdepth, inp):
        out = np.zeros(16, np.int16)
        self.lib.orc_idst_4x4(bitdepth, P(np.ascontiguousarray(inp, np.int16)), P(out))
        return out

    # quant
    @staticmethod
    def qparams(qp, bitdepth=8, intra=1, signhide=0):
        return np.array([qp, bitdepth, intra, signhide], np.int32)

    def scan_table(self, scan_idx, log2):
        p = self.lib.orc_scan_table(scan_idx, log2)
        return np.ctypeslib.as_array(p, shape=(1 << (2 * log2),)).copy()

    def quant(self, qp, coef, w, h, type_, scan_idx, block_type, intra=1, signhide=0, bitdepth=None):
        q = np.zeros(w * h, np.int16)
        prm = self.qparams(qp, bitdepth or self.bitdepth, intra, signhide)
        self.lib.orc_quant(P(prm), P(coef), P(q), w, h, type_, scan_idx, block_type)
        return q

    def dequant(self, qp, q, w, h, type_, block_type, bitdepth=None):
        c = np.zeros(w * h, np.int16)
        prm = self.qparams(qp, bitdepth or self.bitdepth)
        self.lib.orc_dequant(P(prm), P(q), P(c), w, h, type_, block_type)
        return c

    def quantize_residual(self, qp, width, color, scan_idx, trskip, cu_intra, stride, ref, pred, intra_slice=1,
                          signhide=0, bitdepth=None, early_skip=0):
        rec = np.zeros(width * stride, self.pix)
        coeff = np.zeros(width * width, np.int16)
        prm = self.qparams(qp, bitdepth or self.bitdepth, intra_slice, signhide)
        has = self.lib.orc_quantize_residual(P(prm), width, color, scan_idx, trskip, cu_intra, stride, stride,
                                             P(ref), P(pred), P(rec), P(coeff), early_skip)
        return has, rec, coeff

    def coeff_abs_sum(self, c):
        return self.lib.orc_coeff_abs_sum(P(c), c.size)

    def fast_coeff_cost(self, c, width, weights):
        return self.lib.orc_fast_coeff_cost(P(c), width, weights)

    # intra
    def angular(self, log2w, mode, top, left):
        dst = np.zeros(1 << (2 * log2w), self.pix)
        self.lib.orc_angular_pred(log2w, mode, P(top), P(left), P(dst))
        return dst

    def planar(self, log2w, top, left):
        dst = np.zeros(1 << (2 * log2w), self.pix)
        self.lib.orc_intra_pred_planar(log2w, P(top), P(left), P(dst))
        return dst

    def filtered_dc(self, log2w, top, left):
        dst = np.zeros(1 << (2 * log2w), self.pix)
        self.lib.orc_intra_pred_filtered_dc(log2w, P(top), P(left), P(dst))
        return dst

    def intra_predict(self, log2w, mode, color, top, left, filter_boundary):
        dst = np.zeros(1 << (2 * log2w), self.pix)
        self.lib.orc_intra_predict(log2w, mode, color, P(top), P(left), P(dst), filter_boundary)
        return dst

    def intra_build_reference(self, log2w, color, lx, ly, pic_w, pic_h, plane, stride):
        n = 2 * (1 << log2w) + 1
        top = np.zeros(n, self.pix)
        left = np.zeros(n, self.pix)
        self.lib.orc_intra_build_reference(log2w, color, lx, ly, pic_w, pic_h, P(plane), stride, P(top), P(left))
        return top, left

    # ipol
    def sample(self, kind, src_arr, origin_off, stride, w, h, mvx, mvy, dst_stride=None):
        """kind in {'luma','luma_hi','chroma','chroma_hi'}; src_arr flat, origin_off = index of block origin."""
        ds = dst_stride or w
        hi = kind.endswith("_hi")
        dst = np.zeros(h * ds, np.int16 if hi else self.pix)
        fn = {"luma": self.lib.orc_sample_quarterpel_luma, "luma_hi": self.lib.orc_sample_quarterpel_luma_hi,
              "chroma": self.lib.orc_sample_octpel_chroma, "chroma_hi": self.lib.orc_sample_octpel_chroma_hi}[kind]
        fn(C.c_void_p(src_arr.ctypes.data + origin_off * src_arr.itemsize), stride, w, h, P(dst), ds, mvx, mvy)
        return dst

    IM_SIZE = (71 + 1) * 64 + 1
    FIRST_COLS = 71 + 1

    def fme_state(self):
        return (np.zeros(4 * 64 * 64, self.pix), np.zeros(5 * self.IM_SIZE, np.int16),
                np.zeros(5 * self.FIRST_COLS, np.int16))

    def filter_fme(self, stage, src_arr, origin_off, stride, w, h, state, fme_level, off_x, off_y):
        filt, im, cols = state
        self.lib.orc_filter_fme(stage, C.c_void_p(src_arr.ctypes.data + origin_off * src_arr.itemsize), stride, w, h,
                                P(filt), P(im), fme_level, P(cols), off_x, off_y)

    def get_extended_block(self, src, src_w, src_h, src_s, bx, by, bw, bh, pl, pr, pt, pb, pbs):
        buf = np.full((pt + bh + pb + pbs) * (pl + bw + pr) + 1, 0xAB, self.pix)
        out = (C.c_int * 3)()
        r = self.lib.orc_get_extended_block(P(src), src_w, src_h, src_s, bx, by, bw, bh, pl, pr, pt, pb, pbs, P(buf),
                                            C.byref(out, 0), C.byref(out, 4), C.byref(out, 8))
        return r, buf, tuple(out)

    # sao
    def calc_sao_edge_dir(self, bitdepth, orig, rec, eo, bw, bh):
        out = np.zeros(10, np.int32)
        self.lib.orc_calc_sao_edge_dir(bitdepth, P(orig), P(rec), eo, bw, bh, P(out))
        return out

    def sao_edge_ddistortion(self, bitdepth, orig, rec, bw, bh, eo, offsets):
        offsets = np.ascontiguousarray(offsets, np.int32)
        return self.lib.orc_sao_edge_ddistortion(bitdepth, P(orig), P(rec), bw, bh, eo, P(offsets))

    def sao_band_ddistortion(self, bitdepth, orig, rec, bw, bh, band_pos, bands):
        bands = np.ascontiguousarray(bands, np.int32)
        return self.lib.orc_sao_band_ddistortion(bitdepth, P(orig), P(rec), bw, bh, band_pos, P(bands))

    def sao_reconstruct_color(self, bitdepth, rec_arr, origin_off, sao_type, eo, band_position, offsets, stride,
                              new_stride, bw, bh, color):
        out = np.zeros(bh * new_stride, self.pix)
        bp = np.ascontiguousarray(band_position, np.int32)
        of = np.ascontiguousarray(offsets, np.int32)
        self.lib.orc_sao_reconstruct_color(bitdepth, C.c_void_p(rec_arr.ctypes.data + origin_off * rec_arr.itemsize),
                                           P(out), sao_type, eo, P(bp), P(of), stride, new_stride, bw, bh, color)
        return out

    # nal
    def array_checksum(self, data, height, width, stride):
        out = np.zeros(4, np.uint8)
        self.lib.orc_array_checksum(P(data), height, width, stride, P(out))
        return out

    # -- RDOQ
    def rdoq(self, coef, width, qp, lambda_, cabac_ctx, type_=0, scan_mode=0, block_type=1, tr_depth=0, signhide=0, bitdepth=8):
        class P_(C.Structure):
            _fields_ = [("lambda_", C.c_double), ("qp", C.c_int32), ("bitdepth", C.c_int32), ("signhide", C.c_int32), ("pad", C.c_int32)]
        prm = P_(lambda_, qp, bitdepth, signhide, 0)
        co = np.ascontiguousarray(coef, np.int16)
        cc = np.ascontiguousarray(cabac_ctx, np.uint8)
        dest = np.full(width * width, 0x55, np.int16)
        self.lib.orc_rdoq(C.byref(prm), P(cc), P(co), P(dest), width, type_, scan_mode, block_type, tr_depth)
        return dest

    # -- deblocking (frame level)
    def deblock_frame(self, y, u, v, cus, width, height, qp, beta=0, tc=0, slice_is_b=0, per_cu_qp=0, ref_lx=None):
        """y/u/v: flat planes (copied); cus: uint8 [rows_scu, stride_scu, 20].  Returns filtered (y, u, v)."""
        prm = DbkParams(width, height, qp, beta, tc, slice_is_b, per_cu_qp, cus.shape[1])
        if ref_lx is not None:
            C.memmove(prm.ref_LX, np.ascontiguousarray(ref_lx, np.uint8).ctypes.data, 32)
        y, u, v = y.copy(), u.copy(), v.copy()
        cus = np.ascontiguousarray(cus)
        self.lib.orc_deblock_frame(C.byref(prm), P(y), P(u), P(v), P(cus))
        return y, u, v


class Ref:
    """The compiled, unmodified reference (8-bit build, or the -DKVZ_BIT_DEPTH=10 build)."""

    def __init__(self, bitdepth=8):
        so = build_ref(bitdepth)
        if so is None:
            raise FileNotFoundError("oracle/_ref not built (build() builds it when the reference sources are present)")
        self.lib = C.CDLL(so)
        L = self.lib
        L.kvzref_find.restype = C.c_void_p
        L.kvzref_find.argtypes = [C.c_char_p, C.c_char_p]
        L.kvzref_selected.restype = C.c_void_p
        L.kvzref_selected.argtypes = [C.c_char_p]
        L.kvzref_selected_name.restype = C.c_char_p
        L.kvzref_selected_name.argtypes = [C.c_char_p]
        L.kvzref_scan_table.restype = C.POINTER(C.c_uint32)
        L.kvzref_ctx_open.restype = C.c_void_p
        L.kvzref_entry.restype = C.c_char_p
        assert L.kvzref_init() == 1
        self.pix = np.uint8 if L.kvzref_bitdepth() == 8 else np.uint16
        self._ctx = {}

    def ctx(self, qp=22, signhide=0, rdoq=0, w=64, h=64):
        key = (qp, signhide, rdoq, w, h)
        if key not in self._ctx:
            c = self.lib.kvzref_ctx_open(w, h, qp, signhide, rdoq)
            assert c
            self._ctx[key] = C.c_void_p(c)
        return self._ctx[key]

    def entries(self):
        out = []
        for i in range(self.lib.kvzref_count()):
            name = C.c_char_p()
            prio = C.c_int()
            t = self.lib.kvzref_entry(i, C.byref(name), C.byref(prio))
            out.append((t.decode(), name.value.decode(), prio.value))
        return out

    def fn(self, type_, impl, restype, *argtypes):
        p = self.lib.kvzref_find(type_.encode(), impl.encode() if impl else None)
        assert p, (type_, impl)
        return C.CFUNCTYPE(restype, *argtypes)(p)

    def selected_name(self, type_):
        return self.lib.kvzref_selected_name(type_.encode()).decode()

    # -- picture (plain typedefs; called straight through the registry pointer)
    def reg_sad(self, a, b, w, h, s1, s2, impl="generic"):
        f = self.fn("reg_sad", impl, C.c_uint, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_uint, C.c_uint)
        return f(P(a), P(b), w, h, s1, s2)

    def nxn(self, kind, n, a, b, impl="generic"):
        f = self.fn(f"{kind}_{n}x{n}", impl, C.c_uint, C.c_void_p, C.c_void_p)
        return f(P(a), P(b))

    def nxn_dual(self, kind, n, preds, orig, impl="generic"):
        f = self.fn(f"{kind}_{n}x{n}_dual", impl, None, C.c_void_p, C.c_void_p, C.c_uint, C.c_void_p)
        costs = aligned(2, np.uint32)
        f(P(preds), P(orig), 2, P(costs))
        return costs

    def satd_any_size(self, w, h, b1, s1, b2, s2, impl="generic"):
        f = self.fn("satd_any_size", impl, C.c_uint, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int)
        return f(w, h, P(b1), s1, P(b2), s2)

    def satd_any_size_quad(self, w, h, preds4, stride, orig, orig_stride, impl="generic"):
        f = self.fn("satd_any_size_quad", impl, None, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                    C.c_uint, C.c_void_p, C.c_void_p)
        ptrs = (C.c_void_p * 4)(*[p.ctypes.data for p in preds4])
        costs = aligned(4, np.uint32)
        valid = aligned(4, np.int8, fill=1)
        f(w, h, C.cast(ptrs, C.c_void_p), stride, P(orig), orig_stride, 4, P(costs), P(valid))
        return costs

    def pixels_calc_ssd(self, ref, rec, rs, cs, width, impl="generic"):
        f = self.fn("pixels_calc_ssd", impl, C.c_uint, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int)
        return f(P(ref), P(rec), rs, cs, width)

    def ver_sad(self, pic, ref, w, h, ps, impl="generic"):
        f = self.fn("ver_sad", impl, C.c_uint32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_uint32)
        return f(P(pic), P(ref), w, h, ps)

    def hor_sad(self, pic, ref, w, h, ps, rs, left, right, impl="generic"):
        f = self.fn("hor_sad", impl, C.c_uint32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_uint32, C.c_uint32,
                    C.c_uint32, C.c_uint32)
        return f(P(pic), P(ref), w, h, ps, rs, left, right)

    def pixel_var(self, buf, impl="generic"):
        f = self.fn("pixel_var", impl, C.c_double, C.c_void_p, C.c_uint32)
        return f(P(buf), buf.size)

    def bipred_average(self, px0, px1, im0, im1, pu_x, pu_y, pu_w, pu_h, flags0, flags1, impl="generic"):
        """px*/im* = dict(y=,u=,v=) of contiguous arrays; returns (rec_y[64*64], rec_u[32*32], rec_v)."""
        oy = aligned(64 * 64, self.pix)
        ou = aligned(32 * 32, self.pix)
        ov = aligned(32 * 32, self.pix)
        a = []
        for pl in "yuv":
            a += [P(px0[pl]), P(px1[pl]), P(im0[pl]), P(im1[pl])]
        self.lib.kvzref_bipred_average(impl.encode(), *a, pu_x, pu_y, pu_w, pu_h, flags0, flags1, P(oy), P(ou), P(ov))
        return oy, ou, ov

    # -- dct
    def transform(self, name, bitdepth, inp, n, impl="generic"):
        f = self.fn(name, impl, None, C.c_int8, C.c_void_p, C.c_void_p)
        out = aligned(n * n, np.int16)
        inp = al(inp, np.int16)
        f(bitdepth, P(inp), P(out))
        return out

    def dct_coef(self, n, k, i):
        return self.lib.kvzref_dct_coef(n, k, i)

    def scan_table(self, scan_idx, log2):
        p = self.lib.kvzref_scan_table(scan_idx, log2)
        return np.ctypeslib.as_array(p, shape=(1 << (2 * log2),)).copy()

    # -- quant
    def quant(self, qp, coef, w, h, type_, scan_idx, block_type, intra=1, signhide=0, impl="generic"):
        q = aligned(w * h, np.int16)
        coef = al(coef, np.int16)
        self.lib.kvzref_quant(self.ctx(qp, signhide), impl.encode(), qp, intra, P(coef), P(q), w, h, type_, scan_idx,
                              block_type)
        return q

    def dequant(self, qp, q, w, h, type_, block_type, impl="generic"):
        c = aligned(w * h, np.int16)
        q = al(q, np.int16)
        self.lib.kvzref_dequant(self.ctx(qp), impl.encode(), qp, P(q), P(c), w, h, type_, block_type)
        return c

    def quantize_residual(self, qp, width, color, scan_idx, trskip, cu_intra, stride, ref, pred, intra_slice=1,
                          signhide=0, early_skip=0, impl="generic"):
        rec = aligned(width * stride, self.pix)
        coeff = aligned(width * width, np.int16)
        has = self.lib.kvzref_quantize_residual(self.ctx(qp, signhide, 0), impl.encode(), qp, intra_slice, width, color,
                                                scan_idx, trskip, cu_intra, stride, stride, P(ref), P(pred), P(rec),
                                                P(coeff), early_skip)
        return has, rec, coeff

    def coeff_abs_sum(self, c, impl="generic"):
        f = self.fn("coeff_abs_sum", impl, C.c_uint32, C.c_void_p, C.c_size_t)
        return f(P(c), c.size)

    def fast_coeff_cost(self, c, width, weights, impl="generic"):
        f = self.fn("fast_coeff_cost", impl, C.c_double, C.c_void_p, C.c_int32, C.c_uint64)
        return f(P(c), width, weights)

    # -- intra
    def angular(self, log2w, mode, top, left, impl="generic"):
        f = self.fn("angular_pred", impl, None, C.c_int8, C.c_int8, C.c_void_p, C.c_void_p, C.c_void_p)
        dst = aligned(1 << (2 * log2w), self.pix)
        f(log2w, mode, P(top), P(left), P(dst))
        return dst

    def planar(self, log2w, top, left, impl="generic"):
        f = self.fn("intra_pred_planar", impl, None, C.c_int8, C.c_void_p, C.c_void_p, C.c_void_p)
        dst = aligned(1 << (2 * log2w), self.pix)
        f(log2w, P(top), P(left), P(dst))
        return dst

    def filtered_dc(self, log2w, top, left, impl="generic"):
        f = self.fn("intra_pred_filtered_dc", impl, None, C.c_int8, C.c_void_p, C.c_void_p, C.c_void_p)
        dst = aligned(1 << (2 * log2w), self.pix)
        f(log2w, P(top), P(left), P(dst))
        return dst

    def intra_predict(self, log2w, mode, color, top, left, filter_boundary):
        dst = aligned(1 << (2 * log2w), self.pix)
        self.lib.kvzref_intra_predict(log2w, mode, color, P(top), P(left), P(dst), filter_boundary)
        return dst

    def intra_build_reference(self, log2w, color, lx, ly, pic_w, pic_h, plane, stride):
        n = 2 * (1 << log2w) + 1
        top = aligned(n, self.pix)
        left = aligned(n, self.pix)
        self.lib.kvzref_intra_build_reference(log2w, color, lx, ly, pic_w, pic_h, P(plane), stride, P(top), P(left))
        return top, left

    # -- ipol
    def sample(self, kind, src_arr, origin_off, stride, w, h, mvx, mvy, dst_stride=None, impl="generic"):
        ds = dst_stride or w
        hi = kind.endswith("_hi")
        dst = aligned(h * ds, np.int16 if hi else self.pix)
        t = {"luma": "sample_quarterpel_luma", "luma_hi": "sample_quarterpel_luma_hi",
             "chroma": "sample_octpel_chroma", "chroma_hi": "sample_octpel_chroma_hi"}[kind]
        self.lib.kvzref_sample(self.ctx(), t.encode(), impl.encode(),
                               C.c_void_p(src_arr.ctypes.data + origin_off * src_arr.itemsize), stride, w, h, P(dst),
                               ds, mvx, mvy)
        return dst

    def fme_state(self):
        ims = self.lib.kvzref_ipol_im_size()
        fc = self.lib.kvzref_ipol_first_cols()
        return (aligned(4 * 64 * 64, self.pix), aligned(5 * ims, np.int16), aligned(5 * fc, np.int16))

    def filter_fme(self, stage, src_arr, origin_off, stride, w, h, state, fme_level, off_x, off_y, impl="generic"):
        filt, im, cols = state
        self.lib.kvzref_filter_fme(self.ctx(), impl.encode(), stage,
                                   C.c_void_p(src_arr.ctypes.data + origin_off * src_arr.itemsize), stride, w, h,
                                   P(filt), P(im), fme_level, P(cols), off_x, off_y)

    def get_extended_block(self, src, src_w, src_h, src_s, bx, by, bw, bh, pl, pr, pt, pb, pbs, impl="generic"):
        buf = aligned((pt + bh + pb + pbs) * (pl + bw + pr) + 1, self.pix, fill=0xAB)
        out = (C.c_int * 3)()
        r = self.lib.kvzref_get_extended_block(impl.encode(), P(src), src_w, src_h, src_s, bx, by, bw, bh, pl, pr, pt,
                                               pb, pbs, P(buf), C.byref(out, 0), C.byref(out, 4), C.byref(out, 8))
        return r, buf, tuple(out)

    # -- sao
    def calc_sao_edge_dir(self, orig, rec, eo, bw, bh, impl="generic"):
        out = aligned(10, np.int32)
        self.lib.kvzref_calc_sao_edge_dir(self.ctx(), impl.encode(), P(orig), P(rec), eo, bw, bh, P(out))
        return out

    def sao_edge_ddistortion(self, orig, rec, bw, bh, eo, offsets, impl="generic"):
        offsets = al(offsets, np.int32)
        return self.lib.kvzref_sao_edge_ddistortion(self.ctx(), impl.encode(), P(orig), P(rec), bw, bh, eo, P(offsets))

    def sao_band_ddistortion(self, orig, rec, bw, bh, band_pos, bands, impl="generic"):
        bands = al(bands, np.int32)
        return self.lib.kvzref_sao_band_ddistortion(self.ctx(), impl.encode(), P(orig), P(rec), bw, bh, band_pos,
                                                    P(bands))

    def sao_reconstruct_color(self, rec_arr, origin_off, sao_type, eo, band_position, offsets, stride, new_stride, bw,
                              bh, color, impl="generic"):
        out = aligned(bh * new_stride, self.pix)
        bp = al(band_position, np.int32)
        of = al(offsets, np.int32)
        self.lib.kvzref_sao_reconstruct_color(self.ctx(), impl.encode(),
                                              C.c_void_p(rec_arr.ctypes.data + origin_off * rec_arr.itemsize), P(out),
                                              sao_type, eo, P(bp), P(of), stride, new_stride, bw, bh, color)
        return out

    # -- deblocking (kvz_filter_deblock_lcu over every LCU of a frame)
    def deblock_frame(self, y, u, v, cus, width, height, qp, beta=0, tc=0, slice_type=2, per_cu_qp=0, ref_lx=None):
        y, u, v = al(y), al(u), al(v)
        cus = al(np.ascontiguousarray(cus).ravel())
        lx = al(np.asarray(ref_lx, np.uint8).ravel()) if ref_lx is not None else None
        rc = self.lib.kvzref_deblock_frame(self.ctx(qp, 0, 0, width, height), P(y), P(u), P(v), P(cus), cus.size // 20 // ((height + 63) // 64 * 16),
                                           qp, beta, tc, slice_type, per_cu_qp, P(lx))
        assert rc == 0
        return y, u, v

    def make_cu_info(self, type_, depth, part_size, tr_depth, cbf, qp, mv_dir, mv, mv_ref):
        out = aligned(32, np.uint8)
        mv_a, ref_a = al(mv, np.int16), al(mv_ref, np.uint8)          # keep the buffers alive across the call
        self.lib.kvzref_make_cu_info(type_, depth, part_size, tr_depth, cbf, qp, mv_dir, P(mv_a), P(ref_a), P(out))
        return out[:self.lib.kvzref_sizeof_cu_info()].copy()

    # -- RDOQ (kvz_rdoq, not a strategy)
    def cabac_ctx_size(self):
        return self.lib.kvzref_cabac_ctx_size()

    def cabac_ctx_offsets(self):
        out = aligned(16, np.int32)
        self.lib.kvzref_cabac_ctx_offsets(P(out))
        return out[:14].copy()

    def init_contexts(self, qp, slice_type):
        out = aligned(256, np.uint8)
        self.lib.kvzref_init_contexts(self.ctx(qp), qp, slice_type, P(out))
        return out[:self.cabac_ctx_size()].copy()

    def rdoq(self, coef, width, qp, lambda_, cabac_ctx, type_=0, scan_mode=0, block_type=1, tr_depth=0, signhide=0):
        coef = al(coef, np.int16)
        dest = aligned(width * width, np.int16)
        dest[:] = 0x55
        cc = al(cabac_ctx, np.uint8)
        self.lib.kvzref_rdoq(self.ctx(qp, signhide, 1), qp, C.c_double(lambda_), P(cc), P(coef), P(dest), width, type_, scan_mode,
                             block_type, tr_depth)
        return dest.copy()

    def coeff_cost(self, coeff, width, cabac_ctx, type_=0, scan_mode=0, tr_skip=0, signhide=0, trskip_enable=0, update=0, impl="generic"):
        """kvz_encode_coeff_nxn in only_count mode -> (bits, context models afterwards)."""
        self.lib.kvzref_coeff_cost.restype = C.c_double
        after = aligned(256, np.uint8)
        cc = al(cabac_ctx, np.uint8)
        co = al(coeff, np.int16)                                       # keep the buffer alive across the call
        bits = self.lib.kvzref_coeff_cost(self.ctx(27, signhide, 0), impl.encode(), P(cc), update, trskip_enable, P(co), width,
                                          type_, scan_mode, tr_skip, P(after))
        return float(bits), after[:self.cabac_ctx_size()].copy()

    # -- nal
    def array_checksum(self, data, height, width, stride, impl="generic"):
        out = aligned(4, np.uint8)
        self.lib.kvzref_array_checksum(impl.encode(), P(data), height, width, stride, P(out))
        return out


def ref_frame_pass(ref, src, width, height, qp, layout, nthreads=8, signhide=0, blob=None, src_is_aligned=False, rdoq=0, trskip=0):
    """The frame-level pass through the compiled reference's own (AVX2) strategy pointers -> result blob.
    `blob` may be a reusable aligned buffer (bench.py keeps allocation out of the timed region)."""
    L = ref.lib
    if blob is None:
        blob = aligned(int(layout.host_bytes), np.uint8)
    if not src_is_aligned:
        src = al(src)
    ctx = ref.ctx(qp, signhide, rdoq, width, height)
    L.kvzref_set_trskip(ctx, trskip)
    rc = L.kvzref_frame_pass(ctx, P(src), width, height, qp, C.byref(layout), P(blob), nthreads)
    assert rc == 0
    return blob


def ref_inter_pass(ref, cur, refframe, width, height, qp, search_range, layout, nthreads=8):
    """The frame-level inter pass through the compiled reference's own (AVX2) strategy pointers -> result blob."""
    blob = aligned(int(layout.host_bytes), np.uint8)
    cur, refframe = al(cur), al(refframe)
    ctx = ref.ctx(qp, 0, 0, width, height)
    rc = ref.lib.kvzref_inter_pass(ctx, P(cur), P(refframe), width, height, qp, search_range, C.byref(layout), P(blob), nthreads)
    assert rc == 0
    return blob
