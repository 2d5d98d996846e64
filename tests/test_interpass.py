"""The frame-level inter pass (ME full search -> fractional search -> motion compensation -> inter residual coding)."""
import numpy as np
import pytest

from test_framepass import synth_frame


def moving_pair(w, h, seed=5):
    """reference frame + a current frame that is the reference shifted by a fractional, spatially varying motion."""
    ref = synth_frame(w, h, seed=seed, frame_idx=0)
    r = np.random.default_rng(seed)
    y = ref[: w * h].reshape(h, w).astype(np.int32)
    sh = np.roll(y, (2, -3), (0, 1))
    cur_y = np.clip((sh + np.roll(sh, 1, 1) + np.roll(sh, 1, 0)) // 3 + r.integers(-3, 4, y.shape), 0, 255).astype(np.uint8)
    cur = ref.copy()
    cur[: w * h] = cur_y.ravel()
    cu = ref[w * h:].reshape(2, h // 2, w // 2)
    cur[w * h:] = np.roll(cu, (1, -1), (1, 2)).ravel()
    return cur, ref


def test_inter_layout_needs_no_gpu():
    import kvazaar_b200 as kb
    lay = kb.ip_layout_for(1920, 1080)
    assert (lay.pus_x, lay.pus_y, lay.npu) == (118, 65, 118 * 65)


def test_reference_inter_pass_finds_the_motion(ref):
    """Sanity of the CPU arm: the integer search recovers the global shift, SATD improves with the fractional search."""
    import kvazaar_b200 as kb
    from _oracle import ref_inter_pass
    W, H = 128, 96
    cur, rf = moving_pair(W, H)
    lay = kb.ip_layout_for(W, H, 27, 8)
    blob = ref_inter_pass(ref, cur, rf, W, H, 27, 8, lay, nthreads=4)
    sec = kb.ip_sections(lay, W, H)
    mv = kb.fp_section(blob, sec, "mv_int").reshape(-1, 2)
    # most PUs recover the (3, -2) shift (flat / clipped areas legitimately stay at 0); nothing leaves the window
    assert np.mean(mv[:, 1] == -2) >= 0.5 and np.all(np.abs(mv) <= 8), mv
    sat = kb.fp_section(blob, sec, "satd_best")
    assert np.all(sat < 16 * 16 * 255)
    blob1 = ref_inter_pass(ref, cur, rf, W, H, 27, 8, lay, nthreads=1)
    assert np.array_equal(blob, blob1)


PARITY_CASES = [((128, 96), 27, 8), ((208, 136), 32, 5), ((320, 192), 22, 8)]


@pytest.mark.parametrize("dims,qp,rng", PARITY_CASES)
def test_reference_inter_pass_matches_golden(ref, dims, qp, rng):
    """the digests the GPU tests compare with are those of the reference's own pass"""
    import kvazaar_b200 as kb
    from _golden import assert_matches_reference, ip_case
    from _oracle import ref_inter_pass
    W, H = dims
    cur, rf = moving_pair(W, H, seed=W)
    lay = kb.ip_layout_for(W, H, qp, rng)
    want = ref_inter_pass(ref, cur, rf, W, H, qp, rng, lay, nthreads=4)
    assert_matches_reference(want, kb.ip_sections(lay, W, H), ip_case(W, H, qp, rng))


@pytest.mark.gpu
@pytest.mark.parametrize("dims,qp,rng", PARITY_CASES)
def test_cuda_inter_pass_matches_reference(cuda_lib, dims, qp, rng):
    """Byte-identical result blob: CUDA inter pass vs the reference's own strategy functions (its digests, tests/_golden.py)."""
    import torch
    from _golden import assert_matches_reference, ip_case
    kb = cuda_lib
    W, H = dims
    cur, rf = moving_pair(W, H, seed=W)
    ip = kb.InterPass(W, H, qp, rng)
    ip.run_dev(kb.to_dev(cur), kb.to_dev(rf))
    got = ip.result_host()
    sec = kb.ip_sections(ip.layout, W, H)
    assert_matches_reference(got, sec, ip_case(W, H, qp, rng))
    cur_pin, ref_pin = torch.from_numpy(cur.copy()).pin_memory(), torch.from_numpy(rf.copy()).pin_memory()
    res_pin = torch.empty(ip.host_bytes, dtype=torch.uint8).pin_memory()
    ip.run_host(cur_pin, ref_pin, res_pin)
    torch.cuda.synchronize()
    assert_matches_reference(res_pin.numpy(), sec, ip_case(W, H, qp, rng))
    ip.close()
