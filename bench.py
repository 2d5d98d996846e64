#!/usr/bin/env python
"""bench.py -- ENCODED frames/s at fixed QP with a bit-identical bitstream (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # the CUDA CTU search driver inside the reference encoder
    python bench.py --impl reference --steps K --warmup W    # the unmodified reference (its AVX2 strategies, all host threads)

Workload (default): BASELINE config 3 -- 3840x2160 8-bit synthetic I420, --preset veryslow -q 22 -p 1 (all-intra);
`--workload 1080p` = config 2 (1920x1080 --preset medium -q 27 -p 1).

One STEP = `frames_per_step` pictures encoded to HEVC.  Three numbers per run:
  e2e    the headline: pictures in HOST memory go through the unchanged libkvazaar API (kvz_stream_bench.c, the loop of
         src/encmain.c; steps timed from bitstream out to bitstream out, the pipeline kept full by untimed pictures after them) -- host->device copy of every picture, device search, device->host copy of CU records /
         coefficients / SAO / reconstruction, the reference's own CABAC + bitstream writer on the host threads -- and the
         .hevc comes out.  Same program, same loop, for the reference arm (linked against the unmodified library).
  value  the device side alone: pictures resident in HBM -> kvz_cuda_ctu_submit_device / wait_device (search, deblock,
         SAO, final picture; results left on the device), slots pictures in flight, timed with CUDA events.
  cpu_baseline  the unmodified reference on a bounded sample of the same clip; the CUDA arm encodes the same sample and
         the two .hevc files must be byte-identical (`bitstream_identical`).
Multi-GPU: all-intra pictures are independent; every rank encodes its own pictures on its own GPU with its share of
the host threads, no data-path collective ("weak" scaling); times are max over ranks (NCCL all-reduce of the event times).
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

# one hardware queue per picture stream (the default of 8 would cap the overlapping pictures at 8); must be in the
# environment before the CUDA context exists (libkvzcuda sets it too, for hosts that do not)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
REF_DIR = os.path.join(ROOT, "oracle", "_ref")

WORKLOADS = {
    "2160p": dict(w=3840, h=2160, preset="veryslow", qp=22, frames_per_step=16, ref_frames_per_step=12, sample=16, owf=44, slots=40,
                  name="BASELINE config 3: 3840x2160 8-bit synthetic I420, --preset veryslow -q 22 -p 1 (all-intra)"),
    "1080p": dict(w=1920, h=1080, preset="medium", qp=27, frames_per_step=64, ref_frames_per_step=64, sample=64, owf=84, slots=72,
                  name="BASELINE config 2: 1920x1080 8-bit synthetic I420, --preset medium -q 27 -p 1 (all-intra)"),
    "64x64": dict(w=64, h=64, preset="ultrafast", qp=32, frames_per_step=64, ref_frames_per_step=64, sample=16, owf=8, slots=8,
                  name="BASELINE config 1: 64x64 8-bit synthetic I420, --preset ultrafast -q 32 -p 1 (all-intra)"),
}
METRIC = "encoded frames/sec at fixed QP (bit-identical bitstream)"
DISTINCT = 8          # distinct synthetic pictures in the clip (cycled)
REF_COOLDOWN = 16     # untimed pictures after the timed steps (keeps the reference's pipeline full during the last step)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def config_of(wl):
    """identical for both arms: what is encoded, not how"""
    return {"workload": wl["name"], "resolution": f"{wl['w']}x{wl['h']}", "preset": wl["preset"], "qp": wl["qp"], "intra_period": 1,
            "bit_depth": 8, "clip": f"{DISTINCT} distinct synthetic pictures (tools/synth_yuv.py, seed 1234) cycled",
            "l2": "every picture is read once; the pictures in flight (> 126 MB) exceed L2"}


def clip_path(wl):
    from synth_yuv import synth_frame
    d = "/dev/shm" if os.path.isdir("/dev/shm") else "/tmp"
    p = os.path.join(d, f"kvz_bench_{wl['w']}x{wl['h']}_{DISTINCT}.yuv")
    size = wl["w"] * wl["h"] * 3 // 2 * DISTINCT
    if not (os.path.exists(p) and os.path.getsize(p) == size):
        tmp = p + f".{os.getpid()}"
        with open(tmp, "wb") as f:
            for i in range(DISTINCT):
                f.write(synth_frame(wl["w"], wl["h"], 1234, i).tobytes())
        os.replace(tmp, p)
    return p


def stream_bench(binary, clip, wl, out, frames_per_step, steps, warmup, cooldown=0, extra=(), env=None, timeout=1500):
    """one run of the streaming host (integration/kvz_stream_bench.c); returns its JSON line"""
    e = dict(os.environ)
    e.pop("KVZ_CTU_PROVIDER", None)
    e.update(env or {})
    cmd = [binary, clip, f"{wl['w']}x{wl['h']}", out, str(frames_per_step), str(steps), str(warmup), str(cooldown),
           f"preset={wl['preset']}", f"qp={wl['qp']}", "period=1", *extra]
    r = subprocess.run(cmd, env=e, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=timeout)
    if r.returncode != 0:
        raise RuntimeError(f"{os.path.basename(binary)} failed ({r.returncode}): {r.stderr[-1500:]}")
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1]
    res = json.loads(line)
    res["stderr_tail"] = r.stderr[-400:]
    return res


def sha(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for blk in iter(lambda: f.read(1 << 20), b""):
            h.update(blk)
    return h.hexdigest()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (one streaming nvidia-smi process, 100 ms period)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.proc, self.rows = index, None, []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            time.sleep(0.35)
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                out, _ = self.proc.communicate(timeout=5)
            except Exception:
                self.proc.kill()
                out = ""
            for ln in out.splitlines():
                c = [x.strip() for x in ln.split(",")]
                if len(c) >= 7:
                    self.rows.append(c)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows)
        reasons = [name for i, name in enumerate(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"))
                   if any(r[3 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "power_w_max": max(float(r[2]) for r in self.rows), "samples": len(self.rows)}


# ------------------------------------------------------------------------------------------------ reference arm
def run_reference(args, wl):
    """The unmodified reference (oracle/_ref, compiled from /root/reference by oracle/Makefile): its own encoder loop,
    its AVX2 strategies, all the host threads it wants.  Does not load any of this repository's libraries."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    binary = os.path.join(REF_DIR, "kvz_stream_bench_ref")
    clip = clip_path(wl)
    fps_step = args.frames_per_step or wl["ref_frames_per_step"]
    r = stream_bench(binary, clip, wl, "/tmp/kvz_bench_ref_arm.hevc", fps_step, args.steps, args.warmup, cooldown=REF_COOLDOWN)
    cores = os.cpu_count() or 1
    sample = f"{r['frames']} pictures ({args.steps} steps of {fps_step}) after {args.warmup} warm-up steps, unmodified reference through its public API, threads=auto"
    line = {"impl": "reference", "metric": METRIC, "value": r["fps"], "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1000.0 * r["seconds"] / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic", "config": config_of(wl), "frames_per_step": fps_step,
            "cpu_baseline": {"value": r["fps"], "unit": "frames/s", "cores": cores, "kind": "reference", "sample": sample},
            "e2e": {"value": r["fps"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "bitstream_sha256": sha("/tmp/kvz_bench_ref_arm.hevc"), "bitstream_bytes": r["bytes"]}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ CUDA arm
class Config(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "width", "height", "qp", "rdo", "pu_depth_intra_min", "pu_depth_intra_max", "rdoq_enable", "rdoq_skip", "signhide_enable",
        "trskip_enable", "sao_type", "deblock_enable", "deblock_beta", "deblock_tc", "cu_split_termination", "intra_rdo_et",
        "combine_intra_cus", "intra_chroma_search", "full_intra_search", "wpp", "pad")] + [("lambda_", C.c_double), ("lambda_sqrt", C.c_double)]


class DevResult(C.Structure):
    _fields_ = [("cu", C.c_void_p), ("coeff", C.c_void_p), ("sao", C.c_void_p), ("rec", C.c_void_p), ("cu_stride", C.c_int32),
                ("width_in_lcu", C.c_int32), ("height_in_lcu", C.c_int32), ("search_kernel_ms", C.c_float)]


# what the reference's presets set of the fields the intra CTU search reads (src/cfg.c:486-736)
PRESET_FIELDS = {
    "ultrafast": dict(rdo=0, pu=(2, 3), rdoq=0, signhide=0, trskip=0, sao=0),
    "medium": dict(rdo=0, pu=(1, 4), rdoq=1, signhide=0, trskip=0, sao=3),
    "veryslow": dict(rdo=3, pu=(1, 4), rdoq=1, signhide=1, trskip=1, sao=3),
}


def driver_config(wl):
    p = PRESET_FIELDS[wl["preset"]]
    c = Config()
    c.width, c.height, c.qp, c.rdo = wl["w"], wl["h"], wl["qp"], p["rdo"]
    c.pu_depth_intra_min, c.pu_depth_intra_max = p["pu"]
    c.rdoq_enable, c.rdoq_skip, c.signhide_enable, c.trskip_enable = p["rdoq"], 0, p["signhide"], p["trskip"]
    c.sao_type, c.deblock_enable, c.deblock_beta, c.deblock_tc = p["sao"], 1, 0, 0
    c.cu_split_termination, c.intra_rdo_et, c.combine_intra_cus, c.intra_chroma_search, c.full_intra_search, c.wpp = 0, 0, 1, 0, 0, 1
    c.lambda_ = 0.57 * 2.0 ** ((wl["qp"] - 12) / 3.0)        # fixed-QP lambda (rate_control.c:678-691)
    c.lambda_sqrt = float(np.sqrt(c.lambda_))
    return c


class _DevBuf:
    """a device pointer the driver returned, as an object torch.as_tensor can view without a copy"""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


CU_FIELDS = np.dtype([("type", "u1"), ("depth", "u1"), ("part_size", "u1"), ("tr_depth", "u1"), ("tr_skip", "u1"), ("qp", "u1"),
                      ("mode", "i1"), ("mode_chroma", "i1"), ("cbf", "<u2"), ("pad", "<u2")])        # kvz_cuda_ctu_cu
DUMP_ELEMENTS = 3_500_000        # per array: four float32 arrays stay under 64 MB


def dump_outputs(directory, wl, kept):
    """kept: {picture index: (cu, coeff, sao, rec) byte tensors on the device} of the last timed step.  Writes the four result
    arrays of kvz_cuda_ctu_wait_device over those pictures (in picture order) as float32 .npy files; an array larger than
    DUMP_ELEMENTS is replaced by a fixed sample of its elements (seed 0, the same for every build)."""
    os.makedirs(directory, exist_ok=True)
    w, h = wl["w"], wl["h"]
    order = sorted(kept)
    cu = np.stack([kept[i][0].cpu().numpy().view(CU_FIELDS) for i in order])
    arrays = {
        "cu": np.stack([cu[f] for f in CU_FIELDS.names if f != "pad"], -1).reshape(len(order), (h + 63) // 64 * 16, -1, len(CU_FIELDS) - 1),
        "coeff": np.stack([kept[i][1].cpu().numpy().view(np.int16) for i in order]),
        "sao": np.stack([kept[i][2].cpu().numpy().view(np.int32).reshape(-1, 2, 17) for i in order]),
        "rec": np.stack([kept[i][3].cpu().numpy() for i in order]),
    }
    for name, a in arrays.items():
        a = a.astype(np.float32)
        if a.size > DUMP_ELEMENTS:
            a = a.ravel()[np.sort(np.random.default_rng(0).integers(0, a.size, DUMP_ELEMENTS))]
        np.save(os.path.join(directory, f"{name}.npy"), a)


def device_leg(args, wl, local, frames_per_step, barrier):
    """`value`: pictures resident in HBM through the driver alone; returns (seconds for K steps, launches, mean search-kernel ms,
    slots, and with --dump-outputs the results of the last timed step's pictures as device copies)"""
    import torch
    import kvazaar_b200 as kb
    lib = C.CDLL(kb.LIB_PATH)
    lib.kvz_cuda_ctu_open.restype = C.c_void_p
    lib.kvz_cuda_ctu_open.argtypes = [C.POINTER(Config), C.c_int]
    lib.kvz_cuda_ctu_submit_device.argtypes = [C.c_void_p] * 4 + [C.c_int, C.c_int, C.c_void_p, C.c_double, C.c_double, C.c_int]
    lib.kvz_cuda_ctu_wait_device.argtypes = [C.c_void_p, C.c_int, C.POINTER(DevResult)]
    lib.kvz_cuda_ctu_release.argtypes = [C.c_void_p, C.c_int]
    lib.kvz_cuda_ctu_close.argtypes = [C.c_void_p]
    lib.kvz_cuda_ctu_launches.restype = C.c_uint64
    lib.kvz_cuda_ctu_launches.argtypes = [C.c_void_p]
    lib.kvz_cuda_last_error.restype = C.c_char_p
    cfg = driver_config(wl)
    slots = args.slots or (args.owf or wl["owf"]) + 1          # as many pictures in flight as the encoder keeps (owf + 1)
    enc = lib.kvz_cuda_ctu_open(C.byref(cfg), slots)
    if not enc:
        raise RuntimeError(f"kvz_cuda_ctu_open: {lib.kvz_cuda_last_error()}")
    ctx = np.zeros(192, np.uint8)
    assert lib.kvz_cuda_cabac_ctx_init(wl["qp"], 2, ctx.ctypes.data_as(C.c_void_p)) == 0          # KVZ_SLICE_I
    w, h = wl["w"], wl["h"]
    clip = np.fromfile(clip_path(wl), dtype=np.uint8).reshape(DISTINCT, w * h * 3 // 2)
    dev = torch.from_numpy(clip).cuda()
    torch.cuda.synchronize()
    kernel_ms = []

    # one continuous run, `slots` pictures in flight throughout: warm-up pictures, the timed pictures, and `slots` more so
    # that the pipeline is still full while the last timed pictures are searched.  The timed region is completion to
    # completion: from the moment the last warm-up picture is done to the moment the last timed picture is done.
    # A few host threads drive the pipeline (each keeps its share of the pictures in flight) so that a picture that
    # finishes early is not held up behind an older one -- the encoder waits with one worker per picture as well.
    n_warm, n_timed = args.warmup * frames_per_step, args.steps * frames_per_step
    total = n_warm + n_timed + slots
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    state = {"next": 0, "done": 0, "l0": lib.kvz_cuda_ctu_launches(enc), "l1": 0, "err": None}
    if n_warm == 0:
        e0.record()
    lock = threading.Lock()
    n_threads = min(8, slots)
    # --dump-outputs: the results of the last timed step's pictures are copied on the device (a side stream, synchronised
    # before the slot is released) and brought to the host after the run
    last_step = range(n_warm + n_timed - frames_per_step, n_warm + n_timed) if args.dump_outputs else range(0)
    kept = {}
    side = torch.cuda.Stream() if args.dump_outputs else None
    nctu = ((w + 63) // 64) * ((h + 63) // 64)
    sizes = ((h + 63) // 64 * 16 * ((w + 63) // 64) * 16 * CU_FIELDS.itemsize, nctu * 6144 * 2, nctu * 2 * 68, w * h * 3 // 2)

    def drive(share):
        try:
            torch.cuda.set_device(local)
            res = DevResult()
            pending = []
            while True:
                while len(pending) < share:
                    with lock:
                        i = state["next"]
                        if i >= total:
                            break
                        state["next"] = i + 1
                    base = dev[i % DISTINCT].data_ptr()
                    s = lib.kvz_cuda_ctu_submit_device(enc, base, base + w * h, base + w * h * 5 // 4, w, w // 2, ctx.ctypes.data,
                                                       cfg.lambda_, cfg.lambda_sqrt, wl["qp"])
                    if s < 0:
                        raise RuntimeError(f"submit: {lib.kvz_cuda_last_error()}")
                    pending.append((s, i))
                if not pending:
                    return
                s, i = pending.pop(0)
                if lib.kvz_cuda_ctu_wait_device(enc, s, C.byref(res)) != 0:
                    raise RuntimeError(f"wait: {lib.kvz_cuda_last_error()}")
                ms = res.search_kernel_ms
                if i in last_step:
                    with torch.cuda.stream(side):
                        copies = tuple(torch.as_tensor(_DevBuf(p, n), device="cuda").clone()
                                       for p, n in zip((res.cu, res.coeff, res.sao, res.rec), sizes))
                    side.synchronize()
                    with lock:
                        kept[i] = copies
                lib.kvz_cuda_ctu_release(enc, s)
                with lock:
                    state["done"] += 1
                    done = state["done"]
                    if n_warm < done <= n_warm + n_timed:
                        kernel_ms.append(ms)
                    if done == n_warm:
                        e0.record()
                        state["l0"] = lib.kvz_cuda_ctu_launches(enc)
                    if done == n_warm + n_timed:
                        e1.record()
                        state["l1"] = lib.kvz_cuda_ctu_launches(enc)
        except Exception as ex:  # pragma: no cover
            state["err"] = ex

    shares = [slots // n_threads + (1 if t < slots % n_threads else 0) for t in range(n_threads)]
    threads = [threading.Thread(target=drive, args=(sh,)) for sh in shares]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if state["err"]:
        raise state["err"]
    torch.cuda.synchronize()
    seconds = e0.elapsed_time(e1) / 1000.0
    l0, l1 = state["l0"], state["l1"]
    launches = int(l1 - l0)
    lib.kvz_cuda_ctu_close(enc)
    return seconds, launches, float(np.mean(kernel_ms)) if kernel_ms else None, slots, kept


def run_cuda(args, wl):
    import torch
    import torch.distributed as dist
    import kvazaar_b200 as kb

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    kb.init(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    fps_step = args.frames_per_step or wl["frames_per_step"]
    w, h = wl["w"], wl["h"]
    clip = clip_path(wl) if rank == 0 else None
    barrier()
    clip = clip_path(wl)
    ctu_bin = os.path.join(REF_DIR, "kvz_stream_bench_ctu")
    owf = args.owf or wl["owf"]
    # The worker that runs CTU (0,0) of a picture sleeps until the device has searched the picture, so the encoder gets
    # one worker per picture in flight on top of this rank's share of the host cores (the reference's CABAC stage).
    cores = max(4, (os.cpu_count() or 8) // world)
    threads = owf + 1 + cores
    env = {"KVZ_CTU_PROVIDER": kb.LIB_PATH, "CUDA_VISIBLE_DEVICES": os.environ.get("CUDA_VISIBLE_DEVICES", ",".join(str(i) for i in range(world))).split(",")[local]}
    extra = [f"owf={owf}", f"threads={threads}"]

    with ClockSampler(local) as clk:
        # ---- e2e: host pictures -> .hevc through the reference's API with the CTU job on the device
        barrier()
        r = stream_bench(ctu_bin, clip, wl, f"/tmp/kvz_bench_ctu_{rank}.hevc", fps_step, args.steps, args.warmup, cooldown=owf + 1, extra=extra, env=env)
        e2e_seconds = max_over_ranks(r["seconds"])
        # ---- value: the device side alone
        dev_seconds, launches, kernel_ms, slots, kept = device_leg(args, wl, local, fps_step, barrier)
        dev_seconds = max_over_ranks(dev_seconds)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs if world == 1 else os.path.join(args.dump_outputs, f"rank{rank}"), wl, kept)
    # N > 1: the two exchanges of SURVEY 8e (tile all-gather of a 4320p 10-bit picture, reference-frame broadcast) timed on
    # this process group -- they are not on the all-intra data path (pictures shard with no collective), this is their
    # hardware measurement; outside the timed regions, every rank takes part
    exchanges = None
    if world > 1:
        try:
            from kvazaar_b200.dist import measure_exchanges
            exchanges = measure_exchanges(torch.device("cuda", local))
        except Exception as ex:  # pragma: no cover
            exchanges = {"error": repr(ex)[:300]}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    frames = args.steps * fps_step * world
    nctu = ((w + 63) // 64) * ((h + 63) // 64)
    h2d = fps_step * (w * h * 3 // 2 + ((h + 63) // 64) * 192)
    d2h = fps_step * (((w + 63) // 64) * 16 * ((h + 63) // 64) * 16 * 12 + nctu * 6144 * 2 + nctu * 2 * 68 + w * h * 3 // 2)
    peak, peak_src = peaks()
    alg = 2 * w * h * 3 // 2              # SURVEY.md 8(d) frame level: source read once + reconstruction written once
    roof = None
    if kernel_ms:
        ach = alg / (kernel_ms / 1000.0) / 1e9
        roof = {"kernel": "ctu_frame_kernel (one launch per picture: persistent CTAs, a CTU per CTA at a time)", "bound": "hbm", "achieved": ach, "peak": peak,
                "unit": "GB/s", "frac": ach / peak, "traffic": None, "ms_per_launch": kernel_ms, "algorithmic_bytes_per_launch": alg, "peak_source": peak_src,
                "note": "the closed-loop CTU search is a chain of dependent decisions (341 CUs per CTU, CTUs in wavefront order): latency bound by "
                        "construction, its HBM traffic is negligible; the HBM-streaming kernel of the north star is roofline_satd_batch "
                        "(tools/bench_framepass.py, profiles/)"}
    line = {"metric": METRIC, "value": frames / dev_seconds, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1000.0 * e2e_seconds / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic", "config": config_of(wl), "frames_per_step": fps_step,
            "e2e": {"value": frames / e2e_seconds, "unit": "frames/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "pictures_in_flight": owf + 1, "host_threads_per_rank": threads, "host_cores_per_rank": cores,
                    "path": "kvz_stream_bench_ctu: libkvazaar API -> kvz_ctu_hooks -> libkvzcuda.so (kvz_cuda_ctu_submit/wait) -> reference CABAC"},
            "device_only": {"value": frames / dev_seconds, "unit": "frames/s", "pictures_in_flight": slots, "ms_per_step": 1000.0 * dev_seconds / args.steps},
            "gpu_launches": launches, "clocks": clk.summary(), "roofline": roof, "parallelism": f"pictures sharded over {world} GPU(s), no collective"}
    if world > 1:
        line["collective"] = "none on the data path (independent all-intra pictures); measured separately: nccl all_gather (tiles), nccl broadcast (reference picture)"
        line["exchanges"] = exchanges
    if world == 1:
        line.update(parity_and_baseline(args, wl, clip, ctu_bin, env, extra))
        line["me_search"] = side_measurement(env, "bench_me.py")
        line["roofline_satd_batch"] = side_measurement(env, "time_satd.py", "--json")
    else:
        dist.destroy_process_group()
    print(json.dumps(line))


def side_measurement(env, tool, *tool_args):
    """Secondary measurements, outside the timed region and each in its own process (a failure there cannot touch the line):
    tools/bench_me.py -- the motion-search kernels of SURVEY 8f rank 4 on every 16x16 PU of a 1080p picture pair, CUDA events,
    the reference's own functions on one host thread as per-core baseline, identity check;
    tools/time_satd.py -- the HBM-streaming kernel of the north star (batched SATD 8x8) against the measured copy peak."""
    e = dict(os.environ)
    e["CUDA_VISIBLE_DEVICES"] = env["CUDA_VISIBLE_DEVICES"]
    try:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", tool), *tool_args], env=e, stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                           text=True, timeout=300)
        rows = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
        if r.returncode != 0 or not rows:
            return {"error": (r.stderr or r.stdout)[-400:]}
        return json.loads(rows[-1])
    except Exception as ex:  # pragma: no cover
        return {"error": repr(ex)[:400]}


def parity_and_baseline(args, wl, clip, ctu_bin, env, extra):
    """rank 0, N = 1: the unmodified reference on a bounded sample (cpu_baseline) and the byte comparison of the CUDA arm's
    bitstream of the same sample"""
    ref_bin = os.path.join(REF_DIR, "kvz_stream_bench_ref")
    n = args.sample_frames or wl["sample"]
    if not os.path.exists(ref_bin):
        return {"cpu_baseline": {"value": None, "unit": "frames/s", "cores": 0, "kind": "reference", "sample": "oracle/_ref missing"}, "bitstream_identical": None}
    a, b = "/tmp/kvz_bench_sample_ref.hevc", "/tmp/kvz_bench_sample_ctu.hevc"
    rr = stream_bench(ref_bin, clip, wl, a, n, 1, 0, 0)
    rc = stream_bench(ctu_bin, clip, wl, b, n, 1, 0, 0, extra=extra, env=env)
    same = sha(a) == sha(b) and os.path.getsize(a) > 0
    if not same:
        print(f"bench.py: BITSTREAM MISMATCH on the {n}-picture sample ({rr['bytes']} vs {rc['bytes']} bytes)", file=sys.stderr)
    cores = os.cpu_count() or 1
    return {"cpu_baseline": {"value": rr["fps"], "unit": "frames/s", "cores": cores, "kind": "reference",
                             "sample": f"{n} pictures of the same clip, one untimed-ramp-included run of the unmodified reference ({rr['seconds']:.1f} s), threads=auto"},
            "bitstream_identical": bool(same), "bitstream_sha256": sha(b), "bitstream_bytes_sample": rc["bytes"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--workload", default="2160p", choices=sorted(WORKLOADS))
    ap.add_argument("--frames-per-step", type=int, default=0)
    ap.add_argument("--owf", type=int, default=0, help="pictures the encoder keeps in flight (CUDA arm)")
    ap.add_argument("--slots", type=int, default=0, help="pictures in flight of the device-only leg")
    ap.add_argument("--sample-frames", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="CUDA arm: write the results of the last timed step's pictures (CU records, coefficients, SAO parameters, "
                         "final picture) to DIR/<name>.npy as float32, so that two builds can be compared")
    args = ap.parse_args()
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_cuda(args, wl)


if __name__ == "__main__":
    main()
