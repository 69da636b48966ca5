#!/usr/bin/env python
"""bench.py -- throughput of the B200 DSP/scaler hot path (contract: see the task statement / DESIGN.md section 6).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload sws4k|h264|idct_put|me|...] [--impl reference]

BASELINE.json's metric is "Mpixels/s: H.264 1080p decode DSP + 4K yuv420p->rgb24 swscale"; one "step" = one pass of the hot path over
one batch of synthetic input that is already resident in HBM:
  sws4k    (default; configs[4], one GPU's share): sws_scale 3840x2160 yuv420p->rgb24, bicubic|accurate_rnd|bitexact, 16 frames
           per launch                                                            -> 8.29 Mpixel per frame
  h264     (configs[2]): 1920x1088 P pictures of 64 slices, qpel/chroma MC -> idct_add16/add8 -> deblock, 60 pictures per step
  idct_put (configs[1]): IDCTDSPContext.idct_put (FF_IDCT_SIMPLE) over 2^20 dense int16 blocks into an 8192x8192 frame
  me       (configs[3]): pix_abs16 full search +-16 over a 1920x1088 luma pair; with --gpus N the frame's macroblock rows are
           split over the ranks (strong scaling) and the motion-vector field is gathered with ncclAllGather on device buffers
Every other workload runs the same per-GPU batch on every rank (weak scaling, no data-path collective).  `value` is device time
(CUDA events on the launching stream, max over ranks); `e2e` is the same metric through the host-buffer C-ABI call (pinned host
memory, H2D + D2H inside the timed region).  After the timed region (never inside it) the bytes the workload produced are compared
with the CPU checker ("verified").  The line ends with "secondary": {workload: [Mpixels/s, fraction of the HBM roofline]} for the other
workloads and "cpu": their reference-C figures.  --impl reference times the reference's own CPU implementation (oracle/_ref: the
x86 inline-asm build when present, else the portable-C build, else the port) on all host cores for the same workload.
"""
import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

N_BLOCKS = 1 << 20
TILES_PER_ROW = 1024            # 8192-pixel wide frame
SWS_W, SWS_H, SWS_FRAMES = 3840, 2160, 16
SWS_FLAGS = 4 | 0x40000 | 0x80000
IDCT_BYTES_PER_BLOCK = 128 + 64           # algorithmic traffic (SURVEY 8d): coefficients in, pixels out
SWS_BYTES_PER_PIXEL = 1.5 + 3.0


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def traffic_for(kernel):
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        return json.load(open(p)).get(kernel)
    return None


class ClockSampler:
    """Polls NVML for SM clock and throttle reasons while the timed region runs."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz, self._stop, self._t = [], set(), None, False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _poll(self):
        try:
            self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
            r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            for bit, name in self.REASONS.items():
                if r & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def _run(self):
        while not self._stop:
            self._poll()
            time.sleep(0.002)

    def start(self):
        if self.nv:
            self._stop = False
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()

    def stop(self):
        if self.nv and self._t:
            self._poll()
            self._stop = True
            self._t.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ----------------------------------------------------------------------------------------------------
# workloads (GPU arm).  Each returns a dict with run(step_index) launching on `stream`, pixel counts etc.
# ----------------------------------------------------------------------------------------------------
def make_idct_workload(torch, L, stream, rank):
    from libav_b200 import synth
    lib = L.lib
    base = synth.dense_blocks(1 << 14, seed=1 + rank)
    blocks_h = synth.tile_large(base, N_BLOCKS)
    nbuf = 3                                               # rotate buffer sets: 3 x 192 MiB never fits the 126 MB L2
    d_blocks = [torch.from_numpy(blocks_h).cuda() for _ in range(nbuf)]
    stride = TILES_PER_ROW * 8
    rows = (N_BLOCKS // TILES_PER_ROW) * 8
    d_frame = [torch.zeros((rows, stride), dtype=torch.uint8, device="cuda") for _ in range(nbuf)]
    # pinned host buffers for the end-to-end arm
    h_blocks = torch.from_numpy(blocks_h).pin_memory()
    h_frame = torch.zeros((rows, stride), dtype=torch.uint8).pin_memory()

    def run(i):
        k = i % nbuf
        L.check(lib.ff_simple_idct_batch_cuda(0, d_blocks[k].data_ptr(), d_frame[k].data_ptr(), None, stride, N_BLOCKS,
                                              TILES_PER_ROW, 0, stream), "ff_simple_idct_batch_cuda")

    def run_e2e(i):
        L.check(lib.ff_simple_idct_batch_host_cuda(0, h_blocks.data_ptr(), h_frame.data_ptr(), h_frame.numel(), None, stride,
                                                   N_BLOCKS, TILES_PER_ROW), "ff_simple_idct_batch_host_cuda")
        return int(h_frame[0, 0])                          # the step's result is read on the host

    def verify():
        """all 2^20 blocks of the last step's frame against the CPU checker"""
        o, kind = cpu_oracle()
        from oracle.loader import ptr
        want = np.zeros((rows, stride), np.uint8)
        i = np.arange(N_BLOCKS, dtype=np.uint64)
        off = ((i // TILES_PER_ROW) * 8 * stride + (i % TILES_PER_ROW) * 8).astype(np.uint32)
        o.idct_batch(0, ptr(blocks_h.copy()), ptr(want), ptr(off), stride, N_BLOCKS, os.cpu_count() or 1)
        for k in range(nbuf):
            if not np.array_equal(d_frame[k].cpu().numpy(), want):
                raise SystemExit("bench.py: idct_put output differs from the %s checker (buffer %d)" % (kind, k))
        return "all 2^20 blocks of each of the %d frames == %s" % (nbuf, kind)

    return {
        "name": "batched simple_idct_put 8x8, 2^20 dense int16 blocks per GPU -> 8192x8192 u8 frame",
        "run": run, "run_e2e": run_e2e, "verify": verify, "outputs": lambda i: {"frame": d_frame[i % nbuf]},
        "pixels": N_BLOCKS * 64, "alg_bytes": N_BLOCKS * IDCT_BYTES_PER_BLOCK,
        "launches_per_step": 1, "kernel": "simple_idct_kernel<0,false>",  "dtype": "int32 (int16 in, u8 out)",
        "h2d": N_BLOCKS * 128, "d2h": rows * stride,
        "l2": "3 rotating 192 MiB buffer sets (inputs larger than the 126 MB L2)",
        "keep": (d_blocks, d_frame, h_blocks, h_frame),
    }


def make_sws_workload(torch, L, stream, rank):
    from libav_b200 import synth, device
    w, h, K = SWS_W, SWS_H, SWS_FRAMES
    ysz, csz, osz = w * h, (w // 2) * (h // 2), w * h * 3
    frames = [synth.yuv420p_frame(w, h, 1 + rank * 64 + k) for k in range(2)]
    y = np.concatenate([frames[k % 2][0].reshape(-1) for k in range(K)])
    u = np.concatenate([frames[k % 2][1].reshape(-1) for k in range(K)])
    v = np.concatenate([frames[k % 2][2].reshape(-1) for k in range(K)])
    nbuf = 2
    d_y = [torch.from_numpy(y).cuda() for _ in range(nbuf)]
    d_u = [torch.from_numpy(u).cuda() for _ in range(nbuf)]
    d_v = [torch.from_numpy(v).cuda() for _ in range(nbuf)]
    d_o = [torch.empty(osz * K, dtype=torch.uint8, device="cuda") for _ in range(nbuf)]
    ctx = device.SwsContext(w, h, w, h, device.PIX_FMT_RGB24, SWS_FLAGS)
    assert ctx.fused
    # end-to-end arm: one frame per call through the host-pointer sws_scale_cuda (the reference's own call shape), from T host threads
    # with a context each -- config 5's "concurrent streams"; the CPU arm runs one context per host thread the same way.  A call must
    # return a finished picture, so a single caller leaves both PCIe directions idle between frames.
    T = max(1, min(K, int(os.environ.get("AVB200_E2E_STREAMS", "4"))))
    hy, hu, hv = [torch.from_numpy(np.ascontiguousarray(p)).pin_memory() for p in frames[0]]
    ho = torch.empty((h, w * 3), dtype=torch.uint8).pin_memory()
    e2e_ctx = [ctx] + [device.SwsContext(w, h, w, h, device.PIX_FMT_RGB24, SWS_FLAGS) for _ in range(T - 1)]
    e2e_out = [ho] + [torch.empty((h, w * 3), dtype=torch.uint8).pin_memory() for _ in range(T - 1)]
    src = (C.c_void_p * 4)(hy.data_ptr(), hu.data_ptr(), hv.data_ptr(), None)
    sst = (C.c_int * 4)(w, w // 2, w // 2, 0)
    dsts = [(C.c_void_p * 4)(o.data_ptr(), None, None, None) for o in e2e_out]
    dstr = (C.c_int * 4)(w * 3, 0, 0, 0)
    e2e_err = []

    def e2e_worker(t):
        for _ in range(t, K, T):
            if L.lib.sws_scale_cuda(e2e_ctx[t].ctx, src, sst, 0, h, dsts[t], dstr) != h:
                e2e_err.append(t)

    def run(i):
        k = i % nbuf
        ctx.scale_device([d_y[k].data_ptr(), d_u[k].data_ptr(), d_v[k].data_ptr()], [w, w // 2, w // 2], [d_o[k].data_ptr()],
                         [w * 3], nframes=K, src_frame=[ysz, csz, csz], dst_frame=[osz], stream=stream)

    def run_e2e(i):
        ths = [threading.Thread(target=e2e_worker, args=(t,)) for t in range(1, T)]
        [t.start() for t in ths]
        e2e_worker(0)
        [t.join() for t in ths]
        if e2e_err:
            L.check(-1, "sws_scale_cuda")
        return int(ho[0, 0]) + sum(int(o[h - 1, 0]) for o in e2e_out)        # every caller's picture is read on the host

    def verify():
        """first, second and last frame of the last launch + the frame of the host-pointer arm against the CPU checker"""
        o, kind = cpu_oracle()
        from oracle.loader import ptr
        want = []
        for fr in frames:
            w_ = np.zeros((h, w * 3), np.uint8)
            sp = (C.c_void_p * 3)(*[a.ctypes.data for a in fr]); ss = (C.c_int * 3)(w, w // 2, w // 2)
            if o.sws_yuv420p_to_rgb24(sp, ss, w, h, ptr(w_), w * 3, w, h, SWS_FLAGS) != h:
                raise SystemExit("bench.py: the CPU checker refused the frame")
            want.append(w_)
        for k in range(nbuf):
            got = d_o[k].cpu().numpy().reshape(K, h, w * 3)
            for j in (0, 1, K - 1):
                if not np.array_equal(got[j], want[j % 2]):
                    raise SystemExit("bench.py: sws4k frame %d of buffer %d differs from the %s checker" % (j, k, kind))
        for o_ in e2e_out:
            if not np.array_equal(o_.numpy(), want[0]):
                raise SystemExit("bench.py: sws_scale_cuda (host buffers) differs from the %s checker" % kind)
        return "frames 0, 1, %d of each of the %d output batches and the %d host-call pictures == %s" % (K - 1, nbuf, T, kind)

    return {
        "name": "sws_scale 3840x2160 yuv420p->rgb24 bicubic|accurate_rnd|bitexact, %d frames per launch per GPU" % K,
        "run": run, "run_e2e": run_e2e, "verify": verify, "outputs": lambda i: {"rgb24": d_o[i % nbuf].view(K, h, w * 3)},
        "pixels": w * h * K, "alg_bytes": int(w * h * K * SWS_BYTES_PER_PIXEL),
        "launches_per_step": 1, "kernel": "sws_fused_rgb24_tma_kernel", "dtype": "int32 (u8 in, u8 out)",
        "h2d": int(w * h * 1.5) * K, "d2h": osz * K,
        "l2": "2 rotating %d MiB buffer sets (inputs+outputs larger than the 126 MB L2)" % ((ysz + 2 * csz + osz) * K >> 20),
        "keep": (d_y, d_u, d_v, d_o, ctx, hy, hu, hv, ho, e2e_ctx, e2e_out, dsts), "e2e_streams": T,
    }


H264_PICTURES = 30      # 30 x 1088 rows still fit the int16 y of FFH264MCRecord


def make_sws_up_workload(torch, L, stream, rank):
    """secondary row of config 5: a genuine rescale, 1920x1080 -> 3840x2160 yuv420p->rgb24 bicubic (general path:
    hScale8To15 + yuv2rgb24_X vertical pass), 8 frames per step."""
    from libav_b200 import synth, device
    sw, sh, dw, dh, K = 1920, 1080, 3840, 2160, 8
    ysz, csz, osz = sw * sh, (sw // 2) * (sh // 2), dw * dh * 3
    fr = synth.yuv420p_frame(sw, sh, 7 + rank)
    d_y = torch.from_numpy(np.concatenate([fr[0].reshape(-1)] * K)).cuda()
    d_u = torch.from_numpy(np.concatenate([fr[1].reshape(-1)] * K)).cuda()
    d_v = torch.from_numpy(np.concatenate([fr[2].reshape(-1)] * K)).cuda()
    d_o = torch.empty(osz * K, dtype=torch.uint8, device="cuda")
    ctx = device.SwsContext(sw, sh, dw, dh, device.PIX_FMT_RGB24, SWS_FLAGS)
    assert not ctx.fused

    def run(i):
        ctx.scale_device([d_y.data_ptr(), d_u.data_ptr(), d_v.data_ptr()], [sw, sw // 2, sw // 2], [d_o.data_ptr()], [dw * 3], nframes=K,
                         src_frame=[ysz, csz, csz], dst_frame=[osz], stream=stream)

    return {
        "name": "sws_scale 1920x1080 -> 3840x2160 yuv420p->rgb24 bicubic|accurate_rnd|bitexact (true rescale), %d frames per step" % K,
        "run": run, "run_e2e": None, "outputs": lambda i: {"rgb24": d_o.view(K, dh, dw * 3)},
        "pixels": dw * dh * K, "alg_bytes": int((sw * sh * 1.5 + dw * dh * 3) * K),
        "launches_per_step": 1, "kernel": "sws_tile_rgb24_kernel", "dtype": "int32 (u8 in, u8 out)", "h2d": 0, "d2h": 0,
        "l2": "%d MiB of output per step" % (osz * K >> 20), "keep": (d_y, d_u, d_v, d_o, ctx),
    }


def make_h264_workload(torch, L, stream, rank):
    """config 3: 1920x1088 P pictures of 64 slices each, a batch of independent pictures stacked vertically per launch:
    MC (put pass + avg pass) -> residual add -> deblocking.  The consumed coefficient arena is refilled on a side stream (the role the
    entropy decoder plays), double-buffered against the compute stream.  synth.h264_config3_picture is also what the CPU arm runs."""
    from libav_b200 import synth
    lib = L.lib
    G = max(1, int(os.environ.get("AVB200_H264_GROUPS", "2")))         # groups of H264_PICTURES stacked pictures per step
    pic = synth.h264_config3_picture(120, 68, 64, seed=rank)
    mb_w, mb_h, P = pic["mb_w"], pic["mb_h"], H264_PICTURES * G
    W, H = 16 * mb_w, 16 * mb_h
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).cuda()
    refs = pic["refs"]
    d_refs = [[t(np.concatenate([p] * P)) for p in r] for r in refs]              # reference pictures, stacked like the output
    d_planes_g = [torch.tensor([[r[0].data_ptr() + gi * H264_PICTURES * W * H, r[1].data_ptr() + gi * H264_PICTURES * W * H // 4,
                                 r[2].data_ptr() + gi * H264_PICTURES * W * H // 4] for r in d_refs], dtype=torch.int64).cuda() for gi in range(G)]
    mc1 = pic["mc"]
    mcs = []
    for k in range(H264_PICTURES):                         # FFH264MCRecord.y is int16: MC runs per group of 30 stacked pictures
        m = mc1.copy(); m["y"] = m["y"] + k * H; mcs.append(m)
    mc = np.concatenate(mcs)
    res1, coeffs, nnzc = pic["res"], pic["coeffs"], pic["nnzc"]
    ress = []
    for k in range(P):
        r = res1.copy(); r["luma_off"] = r["luma_off"] + k * W * H; r["chroma_off"] = r["chroma_off"] + k * W * H // 4; ress.append(r)
    res = np.concatenate(ress)
    dbk = pic["dbk"]
    d_mc, d_res, d_nnz, d_dbk = t(mc), t(res), t(np.concatenate([nnzc] * P)), t(np.concatenate([dbk] * P))
    d_coef0 = t(np.concatenate([coeffs] * P))
    d_coef = [d_coef0.clone(), d_coef0.clone()]
    d_y = torch.zeros(P * W * H, dtype=torch.uint8, device="cuda")
    d_cb = torch.zeros(P * W * H // 4, dtype=torch.uint8, device="cuda")
    d_cr = torch.zeros(P * W * H // 4, dtype=torch.uint8, device="cuda")
    d_prog = torch.zeros(2 * mb_h * P + 64, dtype=torch.int32, device="cuda")
    side = torch.cuda.Stream()
    main = torch.cuda.current_stream()
    refilled = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]
    for e in refilled + consumed:
        e.record(main)

    # The groups are independent pictures: each runs its own MC -> residual -> deblock chain on its own stream (the decoder threads
    # of the reference would be one per picture too), so the latency-bound wavefront of one group overlaps the other group's kernels.
    chains = [main] + [torch.cuda.Stream() for _ in range(G - 1)] if os.environ.get("AVB200_H264_CHAINS", "1") != "0" else [main] * G
    fork, joined = torch.cuda.Event(), [torch.cuda.Event() for _ in range(G)]
    n_g = mb_w * mb_h * H264_PICTURES                          # macroblocks per group

    def run(i):
        b = i & 1
        main.wait_event(refilled[b])
        fork.record(main)
        for gi in range(G):
            st = chains[gi]
            if st is not main:
                st.wait_event(fork)
            sp = st.cuda_stream
            yo, co = gi * H264_PICTURES * W * H, gi * H264_PICTURES * W * H // 4
            L.check(lib.ff_h264_mc_batch_cuda(d_mc.data_ptr(), mc.shape[0], d_planes_g[gi].data_ptr(), d_y.data_ptr() + yo, d_cb.data_ptr() + co,
                                              d_cr.data_ptr() + co, W, W // 2, W, H, sp), "mc")
            L.check(lib.ff_h264_idct_add_mb_batch_cuda(d_res.data_ptr() + gi * n_g * 12, n_g, d_coef[b].data_ptr() + gi * n_g * 1536, 768,
                                                       d_nnz.data_ptr() + gi * n_g * 120, d_y.data_ptr(), d_cb.data_ptr(), d_cr.data_ptr(), W, W // 2, sp), "residual")
            L.check(lib.ff_h264_deblock_batch_cuda(d_dbk.data_ptr() + gi * n_g * 104, mb_w, mb_h, H264_PICTURES, d_y.data_ptr() + yo, d_cb.data_ptr() + co,
                                                   d_cr.data_ptr() + co, W, W // 2, d_prog.data_ptr() + gi * 8 * mb_h * H264_PICTURES, sp), "deblock")
            if st is not main:
                joined[gi].record(st)
        for gi in range(G):
            if chains[gi] is not main:
                main.wait_event(joined[gi])
        consumed[b].record(main)
        with torch.cuda.stream(side):                      # refill the arena this step consumed while the next step runs
            side.wait_event(consumed[b])
            d_coef[b].copy_(d_coef0, non_blocking=True)
            refilled[b].record(side)

    def verify():
        """every reconstructed picture of the last step against the reference's own tables driven over the same records on the host"""
        o, kind = cpu_oracle()
        if not o.has("h264_pictures"):
            return None
        y, cb, cr, co = np.zeros((H, W), np.uint8), np.zeros((H // 2, W // 2), np.uint8), np.zeros((H // 2, W // 2), np.uint8), coeffs.copy()
        cpu_h264_run(o, pic, 1, y, cb, cr, co, os.cpu_count() or 1)
        gy, gcb, gcr = d_y.cpu().numpy().reshape(P, H, W), d_cb.cpu().numpy().reshape(P, H // 2, W // 2), d_cr.cpu().numpy().reshape(P, H // 2, W // 2)
        for k in range(P):
            if not (np.array_equal(gy[k], y) and np.array_equal(gcb[k], cb) and np.array_equal(gcr[k], cr)):
                raise SystemExit("bench.py: h264 picture %d differs from the %s checker" % (k, kind))
        return "all %d reconstructed pictures (luma + both chroma planes) == %s driver" % (P, kind)

    n_mb = mb_w * mb_h * P
    return {
        "name": NAMES["h264"],
        "run": run, "run_e2e": None, "verify": verify, "pixels": W * H * P, "alg_bytes": int(n_mb * 2.37e3),
        "outputs": lambda i: {"y": d_y.view(P, H, W), "cb": d_cb.view(P, H // 2, W // 2), "cr": d_cr.view(P, H // 2, W // 2)},
        "launches_per_step": 4 * G, "kernel": "h264_mc_kernel_v2", "dtype": "int32 (u8 / int16 in, u8 out)", "h2d": 0, "d2h": 0,
        "l2": "%d pictures (%d MC partitions each) per step: %d MB of pixels + %d MB of coefficients, larger than the 126 MB L2" % (P, mc1.shape[0], P * W * H * 3 // 2 >> 20, d_coef0.numel() >> 20),
        "keep": (d_refs, d_planes_g, d_mc, d_res, d_nnz, d_dbk, d_coef0, d_coef, d_y, d_cb, d_cr, d_prog, side, refilled, consumed, chains, fork, joined),
    }


def make_h264_decide_workload(torch, L, stream, rank):
    """SURVEY 8f rank 1: deblocking decisions (bS / alpha / beta / tc0 per edge) for a batch of stacked 1080p B pictures,
    from the decoder's side-information arrays resident in HBM to FFH264DeblockMB records in HBM."""
    from libav_b200 import synth, tables
    lib = L.lib
    mb_w, mb_h, P = 120, 68, H264_PICTURES
    d = synth.h264_deblock_info(mb_w, mb_h, seed=3 + rank, n_slices=8, bipred=True)
    t = lambda a, reps=P: torch.from_numpy(np.concatenate([np.ascontiguousarray(a)] * reps).view(np.uint8).reshape(-1)).cuda()
    keep = {k: t(d[k]) for k in ("mb_type", "qscale", "nnz", "cbp", "slice_table", "mv0", "mv1", "ref0", "ref1")}
    keep["sp"], keep["cq"] = t(d["slice_params"], 1), t(d["chroma_qp_table"], 1)
    n = mb_w * mb_h * P
    d_out = torch.empty(n * 104, dtype=torch.uint8, device="cuda")
    info = tables.FFH264DeblockInfo(mb_w, mb_h, P, keep["mb_type"].data_ptr(), keep["qscale"].data_ptr(), keep["nnz"].data_ptr(),
                                    keep["cbp"].data_ptr(), keep["slice_table"].data_ptr(),
                                    (C.c_void_p * 2)(keep["mv0"].data_ptr(), keep["mv1"].data_ptr()),
                                    (C.c_void_p * 2)(keep["ref0"].data_ptr(), keep["ref1"].data_ptr()), keep["sp"].data_ptr(), 8,
                                    keep["cq"].data_ptr(), 1, 0)

    def run(i):
        L.check(lib.ff_h264_deblock_params_cuda(C.byref(info), d_out.data_ptr(), stream), "deblock_params")

    per_mb = 4 + 1 + 48 + 2 + 2 + 2 * 64 + 2 * 4 + 104
    return {
        "name": "H.264 deblocking decisions (bS, alpha, beta, tc0) for %d stacked 1080p B pictures of 8 slices" % P,
        "run": run, "run_e2e": None, "outputs": lambda i: {"deblock_records": d_out.view(n, 104)}, "pixels": 256 * n, "alg_bytes": n * per_mb,
        "launches_per_step": 1, "kernel": "h264_deblock_params_kernel", "dtype": "int32 (decoder side information in, records out)",
        "h2d": 0, "d2h": 0, "l2": "%d MB of side information + records per step" % (n * per_mb >> 20), "keep": (keep, d_out, info),
    }


def make_dequant_idct_workload(torch, L, stream, rank):
    """SURVEY 8f rank 2 (mpegvideo half): put_dct() in one kernel -- dct_unquantize_mpeg2_intra (bitexact variant, with
    mismatch control) fused in front of simple_idct_put, same 2^20-block batch and frame as the headline workload."""
    from libav_b200 import synth, tables
    lib = L.lib
    base = synth.dense_blocks(1 << 14, seed=11 + rank) >> 3          # quantised levels
    blocks_h = synth.tile_large(base, N_BLOCKS)
    r = np.random.RandomState(5 + rank)
    rec = np.zeros(N_BLOCKS, np.dtype([("qscale", "u1"), ("last", "i1"), ("dc", "u1"), ("flags", "u1")]))
    rec["qscale"] = r.randint(1, 32, N_BLOCKS); rec["last"] = r.randint(0, 64, N_BLOCKS); rec["dc"] = 8
    t = tables.FFMpegDequantTables()
    perm, rend = synth.zigzag_scan_tables()
    for k in range(64):
        t.intra_matrix[k] = t.inter_matrix[k] = 8 + ((k & 7) + (k >> 3)) * 2
        t.permutated[k], t.raster_end[k] = int(perm[k]), int(rend[k])
    nbuf = 3
    d_blocks = [torch.from_numpy(blocks_h).cuda() for _ in range(nbuf)]
    d_rec = torch.from_numpy(rec.view(np.uint8).reshape(-1)).cuda()
    stride = TILES_PER_ROW * 8
    rows = (N_BLOCKS // TILES_PER_ROW) * 8
    d_frame = [torch.zeros((rows, stride), dtype=torch.uint8, device="cuda") for _ in range(nbuf)]

    def run(i):
        k = i % nbuf
        L.check(lib.ff_mpeg_dequant_idct_batch_cuda(3, C.byref(t), d_rec.data_ptr(), d_blocks[k].data_ptr(), d_frame[k].data_ptr(), None,
                                                    stride, N_BLOCKS, TILES_PER_ROW, 0, stream), "ff_mpeg_dequant_idct_batch_cuda")

    return {
        "name": "fused dct_unquantize_mpeg2_intra (bitexact) + simple_idct_put, 2^20 blocks per GPU -> 8192x8192 u8 frame",
        "run": run, "run_e2e": None, "outputs": lambda i: {"frame": d_frame[i % nbuf]},
        "pixels": N_BLOCKS * 64, "alg_bytes": N_BLOCKS * (IDCT_BYTES_PER_BLOCK + 4),
        "launches_per_step": 1, "kernel": "simple_idct_kernel<0,false,4,false,4>", "dtype": "int32 (int16 levels in, u8 out)",
        "h2d": 0, "d2h": 0, "l2": "3 rotating 196 MiB buffer sets", "keep": (d_blocks, d_rec, d_frame, t),
    }


def make_idct10_workload(torch, L, stream, rank):
    """the 10-bit instance of IDCTDSPContext.idct_put (ff_simple_idct_put_10, bits_per_raw_sample 10): 2^20 blocks -> 8192x8192 16-bit
    samples.  The blocks are modified in place (the C functions leave the row pass there): 384 B of traffic per block."""
    from libav_b200 import synth
    lib = L.lib
    base = synth.dense_blocks(1 << 14, seed=21 + rank) >> 1
    blocks_h = synth.tile_large(base, N_BLOCKS)
    nbuf = 2
    d_blocks0 = torch.from_numpy(blocks_h).cuda()
    d_blocks = [d_blocks0.clone() for _ in range(nbuf)]
    stride = TILES_PER_ROW * 16
    i = np.arange(N_BLOCKS, dtype=np.uint64)
    off = ((i // TILES_PER_ROW) * 8 * stride + (i % TILES_PER_ROW) * 16).astype(np.uint32)
    d_off = torch.from_numpy(off.view(np.int32)).cuda()
    d_frame = [torch.zeros(N_BLOCKS * 64, dtype=torch.int16, device="cuda") for _ in range(nbuf)]

    def run(i):
        k = i % nbuf
        L.check(lib.ff_simple_idct10_batch_cuda(0, d_blocks[k].data_ptr(), d_frame[k].data_ptr(), d_off.data_ptr(), stride, N_BLOCKS, stream), "idct10")

    return {
        "name": "batched simple_idct_put_10 (10-bit), 2^20 int16 blocks per GPU -> 8192x8192 16-bit frame",
        "run": run, "run_e2e": None, "outputs": lambda i: {"frame": d_frame[i % nbuf], "blocks": d_blocks[i % nbuf]},
        "pixels": N_BLOCKS * 64, "alg_bytes": N_BLOCKS * 384,
        "launches_per_step": 1, "kernel": "simple_idct10_staged_kernel<0>", "dtype": "int32 (int16 in, u16 out)", "h2d": 0, "d2h": 0,
        "l2": "2 rotating 384 MiB buffer sets (the row pass is written back over the coefficients, as the C functions leave it)",
        "keep": (d_blocks0, d_blocks, d_off, d_frame),
    }


def make_h264_hbd_workload(torch, L, stream, rank):
    """config 3's chain on 10-bit pictures (the BIT_DEPTH 10 instances: uint16 samples, int32 coefficients): 30 stacked 1920x1088 pictures of 64
    slices per step through ff_h264_mc_batch_hbd_cuda -> ff_h264_idct_add_mb_batch_hbd_cuda -> ff_h264_deblock_batch_hbd_cuda (the functional
    kernels of csrc/h264_hbd_batch.cu).  Same records as the 8-bit workload, byte offsets doubled."""
    from libav_b200 import synth
    lib = L.lib
    pic = synth.h264_config3_picture(120, 68, 64, seed=rank)
    mb_w, mb_h, P = pic["mb_w"], pic["mb_h"], H264_PICTURES
    W, H = 16 * mb_w, 16 * mb_h
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).cuda()
    up = lambda p8: (p8.astype(np.uint16) << 2) | (p8.astype(np.uint16) >> 6)
    d_refs = [[t(np.concatenate([up(p)] * P)) for p in r] for r in pic["refs"]]
    d_planes = torch.tensor([[r[0].data_ptr(), r[1].data_ptr(), r[2].data_ptr()] for r in d_refs], dtype=torch.int64).cuda()
    mcs = []
    for k in range(P):
        m = pic["mc"].copy(); m["y"] = m["y"] + k * H; mcs.append(m)
    mc = np.concatenate(mcs)
    ress = []
    for k in range(P):
        r = pic["res"].copy(); r["luma_off"] = 2 * (r["luma_off"] + k * W * H); r["chroma_off"] = 2 * (r["chroma_off"] + k * W * H // 4); ress.append(r)
    res = np.concatenate(ress)
    n = mb_w * mb_h * P
    d_mc, d_res, d_nnz, d_dbk = t(mc), t(res), t(np.concatenate([pic["nnzc"]] * P)), t(np.concatenate([pic["dbk"]] * P))
    d_coef0 = t(np.concatenate([pic["coeffs"].astype(np.int32) * 4] * P))
    d_coef = d_coef0.clone()
    d_y = torch.zeros(P * W * H * 2, dtype=torch.uint8, device="cuda")
    d_cb = torch.zeros(P * W * H // 2, dtype=torch.uint8, device="cuda")
    d_cr = torch.zeros(P * W * H // 2, dtype=torch.uint8, device="cuda")

    def run(i):
        d_coef.copy_(d_coef0, non_blocking=True)               # (inside the step: the arena the residual pass consumes)
        L.check(lib.ff_h264_mc_batch_hbd_cuda(10, 1, d_mc.data_ptr(), mc.shape[0], d_planes.data_ptr(), d_y.data_ptr(), d_cb.data_ptr(), d_cr.data_ptr(),
                                              2 * W, W, W, H, stream), "mc hbd")
        L.check(lib.ff_h264_idct_add_mb_batch_hbd_cuda(10, 1, d_res.data_ptr(), n, d_coef.data_ptr(), 768, d_nnz.data_ptr(), d_y.data_ptr(), d_cb.data_ptr(),
                                                       d_cr.data_ptr(), 2 * W, W, stream), "residual hbd")
        L.check(lib.ff_h264_deblock_batch_hbd_cuda(10, d_dbk.data_ptr(), mb_w, mb_h, P, d_y.data_ptr(), d_cb.data_ptr(), d_cr.data_ptr(), 2 * W, W, stream), "deblock hbd")

    return {
        "name": "H.264 1080p DSP path on 10-bit pictures (functional kernels): MC + residual + deblock, %d stacked 64-slice pictures per step" % P,
        "run": run, "run_e2e": None, "pixels": P * W * H, "alg_bytes": n * (2 * 768 + 3 * 1536 + 104 + 1536),
        "outputs": lambda i: {"y": d_y.view(torch.int16).view(P, H, W), "cb": d_cb.view(torch.int16).view(P, H // 2, W // 2),
                              "cr": d_cr.view(torch.int16).view(P, H // 2, W // 2)},
        "launches_per_step": 4, "kernel": "h264_deblock_generic_kernel", "dtype": "int32 (u16 samples, int32 coefficients)", "h2d": 0, "d2h": 0,
        "l2": "%d MiB of pictures + coefficients per step" % ((P * W * H * 3 + n * 3072) >> 20),
        "keep": (d_refs, d_planes, d_mc, d_res, d_nnz, d_dbk, d_coef0, d_coef, d_y, d_cb, d_cr),
    }


def make_h264_intra_workload(torch, L, stream, rank):
    """SURVEY 8f rank 2: all-intra 1080p pictures (equal shares of intra 4x4 / 8x8 / 16x16 macroblocks, every prediction
    mode the availability allows, half of the blocks coded) reconstructed by the prediction + residual wavefront; a batch of
    independent pictures stacked per launch, the consumed coefficient arena refilled on a side stream."""
    from libav_b200 import synth
    lib = L.lib
    mb_w, mb_h, P = 120, 68, int(os.environ.get("AVB200_INTRA_PICTURES", "48"))
    W, H = 16 * mb_w, 16 * mb_h
    rec, coeffs, nnzc = synth.h264_intra_work(mb_w, mb_h, seed=9 + rank)
    t = lambda a, reps=P: torch.from_numpy(np.concatenate([np.ascontiguousarray(a)] * reps).view(np.uint8).reshape(-1)).cuda()
    d_rec, d_nnz, d_coef0 = t(rec), t(nnzc), t(coeffs)
    d_coef = [d_coef0.clone(), d_coef0.clone()]
    d_y = torch.zeros(P * W * H, dtype=torch.uint8, device="cuda")
    d_cb = torch.zeros(P * W * H // 4, dtype=torch.uint8, device="cuda")
    d_cr = torch.zeros(P * W * H // 4, dtype=torch.uint8, device="cuda")
    d_prog = torch.zeros(mb_h * P, dtype=torch.int32, device="cuda")
    side, main = torch.cuda.Stream(), torch.cuda.current_stream()
    refilled = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]
    for e in refilled + consumed:
        e.record(main)

    def run(i):
        b = i & 1
        main.wait_event(refilled[b])
        L.check(lib.ff_h264_intra_mb_batch_cuda(d_rec.data_ptr(), mb_w, mb_h, P, d_coef[b].data_ptr(), 768, d_nnz.data_ptr(), d_y.data_ptr(),
                                                d_cb.data_ptr(), d_cr.data_ptr(), W, W // 2, d_prog.data_ptr(), stream), "intra")
        consumed[b].record(main)
        with torch.cuda.stream(side):
            side.wait_event(consumed[b])
            d_coef[b].copy_(d_coef0, non_blocking=True)
            refilled[b].record(side)

    n_mb = mb_w * mb_h * P
    return {
        "name": "H.264 intra reconstruction wavefront: %d all-intra 1080p pictures per step (4x4 / 8x8 / 16x16 mix)" % P,
        "run": run, "run_e2e": None, "pixels": W * H * P, "alg_bytes": n_mb * (768 * 2 + 384 + 120 + 24),
        "outputs": lambda i: {"y": d_y.view(P, H, W), "cb": d_cb.view(P, H // 2, W // 2), "cr": d_cr.view(P, H // 2, W // 2)},
        "launches_per_step": 1, "kernel": "h264_intra_kernel", "dtype": "int32 (u8 / int16 in, u8 out)", "h2d": 0, "d2h": 0,
        "l2": "%d MB of coefficients + pixels per step" % (n_mb * (768 * 2 + 384) >> 20),
        "keep": (d_rec, d_nnz, d_coef0, d_coef, d_y, d_cb, d_cr, d_prog, side, refilled, consumed),
    }


def make_fft_workload(torch, L, stream, rank):
    """SURVEY 8f rank 3: FFTContext.fft_permute + fft_calc, 32768 independent 1024-point complex float transforms per step
    (in place, 256 MiB), followed per step by 32768 imdct_half of size 2048 (AAC long windows) under "also"."""
    lib = L.lib
    nb, T = 10, 32768
    g = torch.Generator(device="cuda"); g.manual_seed(1 + rank)
    bufs = [torch.randn(T * (1 << nb) * 2, generator=g, device="cuda", dtype=torch.float32) for _ in range(2)]
    inputs = [b.clone() for b in bufs]

    def run(i):
        L.check(lib.ff_fft_batch_cuda(nb, 0, bufs[i & 1].data_ptr(), T, stream), "fft")

    def outputs(i):
        """the step's transform applied to its buffer's original contents: the timed buffers are transformed over and over
        without normalisation and soon hold inf / NaN"""
        out = inputs[i & 1].clone()
        L.check(lib.ff_fft_batch_cuda(nb, 0, out.data_ptr(), T, stream), "fft")
        torch.cuda.synchronize()
        return {"transforms": out.view(T, 1 << nb, 2)}

    return {
        "name": "FFTContext fft_permute + fft_calc: %d x %d-point complex float transforms per step" % (T, 1 << nb),
        "run": run, "run_e2e": None, "outputs": outputs,
        "pixels": T * (1 << nb), "alg_bytes": T * (1 << nb) * 16,
        "launches_per_step": 1, "kernel": "fft_kernel", "dtype": "f32 (complex)", "h2d": 0, "d2h": 0,
        "l2": "2 rotating 256 MiB buffers; the metric counts complex points as pixels", "keep": (bufs, inputs),
    }


def make_me_workload(torch, L, stream, rank):
    """config 4: pix_abs16 full search +-16 over a 1920x1088 luma pair (restricted MVs, lambda 0)."""
    from libav_b200 import synth
    lib = L.lib
    w, h = 1920, 1088
    cur, ref = synth.me_frames(w, h, seed=1 + rank)
    d_cur, d_ref = torch.from_numpy(cur).cuda(), torch.from_numpy(ref).cuda()
    n_mb = (w // 16) * (h // 16)
    d_out = torch.zeros(3 * n_mb, dtype=torch.int32, device="cuda")

    def run(i):
        L.check(lib.ff_full_search_cuda(d_cur.data_ptr(), d_ref.data_ptr(), w, w, h, 16, 0, h // 16, d_out.data_ptr(), stream), "full_search")

    def verify():
        o, kind = cpu_oracle()
        from oracle.loader import ptr
        want = np.zeros(3 * n_mb, np.int32)
        o.full_search(ptr(cur), ptr(ref), w, w, h, 16, 0, h // 16, ptr(want), os.cpu_count() or 1)
        if not np.array_equal(d_out.cpu().numpy(), want):
            raise SystemExit("bench.py: full-search motion field differs from the %s checker" % kind)
        return "all %d (mx, my, sad) triples == %s" % (n_mb, kind)

    return {
        "name": "me_cmp pix_abs16 SAD full search, 1920x1088, range 16, whole frame per GPU",
        "run": run, "run_e2e": None, "verify": verify, "outputs": lambda i: {"motion": d_out.view(n_mb, 3)},
        "pixels": w * h, "alg_bytes": 2 * w * h + 12 * n_mb,
        "launches_per_step": 1, "kernel": "full_search_kernel", "dtype": "u8 (vabsdiff4)", "h2d": 0, "d2h": 0,
        "l2": "4 MB working set, ALU/shared-memory bound (2.27 G abs-diff-accumulate per frame), HBM fraction reported for completeness",
        "keep": (d_cur, d_ref, d_out),
    }


def make_me_sharded_workload(torch, dist, L, stream, rank, world):
    """config 4 as BASELINE states it: ONE 1920x1088 frame pair, its 68 macroblock rows split over the ranks (each rank holds only its
    rows of `cur` and those rows +-16 of `ref`), the per-rank pieces of the motion-vector field gathered on every rank with ncclAllGather
    on device buffers inside the timed step.  Strong scaling: the work is fixed, `value` = the frame's pixels / max-over-ranks time."""
    from libav_b200 import synth, shard
    lib = L.lib
    w, h = 1920, 1088
    mb_w, mb_h = w // 16, h // 16
    cur, ref = synth.me_frames(w, h, seed=1)                       # the same frame on every rank: each uploads its shard only
    y0, y1 = shard.mb_row_range(mb_h, rank, world)
    lo, hi = max(0, 16 * y0 - 16), min(h, 16 * y1 + 16)
    rows_max = -(-mb_h // world)
    d_cur = torch.from_numpy(np.ascontiguousarray(cur[16 * y0:16 * y1])).cuda()
    d_ref = torch.from_numpy(np.ascontiguousarray(ref[lo:hi])).cuda()
    d_loc = torch.zeros(rows_max * mb_w * 3, dtype=torch.int32, device="cuda")
    d_all = torch.zeros(world * rows_max * mb_w * 3, dtype=torch.int32, device="cuda")
    # the call addresses rows by their position in the frame: hand it the (virtual) origin of each shard's frame
    p_cur, p_ref, p_out = d_cur.data_ptr() - 16 * y0 * w, d_ref.data_ptr() - lo * w, d_loc.data_ptr() - 12 * y0 * mb_w

    def run(i):
        if y1 > y0:
            L.check(lib.ff_full_search_cuda(p_cur, p_ref, w, w, h, 16, y0, y1, p_out, stream), "full_search")
        dist.all_gather_into_tensor(d_all, d_loc)                  # NCCL all-gather, device to device, on the current stream

    def verify():
        o, kind = cpu_oracle()
        from oracle.loader import ptr
        want = np.zeros((mb_h, mb_w * 3), np.int32)
        o.full_search(ptr(cur), ptr(ref), w, w, h, 16, 0, mb_h, ptr(want), os.cpu_count() or 1)
        got = d_all.cpu().numpy().reshape(world, rows_max, mb_w * 3)
        for r in range(world):
            a, b = shard.mb_row_range(mb_h, r, world)
            if not np.array_equal(got[r, :b - a], want[a:b]):
                raise SystemExit("bench.py: gathered motion field differs from the %s checker in rank %d's rows" % (kind, r))
        return "the gathered field of all %d macroblocks (as rank 0 holds it after ncclAllGather) == %s" % (mb_w * mb_h, kind)

    return {
        "name": "me_cmp pix_abs16 SAD full search, 1920x1088, range 16, frame-shard over %d GPUs + ncclAllGather of the motion field" % world,
        "run": run, "run_e2e": None, "verify": verify, "scaling": "strong", "pixels": w * h, "alg_bytes": 2 * w * h + 12 * mb_w * mb_h,
        "outputs": lambda i: {"motion": d_all.view(world, rows_max * mb_w, 3)},
        "launches_per_step": 1, "kernel": "full_search_kernel", "dtype": "u8 (vabsdiff4)", "h2d": 0, "d2h": 0,
        "l2": "4 MB working set, ALU/shared-memory bound (2.27 G abs-diff-accumulate per frame), HBM fraction reported for completeness",
        "keep": (d_cur, d_ref, d_loc, d_all),
    }


def time_gpu(torch, dist, wl, steps, warmup, world, sampler=None):
    for i in range(warmup):
        wl["run"](i)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if sampler:
        sampler.start()
    e0.record()
    for i in range(steps):
        wl["run"](warmup + i)
    e1.record()
    torch.cuda.synchronize()
    if sampler:
        sampler.stop()
    if world > 1:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms


def time_e2e(torch, dist, wl, steps, warmup, world):
    for i in range(min(warmup, 2)):
        wl["run_e2e"](i)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for i in range(steps):
        wl["run_e2e"](i)
    torch.cuda.synchronize()
    sec = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([sec], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sec = float(t.item())
    return sec


DUMP_BYTES = 60 << 20         # under 64 MB with the .npy headers
DUMP_SEED = 20261017


def dump_outputs(torch, outputs, directory):
    """Writes each array of `outputs` (device tensors) to <directory>/<name>.npy: float32, or float64 where the data is.  An array
    larger than its share of DUMP_BYTES is written as a sample at positions drawn from DUMP_SEED: the same positions for the same
    arguments, so two builds can be compared value for value."""
    os.makedirs(directory, exist_ok=True)
    for name, t in outputs.items():
        flat = t.reshape(-1)
        ftype = torch.float64 if t.dtype == torch.float64 else torch.float32
        share = DUMP_BYTES // len(outputs) // (8 if ftype == torch.float64 else 4)
        if flat.numel() > share:
            pos = np.sort(np.random.default_rng(DUMP_SEED).integers(0, flat.numel(), share))
            flat = flat[torch.from_numpy(pos).to(flat.device)]
        else:
            flat = flat.reshape(t.shape)
        np.save(os.path.join(directory, name + ".npy"), flat.to(ftype).cpu().numpy())


# ----------------------------------------------------------------------------------------------------
# CPU legs (the only place bench.py touches oracle/)
# ----------------------------------------------------------------------------------------------------
def cpu_oracle():
    """the parity checker: the compiled reference's portable-C build, else the port"""
    from oracle import loader
    r = loader.ref()
    if r is not None:
        return r, "reference"
    return loader.port(), "port"


def cpu_timing_arms():
    """[(library, kind, label)] to time: the reference's x86 inline-asm build (what a default build of the reference runs on this host
    without an external assembler: psadbw SAD, MMX simple IDCT under FF_IDCT_AUTO, MMX hpel / blockdsp; every H.264 slot, hScale and
    the bit-exact rgb24 output stage stay C there because their SIMD is external nasm code) and its portable-C build."""
    from oracle import loader
    arms = []
    if loader.ref_simd() is not None:
        arms.append((loader.ref_simd(), "reference", "x86 inline-asm SIMD build (cpu flags unmasked, FF_IDCT_AUTO)"))
    if loader.ref() is not None:
        arms.append((loader.ref(), "reference", "portable C build (ARCH_X86 = 0, av_set_cpu_flags_mask(0))"))
    if not arms:
        arms.append((loader.port(), "port", "plain-C restatement (oracle/port)"))
    return arms


def cpu_idct(nthreads, seconds=3.0, reps=None, arm=None):
    """reference C ff_simple_idct_put_8 over the full 2^20-block workload, all host threads; median of reps."""
    from libav_b200 import synth
    from oracle.loader import ptr
    o, kind = arm[:2] if arm else cpu_oracle()
    base = synth.tile_large(synth.dense_blocks(1 << 14, seed=1), N_BLOCKS)
    stride = TILES_PER_ROW * 8
    frame = np.zeros((N_BLOCKS // TILES_PER_ROW * 8, stride), dtype=np.uint8)
    i = np.arange(N_BLOCKS, dtype=np.uint64)
    off = ((i // TILES_PER_ROW) * 8 * stride + (i % TILES_PER_ROW) * 8).astype(np.uint32)
    times = []
    t_all = time.perf_counter()
    while (len(times) < reps) if reps else (time.perf_counter() - t_all < seconds or len(times) < 3):
        b = base.copy()                                   # the reference clobbers its input block
        t0 = time.perf_counter()
        o.idct_batch(0, ptr(b), ptr(frame), ptr(off), stride, N_BLOCKS, nthreads)
        times.append(time.perf_counter() - t0)
    return {"sec_per_step": float(np.median(times)), "kind": kind, "cores": nthreads, "reps": len(times),
            "sample": "full step: 2^20 dense blocks, %d pthreads, median of %d passes" % (nthreads, len(times)),
            "pixels": N_BLOCKS * 64}


def cpu_sws(nthreads, seconds=3.0, reps=None, arm=None, frames_per_thread=1):
    """reference sws_scale 4K yuv420p->rgb24 on all host threads (one context per thread, one frame each)."""
    from libav_b200 import synth
    from oracle.loader import ptr
    o, kind = arm[:2] if arm else cpu_oracle()
    w, h = SWS_W, SWS_H
    yuv = synth.yuv420p_frame(w, h, 1)
    src = (C.c_void_p * 3)(*[a.ctypes.data for a in yuv])
    sst = (C.c_int * 3)(w, w // 2, w // 2)
    outs = [np.zeros((h, w * 3), np.uint8) for _ in range(nthreads)]

    def work(t):
        for _ in range(frames_per_thread):
            o.sws_yuv420p_to_rgb24(src, sst, w, h, ptr(outs[t]), w * 3, w, h, SWS_FLAGS)

    times = []
    t_all = time.perf_counter()
    while (len(times) < reps) if reps else (time.perf_counter() - t_all < seconds or len(times) < 2):
        ths = [threading.Thread(target=work, args=(t,)) for t in range(nthreads)]
        t0 = time.perf_counter()
        [t.start() for t in ths]
        [t.join() for t in ths]
        times.append(time.perf_counter() - t0)
    sec = float(np.median(times))
    return {"sec_per_step": sec, "kind": kind, "cores": nthreads, "reps": len(times),
            "sample": "%d concurrent 4K frames (one SwsContext per thread, context set-up included), median of %d rounds"
                      % (nthreads * frames_per_thread, len(times)),
            "pixels": w * h * nthreads * frames_per_thread}


def cpu_me(nthreads, seconds=3.0, reps=None, arm=None):
    """reference pix_abs16 (C) driven by the full-search loop over a 1920x1088 frame, MB rows split over host threads."""
    from libav_b200 import synth
    from oracle.loader import ptr
    o, kind = arm[:2] if arm else cpu_oracle()
    w, h = 1920, 1088
    cur, ref = synth.me_frames(w, h, seed=1)
    out = np.zeros(3 * (w // 16) * (h // 16), np.int32)
    times = []
    t_all = time.perf_counter()
    while (len(times) < reps) if reps else (time.perf_counter() - t_all < seconds or len(times) < 2):
        t0 = time.perf_counter()
        o.full_search(ptr(cur), ptr(ref), w, w, h, 16, 0, h // 16, ptr(out), nthreads)
        times.append(time.perf_counter() - t0)
    return {"sec_per_step": float(np.median(times)), "kind": kind, "cores": nthreads, "reps": len(times),
            "sample": "full step: one 1920x1088 frame, %d pthreads over MB rows, median of %d passes" % (nthreads, len(times)),
            "pixels": w * h}


def cpu_h264_run(o, pic, P, y, cb, cr, coeffs, nthreads):
    from oracle.loader import ptr
    refs = (C.c_void_p * 6)(*[p.ctypes.data for r in pic["refs"] for p in r])
    if o.h264_pictures(ptr(pic["mc"]), ptr(pic["mc_first"]), ptr(pic["res"]), ptr(pic["dbk"]), ptr(pic["nnzc"]), ptr(coeffs), refs, 2,
                       ptr(y), ptr(cb), ptr(cr), y.strides[0], cb.strides[0], pic["mb_w"], pic["mb_h"], P, pic["slices"], nthreads) != 0:
        raise SystemExit("bench.py: the CPU H.264 driver refused its arguments")


def cpu_h264(nthreads, seconds=3.0, reps=None, arm=None):
    """config 3 on the host: the reference's H264DSPContext / H264QpelContext / H264ChromaContext / VideoDSPContext tables over the same
    synthetic pictures (MC -> idct_add16 / add8 per macroblock, loop filter per slice; the 64 slices of every picture are independent
    work units handed to pthreads).  A bounded sample: as many pictures per pass as two per thread ... at most the GPU step's 60."""
    from libav_b200 import synth
    o, kind = arm[:2] if arm else cpu_oracle()
    if not o.has("h264_pictures"):
        return None
    pic = synth.h264_config3_picture(120, 68, 64, seed=0)
    W, H = 16 * pic["mb_w"], 16 * pic["mb_h"]
    P = max(2, min(60, (2 * nthreads + 63) // 64))
    y, cb, cr = np.zeros((P * H, W), np.uint8), np.zeros((P * H // 2, W // 2), np.uint8), np.zeros((P * H // 2, W // 2), np.uint8)
    co0 = np.concatenate([pic["coeffs"]] * P)
    times = []
    t_all = time.perf_counter()
    while (len(times) < reps) if reps else (time.perf_counter() - t_all < seconds or len(times) < 3):
        co = co0.copy()                                   # the residual functions consume (zero) their coefficients: refill outside the timing
        t0 = time.perf_counter()
        cpu_h264_run(o, pic, P, y, cb, cr, co, nthreads)
        times.append(time.perf_counter() - t0)
    return {"sec_per_step": float(np.median(times)), "kind": kind, "cores": nthreads, "reps": len(times),
            "sample": "%d 1920x1088 pictures x 64 slices per pass, slices handed to %d pthreads, median of %d passes" % (P, nthreads, len(times)),
            "pixels": W * H * P}


def bind_to_gpu_numa_node(index):
    """One rank drives one GPU: run this process on the CPUs next to that GPU and prefer their memory node, BEFORE the pinned staging
    buffers are allocated -- with four ranks per socket copying at once the host side is the limiter of the end-to-end arm."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        dev = "/sys/bus/pci/devices/" + bus.lower()[-12:]
        node = int(open(dev + "/numa_node").read())
        cpus = open(dev + "/local_cpulist").read().strip()
        ids = set()
        for part in cpus.split(","):
            lo, _, hi = part.partition("-")
            ids.update(range(int(lo), int(hi or lo) + 1))
        if ids:
            os.sched_setaffinity(0, ids)
        if node >= 0:
            libc = C.CDLL(None, use_errno=True)
            mask = C.c_ulong(1 << node)
            libc.syscall(238, 1, C.byref(mask), C.c_ulong(64))       # set_mempolicy(MPOL_PREFERRED, {node})
        return {"numa_node": node, "cpus": cpus}
    except Exception as e:                                            # containers without sysfs / NVML: stay unbound
        return {"numa_node": None, "error": str(e)[:80]}


CPU_LEGS = {"idct_put": cpu_idct, "sws4k": cpu_sws, "me": cpu_me, "h264": cpu_h264}
NAMES = {"idct_put": "batched simple_idct_put 8x8, 2^20 dense int16 blocks per GPU -> 8192x8192 u8 frame",
         "sws4k": "sws_scale 3840x2160 yuv420p->rgb24 bicubic|accurate_rnd|bitexact, %d frames per launch per GPU" % SWS_FRAMES,
         "me": "me_cmp pix_abs16 SAD full search, 1920x1088, range 16, whole frame per GPU",
         "h264": "H.264 1080p DSP path: qpel/chroma MC + idct_add16/add8 + deblock, 64 synthetic slices per picture"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="sws4k", choices=["sws4k", "h264", "idct_put", "me", "sws_up", "h264_decide", "dequant_idct", "h264_intra", "fft", "idct10", "h264_hbd"])
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary workloads and the CPU baselines")
    ap.add_argument("--no-verify", action="store_true", help="skip the post-timing comparison with the CPU checker")
    ap.add_argument("--tune", action="append", default=[], help="kernel-variant knob key=value (avb200_set_tuning), profiling only")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed path computed in its last step to DIR/<name>.npy (at most 64 MB)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    steps, warmup = max(1, args.steps), max(3, args.warmup)
    hbm_peak, peak_src = peaks()
    ncores = os.cpu_count() or 1

    if args.impl == "reference":
        if rank != 0:
            return 0
        steps = min(steps, 20)
        fn = CPU_LEGS.get(args.workload)
        arms = [a for a in cpu_timing_arms() if args.workload != "h264" or a[0].has("h264_pictures")]
        if fn is None or not arms:
            print(json.dumps({"impl": "reference", "unavailable": "no batched CPU driver for workload %s (its per-function parity against the reference is in tests/)" % args.workload}))
            return 0
        # the reference's fastest build on this host for this workload (its x86 inline-asm build is not always the faster one: the MMX
        # code paths it enables in libswscale lose to gcc -O3 C on current cores); the probe doubles as the warm-up pass
        probes = []
        for a in arms:
            fn(ncores, reps=1, arm=a)
            p = fn(ncores, seconds=1.5, arm=a)               # (at least three passes: the first ones still pay page faults and thread start-up)
            probes.append((p["pixels"] / p["sec_per_step"] / 1e6, a))
        arm = max(probes, key=lambda t: t[0])[1]
        r = fn(ncores, reps=steps, arm=arm)
        mpix = r["pixels"] / r["sec_per_step"] / 1e6
        # the same workload names as the GPU arm's config.workload (the driver pairs the two lines by them)
        print(json.dumps({
            "impl": "reference", "metric": "Mpixels/s", "value": mpix, "unit": "Mpixels/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": r["sec_per_step"] * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": NAMES[args.workload], "per_gpu_batch": "one batch of the same shape on the host cores (a bounded sample: %s)" % r["sample"],
                       "host_threads": ncores, "build": arm[2], "builds_probed": {a[2]: round(v, 1) for v, a in probes}, "idct_algo": "FF_IDCT_SIMPLE (C build) / FF_IDCT_AUTO (x86 build)",
                       "sws_flags": "SWS_BICUBIC|SWS_ACCURATE_RND|SWS_BITEXACT"},
            "cpu_baseline": {"value": mpix, "unit": "Mpixels/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"], "build": arm[2]},
            "e2e": {"value": mpix, "unit": "Mpixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }))
        return 0

    numa = bind_to_gpu_numa_node(local_rank)                  # before torch / the library allocate their pinned staging buffers
    import torch
    import torch.distributed as dist
    import libav_b200._lib as L
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the CUDA path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    L.init(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    stream = torch.cuda.current_stream().cuda_stream
    for kv in args.tune:
        k, v = kv.split("=")
        L.lib.avb200_set_tuning(k.encode(), int(v))

    makers = {"sws4k": make_sws_workload, "h264": make_h264_workload, "idct_put": make_idct_workload, "me": make_me_workload,
              "sws_up": make_sws_up_workload, "dequant_idct": make_dequant_idct_workload, "h264_intra": make_h264_intra_workload,
              "fft": make_fft_workload, "h264_decide": make_h264_decide_workload, "idct10": make_idct10_workload, "h264_hbd": make_h264_hbd_workload}
    if args.workload == "me" and world > 1:
        makers["me"] = make_me_sharded_workload
    order = [args.workload] + ([w for w in makers if w != args.workload] if not args.no_secondary else [])
    results = {}
    for idx, wname in enumerate(order):
        sharded = wname == "me" and makers[wname] is make_me_sharded_workload
        wl = makers[wname](torch, dist, L, stream, rank, world) if sharded else makers[wname](torch, L, stream, rank)
        st = steps if idx == 0 else max(5, min(steps, 30))   # the secondaries get a shorter timed region
        sampler = ClockSampler(local_rank) if rank == 0 else None
        ms = time_gpu(torch, dist, wl, st, warmup, world, sampler)
        if args.dump_outputs and idx == 0 and rank == 0:
            dump_outputs(torch, wl["outputs"](warmup + st - 1), args.dump_outputs)
        e2e_steps = max(1, min(st, 5))
        e2e_sec = time_e2e(torch, dist, wl, e2e_steps, warmup, world) if wl["run_e2e"] else None
        verified = None
        if not args.no_verify and wl.get("verify") and rank == 0:
            torch.cuda.synchronize()
            verified = wl["verify"]()
        ms_step = ms / st
        strong = wl.get("scaling") == "strong"
        mpix = wl["pixels"] * (1 if strong else world) / (ms_step * 1e-3) / 1e6
        gbs = wl["alg_bytes"] / (ms_step * 1e-3) / 1e9
        results[wname] = {
            "workload": wl["name"], "value": mpix, "ms_per_step": ms_step, "steps": st, "scaling": wl.get("scaling", "weak"),
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                         "traffic": traffic_for(wl["kernel"]), "kernel": wl["kernel"], "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": wl["alg_bytes"]},
            "e2e": ({"value": wl["pixels"] * world / (e2e_sec / e2e_steps) / 1e6, "unit": "Mpixels/s",
                     "h2d_bytes_per_step": wl["h2d"], "d2h_bytes_per_step": wl["d2h"], "steps": e2e_steps,
                     "host_threads": wl.get("e2e_streams", 1)} if e2e_sec else None),
            "gpu_launches": wl["launches_per_step"] * st * world, "verified": verified,
            "clocks": sampler.summary() if sampler else None, "dtype": wl["dtype"], "l2": wl["l2"],
        }
        del wl
        torch.cuda.empty_cache()

    cpu, cpu_others = None, {}
    if rank == 0 and world == 1 and not args.no_secondary:
        arms = cpu_timing_arms()
        leg = CPU_LEGS.get(args.workload, cpu_sws)
        timed = []
        for a in arms:                                        # every build of the reference; the fastest is the baseline, the others are listed
            r_ = leg(ncores, seconds=2.5, arm=a)
            if r_:
                timed.append((r_["pixels"] / r_["sec_per_step"] / 1e6, r_, a))
        timed.sort(key=lambda t: -t[0])
        v0, r, a0 = timed[0]
        cpu = {"value": v0, "unit": "Mpixels/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"], "build": a0[2]}
        for v_, r2, a_ in timed[1:]:
            cpu.setdefault("other_builds", []).append({"build": a_[2], "value": v_, "cores": r2["cores"]})
        arms = [a0] + [a for a in arms if a is not a0]
        r1 = leg(1, reps=2, arm=arms[0])                      # SURVEY 8d also asks for the one-thread number
        if r1:
            cpu["single_thread"] = {"value": r1["pixels"] / r1["sec_per_step"] / 1e6, "unit": "Mpixels/s", "cores": 1}
        cpu["note"] = ("x86 build = the reference's inline-asm SIMD (psadbw SAD, MMX simple IDCT / hpel / blockdsp); all H.264 slots, hScale and "
                       "the bit-exact rgb24 output stage are C in it too: their SIMD is external nasm code and no assembler exists here")
        for wname, fn in CPU_LEGS.items():                    # reference figures of the other headline workloads, all host threads
            if wname == args.workload or wname not in results:
                continue
            r3 = fn(ncores, seconds=2.0, arm=arms[0])
            if r3:
                cpu_others[wname] = round(r3["pixels"] / r3["sec_per_step"] / 1e6, 1)

    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        m = results[args.workload]
        line = {
            "metric": "Mpixels/s", "value": m["value"], "unit": "Mpixels/s", "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": m["ms_per_step"], "higher_is_better": True, "scaling": m["scaling"], "vs_baseline": None,
            "dtype": m["dtype"], "data": "synthetic",
            "config": {"workload": m["workload"], "per_gpu_batch": ("one frame's macroblock rows split over the ranks, ncclAllGather of the motion field" if m["scaling"] == "strong"
                                                                    else "identical on every rank (weak scaling, no collective on the data path)"),
                       "l2": m["l2"], "idct_algo": "FF_IDCT_SIMPLE", "sws_flags": "SWS_BICUBIC|SWS_ACCURATE_RND|SWS_BITEXACT"},
            "tuning": args.tune, "roofline": m["roofline"], "e2e": m["e2e"], "gpu_launches": m["gpu_launches"], "clocks": m["clocks"],
            "verified": m["verified"], "numa": numa, "cpu_baseline": cpu,
            # compact tail: [Mpixels/s on this many GPUs, fraction of the HBM roofline, verified against the checker]
            "secondary": {k: [round(v["value"], 1), round(v["roofline"]["frac"], 4), bool(v["verified"])] for k, v in results.items() if k != args.workload},
            "secondary_ms_per_step": {k: round(v["ms_per_step"], 4) for k, v in results.items() if k != args.workload},
            "cpu": cpu_others,
        }
        print(json.dumps(line))
    return 0


if __name__ == "__main__":
    sys.exit(main())
