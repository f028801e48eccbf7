#!/usr/bin/env python
"""Headline benchmark: Mpixel/s of `apply` + `combine_with(mode=3)` on batched 1080p frames (BASELINE.json, cfg 4).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl ours|reference] [--dump-outputs DIR]

A step = one pass of the target-referenced hot path over one batch of B synthetic 1920x1080 frames per GPU:
  (1) FlowBatch.apply(uint8x3 images, return_valid_area=True)   -> ofk_warp_t      (16 B/px algorithmic)
  (2) FlowBatch.combine_with(other, mode=3)                      -> ofk_combine3    (27 B/px algorithmic)
Pixels are counted once per pair of calls (SURVEY section 8d). `value` is device-resident throughput (CUDA events,
max over ranks), `e2e` is the same pair of operations through the host-buffer API (pinned numpy in / numpy out, copies
inside the timed region). `--impl reference` times the CPU oracle port of the reference (cv2.remap + numpy glue, all
host threads OpenCV uses) on a bounded sample of the same workload.

Multi-GPU: one process per GPU (torchrun), contiguous batch shards, no data-path collective; weak scaling.

--dump-outputs DIR writes rank 0's outputs of the last timed step as float32 .npy files (see dump_outputs). The inputs
depend on the arguments only, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

H, W = 1080, 1920
BYTES_WARP = 16       # flow 8 + image 3 in + 3 out + flow mask 1 + valid 1
BYTES_COMBINE = 27    # A 8+1, B 8+1, out 8+1
METRIC = "Mpixel/s for apply + combine_with(mode=3) at 1080p"


def frame_transforms(i):
    import golden_inputs as gi
    return gi.cfg4_transforms(i), gi.cfg4_transforms(i + 100000)


def host_inputs(n_distinct, seed=0):
    """Distinct host frames (masks 2 % invalid, uint8x3 images); tiled over the batch on the device."""
    rng = np.random.default_rng(seed)
    am = rng.random((n_distinct, H, W)) > 0.02
    bm = rng.random((n_distinct, H, W)) > 0.02
    img = rng.integers(0, 256, (n_distinct, H, W, 3), dtype=np.uint8)
    return am, bm, img


def dump_outputs(out_dir, arrays, n_sample=1 << 20, seed=0):
    """Writes arrays (name -> DeviceArray of shape (B, H, W) or (B, H, W, C)) as out_dir/<name>.npy, float32, at the
    same fixed, seeded sample of about n_sample pixels for every array: (n,) or (n, C). A full batch of outputs is
    gigabytes; 2**20 pixels of the four outputs are 28 MiB."""
    os.makedirs(out_dir, exist_ok=True)
    B = next(iter(arrays.values())).shape[0]
    idx = np.unique(np.random.default_rng(seed).integers(0, B * H * W, n_sample))
    frame, pix = np.divmod(idx, H * W)
    bounds = np.searchsorted(frame, np.arange(B + 1))
    for name, dev in arrays.items():
        tail = dev.shape[3:]
        out = np.empty((len(idx),) + tail, np.float32)
        for i in range(B):
            a, b = bounds[i], bounds[i + 1]
            if b > a:
                out[a:b] = dev.frames(i, i + 1).numpy().reshape((H * W,) + tail)[pix[a:b]]
        np.save(os.path.join(out_dir, name + '.npy'), out)


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.stop_flag = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {'hw_slowdown': getattr(nv, 'nvmlClocksEventReasonHwSlowdown', 0x8),
                 'hw_thermal_slowdown': getattr(nv, 'nvmlClocksEventReasonHwThermalSlowdown', 0x40),
                 'sw_thermal_slowdown': getattr(nv, 'nvmlClocksEventReasonSwThermalSlowdown', 0x20),
                 'sw_power_cap': getattr(nv, 'nvmlClocksEventReasonSwPowerCap', 0x4),
                 'hw_power_brake': getattr(nv, 'nvmlClocksEventReasonHwPowerBrakeSlowdown', 0x80)}
        while not self.stop_flag.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.005)

    def result(self):
        self.stop_flag.set()
        if self.is_alive():
            self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def reference_module():
    """The UNMODIFIED reference (oflibnumpy 1.1.1), installed into baseline/_ref by __graft_entry__.build() in the build
    container; the directory is git-ignored and travels to the GPU box with the snapshot. None if it is not there."""
    path = os.path.join(ROOT, 'baseline', '_ref')
    if not os.path.isdir(os.path.join(path, 'oflibnumpy')):
        return None
    if path not in sys.path:
        sys.path.insert(0, path)
    try:
        import oflibnumpy
        return oflibnumpy
    except Exception:
        return None


def cpu_reference_step(frames, sample, repeat=1, ref=None):
    """The reference's CPU path on `sample` frames, `repeat` times over; returns seconds. ref = the reference module
    (oflibnumpy.Flow(...).apply / .combine_with, exactly what a user of the reference runs); without it the oracle port
    (cv2.remap + the numpy glue of Flow.apply / combine_with, restated)."""
    if ref is not None:
        t0 = time.perf_counter()
        for _ in range(repeat):
            for (fa, fam, fb, fbm, img) in frames[:sample]:
                a, b = ref.Flow(fa, 't', fam), ref.Flow(fb, 't', fbm)
                a.apply(img, return_valid_area=True)
                a.combine_with(b, 3)
        return time.perf_counter() - t0
    from oracle import flowref as R
    t0 = time.perf_counter()
    for _ in range(repeat):
        for (fa, fam, fb, fbm, img) in frames[:sample]:
            a, b = R.make(fa, 't', fam), R.make(fb, 't', fbm)
            R.apply(a, img, return_valid_area=True)
            R.combine(a, b, 3)
    return time.perf_counter() - t0


def cpu_frames(count, ref=None):
    am, bm, img = host_inputs(count, seed=0)
    if ref is not None:
        gen = ref.from_transforms
    else:
        from oracle import flowref as R
        gen = R.from_transforms
    frames = []
    for i in range(count):
        ta, tb = frame_transforms(i)
        frames.append((gen(ta, (H, W), 't'), am[i], gen(tb, (H, W), 't'), bm[i], img[i]))
    return frames


def run_reference(args, rank, world, restore_stdout=lambda: None):
    if rank != 0:
        return
    import cv2
    sample = args.cpu_sample
    ref = reference_module()
    kind = "reference" if ref is not None else "port"
    frames = cpu_frames(sample, ref)
    for _ in range(args.warmup):
        cpu_reference_step(frames, 1, ref=ref)
    secs = [cpu_reference_step(frames, sample, ref=ref) for _ in range(args.steps)]
    t = float(np.mean(secs))
    value = sample * H * W / t / 1e6
    cores = cv2.getNumThreads()
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "Mpixel/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8+f32", "data": "synthetic",
            "config": {"workload": "cfg4: 1920x1080 apply(uint8x3, valid area) + combine_with(mode=3), ref 't'",
                       "frames_per_step": sample},
            "cpu_baseline": {"value": value, "unit": "Mpixel/s", "cores": cores, "kind": kind,
                             "sample": "%d frames of 1920x1080 per step, per-frame Python loop of %s (the reference has "
                                       "no batch axis); cv2.remap uses %d threads, numpy glue 1" %
                                       (sample, "oflibnumpy 1.1.1 itself (baseline/_ref: Flow.apply + Flow.combine_with)"
                                        if ref is not None else "the oracle port", cores)},
            "e2e": {"value": value, "unit": "Mpixel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    restore_stdout()
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=30)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--batch', type=int, default=256, help='frames per GPU per step')
    ap.add_argument('--e2e-batch', type=int, default=32, help='frames per GPU per end-to-end step (pinned host)')
    ap.add_argument('--e2e-steps', type=int, default=10)
    ap.add_argument('--cpu-sample', type=int, default=8, help='distinct frames per CPU-baseline step')
    ap.add_argument('--cpu-repeat', type=int, default=12, help='passes over the CPU sample (about 13 s of CPU work)')
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-gather', action='store_true', help='skip the optional NCCL gather of the outputs (N > 1)')
    ap.add_argument('--no-modes12', action='store_true', help='skip the modes 1 / 2 block')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write a seeded sample of the outputs of the last timed step to DIR/<name>.npy (float32)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs needs --impl ours')
    if args.warmup < 3 and args.impl == 'ours':
        args.warmup = 3

    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))

    # stdout carries the ONE JSON line and nothing else: whatever libraries print there meanwhile (NCCL announces its
    # version on stdout) goes to stderr
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)

    def restore_stdout():
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)

    if args.impl == 'reference':
        run_reference(args, rank, world, restore_stdout)
        return

    import oflibnumpy_b200 as of
    from oflibnumpy_b200 import _lib, _ops
    from oflibnumpy_b200.device import DeviceArray, Event, Stream
    of.device.require_gpu()

    dist = None
    cpus = []
    if world > 1:
        from oflibnumpy_b200 import dist as ofd0
        # disjoint GPU-local cores per rank: pinned buffers / copy threads of the e2e leg do not fight over one core set
        cpus = ofd0.bind_to_gpu_cpus(local_rank, local_rank, int(os.environ.get('LOCAL_WORLD_SIZE', world)))
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    of.device.set_device(local_rank)
    stream = Stream()
    of.device.set_stream(stream)

    # ---------------------------------------------------------------- device-resident inputs (this rank's shard)
    B = args.batch
    base = rank * B                                   # weak scaling: every rank owns B frames of the global batch
    n_distinct = min(B, 8)
    am_h, bm_h, img_h = host_inputs(n_distinct, seed=rank)
    ta, tb = zip(*[frame_transforms(base + i) for i in range(B)])
    fa = of.FlowBatch.from_transforms(list(ta), (H, W), 't')
    fb = of.FlowBatch.from_transforms(list(tb), (H, W), 't')
    imgs = DeviceArray.empty((B, H, W, 3), np.uint8)
    for i in range(B):
        j = i % n_distinct
        for dst, src in ((fa.masks, am_h), (fb.masks, bm_h), (imgs, img_h)):
            d = dst.frames(i, i + 1)
            _lib.call('ofk_rt_memcpy_h2d', d.ptr, np.ascontiguousarray(src[j]).ctypes.data, d.nbytes, stream.handle)
        if i % 32 == 31:
            stream.synchronize()
    stream.synchronize()

    # persistent outputs: the timed region launches kernels only (no allocation)
    out_img = DeviceArray.empty((B, H, W, 3), np.uint8)
    out_valid = DeviceArray.empty((B, H, W), np.uint8)
    out_vecs = DeviceArray.empty((B, H, W, 2), np.float32)
    out_mask = DeviceArray.empty((B, H, W), np.uint8)
    flags = DeviceArray.empty((B, 2), np.int32)
    arith, rule = _ops.promoted_rule(np.uint8, False)

    def step(evs=None):
        if evs:
            evs[0].record(stream)
        _lib.call('ofk_warp_t', imgs.ptr, _lib.U8, 3, arith, fa.vecs.ptr, -1.0, None, fa.masks.ptr, out_img.ptr,
                  out_valid.ptr, rule, B, H, W, H, W, 0, 0, 1, stream.handle)
        if evs:
            evs[1].record(stream)
        _lib.call('ofk_combine3', fa.vecs.ptr, fa.masks.ptr, fb.vecs.ptr, fb.masks.ptr, ord('t'), 0.0, out_vecs.ptr,
                  out_mask.ptr, flags.ptr, B, H, W, stream.handle)
        if evs:
            evs[2].record(stream)

    def barrier():
        stream.synchronize()
        of.device.synchronize()
        if dist is not None:
            dist.barrier()

    for _ in range(args.warmup):
        step()
    barrier()

    sampler = ClockSampler(local_rank)
    sampler.start()
    ev = [[Event(), Event(), Event()] for _ in range(args.steps)]
    launches0 = _lib.load().ofk_rt_launch_count()
    t_start, t_stop = Event(), Event()
    barrier()
    t_start.record(stream)
    for k in range(args.steps):
        step(ev[k])
    t_stop.record(stream)
    barrier()
    launches = _lib.load().ofk_rt_launch_count() - launches0
    clocks = sampler.result()
    total_ms = t_start.elapsed_ms(t_stop)
    warp_ms = float(np.mean([e[0].elapsed_ms(e[1]) for e in ev]))
    comb_ms = float(np.mean([e[1].elapsed_ms(e[2]) for e in ev]))

    if dist is not None:
        from oflibnumpy_b200 import dist as ofd
        total_ms, warp_ms, comb_ms = ofd.max_over_ranks([total_ms, warp_ms, comb_ms])
    if args.dump_outputs and rank == 0:
        # what callers of FlowBatch.apply(images, return_valid_area=True) and FlowBatch.combine_with(other, 3) receive
        dump_outputs(args.dump_outputs, {'apply_image': out_img, 'apply_valid': out_valid, 'combine_vecs': out_vecs,
                                         'combine_mask': out_mask})
    # ---------------------------------------------------------------- optional gather of the outputs (SURVEY 8e)
    # The combined flows of all ranks are collected on rank 0 over NCCL / NVLink, in chunks on a side stream, while
    # this rank's stream already runs the next step (outputs double-buffered). Reported beside the headline: the
    # gather alone (ms, GB/s into rank 0) and the throughput of steps with their gathers overlapped.
    gather = None
    if dist is not None and not args.no_gather:
        import torch
        ext = torch.cuda.ExternalStream(stream.handle)
        comm = torch.cuda.Stream()
        out_vecs2 = DeviceArray.empty((B, H, W, 2), np.float32)
        bufs = [out_vecs, out_vecs2]
        chunks = 4
        full = torch.empty((world * B, H, W, 2), dtype=torch.float32, device='cuda') if rank == 0 else None

        def gather_chunked(src):
            """Chunk c of every rank's shard goes to rank 0 as one batched send/recv group (the NVSwitch serves all
            peers at once); chunking lets the first bytes leave before the step's last tile is written."""
            t = ofd.as_torch(src)
            per = (B + chunks - 1) // chunks
            for c in range(chunks):
                a, b = c * per, min(B, (c + 1) * per)
                if b <= a:
                    break
                ops = []
                if rank == 0:
                    full[a:b].copy_(t[a:b], non_blocking=True)
                    for r in range(1, world):
                        ops.append(dist.P2POp(dist.irecv, full[r * B + a:r * B + b], r))
                else:
                    ops.append(dist.P2POp(dist.isend, t[a:b], 0))
                for q in dist.batch_isend_irecv(ops):
                    q.wait()

        with torch.cuda.stream(comm):
            gather_chunked(out_vecs)                   # warm-up: NCCL connects lazily
        torch.cuda.synchronize()
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(comm):
            g0.record()
            gather_chunked(out_vecs)
            g1.record()
        torch.cuda.synchronize()
        alone_ms = ofd.max_over_ranks([g0.elapsed_time(g1)])[0]
        gsteps = min(args.steps, 8)

        def step_into(dst_vecs):
            _lib.call('ofk_warp_t', imgs.ptr, _lib.U8, 3, arith, fa.vecs.ptr, -1.0, None, fa.masks.ptr, out_img.ptr,
                      out_valid.ptr, rule, B, H, W, H, W, 0, 0, 1, stream.handle)
            _lib.call('ofk_combine3', fa.vecs.ptr, fa.masks.ptr, fb.vecs.ptr, fb.masks.ptr, ord('t'), 0.0, dst_vecs.ptr,
                      out_mask.ptr, flags.ptr, B, H, W, stream.handle)

        barrier()
        w0, w1 = Event(), Event()
        w0.record(stream)
        done = []
        for k in range(gsteps):
            buf = bufs[k % 2]
            if k >= 2:
                ext.wait_event(done[k - 2])            # the gather that read this buffer two steps ago has finished
            step_into(buf)
            comm.wait_stream(ext)
            with torch.cuda.stream(comm):
                gather_chunked(buf)
                e = torch.cuda.Event()
                e.record()
                done.append(e)
        ext.wait_stream(comm)
        w1.record(stream)
        barrier()
        torch.cuda.synchronize()
        with_ms = ofd.max_over_ranks([w0.elapsed_ms(w1)])[0] / gsteps
        gbytes = (world - 1) * B * H * W * 8
        gather = {"ms_alone": alone_ms, "bytes_into_rank0": gbytes, "gbs_into_rank0": gbytes / alone_ms / 1e6,
                  "chunks": chunks, "steps": gsteps, "ms_per_step_with_gather": with_ms,
                  "value_with_gather": world * B * H * W / (with_ms * 1e-3) / 1e6,
                  "what": "combined flows of all ranks -> rank 0 (batched isend/irecv over NCCL, %d chunks on a side "
                          "stream, overlapped with the next step; outputs double-buffered)" % chunks}
        del full
    ms_per_step = total_ms / args.steps
    px_step = world * B * H * W
    value = px_step / (ms_per_step * 1e-3) / 1e6

    # ---------------------------------------------------------------- end to end through the host-buffer API
    e2e = None
    if not args.no_e2e:
        EB = min(args.e2e_batch, B)
        pin = {}
        keep = []
        for name, shape, dt in (('a', (EB, H, W, 2), np.float32), ('b', (EB, H, W, 2), np.float32),
                                ('am', (EB, H, W), np.bool_), ('bm', (EB, H, W), np.bool_),
                                ('img', (EB, H, W, 3), np.uint8), ('o_img', (EB, H, W, 3), np.uint8),
                                ('o_valid', (EB, H, W), np.bool_), ('o_vecs', (EB, H, W, 2), np.float32),
                                ('o_mask', (EB, H, W), np.bool_)):
            arr, handle = of.device.pinned_empty(shape, dt)
            pin[name] = arr
            keep.append(handle)
        fa.vecs.frames(0, EB).numpy(out=pin['a'])
        fb.vecs.frames(0, EB).numpy(out=pin['b'])
        for i in range(EB):
            pin['am'][i], pin['bm'][i], pin['img'][i] = am_h[i % n_distinct], bm_h[i % n_distinct], img_h[i % n_distinct]

        def e2e_step():
            of.batch.apply_combine_host(pin['a'], pin['b'], pin['img'], 't', pin['am'], pin['bm'],
                                        out_images=pin['o_img'], out_valid=pin['o_valid'], out=pin['o_vecs'],
                                        out_masks=pin['o_mask'], device=local_rank)

        def e2e_two_calls():
            of.batch.apply_flow_host(pin['a'], pin['img'], flow_masks=pin['am'], return_valid_area=True,
                                     out=pin['o_img'], out_valid=pin['o_valid'], device=local_rank)
            of.batch.combine_flows_host(pin['a'], pin['b'], 3, 't', pin['am'], pin['bm'], out=pin['o_vecs'],
                                        out_masks=pin['o_mask'], device=local_rank)

        def timed(fn, steps):
            fn()
            barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                fn()
            barrier()
            dt = (time.perf_counter() - t0) / steps
            return ofd.max_over_ranks([dt])[0] if dist is not None else dt

        dt2 = timed(e2e_two_calls, max(3, args.e2e_steps // 3))
        pin['o_vecs'][...] = 0
        pin['o_img'][...] = 0
        dt = timed(e2e_step, args.e2e_steps)
        px = EB * H * W
        h2d = px * (8 + 1 + 3 + 8 + 1)                    # A, A mask, image, B, B mask: every input once
        d2h = px * (3 + 1) + px * (8 + 1) + EB * 8
        e2e = {"value": world * px / dt / 1e6, "unit": "Mpixel/s", "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "frames_per_step": EB, "steps": args.e2e_steps,
               "api": "batch.apply_combine_host (ofh_apply_combine3: one pass of the pinned ring, A and its mask "
                      "uploaded once for both kernels), pinned numpy buffers",
               "h2d_gbs_per_gpu": px * 21 / dt / 1e9, "d2h_gbs_per_gpu": px * 13 / dt / 1e9,
               "two_calls": {"value": world * px / dt2 / 1e6, "h2d_bytes_per_step": px * 30,
                             "api": "batch.apply_flow_host + batch.combine_flows_host (round 1: A uploaded twice)"}}
        # results of the two paths must agree
        assert np.array_equal(pin['o_vecs'], out_vecs.frames(0, EB).numpy())
        assert np.array_equal(pin['o_img'], out_img.frames(0, EB).numpy())

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---------------------------------------------------------------- roofline of the dominant kernel + CPU baseline
    peaks_path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    else:
        peak, peak_src = 6650.0, 'fallback (B200_PROFILING.md)'
    px_rank = B * H * W
    comb_gbs = px_rank * BYTES_COMBINE / (comb_ms * 1e-3) / 1e9
    warp_gbs = px_rank * BYTES_WARP / (warp_ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get('combine3_ws_dram_bytes_per_px')
            traffic = traffic * px_rank if traffic else None       # bytes per launch, like `achieved`
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "kernel": "c3_ws_kernel<masks> (ofk_combine3, ref t)", "achieved": comb_gbs, "peak": peak,
                "unit": "GB/s", "frac": comb_gbs / peak, "traffic": traffic,
                "traffic_source": "profiles/traffic.json: ncu dram bytes per pixel of this kernel captured at batch 64, "
                                  "scaled to this launch (not measured in this run)", "peak_source": peak_src,
                "bytes_per_px": BYTES_COMBINE, "ms_per_launch": comb_ms,
                "other_kernels": {"warp_u8x3_ws_kernel<half_even, geometry mask, flow mask> (ofk_warp_t)": {"achieved": warp_gbs, "frac": warp_gbs / peak,
                                                            "bytes_per_px": BYTES_WARP, "ms_per_launch": warp_ms}},
                "frac_of_nominal_8TBs": comb_gbs / 8000.0}
    # ---------------------------------------------------------------- modes 1 / 2 of configuration 4 (device-resident)
    modes12 = None
    if not args.no_modes12:
        MB = min(B, 8)
        sa = of.FlowBatch._wrap(fa.vecs.frames(0, MB), 't', fa.masks.frames(0, MB))
        sb = of.FlowBatch._wrap(fb.vecs.frames(0, MB), 't', fb.masks.frames(0, MB))
        modes12 = {"frames": MB, "what": "FlowBatch.combine_with(mode) on %d of the bench's 1080p frame pairs (2 %% "
                   "invalid masks, ref 't'), device-resident, one ofk_combine12 chain per call; Mpixel/s" % MB}
        for mode in (2, 1):
            sa.combine_with(sb, mode)
            stream.synchronize()
            best = 1e30
            for _ in range(3):
                e0, e1 = Event(), Event()
                e0.record(stream)
                sa.combine_with(sb, mode)
                e1.record(stream)
                stream.synchronize()
                best = min(best, e0.elapsed_ms(e1))
            modes12["mode%d_t" % mode] = {"ms": best, "value": MB * H * W / best / 1e3}
    # ---------------------------------------------------------------- source-referenced resampler (cfg 3 operations)
    forward = None
    if not args.no_modes12:
        import golden_inputs as gi
        FB = min(B, 8)
        rot = of.FlowBatch.from_transforms([gi.cfg4_transforms(i) for i in range(FB)], (H, W), 's')
        smooth = of.FlowBatch(np.ascontiguousarray(np.broadcast_to(gi.smooth_field(H, W)[None], (FB, H, W, 2))), 's')
        rot_m = of.FlowBatch._wrap(rot.vecs, 's', fa.masks.frames(0, FB))
        forward = {"frames": FB, "what": "FlowBatch.invert() (same reference: ofk_forward_s, 18 B/px) on %d 1080p 's' "
                   "flows, device-resident: cfg-4 similarity transforms with full masks, the smooth non-affine field of "
                   "SURVEY 8d with full masks (hull pockets), the transforms with 2 %% of the points removed "
                   "(consider_mask: holes bridged); Mpixel/s, fraction of the HBM roofline" % FB}
        for name, fl in (("rotation", rot), ("smooth", smooth), ("rotation_2pct_removed", rot_m)):
            fl.invert()
            stream.synchronize()
            best = 1e30
            for _ in range(3):
                e0, e1 = Event(), Event()
                e0.record(stream)
                fl.invert()
                e1.record(stream)
                stream.synchronize()
                best = min(best, e0.elapsed_ms(e1))
            forward[name] = {"ms": best, "value": FB * H * W / best / 1e3,
                             "frac": FB * H * W * 18 / (best * 1e-3) / 1e9 / peak}
    cpu = None
    if not args.no_cpu_baseline:
        import cv2
        ref = reference_module()
        frames = cpu_frames(args.cpu_sample, ref)
        cpu_reference_step(frames, 1, ref=ref)
        rep = args.cpu_repeat if ref is None else max(1, args.cpu_repeat // 2)
        secs = cpu_reference_step(frames, args.cpu_sample, rep, ref=ref)
        cpu = {"value": rep * args.cpu_sample * H * W / secs / 1e6, "unit": "Mpixel/s", "cores": cv2.getNumThreads(),
               "kind": "reference" if ref is not None else "port", "host_cpus": os.cpu_count(),
               "sample": "%d frame pairs of 1920x1080 (%d distinct x %d), per-frame loop of %s (cv2.remap on %d threads + "
                         "single-threaded numpy glue), %.1f s" %
                         (rep * args.cpu_sample, args.cpu_sample, rep,
                          "oflibnumpy 1.1.1 itself (baseline/_ref)" if ref is not None else "the oracle port",
                          cv2.getNumThreads(), secs)}
        if ref is not None:       # the restated port beside it (it skips the per-Flow isfinite / astype copies)
            pframes = cpu_frames(args.cpu_sample, None)
            cpu_reference_step(pframes, 1)
            psecs = cpu_reference_step(pframes, args.cpu_sample, 2)
            cpu["port_value"] = 2 * args.cpu_sample * H * W / psecs / 1e6
    line = {"metric": METRIC, "value": value, "unit": "Mpixel/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8+f32", "data": "synthetic",
            "config": {"workload": "cfg4: batched 1920x1080 apply(uint8x3, return_valid_area) + "
                                   "combine_with(mode=3), ref 't'", "frames_per_gpu": B, "global_batch": world * B,
                       "parallelism": "batch-sharded x%d, no collective" % world,
                       "cpu_binding": ("rank 0 bound to %d GPU-local cores" % len(cpus)) if cpus else "none",
                       "l2": "inputs (%.1f GB per GPU) exceed L2; no flush needed" %
                             (px_rank * (8 + 8 + 1 + 1 + 3) / 1e9)},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu}
    if modes12 is not None:
        line["modes12"] = modes12
    if forward is not None:
        line["forward_s"] = forward
    if gather is not None:
        line["gather"] = gather
    restore_stdout()
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
