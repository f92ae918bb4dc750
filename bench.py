#!/usr/bin/env python
"""bench.py -- RANSAC-vote throughput (images*keypoints/s) of the B200-native voting layer.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]   # our arm (torchrun for N>1)
    python bench.py --impl reference [--gpus N] --steps K --warmup W   # the reference's own path

One "step" = one ransac_voting_layer_v3(mask, vertex, 512, inlier_thresh=0.99) call over one batch of
BASELINE.json's configs[1] ("cfg2": B=16, 480x640, K=9, 512 hypotheses, ~30 % mask fill, int64 mask,
contiguous [B,H,W,K,2] vertex) per GPU; weak scaling (every rank owns a full batch; every rank's keypoints
reach every rank inside the step: the refit kernel stores them into the peers' HBM over NVLink, see
clean_pvnet_b200/parallel.py).  `--workload cfg4` runs BASELINE.json's configs[3] instead (B=128, 720x540, K=17,
sharded over the ranks: strong scaling).  Prints ONE JSON line on rank 0.

  value      whole-job images*keypoints/s, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e        same metric through the host-buffer entry (pinned host inputs -> H2D -> kernels -> D2H)
  roofline   dominant kernel (vote) : algorithmic bytes of the op / its CUDA-event duration vs measured HBM peak
  cpu_baseline  the CPU oracle port timed on this box's host cores (bounded sample), rank 0, N=1 only

--impl reference times the UNMODIFIED reference (its CUDA extension compiled for sm_100 by
oracle/build_ref.py + its own Python operator, loaded from oracle/_ref) on the same tensors; the
reference has no CPU implementation (ransac_voting.cpp:7-9 asserts CUDA), so where oracle/_ref cannot
be loaded the CPU oracle port is timed instead and the line says so (cpu_baseline.kind).
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT,):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "ransac_vote_throughput"
UNIT = "images*keypoints/s"
WORKLOAD = "cfg2"
HN = 512
THRESH = 0.99
KERNELS_PER_STEP = 5   # mask_bits, thin_gather, generate, vote, refit (+1 exchange_wait per step when N > 1)


def workload_string(name, cfg, layout, per_gpu_images):
    """The SAME string in both arms (ours / --impl reference): what one GPU processes per step."""
    return (f"{name}: B={per_gpu_images} images per GPU per step, {cfg['H']}x{cfg['W']}, K={cfg['K']}, hn={HN}, "
            f"inlier_thresh={THRESH}, fill~30%, int64 mask, vertex layout={layout}, max_num=30000")
# dram__bytes_read.sum + dram__bytes_write.sum of one vote_kernel launch on this workload, from the committed
# `ncu --set full` capture (profiles/r02_ncu_select_vote_refit.txt; ncu flushes the caches before the launch): 39 422 976 + 0.
# In a real step the compacted arrays are still in L2: 4.40 MB + 1.79 MB (profiles/r02_traffic_warm.csv, --cache-control none)
VOTE_KERNEL_DRAM_BYTES = 39422976
VOTE_KERNEL_DRAM_BYTES_WARM = 6190000


def _env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index, period=0.01, reasons_every=1, clock=True):
        # every NVML query stalls the GPU it asks about (tools/scale_diag.py: clock + reasons at 100 Hz cost 31 us per
        # 0.65 ms step), so the sampler asks as rarely as the contract allows: see run_ours()
        self.index, self.period, self.reasons_every, self.clock = index, period, max(1, int(reasons_every)), clock
        self.samples, self.reasons = [], set()
        self.reason_samples = 0
        self.max_mhz = None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = index
            if vis:
                try:
                    phys = int(vis.split(",")[index])
                except Exception:
                    phys = index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        it = 0
        self._stop.wait(min(0.002, self.period))      # first sample 2 ms into the region: the GPU is under load by then
        while not self._stop.is_set():
            try:
                if self.clock:
                    self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                if it % self.reasons_every == 0:
                    try:
                        mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                    except Exception:
                        mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    self.reason_samples += 1
                    for bit, name in names.items():
                        if mask & bit:
                            self.reasons.add(name)
            except Exception:
                pass
            it += 1
            self._stop.wait(self.period)

    def start(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()

    def stop(self):
        self._stop.set()
        if self._thr is not None:
            self._thr.join(timeout=2)
        if not self.samples:
            return None
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s), "reason_samples": self.reason_samples, "period_ms": self.period * 1e3}


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            p = json.load(fh)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def _algorithmic_bytes(B, H, W, K, tn_sum, mask_elt=8):
    # SURVEY.md 8(d): B*[H*W*sizeof(mask) + tn*K*8 + K*8]  (read each mask element once, the selected
    # pixels' K vectors once, write K keypoints)
    return B * H * W * mask_elt + tn_sum * K * 8 + B * K * 8


def _usable_cores():
    """Host threads this process can really run: affinity mask capped by the cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as fh:
            quota, period = fh.read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    return n


def _bind_to_gpu_numa_node(index):
    """One process per GPU on a two-socket box: run this rank's host thread -- and therefore allocate its pinned buffers --
    on the CPUs NVML lists as local to its GPU (`nvidia-smi topo -m`, "CPU Affinity"), so that the end-to-end path's PCIe
    reads do not cross the socket interconnect.  Best effort: returns the number of CPUs bound to, or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[index]) if vis else index
        h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {w * 64 + b for w, m in enumerate(words) for b in range(64) if (m >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if len(cpus) >= 2:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def _cpu_baseline(mask, vertex, K, seconds_target=15.0):
    """Oracle port (oracle/pvnet_oracle.c) on the host cores: one image per thread at a time."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import pvnet_oracle
    pvnet_oracle.build()
    cores = _usable_cores()
    m = mask.cpu().numpy().astype(np.int64)
    v = vertex.cpu().numpy()
    B = m.shape[0]
    t0 = time.perf_counter()
    pvnet_oracle.ransac_voting_layer_v3(m[:1], v[:1], HN, inlier_thresh=THRESH, seed=1)
    t_one = time.perf_counter() - t0
    # bounded sample: about `seconds_target` seconds of wall time assuming perfect scaling, at most
    # two images per thread (host cores share memory bandwidth and, on SMT, FMA pipes)
    n_img = int(max(1, min(cores * max(1, int(seconds_target / max(t_one, 1e-3))), 2 * cores)))
    done = [0]
    lock = threading.Lock()

    def work():
        while True:
            with lock:
                i = done[0]
                if i >= n_img:
                    return
                done[0] += 1
            b = i % B
            pvnet_oracle.ransac_voting_layer_v3(m[b:b + 1], v[b:b + 1], HN, inlier_thresh=THRESH, seed=1, img_base=i)

    t0 = time.perf_counter()
    thr = [threading.Thread(target=work) for _ in range(min(cores, n_img))]
    for t in thr:
        t.start()
    for t in thr:
        t.join()
    dt = time.perf_counter() - t0
    return {"value": n_img * K / dt, "unit": UNIT, "cores": min(cores, n_img), "kind": "port",
            "sample": f"{n_img} images of {WORKLOAD} (480x640, K={K}, hn={HN}) through oracle/pvnet_oracle.c, "
                      f"{min(cores, n_img)} threads, {dt:.1f} s", "single_image_s": t_one}


def _dump_outputs(out_dir, **arrays):
    """Writes each array as out_dir/<name>.npy in float32, so that two builds can be compared output for output."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy().astype(np.float32))


def run_ours(args):
    import torch
    import torch.distributed as dist
    import clean_pvnet_b200 as pvb
    from clean_pvnet_b200 import _lib, parallel, synth

    rank, world, local = _env_int("RANK", 0), _env_int("WORLD_SIZE", 1), _env_int("LOCAL_RANK", 0)
    if world > 1:
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = _bind_to_gpu_numa_node(local) if world > 1 else None
    lib = _lib.load()
    wl = args.workload
    cfg = synth.CONFIGS[wl]
    H, W, K = cfg["H"], cfg["W"], cfg["K"]
    if wl == "cfg2":                       # weak scaling: a full cfg-2 batch on every rank
        B = cfg["B"]
        total = B * world
        scaling = "weak"
    else:                                  # cfg-4: the named batch sharded over the ranks
        total = cfg["B"]
        lo_, hi_ = parallel.shard_bounds(total, world, rank)
        B = hi_ - lo_
        scaling = "strong"
        if total % world:
            raise SystemExit(f"{wl}: {total} images do not split evenly over {world} ranks")
    mask, vertex, _ = synth.make_inputs(wl, device=dev, seed=1234 + 2 + rank, layout=args.layout, B=B)
    layer = None
    if world > 1:
        layer = parallel.ShardedVotingLayer(total, K, depth=4, gather=args.gather, device=dev)
    pending = []

    # --streams S > 1 (experiment, off by default): consecutive steps go round-robin onto S CUDA streams, so the HBM- and
    # latency-bound kernels of one step (select, generate, refit) can fill the SMs the other step's ALU-bound vote kernel
    # leaves idle in its last wave -- the double-buffered way a serving loop would call the layer.  Every step is still a
    # complete call on a complete batch; ms_per_step is then throughput^-1, not the latency of one call.
    streams = [torch.cuda.Stream(device=dev) for _ in range(args.streams)] if args.streams > 1 else None

    def step(i):
        if streams is not None:
            with torch.cuda.stream(streams[i % len(streams)]):
                return step_on_current_stream(i)
        return step_on_current_stream(i)

    def join_streams():
        if streams is not None:
            cur = torch.cuda.current_stream(dev)
            for st_ in streams:
                cur.wait_stream(st_)

    def fork_streams():
        if streams is not None:
            cur = torch.cuda.current_stream(dev)
            for st_ in streams:
                st_.wait_stream(cur)

    def step_on_current_stream(i):
        if layer is not None:
            # the refit kernel pushes this rank's [B,K,2] into every peer's ring (NVLink stores); the wait of step i-4
            # is enqueued by the layer before step i; everything still pending is waited for inside the timed region (drain)
            p = layer(mask, vertex, HN, inlier_thresh=THRESH, seed=1000 + i)
            pending.append(p)
            return p
        return pvb.ransac_voting_layer_v3(mask, vertex, HN, inlier_thresh=THRESH, seed=1000 + i, img_base=rank * B)

    def drain():
        res = None
        if layer is not None:
            layer.drain()
            if pending:
                res = pending[-1].result()
            pending.clear()
        return res

    # one debug call for the workload's tn (units of algorithmic bytes / tests)
    _, dbg = pvb.ransac_voting_layer_v3(mask, vertex, HN, inlier_thresh=THRESH, seed=999, img_base=rank * B, debug=True)
    tn_sum = int(dbg["tn"].sum().item())
    del dbg
    for i in range(max(args.warmup, 3)):
        step(i)
    join_streams()
    drain()
    torch.cuda.synchronize()
    # NVML polling is free with one process (tools/scale_diag.py at N=1: +1 us/step at 100 Hz) but 8 processes polling at
    # 100 Hz cost every rank 31 us per 0.65 ms step (profiles/r02_scale_diag_n8.txt): rank 0 samples its GPU, the others do not
    sampler = ClockSampler(local) if rank == 0 else None
    lib.pvb_profile_reset()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    if layer is not None:
        # GPU-side alignment of the ranks' timelines (untimed): one more step whose gathered result is waited for on the
        # compute stream -- its wait kernel ends when the LAST rank's results have arrived, i.e. at the same moment (+- an
        # NVLink hop) on every rank, so ev0 below is recorded simultaneously everywhere.  The host-side barrier above lets
        # ranks leave up to a few hundred microseconds apart, which a 20-step region would pay as 10-20 us per step.
        layer(mask, vertex, HN, inlier_thresh=THRESH, seed=999).result()
    lib.pvb_profile_enable(args.profile_every)     # stage events on every n-th step only: each record drains the pipeline
    if sampler is not None:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    fork_streams()
    last = None
    t_host0 = time.perf_counter()
    for i in range(args.steps):
        last = step(i)
    t_host1 = time.perf_counter()            # host time to ENQUEUE the steps (the GPU runs behind unless the host is the bottleneck)
    join_streams()
    gathered = drain()
    ev1.record()
    torch.cuda.synchronize()
    out = gathered if gathered is not None else last
    dumped = out.cpu() if args.dump_outputs and rank == 0 else None   # before the extras below call the layer again
    if world > 1:
        dist.barrier()
    clocks = sampler.stop() if sampler is not None else None
    # ---- outside the timed region: the gathered result is what N single-GPU calls produce
    gather_check = None
    if layer is not None:
        layer.check()                                    # raises if any exchange wait timed out
        mine = last.local                                # this rank's own result of the last step
        lo_g = rank * B
        ok = bool(torch.equal(out[lo_g:lo_g + B], mine))
        every = [torch.empty_like(out) for _ in range(world)]
        dist.all_gather(every, out.contiguous())         # NCCL, check only
        ok = ok and all(bool(torch.equal(e, out)) for e in every)
        # and equal to a plain single-GPU call on this rank's shard with the same seed / global image index
        again = pvb.ransac_voting_layer_v3(mask, vertex, HN, inlier_thresh=THRESH, seed=1000 + args.steps - 1, img_base=lo_g)
        ok = ok and bool(torch.equal(again, mine))
        flag = torch.tensor([1 if ok else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        gather_check = "ok" if int(flag.item()) == 1 else "MISMATCH"
    ms = ev0.elapsed_time(ev1)
    import ctypes
    stage = (ctypes.c_double * 4)()
    calls = lib.pvb_profile_read(stage, 4)
    lib.pvb_profile_enable(0)
    stage_ms = [stage[i] / max(calls, 1) for i in range(4)]
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    ms_per_step = ms_max / args.steps
    value = total * K / (ms_per_step * 1e-3)

    # ---- extras (context, not the headline): the un_pnp production pair (resnet18.py:71-72) and B=1 latency
    extras = {}
    try:
        if args.quick:
            raise RuntimeError("skipped (--quick)")

        def timed(fn, n):
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(n):
                fn()
            a1.record()
            torch.cuda.synchronize()
            return a0.elapsed_time(a1) / n
        mean = out[rank * B:(rank + 1) * B] if world > 1 else out
        extras["estimate_voting_distribution_ms"] = timed(
            lambda: pvb.estimate_voting_distribution_with_mean(mask, vertex, mean, seed=7, img_base=rank * B), 10)
        extras["v3_plain_call_ms"] = timed(
            lambda: pvb.ransac_voting_layer_v3(mask, vertex, HN, inlier_thresh=THRESH, seed=7, img_base=rank * B), 30)
        extras["v3_latency_b1_ms"] = timed(
            lambda: pvb.ransac_voting_layer_v3(mask[:1], vertex[:1], HN, inlier_thresh=THRESH, seed=7), 50)
        # SURVEY 8f row 1: decode_keypoint's argmax fused into the select kernel (pvb_decode_v3) vs torch.argmax + v3
        from clean_pvnet_b200 import decode as _dec
        seg = torch.stack([1.0 - mask.float(), mask.float()], dim=1).contiguous()
        extras["decode_front_fused_ms"] = timed(
            lambda: _dec._decode_v3(seg, vertex, HN, THRESH, 5, 30000, 7, rank * B), 30)
        extras["decode_front_unfused_ms"] = timed(
            lambda: pvb.ransac_voting_layer_v3(torch.argmax(seg, 1), vertex, HN, inlier_thresh=THRESH, seed=7,
                                               img_base=rank * B), 30)
    except Exception as e:
        extras["error"] = str(e)
    try:
        # context, NOT the headline: the same calls issued round-robin on 3 CUDA streams -- the HBM- and latency-bound
        # kernels of one step (select, generate, refit) fill the SMs another step's ALU-bound vote kernel leaves idle in its
        # last wave, the way a double-buffered serving loop would call the layer.  The headline stays single-stream so that
        # stage times, kernel shares and the roofline refer to kernels that ran alone.
        if world == 1 and streams is None:
            ms3 = []
            side = [torch.cuda.Stream(device=dev) for _ in range(3)]
            for rep in range(2):
                torch.cuda.synchronize()
                b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                b0.record()
                cur = torch.cuda.current_stream(dev)
                for st_ in side:
                    st_.wait_stream(cur)
                n3 = 60
                for i in range(n3):
                    with torch.cuda.stream(side[i % 3]):
                        pvb.ransac_voting_layer_v3(mask, vertex, HN, inlier_thresh=THRESH, seed=3000 + i, img_base=rank * B)
                for st_ in side:
                    cur.wait_stream(st_)
                b1.record()
                torch.cuda.synchronize()
                ms3.append(b0.elapsed_time(b1) / n3)
            extras["three_streams"] = {"ms_per_step": ms3[-1], "value": total * K / (ms3[-1] * 1e-3),
                                       "note": "60 calls round-robin on 3 streams; throughput, not the latency of a call"}
    except Exception as e:
        extras["three_streams_error"] = str(e)
    try:
        if args.quick:
            raise RuntimeError("skipped (--quick)")
        # SURVEY 8f rows 2+3: the un_pnp tail for this batch -- cov -> inv(sqrtm(cov)) weights, then the batched LM pose
        # refinement (one warp per image), from the keypoints / covariances the voting layer just produced
        kp2d, var = pvb.estimate_voting_distribution_with_mean(mask, vertex, mean, seed=7, img_base=rank * B)
        model = torch.rand((K, 3), device=dev, dtype=torch.float64) * 0.2 - 0.1
        cam = torch.tensor([[572.4114, 0.0, 325.2611], [0.0, 573.57043, 242.04899], [0.0, 0.0, 1.0]], device=dev, dtype=torch.float64)
        init = torch.tensor([0.1, -0.2, 0.3, 0.0, 0.0, 0.9], device=dev, dtype=torch.float64).repeat(B, 1)
        extras["un_pnp_tail_ms"] = timed(
            lambda: pvb.uncertainty_pnp_batch(kp2d, pvb.uncertainty_pnp_weights(var), model, cam, init), 20)
        # the same tail as ONE launch straight from the fp32 outputs (pvb_uncertainty_pnp_from_votes), same initial pose ...
        extras["un_pnp_tail_fused_ms"] = timed(
            lambda: pvb.uncertainty_pnp_from_votes(kp2d, var, model, cam, init), 20)
        # ... and the evaluator's real recipe, P3P initial pose included: three entry points vs one launch
        def three_step():
            w = pvb.uncertainty_pnp_weights(var)
            return pvb.uncertainty_pnp_batch(kp2d, w, model, cam, pvb.p3p_init_batch(kp2d, w, model, cam))
        extras["un_pnp_tail_p3p_3calls_ms"] = timed(three_step, 20)
        extras["un_pnp_tail_p3p_fused_ms"] = timed(lambda: pvb.uncertainty_pnp_from_votes(kp2d, var, model, cam), 20)
    except Exception as e:
        extras["un_pnp_error"] = str(e)

    # ---- end-to-end: pinned host inputs -> H2D -> kernels -> D2H, through the public host entry
    mh, vh = mask.cpu().pin_memory(), vertex.contiguous().cpu().pin_memory()
    oh = torch.empty((B, K, 2), dtype=torch.float32).pin_memory()
    e2e_steps = max(3, min(args.steps, 20)) if not args.quick else 1

    def e2e_run(mode):
        for i in range(3):
            pvb.ransac_voting_layer_v3_host(mh, vh, HN, inlier_thresh=THRESH, seed=1, img_base=rank * B,
                                            chunk_images=args.chunk, out=oh, device=dev, mode=mode)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(e2e_steps):
            pvb.ransac_voting_layer_v3_host(mh, vh, HN, inlier_thresh=THRESH, seed=1000 + i, img_base=rank * B,
                                            chunk_images=args.chunk, out=oh, device=dev, mode=mode)
        e1.record()
        torch.cuda.synchronize()
        te = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        return float(te.item()) / e2e_steps

    e2e_staged_ms = e2e_run("staged")     # both tensors copied host->device (393 MB per step and GPU at cfg-2)
    e2e_inplace_ms = e2e_run("inplace")   # both tensors read in place by the kernels (round 1's mode)
    e2e_ms = e2e_run("auto")              # mask by DMA, selected vertex rows read in place
    staged_bytes = mh.numel() * mh.element_size() + vh.numel() * vh.element_size()
    # bytes that cross the bus in the default mode: the whole mask (DMA) + K float2 per SELECTED pixel (in-place reads)
    h2d = mh.numel() * mh.element_size() + tn_sum * K * 8
    d2h = oh.numel() * oh.element_size()

    if rank == 0:
        hbm_peak, peak_src = _peaks()
        bytes_alg = _algorithmic_bytes(B, H, W, K, tn_sum, mask.element_size())
        vote_ms = stage_ms[2]
        achieved = bytes_alg / (vote_ms * 1e-3) / 1e9 if vote_ms > 0 else None
        tests = K * HN * tn_sum
        sm_mhz = (clocks or {}).get("sm_mhz") or 1965
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {
                "workload": workload_string(wl, cfg, args.layout, B),
                "global_batch": total, "selected_pixels_per_image": tn_sum / B,
                "l2": "inputs larger than L2 (mask+vertex = %.0f MB per GPU > 126 MB); no explicit flush" % (staged_bytes / 1e6),
                "parallelism": (f"dp{world} (images sharded; gather={layer.mode}: "
                                + ("every rank's [B,K,2] stored into all peers' HBM over NVLink by the refit kernel, flag-"
                                   "synchronised, no collective in the steady state; all waits inside the timed region)"
                                   if layer.mode == "peer" else
                                   "one torch.distributed all_gather per step, all waited for inside the timed region)"))
                               if world > 1 else "single GPU",
                "sampling": "philox (in-kernel), new seed every step",
                "streams": args.streams,
            },
            "clocks": clocks,
            "e2e": {"value": total * K / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms, "steps": e2e_steps,
                    "chunk_images": args.chunk,
                    "api": "ransac_voting_layer_v3_host -> pvb_ransac_voting_v3_host (pinned host buffers; mask by DMA, "
                           "only the selected pixels' vertex rows fetched in place over PCIe)",
                    "pcie_gb_s": h2d / (e2e_ms * 1e-3) / 1e9,
                    "inplace": {"value": total * K / (e2e_inplace_ms * 1e-3), "ms_per_step": e2e_inplace_ms,
                                "h2d_bytes_per_step": h2d,
                                "note": "same entry, mode='inplace': mask and vertex rows both read in place (round 1's mode)"},
                    "staged": {"value": total * K / (e2e_staged_ms * 1e-3), "ms_per_step": e2e_staged_ms,
                               "h2d_bytes_per_step": staged_bytes,
                               "note": "same entry, mode='staged': both tensors copied with cudaMemcpyAsync"}},
            "gpu_launches": (KERNELS_PER_STEP + (1 if world > 1 and layer.mode == "peer" else 0)) * args.steps,
            "roofline": {
                "bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                "frac": (achieved / hbm_peak) if achieved else None,
                "traffic": args.traffic if args.traffic is not None else (VOTE_KERNEL_DRAM_BYTES if wl == "cfg2" else None),
                "traffic_warm_caches": VOTE_KERNEL_DRAM_BYTES_WARM if wl == "cfg2" else None,
                "traffic_source": "constants from the committed ncu captures of this kernel on this workload: `--set full` with "
                                  "ncu's cache flush (profiles/r02_ncu_select_vote_refit.txt) and `--cache-control none` "
                                  "(profiles/r02_traffic_warm.csv); not re-measured per run",
                "kernel": "pvb::vote_kernel<4,128,8,512,4>",
                "kernel_ms": vote_ms, "algorithmic_bytes": bytes_alg,
                "peak_source": peak_src,
                "note": "the vote kernel is FP32-issue bound by construction (hn inlier tests per 16 loaded bytes); "
                        "see 'alu' and DESIGN.md",
            },
            "alu": {"inlier_tests_per_step": tests, "tests_per_s_vote_kernel": tests / (vote_ms * 1e-3) if vote_ms else None,
                    "lane_ops_peak_per_s": 148 * 128 * sm_mhz * 1e6,
                    "sass_instr_per_test": 7.1,
                    "note": ("454 SASS instr per 16 pixels x 4 hypotheses per thread (256 FFMA, 64 FADD, 64 LEA.HI, 32 FMNMX3, "
                             "24 LDS); tools/microbench.cu bounds this mix at 610 cycles/block/SMSP => ~4.2 T tests/s")},
            "stages_ms": {"select": stage_ms[0], "generate": stage_ms[1], "vote": stage_ms[2], "refit": stage_ms[3],
                          "profiled_steps": calls, "note": f"CUDA events at the stage boundaries of every {args.profile_every}-th timed step"},
            "host": {"enqueue_ms_per_step": (t_host1 - t_host0) * 1e3 / args.steps, "usable_cores": _usable_cores(),
                     "bound_to_gpu_local_cpus": numa,
                     "note": "host time spent enqueueing one step (rank 0); if it approaches ms_per_step the GPU is launch-starved"},
            "extras": extras,
        }
        if gather_check is not None:
            line["gather_check"] = gather_check
            if layer.gather_error:
                line["gather_fallback_reason"] = layer.gather_error
        if world == 1 and not args.no_cpu_baseline and not args.quick:
            try:
                line["cpu_baseline"] = _cpu_baseline(mask, vertex, K, args.cpu_seconds)
            except Exception as e:   # the oracle is a checker; its absence must not hide the GPU number
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"failed: {e}"}
        if dumped is not None:
            _dump_outputs(args.dump_outputs, keypoints=dumped)
        print(json.dumps(line))
        sys.stdout.flush()
    if world > 1:
        dist.barrier()
        layer.close()
        dist.destroy_process_group()


def run_reference(args):
    rank = _env_int("RANK", 0)
    if rank != 0:
        return          # the reference has no multi-GPU path: rank 0 alone runs it
    import torch
    from clean_pvnet_b200 import synth
    wl = args.workload
    cfg = synth.CONFIGS[wl]
    H, W, K = cfg["H"], cfg["W"], cfg["K"]
    world = _env_int("WORLD_SIZE", 1)
    B = cfg["B"] if wl == "cfg2" else cfg["B"] // world     # what ONE GPU of our arm processes per step
    local = _env_int("LOCAL_RANK", 0)
    gpu_ref = None
    if torch.cuda.is_available():
        try:
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            from refload import load_reference
            _, gpu_ref = load_reference()
        except Exception as e:
            gpu_ref, why = None, str(e)
    base = {"metric": METRIC, "unit": UNIT, "n_gpus": _env_int("WORLD_SIZE", 1), "steps": args.steps,
            "warmup": max(args.warmup, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "impl": "reference"}
    if gpu_ref is not None:
        torch.cuda.set_device(local)
        dev = torch.device("cuda", local)
        mask, vertex, _ = synth.make_inputs(wl, device=dev, seed=1234 + 2, layout=args.layout, B=B)
        for i in range(max(args.warmup, 3)):
            torch.manual_seed(i)
            gpu_ref.ransac_voting_layer_v3(mask, vertex, HN, inlier_thresh=THRESH)
        torch.cuda.synchronize()
        sampler = ClockSampler(local)
        sampler.start()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for i in range(args.steps):
            torch.manual_seed(1000 + i)
            gpu_ref.ransac_voting_layer_v3(mask, vertex, HN, inlier_thresh=THRESH)
        ev1.record()
        torch.cuda.synchronize()
        clocks = sampler.stop()
        ms_per_step = ev0.elapsed_time(ev1) / args.steps
        value = B * K / (ms_per_step * 1e-3)
        extras = {}
        try:   # context: the other half of the un_pnp production pair (resnet18.py:71-72) and B=1 latency
            mean = gpu_ref.ransac_voting_layer_v3(mask, vertex, HN, inlier_thresh=THRESH)
            gpu_ref.estimate_voting_distribution_with_mean(mask[:2], vertex[:2], mean[:2])
            torch.cuda.synchronize()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            gpu_ref.estimate_voting_distribution_with_mean(mask, vertex, mean)
            a1.record()
            torch.cuda.synchronize()
            extras["estimate_voting_distribution_ms"] = a0.elapsed_time(a1)
            a0.record()
            for _ in range(5):
                gpu_ref.ransac_voting_layer_v3(mask[:1], vertex[:1], HN, inlier_thresh=THRESH)
            a1.record()
            torch.cuda.synchronize()
            extras["v3_latency_b1_ms"] = a0.elapsed_time(a1) / 5
        except Exception as e:
            extras["error"] = str(e)
        line = dict(base, value=value, ms_per_step=ms_per_step, clocks=clocks, extras=extras,
                    config={"workload": workload_string(wl, cfg, args.layout, B),
                            "global_batch": B, "parallelism": "single GPU (the reference has no multi-GPU path)",
                            "implementation": "unmodified clean-pvnet lib/csrc/ransac_voting (CUDA ext compiled for sm_100 "
                                              "by oracle/build_ref.py) through its own ransac_voting_layer_v3"},
                    cpu_baseline={"value": value, "unit": UNIT, "cores": 0, "kind": "reference",
                                  "sample": f"{args.steps} batches of {B} {wl} images on 1 GPU (the reference path is CUDA-only, "
                                            "ransac_voting.cpp:7-9)"},
                    e2e={"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})
    else:
        mask, vertex, _ = synth.make_inputs(wl, device="cpu", seed=1234 + 2, B=min(B, 4))
        cb = _cpu_baseline(mask, vertex, K, args.cpu_seconds)
        line = dict(base, value=cb["value"], ms_per_step=None,
                    config={"workload": workload_string(wl, cfg, args.layout, B),
                            "implementation": "bounded sample through the CPU oracle port; the reference CUDA extension "
                                              "is not loadable here"},
                    cpu_baseline=cb, e2e={"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0,
                                          "d2h_bytes_per_step": 0})
    print(json.dumps(line))
    sys.stdout.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--layout", default="interleaved", choices=["interleaved", "planar"])
    ap.add_argument("--workload", default=WORKLOAD, choices=["cfg2", "cfg4"])
    ap.add_argument("--gather", default="auto", choices=["auto", "peer", "collective"],
                    help="N>1: how every rank's keypoints reach every rank (clean_pvnet_b200/parallel.py)")
    ap.add_argument("--chunk", type=int, default=4, help="images per H2D chunk of the end-to-end path")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--streams", type=int, default=1,
                    help="experiment: issue consecutive steps round-robin on this many CUDA streams (default 1)")
    ap.add_argument("--profile-every", type=int, default=4,
                    help="record the stage events (stages_ms, roofline.kernel_ms) on every n-th timed step")
    ap.add_argument("--quick", action="store_true",
                    help="profiling passes (ncu): timed steps only -- no extras, no end-to-end runs, no CPU baseline")
    ap.add_argument("--traffic", type=float, default=None,
                    help="dram bytes/launch of the vote kernel from the committed ncu capture (profiles/)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the keypoints [images of all ranks,K,2] of the last timed step to DIR/keypoints.npy (float32); the inputs "
                         "and the step's seed depend only on the arguments, so two builds can be compared")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
