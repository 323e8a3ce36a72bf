#!/usr/bin/env python
"""bench.py -- update-iteration throughput of the DPVO hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config default|fast] [--dump-outputs DIR]

One "step" = one DPVO.update() (dpvo/dpvo.py:328-360): reprojection, 2-level patch correlation,
update operator, 2 Gauss-Newton BA iterations, on the steady-state synthetic patch graph of
BASELINE.json configs[1] (480x640, 96 patches/frame, 10-pose window, E = 47,712 edges; one update per
frame in steady state, so steps/s == frames/s of the hot path).  N > 1 runs one independent stream per
GPU (no collective on the data path): whole-job value = N * stream rate, scaling "weak".

Prints ONE JSON line (rank 0).  `value` is device-resident throughput, `e2e` the same step through the
public API with the new frame coming from pinned host memory and poses/depths read back to the host.
`roofline` is for the dominant kernel CLASS of the step, the update operator's dense layers
(linear_f16_kernel, 15 launches): algorithmic FLOPs (SURVEY 8(d): 5.396 MFLOP/edge) / the summed CUDA-event
time of those launches in the eager pass, vs the measured sustained dense tensor peak in MEASURED_PEAKS.json.
`roofline_corr` keeps the correlation kernel's numbers: algorithmic bytes/time (served mostly by L2, so NOT an
HBM fraction) next to the DRAM and L2 bytes of one launch from the committed ncu capture.
`reference_cuda` = the reference's OWN CUDA pipeline for the same update on the same state, timed in the same
run (oracle/ref_pipeline.py:RefCudaStep: ref_cuda_corr x2 + stack, torch Update under autocast, ref_cuda_ba
from oracle/_ref) -- the same-box denominator of north_star's ">= 5x the reference CUDA build".
`--dump-outputs DIR` writes what the timed path computed in its last timed step (rank 0) as DIR/<name>.npy; the inputs
are seeded, so two builds run with the same arguments can be compared output for output.
`--impl reference` times the reference's CPU path (oracle port of F.grid_sample correlation + PyTorch
Update + dpvo/ba.py BA, BASELINE.json configs[0] style) on a bounded sample of the same workload.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BYTES_PER_EDGE_FP16 = 50492      # SURVEY 8(d), both pyramid levels, s = 2 bytes
METRIC = "update-iterations/sec of the DPVO hot path (reproject + corr + update operator + 2 BA iterations; one update per frame in steady state)"
FLOP_PER_EDGE = 2 * (882 * 384 + 16 * 384 * 384)      # SURVEY 8(d): the 17 dense layers of the update operator


def peaks():
    """(HBM GB/s, dense 16-bit TFLOP/s sustained, source).  Sustained, not burst: the kernels are timed inside a step."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        tf = d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1416.5))
        return d.get("hbm_gbs", 6650.0), tf, "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1416.5, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def wait_first(self, timeout=8.0):
        """nvidia-smi needs up to a second before its first row; block until the stream is live"""
        t0 = time.time()
        while self.proc is not None and not self.rows and time.time() - t0 < timeout:
            time.sleep(0.02)

    def count_in(self, windows):
        return sum(1 for t, _ in self.rows if any(a <= t <= b for a, b in windows))

    def stop(self, windows=None):
        """median SM clock / union of throttle reasons over the rows sampled inside `windows` (host times)"""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for t, r in self.rows:
            if windows is not None and not any(a <= t <= b for a, b in windows):
                continue
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------ CPU path
def cpu_reference_step_factory(config, sample_stride, threads):
    """The reference's CPU implementation of one update() on the edges of every `sample_stride`-th
    patch of the SAME synthetic graph: grid_sample correlation (2 levels) + Update (fp32 torch) +
    2 x dpvo/ba.py BA.  Returns (step_fn, E_sample, E_full)."""
    import torch
    from dpvo_b200 import synthetic
    from oracle import ba as OB, corr as OC, update as OU
    torch.set_num_threads(threads)
    st = synthetic.make_state(config, 36 if config == "default" else 30, device="cpu", features=False)
    M = st.cfg["M"]
    keep = (st.kk % sample_stride) == 0
    ii, jj, kk = st.ii[keep], st.jj[keep], st.kk[keep]
    E = int(keep.sum())
    g = torch.Generator().manual_seed(5)
    frames = sorted(set(jj.tolist()))
    h, w = st.cfg["ht"] // 4, st.cfg["wd"] // 4
    remap = {f: i for i, f in enumerate(frames)}
    jl = torch.tensor([remap[int(j)] for j in jj])
    fmap1 = torch.randn(1, len(frames), 128, h, w, generator=g) / 4
    fmap2 = torch.nn.functional.avg_pool2d(fmap1[0], 4, 4)[None]
    pk = torch.unique(kk)
    kl = torch.searchsorted(pk, kk)
    gmap = torch.randn(1, len(pk), 128, 3, 3, generator=g) / 4
    imap = torch.randn(1, len(pk), 384, generator=g) / 4
    torch.manual_seed(1234)
    upd = OU.Update(3).eval()
    net = torch.zeros(1, E, 384)
    poses, patches, intr = st.poses[None], st.patches[None], st.intrinsics[None]
    bounds = [-64, -64, w + 64, h + 64]

    def step():
        with torch.no_grad():
            coords = OB.transform(poses, patches, intr, ii, jj, kk).permute(0, 1, 4, 2, 3).contiguous()
            c0 = OC.corr_grid_sample(gmap, fmap1, coords, kl, jl, 3)
            c1 = OC.corr_grid_sample(gmap, fmap2, coords / 4, kl, jl, 3)
            corr = torch.stack([c0, c1], -1).view(1, E, -1)
            n2, (delta, weight, _) = upd(net, imap[:, kl], corr, None, ii, jj, kk)
            target = coords[..., 1, 1] + delta
            P, Q = poses, patches
            for _ in range(2):
                P, Q = OB.python_ba(P, Q, intr, target, weight, 1e-4, ii, jj, kk, bounds, ep=10.0, fixedp=1)
        return P

    return step, E, st.E


def cpu_reference_measure(config, steps, warmup, budget_s, full_check=False):
    """Times the CPU implementation of the update on a bounded sample; returns (frames/s scaled to the full graph,
    threads used, sample description, E_full).  The per-step sample is sized so that warmup + steps take about
    `budget_s` on this host: the cost of one step is probed on a thin sample first (cost is linear in the edges)."""
    import torch
    threads = os.cpu_count() or 1
    probe_stride = 96 if config == "default" else 32
    step, Es, Ef = cpu_reference_step_factory(config, probe_stride, threads)
    step()
    # the update is many mid-sized ops: past a few dozen threads torch's intra-op pool only adds contention,
    # so time the probe at several pool sizes and keep the fastest (reported as `cores`)
    best = None
    for nt in sorted({threads, min(threads, 64), min(threads, 32), min(threads, 16), min(threads, 8)}, reverse=True):
        torch.set_num_threads(nt)
        step()
        t0 = time.perf_counter(); step(); dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, nt)
    t_probe, threads = best
    want = budget_s / max(1, steps + warmup)
    stride = int(min(probe_stride * 4, max(probe_stride // 4, -(-probe_stride * t_probe // want))))
    if stride != probe_stride:
        step, Es, Ef = cpu_reference_step_factory(config, stride, threads)
    torch.set_num_threads(threads)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    full = dt * Ef / Es                      # seconds per full update, linear in the edge count
    sample = "edges of every %dth patch: %d of %d edges per step, time scaled by %d/%d" % (stride, Es, Ef, Ef, Es)
    check = None
    if full_check and stride > 1:
        # ONE update on the whole graph (no sampling), to show what the scaling is worth: BA and the grouped
        # softmax are not strictly linear in the edges
        fstep, _, _ = cpu_reference_step_factory(config, 1, threads)
        t0 = time.perf_counter(); fstep(); t_full = time.perf_counter() - t0
        check = {"full_graph_one_step_s": t_full, "scaled_sample_s": full, "ratio": t_full / full}
        full = t_full                        # the measured full-graph time is the number reported
        sample += "; plus ONE untimed-loop step on all %d edges: %.2f s measured vs %.2f s scaled (reported value = measured full-graph step)" % (Ef, t_full, check["scaled_sample_s"])
    return 1.0 / full, threads, sample, Ef, dt, check


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # all host cores serve one stream at a time: the whole-job CPU rate does not grow with --gpus
    val, threads, sample, Ef, dt, check = cpu_reference_measure(args.config, args.steps, args.warmup, 100.0, full_check=True)
    out = {"impl": "reference", "metric": METRIC, "value": val, "unit": "frames/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
           "ms_per_step_is": "measured wall time of one SAMPLED step (see cpu_baseline.sample); value = full-graph updates/s",
           "full_graph_check": check, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": workload_config(args.config, Ef),
           "cpu_baseline": {"value": val, "unit": "frames/s", "cores": threads, "kind": "port", "sample": sample},
           "e2e": {"value": val, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def _bytes(txt):
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    val, unit = txt.split()
    return float(val) * scale[unit]


def ncu_summaries():
    """hardware counters of the committed `ncu --set full` captures (profiles/): newest round first"""
    out = {}
    prof = os.path.join(ROOT, "profiles")
    for rnd in ("r02", "r01"):
        path = os.path.join(prof, "%s_ncu_corr_fwd_tc.json" % rnd)
        if "corr_dram_bytes" not in out and os.path.exists(path):
            try:
                k = json.load(open(path))["kernels"][0]
                out["corr_dram_bytes"] = _bytes(k["dram_read"]) + _bytes(k["dram_write"])
                out["corr_l2_bytes"] = _bytes(k["l2_to_sm_read"]) if "l2_to_sm_read" in k else None
                out["corr_source"] = "profiles/" + os.path.basename(path)
            except Exception:
                pass
        path = os.path.join(prof, "%s_ncu_gemm_step.json" % rnd)
        if "gemm_dram_bytes" not in out and os.path.exists(path):
            try:
                out["gemm_dram_bytes"] = sum(_bytes(k["dram_read"]) + _bytes(k["dram_write"]) for k in json.load(open(path))["kernels"])
            except Exception:
                pass
    return out


def reference_cuda_leg(st, run, our_ms, iters=10, warmup=3):
    """The reference's own CUDA pipeline for the SAME update on the SAME state, timed here with CUDA events:
    ref_cuda_corr.forward x2 + stack (dpvo.py:200-207), the torch Update under autocast (dpvo.py:332) with the same
    weights, ref_cuda_ba.forward (2 iterations) -- oracle/ref_pipeline.py:RefCudaStep over oracle/_ref.  This is the
    checker used as a baseline (allowed for bench.py); none of our kernels run inside it."""
    import torch
    try:
        from oracle import update as OU
        from oracle.ref_pipeline import RefCudaStep
        mod = OU.Update(3).to(st.poses.device).eval()
        mod.load_state_dict(run.update.state_dict())
        ref = RefCudaStep(st, mod)
    except Exception as exc:                               # noqa: BLE001 -- oracle/_ref not shipped: say so
        return {"unavailable": str(exc).splitlines()[0][:160]}
    for _ in range(warmup):
        ref.reset(); ref.step()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        ref.reset()
        ref.step()
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / iters
    return {"ms_per_step": ms, "value": 1e3 / ms, "unit": "frames/s", "iters": iters, "speedup_ours": ms / our_ms,
            "what": "reference CUDA kernels (oracle/_ref: correlation_kernel.cu, ba_cuda.cu compiled for sm_100a) + torch Update under "
                    "autocast, eager launches as in dpvo.py:328-360, same synthetic state and weights, same GPU, same process"}


def workload_config(config, E):
    if config == "default":
        w = "BASELINE configs[1]: synthetic 480x640 stream, default.yaml (96 patches, 10-pose window), E=%d edges, 2208 live patches" % E
    else:
        w = "BASELINE configs[2]: synthetic 480x752 stream, fast.yaml (48 patches, 7-pose window), E=%d edges" % E
    return {"workload": w, "edges": E, "l2_policy": "inputs larger than L2 (fp16 feature ring 188 MB > 126 MB L2); no flush",
            "parallelism": "one independent stream per GPU, no collectives"}


# ------------------------------------------------------------------------------------ GPU path
DUMP_NET_ROWS = 4096          # rows of the recurrent state kept by --dump-outputs (a fixed seeded sample of E)


def step_outputs(st, run, target, weight):
    """host copies of what one update hands its caller: the BA-refined poses and patch inverse depths of the
    window, the flow target / confidence of every edge, and a fixed seeded sample of the recurrent state rows"""
    import torch
    rows = torch.randperm(st.E, generator=torch.Generator().manual_seed(0))[:DUMP_NET_ROWS].sort().values
    return {"poses": st.poses[:st.n].float().cpu(), "depths": st.patches[:st.n * run.M, 2, 1, 1].float().cpu(),
            "target": target[0].float().cpu(), "weight": weight[0].float().cpu(),
            "net_rows": rows, "net_sample": run.net[0, rows.to(run.net.device)].float().cpu()}


def dump_outputs(out_dir, outputs):
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for k, v in outputs.items():
        a = v.numpy()
        np.save(os.path.join(out_dir, k + ".npy"), a.astype(np.float64 if a.dtype.kind in "iu" else np.float32))


def run_ours(args):
    import torch
    import dpvo_b200
    from dpvo_b200 import synthetic, multigpu
    from dpvo_b200.runner import UpdateRunner
    rank, world, local = multigpu.env_rank()
    torch.cuda.set_device(local)
    dev = "cuda:%d" % local
    multigpu.init("nccl", dev)
    ex = dpvo_b200.extensions()[3]

    n_frames = 36 if args.config == "default" else 30
    st = synthetic.make_state(args.config, n_frames, device=dev, seed=1234 + rank)
    run = UpdateRunner(st)
    E = st.E

    def barrier():
        torch.cuda.synchronize()
        multigpu.barrier()
        torch.cuda.synchronize()

    # ---- device-resident loop
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        run.reset(); run.step()
    if rank == 0:
        sampler.wait_first()
    windows = []
    ev = {k: [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)] for k in ("corr0", "corr1", "ba0", "ba1")}
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    w0 = time.time()
    l0 = ex.launch_count()
    t_start.record()
    gemm_events = []
    run.update.gemm_events = gemm_events                 # (start, end) CUDA events around every dense-layer launch
    for i in range(args.steps):
        run.timers = {k: v[i] for k, v in ev.items()}
        run.reset()
        out = run.step()
    t_end.record()
    barrier()
    windows.append((w0, time.time()))
    launches = ex.launch_count() - l0
    run.timers = None
    outputs = step_outputs(st, run, *out) if args.dump_outputs and rank == 0 else None
    run.update.gemm_events = None
    gemm_ms = sum(a.elapsed_time(b) for a, b in gemm_events) / args.steps
    gemm_launches = len(gemm_events) // args.steps
    ms_eager = t_start.elapsed_time(t_end) / args.steps
    ms = ms_eager
    corr_ms = statistics.mean(a.elapsed_time(b) for a, b in zip(ev["corr0"], ev["corr1"]))
    ba_ms = statistics.mean(a.elapsed_time(b) for a, b in zip(ev["ba0"], ev["ba1"]))

    # ---- the same step as a CUDA graph (how the runner is meant to be driven): timed the same way.  The eager
    # pass above stays for the per-stage breakdown (events cannot be recorded inside a graph).
    launch_mode = "eager launches"
    graph_out = None
    if not args.no_graph:
        try:
            run.capture()
            for _ in range(3):
                run.reset(); run.step_graph()
            barrier()
            w0 = time.time()
            t_start.record()
            for i in range(args.steps):
                run.reset()
                out = run.step_graph()
            t_end.record()
            barrier()
            windows.append((w0, time.time()))
            ms = t_start.elapsed_time(t_end) / args.steps
            launch_mode = "CUDA graph replay (%d kernel nodes per step)" % (launches // args.steps)
            launches *= 2                                  # kernels of the eager pass + of the replays
            graph_out = out
        except Exception as exc:                           # noqa: BLE001 -- report and keep the eager number
            run.graph = None
            launch_mode = "eager launches (graph capture failed: %s)" % str(exc).splitlines()[0][:120]
    if outputs is not None and graph_out is not None:      # the reported rate is the graph loop's: dump its last step
        outputs = step_outputs(st, run, *graph_out)

    # ---- end to end: new frame from pinned host memory every step, poses + depths back to host
    hf = run.make_host_frame()
    out_p = [torch.empty(st.n, 7, pin_memory=True) for _ in range(2)]       # two result buffers in rotation: the host reads
    out_d = [torch.empty(st.n * run.M, pin_memory=True) for _ in range(2)]  # frame t while the device computes frame t+1
    # frame t+1 is uploaded (pinned host -> staging, copy stream) while update t runs, as a streaming front end
    # would; the first upload of the timed region is exposed, and there are exactly `steps` uploads in it
    run.upload(hf)
    for _ in range(3):
        run.reset(); run.step_e2e_pipelined(hf, out_p[0], out_d[0])
    torch.cuda.synchronize()
    run.step_e2e_pipelined(None, out_p[0], out_d[0])           # drain the last warm-up upload
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.time()
    e0.record()
    h2d = run.upload(hf)
    prev, checksum = None, 0.0
    for i in range(args.steps):
        run.reset()
        _, d2h, done = run.step_e2e_pipelined(hf if i + 1 < args.steps else None, out_p[i & 1], out_d[i & 1])
        if prev is not None:                               # the host consumes frame i-1 (its copies have landed) while frame i runs
            prev.synchronize()
            checksum += float(out_p[(i - 1) & 1][-1, 0]) + float(out_d[(i - 1) & 1][0])
        prev = done
    prev.synchronize()
    checksum += float(out_p[(args.steps - 1) & 1][-1, 0]) + float(out_d[(args.steps - 1) & 1][0])
    e1.record()
    barrier()
    windows.append((w0, time.time()))
    clocks = None
    if rank == 0:
        # nvidia-smi delivers a row every 100 ms; when the timed regions are shorter than a few rows, keep the
        # identical step loop running (untimed) until the sampler has seen the GPU under this load
        cont = 0
        tc0 = time.time()
        while sampler.proc is not None and sampler.count_in(windows + [(tc0, time.time())]) < 5 and time.time() - tc0 < 3.0:
            run.reset(); run.step(); cont += 1
            if cont % 16 == 0:
                torch.cuda.synchronize()
        torch.cuda.synchronize()
        if cont:
            windows.append((tc0, time.time()))
        clocks = sampler.stop(windows)
        clocks["window"] = "timed regions" if not cont else "timed regions + %d untimed steps of the same loop" % cont
    barrier()
    e2e_ms = e0.elapsed_time(e1) / args.steps

    # one stream per rank: whole-job rate = (steps of all ranks) / (slowest rank's time)
    ms, e2e_ms, corr_ms, ba_ms, gemm_ms = multigpu.max_over_ranks([ms, e2e_ms, corr_ms, ba_ms, gemm_ms], dev)
    if rank != 0:
        multigpu.finalize()
        return

    hbm, tensor_tf, which = peaks()
    corr_alg = BYTES_PER_EDGE_FP16 * E / (corr_ms * 1e-3) / 1e9
    # dense layers: 17 layers x E rows (+ the two h layers on the group rows, < 1 % and not counted)
    gemm_flop = FLOP_PER_EDGE * E
    gemm_tf = gemm_flop / (gemm_ms * 1e-3) / 1e12
    ncu = ncu_summaries()
    out = {"metric": METRIC, "value": world * 1e3 / ms, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
           "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f16 operands, f32 accumulate/state (BA f32)", "data": "synthetic", "config": workload_config(args.config, E),
           "breakdown_ms": {"corr": corr_ms, "ba": ba_ms, "dense_layers": gemm_ms, "dense_layer_launches": gemm_launches,
                            "row_kernels_grouping_and_rest": ms_eager - corr_ms - ba_ms - gemm_ms,
                            "gemm_backend": "tcgen05: fused layer chains (dpvo_update_corr_norm / neighbor_mlp x2 / gru_heads) + dpvo_linear_f16 for the SoftAgg layers", "eager_ms_per_step": ms_eager, "launch": launch_mode},
           "e2e": {"value": world * 1e3 / e2e_ms, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                   "pipeline": "frame t+1: pinned host -> staging on a copy stream while update t runs; staging -> ring slots, update (CUDA graph), "
                               "D2H of poses + depths into one of two pinned result buffers; the host waits for and reads frame t's results after it has issued frame t+1"},
           "gpu_launches": int(launches), "clocks": clocks,
           "roofline": {"kernel": "chain_kernel x4 + linear_f16_kernel x4 (%d launches: the 17 dense layers of the update operator with their LayerNorm / gating / heads epilogues, tcgen05.mma + TMA + TMEM)" % gemm_launches,
                        "bound": "tensor", "achieved": gemm_tf, "peak": tensor_tf, "unit": "TFLOP/s", "frac": gemm_tf / tensor_tf,
                        "traffic": ncu.get("gemm_dram_bytes"), "peak_source": which + ", sustained dense 16-bit (kernels timed inside a step)",
                        "algorithmic_flop_per_step": gemm_flop, "kernel_ms": gemm_ms,
                        "timing": "sum of CUDA-event intervals around each of the launches, eager pass, same stream; since round 2 the intervals also contain the LayerNorm, gating, residual and heads work that is fused into the chain kernels' epilogues",
                        "traffic_note": "sum of dram__bytes_read+write over the 8 dense-layer launches of one update, ncu --set full capture of this build: profiles/r02_ncu_gemm_step.json"},
           "roofline_corr": {"kernel": "corr_fwd_tc (2-level patch correlation, tcgen05 + TMA)", "kernel_ms": corr_ms,
                             "algorithmic_bytes_per_launch": BYTES_PER_EDGE_FP16 * E, "algorithmic_GBps": corr_alg,
                             "note": "SURVEY 8(d)'s per-edge window bytes are served by L2 (each frame is reused ~11x), so algorithmic/HBM-peak (%.2f) is "
                                     "NOT a DRAM fraction; the hardware counters of one launch are below" % (corr_alg / hbm),
                             "dram_bytes": ncu.get("corr_dram_bytes"), "l2_to_sm_bytes": ncu.get("corr_l2_bytes"),
                             "dram_frac_of_hbm_peak": (ncu["corr_dram_bytes"] / (corr_ms * 1e-3) / 1e9 / hbm) if ncu.get("corr_dram_bytes") else None,
                             "ncu_source": ncu.get("corr_source")}}
    if not args.no_reference_cuda and world == 1:
        out["reference_cuda"] = reference_cuda_leg(st, run, ms)
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    if not args.no_cpu_baseline and world == 1:          # the CPU leg is timed at N = 1 only
        # same figure as the reference arm reports: one measured update on the whole graph (the strided sample only picks the pool size)
        val, threads, sample, _, _, chk = cpu_reference_measure(args.config, 2, 1, 20.0, full_check=True)
        out["cpu_baseline"] = {"value": val, "unit": "frames/s", "cores": threads, "kind": "port", "sample": sample, "full_graph_check": chk}
    print(json.dumps(out))
    multigpu.finalize()


# ------------------------------------------------------------------------------------ training step (configs[3])
TRAIN_METRIC = ("training clips/sec: batch of 8 synthetic 15-frame 480x640 subsequences per optimiser step, 18 unrolled updates "
                "(altcorr fwd+bwd, differentiable update operator and BA), NCCL gradient all-reduce, AdamW")


def synthetic_clip(device, seed, n_frames=15, ht=480, wd=640):
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    images = (torch.rand(1, n_frames, 3, ht, wd, generator=g, device=device) * 255).floor()
    k = torch.ones(3, 1, 5, 5, device=device) / 25
    images = torch.nn.functional.conv2d(images[0], k, padding=2, groups=3)[None]          # uint8-valued-ish smooth frames
    disps = 0.1 + 0.9 * torch.rand(1, n_frames, ht, wd, generator=g, device=device)
    poses = torch.zeros(1, n_frames, 7, device=device)
    poses[..., 6] = 1.0
    poses[0, :, 0] = 0.05 * torch.arange(n_frames, device=device)
    intr = torch.tensor([320.0, 320.0, 320.0, 240.0], device=device).view(1, 1, 4).repeat(1, n_frames, 1)
    return images, poses, disps, intr


def run_train(args):
    """BASELINE configs[3]: global batch 8 clips per optimiser step, split over the ranks (strong scaling: 1 GPU runs
    8 clips with gradient accumulation, 8 GPUs one clip each), gradients averaged over NVLink by
    dpvo_b200.multigpu.GradReducer (bucketed NCCL all-reduce launched from autograd hooks)."""
    import numpy as np
    import torch
    import dpvo_b200
    from dpvo_b200 import multigpu
    from dpvo_b200.train import VONet, TrainStep
    rank, world, local = multigpu.env_rank()
    torch.cuda.set_device(local)
    dev = "cuda:%d" % local
    multigpu.init("nccl", dev)
    ex = dpvo_b200.extensions()[3]
    torch.manual_seed(1234); np.random.seed(1234 + rank)
    net = VONet().to(dev).train()
    red = multigpu.GradReducer(net.parameters())
    step = TrainStep(net, steps_unrolled=18, total_steps=100000, reducer=red)
    global_batch = 8
    local_clips = max(1, global_batch // world)
    pinned = [[t.cpu().pin_memory() for t in synthetic_clip(dev, 1234 + rank * 100 + c)] for c in range(local_clips)]

    def one_step():
        clips = [[t.to(dev, non_blocking=True) for t in c] for c in pinned]          # H2D of this step's inputs
        loss, _ = step.step_clips(clips, structure_only=False)
        return float(loss)                                                             # D2H of the loss

    def barrier():
        torch.cuda.synchronize(); multigpu.barrier(); torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 1)):
        one_step()
    if rank == 0:
        sampler.wait_first()
    barrier()
    w0 = time.time()
    l0 = ex.launch_count()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(args.steps):
        loss = one_step()
    b.record()
    barrier()
    w1 = time.time()
    launches = ex.launch_count() - l0
    ms, = multigpu.max_over_ranks([a.elapsed_time(b) / args.steps], dev)
    clocks = sampler.stop([(w0, w1)]) if rank == 0 else None
    if rank == 0:
        h2d = sum(t.numel() * t.element_size() for c in pinned for t in c)
        clips_per_s = local_clips * world / (ms * 1e-3)
        out = {"metric": TRAIN_METRIC, "value": clips_per_s, "unit": "clips/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 1),
               "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32 (training runs without autocast, net.py:187)",
               "data": "synthetic", "gpu_launches": int(launches), "clocks": clocks, "last_loss": loss,
               "config": {"workload": "BASELINE configs[3]: training step, global batch 8 x 15 frames x 480x640, 80 patches/frame, STEPS=18", "global_batch": global_batch,
                          "clips_per_rank": local_clips, "parallelism": "dp%d: one clip at a time per rank, NCCL all-reduce of %.2f MB fp32 gradients per step in %d buckets"
                          % (world, red.bytes_per_step / 1e6, len(red.buckets)), "l2_policy": "inputs larger than L2 (15-frame fp32 feature pyramid 147 MB + activations)"},
               "e2e": {"value": clips_per_s, "unit": "clips/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                       "note": "the timed step IS end to end: clips come from pinned host memory every step and the loss is read back"}}
        print(json.dumps(out))
    multigpu.finalize()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", default="infer", choices=["infer", "train"], help="train = BASELINE configs[3] (training step, NCCL grad all-reduce)")
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="default", choices=["default", "fast"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-reference-cuda", action="store_true", help="skip the reference-CUDA-pipeline leg")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches only")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32 / float64, rank 0; --impl ours inference only)")
    args = ap.parse_args()
    if args.dump_outputs and (args.mode == "train" or args.impl == "reference"):
        ap.error("--dump-outputs writes the outputs of the timed inference step of --impl ours; "
                 "it is not available with --mode train or --impl reference")
    if args.mode == "train":
        args.steps = 3 if args.steps is None else args.steps
        args.warmup = 1 if args.warmup is None else args.warmup
        return run_train(args)
    if args.steps is None:
        args.steps = 200 if args.impl == "ours" else 4
    if args.warmup is None:
        args.warmup = 10 if args.impl == "ours" else 1
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
