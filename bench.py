#!/usr/bin/env python
"""bench.py -- the headline measurement (BASELINE.json metric) of the B200-native LightCTR hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload fm_c2|ffm_c3] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path (gather -> interaction -> loss -> scatter-add -> updater) over one batch of
synthetic Criteo-shaped input.  N=1 workload = BASELINE.json configs[1]: FM k=16, 1M features, 39 fields,
~77 nnz/row, batch 4096, Adagrad.  Prints ONE JSON line (rank 0).

--dump-outputs DIR writes what the last timed step computed as DIR/<name>.npy (float32; see dump_outputs), so that two
builds run with the same arguments -- hence the same seeded inputs -- can be compared output for output.
The benchmark reads the library build() compiled and writes nothing into the tree.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (model, k, F, batch, optimizer)
    "fm_c2": dict(model="fm", k=16, F=1_000_000, batch=4096, opt="adagrad",
                  desc="FM k=16, 1M synthetic Criteo-shape features (39 fields, ~77 nnz/row), batch 4096, Adagrad"),
    "ffm_c3": dict(model="ffm", k=4, F=1_000_000, batch=8192, opt="ftrl",
                   desc="FFM k=4, 39 fields, 1M features, batch 8192, FTRL"),
    "nfm_c4": dict(model="nfm", k=16, F=1_000_000, batch=16384, opt="adagrad", hidden=[256, 128, 64], nb=4,
                   desc="NFM k=16 + MLP [256,128,64], 1M features, batch 16384, Adagrad"),
    "ffm_c5": dict(model="ffm", k=8, F=10_000_000, batch=65536, opt="adagrad", nb=2,
                   desc="FFM k=8, 39 fields, 10M features, batch 65536 per GPU, Adagrad"),
}
N_FIELDS = 39


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index=0, period_ms=100):
        super().__init__(daemon=True)
        self.q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                  "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                  "clocks_event_reasons.sw_power_cap")
        self.gpu, self.period, self.samples, self.proc = gpu_index, period_ms, [], None
        self.stop_flag = False

    def run(self):
        # NVML (same counters as nvidia-smi, ~50 us per query) gives hundreds of samples inside a 20 ms timed region;
        # the nvidia-smi loop of the recipe is the fallback (its process start alone outlasts a short region)
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            bits = {"hw_slowdown": pynvml.nvmlClocksThrottleReasonHwSlowdown,
                    "hw_thermal_slowdown": pynvml.nvmlClocksThrottleReasonHwThermalSlowdown,
                    "sw_thermal_slowdown": pynvml.nvmlClocksThrottleReasonSwThermalSlowdown,
                    "sw_power_cap": pynvml.nvmlClocksThrottleReasonSwPowerCap}
            while not self.stop_flag:
                sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.samples.append("%d,%d,%g,0,%s" % (self.gpu, sm, mx, ",".join(
                    "Active" if r & bits[k] else "Not Active"
                    for k in ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"))))
                time.sleep(0.002)
            return
        except Exception:
            pass
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.q,
                                          "--format=csv,noheader,nounits", "-lms", str(self.period)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.samples.append(line.strip())
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], 0, set()
        for s in self.samples:
            p = [x.strip() for x in s.split(",")]
            if len(p) < 8:
                continue
            try:
                sm.append(float(p[1]))
                mx = max(mx, float(p[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_tensor_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        if "bf16_tflops" in d:
            return d["bf16_tflops"], "measured burst cuBLAS bf16 (MEASURED_PEAKS.json)"
    return 1600.0, "fallback (B200_PROFILING.md)"


def make_batches(wl, n_batches, seed_offset=0):
    from lightctr_b200.data import BASE_SEED, CriteoSynth
    gen = CriteoSynth(wl["F"], seed=BASE_SEED + seed_offset, alpha=float(os.environ.get("LCTR_BENCH_ALPHA", "1.1")))
    return [gen.batch(wl["batch"]) for _ in range(n_batches)]


# ------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's own Train() on the host cores
# ------------------------------------------------------------------------------------------------
def run_reference(wl, steps, warmup, budget_s=20.0):
    if wl["model"] == "nfm":
        return run_port_nfm(wl, budget_s)
    return _run_reference(wl, steps, warmup, budget_s)


def run_port_nfm(wl, budget_s):
    """The reference's NFM takes ONE hidden layer (train_nfm_algo.h:21); the [256,128,64] chain of config C4 is a
    Fully_Conn_Layer chain only the oracle port can instantiate, so this arm is kind="port", single-threaded."""
    from oracle import api
    rp, fid, fld, lab = make_batches(wl, 1)[0]
    sub = min(wl["batch"], 1024)  # bounded sample: the first `sub` rows of the batch as one minibatch
    nz = rp[sub]
    ds = api.Dataset(rp[:sub + 1], fid[:nz], fld[:nz].astype(np.uint32), np.ones(nz, np.float32), lab[:sub], wl["F"], 0)
    o = api.NFMOracle(ds, wl["k"], wl["hidden"], seed=1, batch_size=sub, minibatch=sub)
    t0 = time.time()
    n = 0
    while time.time() - t0 < budget_s and n < 50:
        o.epoch()
        n += 1
    secs = time.time() - t0
    return dict(value=sub * n / secs, cores=1, steps=n, ms_per_step=1e3 * secs / n, rows=sub, kind="port",
                sample="%d minibatch steps of %d rows (first rows of one synthetic batch), oracle C port, 1 thread" % (n, sub))


def _run_reference(wl, steps, warmup, budget_s=20.0):
    """Times Train_FM_Algo / Train_FFM_Algo::Train() of the UNMODIFIED reference (oracle/_ref/libref.so) on one
    synthetic batch written in its libffm text format; one epoch over the B-row file == one step (SURVEY 8 C2)."""
    from lightctr_b200.data import write_libffm
    from oracle import api
    if not api.ref_available():
        return None
    rp, fid, fld, lab = make_batches(wl, 1)[0]
    path = "/tmp/lctr_bench_%s_%d.txt" % (wl["model"], os.getpid())
    write_libffm(path, rp, fid, fld, lab)
    cores = int(api.ref().ref_hw_threads())
    if wl["model"] == "fm":
        t = api.RefTrainer("fm", path, wl["k"], seed=1, proc_cnt=0)
    else:
        t = api.RefTrainer("ffm", path, wl["k"], seed=1, proc_cnt=0, field_cnt=N_FIELDS)
    rows = t.rows
    t0 = time.time()
    t.time_train(max(1, warmup))
    per = (time.time() - t0) / max(1, warmup)
    steps = max(1, min(steps, int(budget_s / max(per, 1e-6))))
    secs = t.time_train(steps)
    t.close()
    os.unlink(path)
    return dict(value=rows * steps / secs, cores=cores, steps=steps, ms_per_step=1e3 * secs / steps, rows=rows,
                sample="%d epochs of Train() over one %d-row synthetic batch (%d features), all %d host threads"
                       % (steps, rows, wl["F"], cores))


def ncu_traffic(wname, kernel):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of the CURRENT kernels, from the ncu
    --set full capture summarised by scripts/ncu_summary.py --json into profiles/ncu_traffic.json (the bench itself
    never runs under a profiler).  None where no capture exists."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(p):
        return None, None
    d = json.load(open(p)).get(wname, {})
    import re
    pat = {"fm_fused": r"fm_fused_kernel<\d+, \d, 1,", "fm_forward": r"fm_fused_kernel<\d+, \d, 0,|fm_forward", "apply_compact": r"apply_compact",
           "ffm_fused": r"ffm_warp_kernel|ffm_fused_kernel|ffm_tma_kernel", "apply": r"apply_kernel", "fm_backward_red": r"fm_backward_kernel"}.get(kernel, re.escape(kernel))
    for name, rec in d.get("kernels", {}).items():
        if re.search(pat, name):
            return rec.get("dram_bytes"), "profiles/ncu_traffic.json <- %s (%s)" % (d.get("source", "?"), name.strip())
    return None, None


def check_against_oracle(ctx, wl, batch, Fc):
    """--check: step 0 of the benched batch against the CPU oracle from the same (downloaded) parameters."""
    from oracle import api
    rp, fid, fld, lab = batch
    W0, V0 = ctx.download_params()
    F, k = wl["F"], wl["k"]
    ds = api.Dataset(rp, fid, fld.astype(np.uint32), np.ones(len(fid), np.float32), lab, F, Fc)
    if wl["model"] == "fm":
        o = api.FMOracle(ds, k, W0, V0)
    elif wl["model"] == "ffm":
        o = api.FFMOracle(ds, k, W0, V0, optimizer=wl["opt"])
    else:
        return {"supported": False, "why": "NFM chain check lives in tests/test_shapes_gpu.py"}
    lg, _ = ctx.train_step(0)
    lo, _ = o.epoch()
    Wg, Vg = ctx.download_params()
    rel = abs(lg - lo) / max(abs(lo), 1e-30)
    out = {"supported": True, "loss_gpu": lg, "loss_oracle": lo, "loss_rel": rel, "max_dW": float(np.max(np.abs(Wg - o.W))),
           "max_dV": float(np.max(np.abs(Vg - o.V))), "ok": bool(rel < 1e-5)}
    ctx.upload_params(W0, V0)  # the timed run starts from the same parameters (updater state keeps one step: harmless)
    return out


DUMP_MAX_BYTES = 64 << 20
DUMP_RANDOM_ROWS = 65536


def dump_outputs(ctx, wl, batch, slot, out_dir):
    """Write what the last timed step handed its caller: the batch's pCTR (`pred`), and the parameter rows W[rows] (`W_rows`)
    and V[rows] (`V_rows`, one row of the factor table per id) after the update.  `rows` is the sorted union of the ids the
    step read and updated and a fixed seeded sample of all ids (mostly ids the step must leave unchanged), trimmed by the
    same seeded draw to keep the files under DUMP_MAX_BYTES; NFM adds its dense layers (`mlp<l>_weight`, `mlp<l>_bias`)."""
    W, V = ctx.download_params()
    F, rowlen = wl["F"], ctx.rowlen
    rng = np.random.default_rng(0)
    rows = np.union1d(batch[1].astype(np.int64), rng.choice(F, min(F, DUMP_RANDOM_ROWS), replace=False))
    cap = (DUMP_MAX_BYTES // 2) // (4 * (rowlen + 1))
    if len(rows) > cap:
        rows = np.sort(rng.choice(rows, cap, replace=False))
    out = {"pred": ctx.download_pred(slot), "W_rows": W[rows], "V_rows": V.reshape(F, rowlen)[rows]}
    if wl["model"] == "nfm":
        dims = [wl["k"]] + list(wl["hidden"]) + [1]
        for li in range(len(dims) - 1):
            out["mlp%d_weight" % li], out["mlp%d_bias" % li] = ctx.mlp_download(li, dims[li], dims[li + 1])
    assert sum(a.nbytes for a in out.values()) <= DUMP_MAX_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, np.float32))


def measure(wname, wl, args, rank, world, local_rank, dist, steps, warmup, do_e2e=True, split_global=0, dump_dir=None):
    """One workload on this process group: K device-timed steps on resident batches (+ the end-to-end arm)."""
    import torch
    from lightctr_b200 import capi
    model = {"fm": capi.MODEL_FM, "ffm": capi.MODEL_FFM, "nfm": capi.MODEL_NFM}[wl["model"]]
    opt = {"adagrad": capi.OPT_ADAGRAD, "ftrl": capi.OPT_FTRL, "adam": capi.OPT_ADAM}[wl["opt"]]
    F, k = wl["F"], wl["k"]
    B = wl["batch"] if not split_global else split_global // world  # rows per GPU per step
    Fc = N_FIELDS if wl["model"] == "ffm" else 0
    # FM on one GPU: the order-free fused step (csrc/fm_fused.cu).  LCTR_BENCH_BACKWARD=grouped selects the
    # feature-grouped modes of csc.cu / ffm_grouped.cu (their grouping kernels: at upload for FM, inside the step for FFM).
    det = 2 if (world == 1 and wl["model"] in ("fm", "ffm") and os.environ.get("LCTR_BENCH_BACKWARD", "red") == "grouped") else 0
    if det == 2 and wl["model"] == "ffm":
        os.environ["LCTR_CSC_IN_STEP"] = "1"
    mlp_bf16 = wl["model"] == "nfm" and os.environ.get("LCTR_BENCH_MLP", "bf16") == "bf16"
    ctx = capi.Context(model, F, k, Fc, optimizer=opt, device=local_rank, deterministic=det, rank=rank, world=world,
                       minibatch_size=(world * B if world > 1 else 0), max_nnz=B * 100, hidden=wl.get("hidden", ()),
                       mlp_precision=capi.MLP_BF16 if mlp_bf16 else capi.MLP_FP32)
    if wl["model"] == "nfm":  # FC chain initialised like fullyconnLayer.h:48-54 (U(-0.5,0.5), bias 0), masks all-ones
        rng0 = np.random.default_rng(99)
        dims = [k] + list(wl["hidden"]) + [1]
        for li in range(len(dims) - 1):
            ctx.mlp_upload(li, (rng0.random((dims[li + 1], dims[li]), dtype=np.float32) - 0.5), np.zeros(dims[li + 1], np.float32))
    ctx.fill_params(1234, float(1.0 / np.sqrt(k)))  # random-init weights (W = 0, V ~ N(0,1)/sqrt(k)), on the device
    if world > 1:
        from lightctr_b200 import dist as ldist
        ldist.connect(ctx)
        if wl["model"] == "nfm":  # replicated dense layers: dW / db summed with NCCL on the context's stream every step
            ldist.attach_dense_allreduce(ctx)
    NB = wl.get("nb", 8)
    wl_b = dict(wl, batch=B)
    batches = make_batches(wl_b, NB, seed_offset=rank)
    pinned = []
    if do_e2e:  # pinned host copies (the end-to-end arm copies from these every step)
        for (rp, fid, fld, lab) in batches:
            pinned.append((torch.from_numpy(rp).pin_memory(), torch.from_numpy(fid.astype(np.int32)).pin_memory(),
                           torch.from_numpy(fld.astype(np.int16)).pin_memory(), torch.from_numpy(lab).pin_memory()))
    for i, (rp, fid, fld, lab) in enumerate(batches):
        ctx.upload_batch(i, rp, fid, fld if Fc else None, None, lab)
    nnz_mean = float(np.mean([len(b[1]) for b in batches]))
    check = None
    if args.check and world == 1:
        check = check_against_oracle(ctx, wl_b, batches[0], Fc)
    stream = torch.cuda.ExternalStream(ctx.stream())
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    do_flush = os.environ.get("LCTR_BENCH_NOFLUSH", "0") != "1"

    def one_step(i, timed_events=None):
        with torch.cuda.stream(stream):
            if do_flush:
                flush.zero_()
            if world > 1 and do_flush:
                # the 256 MB flush saturates THIS GPU's memory system for ~80 us; a peer that is already inside its step
                # would have its NVLink stores into this GPU queue behind it (measured: 3 MB pull / push kernels stretched
                # from ~10 to ~45 us).  Ranks therefore leave the flush together; the timed region starts after it.
                stream.synchronize()
                dist.barrier()
            if timed_events is not None:
                timed_events[0].record(stream)
        ctx.train_step(i % NB, want_stats=False)
        if timed_events is not None:
            with torch.cuda.stream(stream):
                timed_events[1].record(stream)

    for i in range(max(warmup, 3)):
        one_step(i)
    ctx.sync()
    # The timed region: EXACTLY `steps` steps, one CUDA-event pair per step, no per-kernel instrumentation -- an event recorded
    # between two kernels would defeat the programmatic dependent launch of the updater behind the gradient kernel, i.e. time
    # something a user never runs.  The per-kernel buckets (kernels_ms, roofline.kernel_ms) come from a second pass of the
    # same `steps` steps with the library's per-launch events switched on.
    launches0 = ctx.launch_count()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    sampler = ClockSampler(local_rank)
    sampler.start()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t_wall0 = time.time()
    for i in range(steps):
        one_step(i, evs[i])
    ctx.sync()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t_wall = time.time() - t_wall0
    launches = ctx.launch_count() - launches0
    if dump_dir:
        dump_outputs(ctx, wl_b, batches[(steps - 1) % NB], (steps - 1) % NB, dump_dir)
    ctx.profile(True)
    ctx.profile_read(reset=True)
    for i in range(steps):
        one_step(i)
    ctx.sync()
    prof = ctx.profile_read(reset=True)
    step_ms = [a.elapsed_time(b) for a, b in evs]
    ms_per_step = float(np.mean(step_ms))
    if world > 1:  # device time, max over ranks
        t = torch.tensor([ms_per_step], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_per_step = float(t[0])
    value = world * B / (ms_per_step * 1e-3)

    # ---- the embedding gather alone (BASELINE metric "embed-gather HBM GB/s vs peak"): the forward kernel of the model
    # on the same resident batches, L2 flushed before every launch, timed with the per-kernel CUDA events -------------
    gather = None
    if wl["model"] == "fm" and world == 1:
        for i in range(3 + min(steps, 50)):
            with torch.cuda.stream(stream):
                if do_flush:
                    flush.zero_()
            if i == 3:
                ctx.sync()
                ctx.profile_read(reset=True)
            ctx.predict_resident(i % NB)
        pg = ctx.profile_read(reset=True)
        if "fm_forward" in pg:
            gms, gcnt = pg["fm_forward"]
            gather = {"ms": gms / gcnt, "launches": gcnt}
    ctx.profile(False)

    # ---- end-to-end arm: host buffers in, loss out, every step (C-ABI lctr_train_batch_async / lctr_wait) -------------
    e2e = None
    clocks = None
    if do_e2e:
        h2d = 8 * (B + 1) + 4 * nnz_mean + 4 * B + (2 * nnz_mean if Fc else 0)
        host = [_host_arrays(p, Fc) for p in pinned]
        for i in range(NB + 3):  # warm-up through the same pipelined entry points (allocates both pipeline slots)
            ctx.wait(ctx.train_batch_async(*host[i % NB]))
        ctx.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.time()
        from collections import deque
        from lightctr_b200 import capi as _capi
        pending = deque()  # the API's pipeline depth: step t computes, t+1 has its slot map built, t+2 is being copied
        e2e_loss = 0.0
        t_issue = 0.0  # host time inside the issuing call (numpy -> pointers, copies / graph launches / events enqueued)
        for i in range(steps):
            ti = time.perf_counter()
            pending.append(ctx.train_batch_async(*host[i % NB]))
            t_issue += time.perf_counter() - ti
            if len(pending) >= _capi.PIPE_DEPTH:
                e2e_loss += ctx.wait(pending.popleft())[0]
        while pending:
            e2e_loss += ctx.wait(pending.popleft())[0]
        ctx.sync()
        e2e_s = time.time() - t0
        if world > 1:
            t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_s = float(t[0])
        e2e = {"value": world * B * steps / e2e_s, "unit": "samples/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 16,
               "us_per_step": 1e6 * e2e_s / steps, "host_issue_us_per_step": 1e6 * t_issue / steps, "pipeline_depth": _capi.PIPE_DEPTH,
               "l2": "not flushed: every step's batch arrives from pinned host memory, parameters stay L2-resident between "
                     "steps as in a real training loop (the device-timed `value` flushes L2 before every step)"}
    clocks = sampler.finish()
    if world > 1:
        dist.barrier()
    ctx.close()
    del flush
    torch.cuda.empty_cache()
    return dict(value=value, ms_per_step=ms_per_step, prof=prof, launches=launches, nnz_mean=nnz_mean, B=B, Fc=Fc, det=det,
                mlp_bf16=mlp_bf16, e2e=e2e, clocks=clocks, t_wall=t_wall, gather=gather, check=check)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-c5", action="store_true", help="skip the FFM C5 split-batch scaling measurement")
    ap.add_argument("--check", action="store_true", help="compare step 0 of the benched batch with the CPU oracle")
    ap.add_argument("--batch", type=int, default=0, help="override the workload's rows per GPU per step (sweeps; "
                    "the headline configs are the defaults)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (one GPU)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs needs --impl ours on one GPU")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    wname = args.workload or "fm_c2"
    wl = dict(WORKLOADS[wname])
    if args.batch:
        wl["desc"] = wl["desc"].replace("batch %d" % wl["batch"], "batch %d (--batch override)" % args.batch)
        wl["batch"] = args.batch
        wl["nb"] = min(wl.get("nb", 8), max(2, (1 << 21) // args.batch))
    metric = "samples/sec (device-timed) %s train step on Criteo-shape" % wl["model"].upper()

    if args.impl == "reference":
        if rank != 0:
            return 0
        r = run_reference(wl, args.steps, max(args.warmup, 1))
        if r is None:
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libref.so not built"}))
            return 0
        line = {"impl": "reference", "metric": metric, "value": r["value"], "unit": "samples/s", "n_gpus": args.gpus,
                "steps": r["steps"], "warmup": max(args.warmup, 1), "ms_per_step": r["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": wl["desc"]},
                "cpu_baseline": {"value": r["value"], "unit": "samples/s", "cores": r["cores"],
                                 "kind": r.get("kind", "reference"), "sample": r["sample"]},
                "e2e": {"value": r["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    import torch
    from lightctr_b200 import capi
    capi.load_library()  # the library build() compiled; raises when it is missing
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product has no CPU path)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    m = measure(wname, wl, args, rank, world, local_rank, dist, args.steps, args.warmup, dump_dir=args.dump_outputs)
    value, ms_per_step, prof, B, Fc, det, nnz_mean = m["value"], m["ms_per_step"], m["prof"], m["B"], m["Fc"], m["det"], m["nnz_mean"]
    mlp_bf16 = m["mlp_bf16"]
    k = wl["k"]

    # ---- roofline of the dominant kernel (algorithmic bytes per SURVEY.md 8d / DESIGN.md) -----------------
    peak, peak_src = measured_peaks()
    compute = {kk: vv for kk, vv in prof.items() if not kk.startswith("dist_")}
    dom = max(compute.items(), key=lambda kv: kv[1][0]) if compute else (None, (0.0, 0))
    n = nnz_mean / B
    gather_bps = n * (4 * k + 12) + 8          # SURVEY 8d: V row + W + fid + slot per entry, row_ptr per sample
    scatter_bps = n * (4 * k + 4)              # one gradient row [gV | gW] per entry, RED into the compact buffer
    if wl["model"] in ("fm", "nfm"):
        bytes_per_sample = {"fm_forward": gather_bps, "fm_backward_red": gather_bps, "fm_fused": gather_bps + scatter_bps,
                            "fm_backward_csc": gather_bps, "apply": None, "apply_compact": None, "mlp": None}
    else:
        # fused: one row gather per entry (+ the sample's Fc x Fc x k tile written once in grouped mode);
        # grouped backward: one contiguous tile row per entry
        bytes_per_sample = {"ffm_fused": n * (Fc * k * 4 + 12) + (Fc * Fc * k * 4 if det == 2 else 0),
                            "fm_backward_csc": n * (Fc * k * 4 + 10)}
    roof = None
    cnt = 0
    if dom[0] is not None:
        ms, cnt = dom[1]
        bps = bytes_per_sample.get(dom[0])
        if bps is not None and cnt:
            achieved = bps * B / (ms / cnt * 1e-3) / 1e9
            roof = {"bound": "hbm", "kernel": dom[0], "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": bps * B, "kernel_ms": ms / cnt,
                    "bytes": ("gather n(4k+12)+8 + scatter n(4k+4) per sample" if dom[0] == "fm_fused" else "gather bytes per sample (SURVEY 8d)")}
            if not args.batch and world == 1:
                roof["traffic"], src = ncu_traffic(wname, dom[0])
                if src:
                    roof["traffic_source"] = src
    if dom[0] == "mlp" and cnt:  # dense layers: fwd + dX + dW = 6 flops per weight per sample
        dims = [k] + list(wl["hidden"]) + [1]
        flops = 6.0 * sum(dims[i] * dims[i + 1] for i in range(len(dims) - 1)) * B
        tpeak, tsrc = measured_tensor_peak()
        achieved = flops / (ms / cnt * 1e-3) / 1e12
        umma = os.environ.get("LCTR_MLP_UMMA", "1") != "0"
        roof = {"bound": "tensor", "kernel": ("mlp (nfm_mlp_umma_kernel: tcgen05.mma, TMEM accumulators; + dense Adagrad)" if umma
                                              else "mlp (nfm_mlp_fused_kernel: mma.sync; + dense Adagrad)"), "achieved": achieved, "peak": tpeak,
                "unit": "TFLOP/s", "frac": achieved / tpeak, "traffic": None, "peak_source": tsrc,
                "algorithmic_flops_per_launch": flops, "kernel_ms": ms / cnt}
        if world == 1:
            tr, src = ncu_traffic(wname, "nfm_mlp_umma" if umma else "nfm_mlp_fused")
            if tr is not None:
                roof["traffic"], roof["traffic_source"] = tr, src
    roof_gather = None
    if m["gather"]:
        gms = m["gather"]["ms"]
        ach = gather_bps * B / (gms * 1e-3) / 1e9
        roof_gather = {"bound": "hbm", "kernel": "fm_fused_kernel<MODE 0> (forward gather alone, lctr_predict)", "achieved": ach,
                       "peak": peak, "unit": "GB/s", "frac": ach / peak, "kernel_ms": gms, "launches": m["gather"]["launches"],
                       "algorithmic_bytes_per_launch": gather_bps * B, "peak_source": peak_src}
        tr, src = ncu_traffic(wname, "fm_forward") if not args.batch else (None, None)
        roof_gather["traffic"] = tr
        if src:
            roof_gather["traffic_source"] = src
    kernels = {name: {"ms": v[0] / max(v[1], 1), "launches": v[1]} for name, v in prof.items()}
    bw_desc = ("RED scatter + sparse apply" if not (wl["model"] == "fm" and world == 1) else
               "order-free fused step: one gather, RED scatter into the batch-compact buffer (hot-slot replicas), compact updater")
    if det == 2:
        bw_desc = ("feature-grouped on device + fused updater (csc.cu)" if wl["model"] == "fm" else
                   "feature-grouped, atomic-free, fused updater (ffm_grouped.cu); grouping kernels inside the timed step")
    line = {"metric": metric, "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16 dense layers (fp32 accumulate, fp32 masters) + f32 embeddings" if mlp_bf16 else "f32",
            "data": "synthetic",
            "config": {"workload": wl["desc"], "l2": "flushed between timed steps (256 MB write)" + ("; ranks barrier after the flush, before the timed region" if world > 1 else ""),
                       "kernel_buckets": "kernels_ms / roofline.kernel_ms: a second pass of the same steps with per-launch CUDA events (the timed region carries one event pair per step only)",
                       "batch_per_gpu": B,
                       "global_batch": world * B, "nnz_per_row": n,
                       **({"mlp": ("bf16 tcgen05.mma with TMEM accumulators, fused fwd+bwd per 128-sample CTA" if os.environ.get("LCTR_MLP_UMMA", "1") != "0"
                                   else "bf16 mma.sync, fused fwd+bwd per 128-sample tile") if mlp_bf16 else "fp32 reference-order"}
                          if wl["model"] == "nfm" else {}),
                       "backward": bw_desc,
                       "parallelism": "1 GPU" if world == 1 else
                       ("dp%d rows + owner-sharded tables (fid mod %d), unique-id pull/push over NVLink peer memory" % (world, world))
                       + ("; dense layers replicated, gradients NCCL all-reduced" if wl["model"] == "nfm" else "")},
            "clocks": m["clocks"], "gpu_launches": int(m["launches"]), "kernels_ms": kernels,
            "e2e": m["e2e"], "roofline": roof, "roofline_gather": roof_gather, "wall_s_timed_region": m["t_wall"]}
    if m["check"] is not None:
        line["check"] = m["check"]
    # ---- north-star scaling config: FFM C5 (k=8, 10 M features) with the GLOBAL batch 65 536 split across the ranks
    # (SURVEY 8d; strong scaling), measured by every default run so that the driver's N = 1, 2, 4, 8 records carry it ----
    if not args.no_c5 and not args.workload and not args.batch:
        wl5 = dict(WORKLOADS["ffm_c5"])
        c5 = measure("ffm_c5", wl5, args, rank, world, local_rank, dist, steps=max(5, min(args.steps, 10)), warmup=3, do_e2e=False,
                     split_global=wl5["batch"])
        line["c5"] = {"workload": "FFM k=8, 39 fields, 10M features, GLOBAL batch 65536 split across %d GPU(s), Adagrad" % world,
                      "n": world, "split": "strong (global batch fixed at 65536)", "rows_per_gpu": c5["B"], "value": c5["value"],
                      "unit": "samples/s", "ms_per_step": c5["ms_per_step"],
                      "kernels_ms": {nm: {"ms": v[0] / max(v[1], 1), "launches": v[1]} for nm, v in c5["prof"].items()}}
    if not args.no_cpu_baseline and rank == 0 and world == 1:
        r = run_reference(wl, 50, 1, budget_s=15.0)
        if r is not None:
            line["cpu_baseline"] = {"value": r["value"], "unit": "samples/s", "cores": r["cores"],
                                    "kind": r.get("kind", "reference"), "sample": r["sample"]}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def _host_arrays(p, Fc):
    t_rp, t_fid, t_fld, t_lab = p
    return (t_rp.numpy(), t_fid.numpy().view(np.uint32), t_fld.numpy().view(np.uint16) if Fc else None, None,
            t_lab.numpy())


if __name__ == "__main__":
    sys.exit(main())
