#!/usr/bin/env python
"""bench.py — headline metric of BASELINE.json: utterances/s (2 s @ 16 kHz) embedding extraction; PLDA scores/s.

    python bench.py [--gpus N --steps K --warmup W] [--impl reference] [--workload NAME] [--no-configs] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...

A "step" is one pass of the hot path (fbank -> CMN -> model forward) over one batch of synthetic utterances per GPU.
Default workload = BASELINE.json configs[1]: ECAPA-TDNN-1024, bf16 tensor-core path, batch 256 of 2.02 s utterances
(32320 samples -> 200 frames, the "256 x 200-frame" case).  `value` is measured with the waveforms already resident in
HBM; `e2e` is the same metric through the public host-buffer API (B200SpeakerModel.extract_stream on pinned host int16
PCM: H2D + kernels + D2H inside the timed region).  Multi-GPU: one rank per GPU, utterances sharded with no data-path
collective (weak scaling), ONE NCCL all-gather of the embeddings at the end of the job, inside the timed region.

The same JSON line carries a `configs` block with one short timed leg per remaining BASELINE.json config (the driver
only runs the default command): ECAPA-TDNN-512 in tf32x3 (the <= 1e-4 tensor-core path) and bf16, ResNet34 fp16 at 64
utterances per GPU (= batch 512 sharded when 8 ranks run), CAM++ bf16 on the seed-2 mix of 1-10 s utterances, and the full
10^6 x 10^5 TwoCov-PLDA scoring job tiled over enroll rows (sharded over ranks).  Every model leg reports
`parity_rel_l2`: embeddings of utterances OF THE TIMED BATCH against the CPU oracle on identical fbank inputs.

`--impl reference` times the oracle port of the reference's CPU PyTorch path (torch fp32) on the same config, rank 0
only, using all host cores as a pool of worker processes (the reference's own parallelism is process-level sharding,
tools/extract_embedding.sh:39-63).
"""
import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (model, precision, batch per GPU, samples per utterance, GFLOP/utt of conv+linear layers at that T)
    "ecapa1024_bf16_b256": ("ECAPA_TDNN_c1024", "bf16", 256, 32320, 5.141),
    "ecapa512_bf16_b256": ("ECAPA_TDNN_c512", "bf16", 256, 32320, 1.917),
    "ecapa1024_bf16_b128": ("ECAPA_TDNN_c1024", "bf16", 128, 32320, 5.141),
    "ecapa1024_bf16_b64": ("ECAPA_TDNN_c1024", "bf16", 64, 32320, 5.141),
    "ecapa1024_bf16_b512": ("ECAPA_TDNN_c1024", "bf16", 512, 32320, 5.141),
    "ecapa512_fp32_b16": ("ECAPA_TDNN_c512", "fp32", 16, 32000, 1.898),
    "resnet34_fp16_b64": ("ResNet34", "fp16", 64, 32320, 9.056),
    "campplus_bf16_b64": ("CAMPPlus", "bf16", 64, 32320, 2.252),
    "ecapa512_tf32x3_b256": ("ECAPA_TDNN_c512", "tf32x3", 256, 32320, 1.917),
    "ecapa512_fp32_b256": ("ECAPA_TDNN_c512", "fp32", 256, 32320, 1.917),
    "ecapa1024_tf32x3_b256": ("ECAPA_TDNN_c1024", "tf32x3", 256, 32320, 5.141),
}
DEFAULT_WORKLOAD = "ecapa1024_bf16_b256"
# Not BASELINE configs: reported beside them in "extras" (N = 1 only).  Batch 1 is how the reference extracts every test set
# (examples/voxceleb/v2/local/extract_vox.sh:31: one whole utterance per forward); the last two are SURVEY section 8(f) rank-4
# families on the existing operators.  (model, precision, batch, samples per utterance)
EXTRA_WORKLOADS = {
    "ecapa512_tf32x3_b1": ("ECAPA_TDNN_c512", "tf32x3", 1, 32320),
    "ecapa512_bf16_b1": ("ECAPA_TDNN_c512", "bf16", 1, 32320),
    "res2net34_fp16_b64": ("Res2Net34_Base", "fp16", 64, 32320),
    "eres2net34_fp16_b64": ("ERes2Net34_Base", "fp16", 64, 32320),
}
METRIC = "utterances/s (2s@16kHz) embedding extraction"
DTYPE_NAME = {"fp32": "f32", "tf32": "tf32", "tf32x3": "tf32x3", "bf16": "bf16", "fp16": "f16"}
# bars for `parity_rel_l2` (max over the checked utterances of |e - e_ref|_2 / |e_ref|_2), as in tests/test_gpu_parity.py
PARITY_BAR = {"fp32": 1e-4, "tf32x3": 1e-4, "tf32": 1e-2, "bf16": 1e-2, "fp16": 1e-2}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md).  NVML polled every 5 ms from a
    thread (the timed region is only tens of ms long); falls back to `nvidia-smi -lms 100` if NVML is unavailable.
    start() is called BEFORE the pre-timing barrier (NVML init costs milliseconds: inside the window it skewed rank 0
    against the other ranks in round 1); mark() / stop() bracket the samples that are kept."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []
        self.nvml, self.samples, self.reasons, self.maxclk, self._stop = None, [], set(), None, False
        self._on = False

    def _poll(self):
        n = self.nvml
        while not self._stop:
            if self._on:
                try:
                    self.samples.append(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM))
                    try:
                        r = n.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                    except Exception:
                        r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    for bit, name in self.BITS.items():
                        if r & bit:
                            self.reasons.add(name)
                except Exception:
                    pass
            time.sleep(0.005)

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            try:
                bus = torch.cuda.get_device_properties(self.index).pci_bus_id
                self.h = pynvml.nvmlDeviceGetHandleByPciBusId(f"00000000:{bus:02x}:00.0".encode()) if isinstance(bus, int) \
                    else pynvml.nvmlDeviceGetHandleByIndex(self.index)
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.maxclk = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.nvml = pynvml
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def mark(self, on=True):
        """mark(True) opens a new sampling window (previous samples are dropped); mark(False) closes it."""
        if on:
            self.samples, self.reasons = [], set()
        self._on = on

    def read(self):
        """Statistics of the last window (NVML mode)."""
        smp = list(self.samples)
        return {"sm_mhz": float(np.median(smp)) if smp else None, "sm_min_mhz": float(min(smp)) if smp else None,
                "sm_max_mhz": float(self.maxclk) if self.maxclk else None, "reasons": sorted(self.reasons),
                "samples": len(smp), "source": "nvml, 5 ms polling during the timed region"}

    def stop(self):
        if self.nvml is not None:
            self._stop = True
            self.t.join(timeout=1)
            return self.read()
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvidia-smi -lms 100"}


# ------------------------------------------------------------------------------------------------ CPU arm (oracle port)
def _cpu_path(model_name, nsamples, batch, seed=0):
    """Oracle port of the reference CPU path: numpy fbank+CMN, torch-CPU fp32 forward."""
    from oracle import fbank_np, models_torch
    from wespeaker_b200 import synthetic as syn
    sd = {k: torch.from_numpy(np.asarray(v)) for k, v in syn.make_state_dict(model_name, 0).items()}
    wavs = syn.make_wavs(batch, nsamples, seed=seed)

    def one():
        feats = np.stack([fbank_np.cmn(fbank_np.fbank(w)) for w in wavs])
        return models_torch.forward(model_name, sd, torch.from_numpy(feats))
    return one


def _cpu_worker(model_name, nsamples, batch, threads, seed, cpus, conn):
    if cpus:
        try:
            os.sched_setaffinity(0, cpus)   # a disjoint core set per worker: no migration, no oversubscription
        except Exception:
            pass
    torch.set_num_threads(threads)
    one = _cpu_path(model_name, nsamples, batch, seed)
    one(); one()
    conn.send("ready")
    while True:
        n = conn.recv()
        if n is None:
            break
        for _ in range(n):
            one()
        conn.send("done")


class CpuPool:
    """All host cores as P worker processes x `threads` torch threads each (torch's intra-op scaling of these small convs
    collapses beyond ~8 threads, while independent processes over disjoint utterance lists scale — which is also how
    the reference parallelises extraction, tools/extract_embedding.sh:39-63).  One pool step = every worker runs one
    batch of `batch` utterances through fbank + CMN + forward."""

    def __init__(self, model_name, nsamples, batch=16, threads=8):
        try:
            cores = len(os.sched_getaffinity(0))
        except Exception:
            cores = os.cpu_count() or 1
        self.cores, self.threads, self.batch = cores, min(threads, cores), batch
        self.nproc = max(1, min(16, cores // self.threads))
        try:
            cpu_list = sorted(os.sched_getaffinity(0))
        except Exception:
            cpu_list = []
        ctx = mp.get_context("spawn")
        self.conns, self.procs = [], []
        # BLAS / OpenMP pools of the children are sized by the environment they are spawned with (numpy's matmul in the
        # fbank would otherwise start one thread per host core in EVERY worker)
        keys = ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS", "NUMEXPR_NUM_THREADS")
        saved = {k: os.environ.get(k) for k in keys}
        for k in keys:
            os.environ[k] = str(self.threads)
        try:
            for i in range(self.nproc):
                a, b = ctx.Pipe()
                cpus = set(cpu_list[i * self.threads:(i + 1) * self.threads]) if len(cpu_list) >= self.nproc * self.threads else None
                p = ctx.Process(target=_cpu_worker, args=(model_name, nsamples, batch, self.threads, i, cpus, b), daemon=True)
                p.start()
                self.conns.append(a); self.procs.append(p)
        finally:
            for k, v in saved.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
        for c in self.conns:
            assert c.recv() == "ready"
        self.active = self.nproc

    def run(self, nsteps, active=None):
        conns = self.conns[: (active or self.active)]
        t0 = time.perf_counter()
        for c in conns:
            c.send(nsteps)
        for c in conns:
            c.recv()
        return time.perf_counter() - t0

    def calibrate(self):
        """How many of the workers actually help: `nproc` may exceed what the container is allowed to use (a CPU quota
        makes 16 x 8 threads run no faster than 1 x 8), so time one pool step with P, P/2, ... 1 active workers and keep
        the fastest setting.  The count in use is what `cores` reports."""
        best, k = None, self.nproc
        while k >= 1:
            dt = self.run(1, active=k)
            rate = k * self.batch / dt
            if best is None or rate > best[0]:
                best = (rate, k)
            k //= 2
        self.active = best[1]
        return self.active

    @property
    def utts_per_step(self):
        return self.active * self.batch

    def close(self):
        for c in self.conns:
            try:
                c.send(None)
            except Exception:
                pass
        for p in self.procs:
            p.join(timeout=5)

    def describe(self, nsamples):
        return (f"{self.active} worker processes x {self.threads} torch threads = {self.active * self.threads} threads (fastest of "
                f"{self.nproc}, {self.nproc // 2}, ... 1 workers on this host: {self.cores} logical CPUs visible), each step = "
                f"{self.active} x {self.batch} utterances of {nsamples} samples: numpy fbank+CMN + torch-CPU fp32 forward (oracle "
                f"port of the reference CPU path)")


def run_reference(args, wl):
    model, _, _, nsamples, _ = WORKLOADS[wl]
    if int(os.environ.get("RANK", 0)) != 0:
        return
    pool = CpuPool(model, nsamples)
    pool.calibrate()
    pool.run(max(1, min(args.warmup, 2)))
    dt = pool.run(args.steps)
    v = args.steps * pool.utts_per_step / dt
    sample = f"{args.steps} pool steps; " + pool.describe(nsamples)
    cores = pool.active * pool.threads
    pool.close()
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "utt/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl, "model": model, "utts_per_step": pool.utts_per_step, "samples_per_utt": nsamples},
        "cpu_baseline": {"value": v, "unit": "utt/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "utt/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------------ helpers
def _timed(fn, dev, parallel, world, reps=1):
    """Device time of fn() (CUDA events on torch's current stream, which every engine call joins), bracketed by barrier +
    synchronize, streams aligned by an on-device all-reduce right before the start event; max over ranks; best of reps."""
    import torch.distributed as dist
    best, ret = None, None
    tiny = torch.zeros(1, device=dev)
    for _ in range(reps):
        parallel.barrier(); torch.cuda.synchronize()
        if world > 1:
            dist.all_reduce(tiny)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ret = fn()
        e1.record()
        torch.cuda.synchronize(); parallel.barrier()
        ms = parallel.max_over_ranks(e0.elapsed_time(e1), dev)
        best = ms if best is None else min(best, ms)
    return best, ret


def _parity(model_name, emb_rows, feats_rows):
    """max rel-L2 of GPU embedding rows against the CPU oracle on the identical fbank+CMN inputs."""
    from oracle import models_torch
    from wespeaker_b200 import synthetic as syn
    sd = {k: torch.from_numpy(np.asarray(v)) for k, v in syn.make_state_dict(model_name, 0).items()}
    worst = 0.0
    for e, f in zip(emb_rows, feats_rows):
        ref = models_torch.forward(model_name, sd, f[None].float().cpu())
        ref = (ref[-1] if isinstance(ref, tuple) else ref)[0].double()
        worst = max(worst, float(torch.linalg.norm(e.double().cpu() - ref) / torch.linalg.norm(ref)))
    return worst


def model_leg(name, model_name, prec, B, nsamples, gflop_utt, steps, warmup, dev, rank, world, parallel, peaks, sampler,
              parity_n=4):
    """One fixed-length config: K timed steps of wav -> fbank -> CMN -> forward on a batch of B per GPU."""
    from wespeaker_b200.models import from_synthetic
    from wespeaker_b200 import synthetic as syn
    model = from_synthetic(model_name, 0, precision=prec).to(dev)
    base = syn.make_wavs(B, nsamples, seed=300 + rank)
    wavs = [torch.from_numpy(np.roll(base, i, axis=0)).to(dev) for i in range(2)]
    for i in range(max(3, warmup)):
        model.extract_from_wav(wavs[i % 2])
    launches = model.last_launches()

    def run():
        out = None
        for i in range(steps):
            out = model.extract_from_wav(wavs[i % 2])
        return out
    ms, _ = _timed(run, dev, parallel, world)
    value = world * B * steps / (ms * 1e-3)
    res = {"workload": name, "model": model_name, "precision": prec, "batch_per_gpu": B, "frames": 1 + (nsamples - 400) // 160,
           "value": value, "unit": "utt/s", "ms_per_step": ms / steps, "launches_per_step": int(launches),
           "step_tflops_per_gpu": value / world * gflop_utt / 1e3,
           "step_frac_of_sustained": value / world * gflop_utt / 1e3 / peaks["tf_sustained"]}
    if prec == "tf32x3":
        # the algorithmic FLOPs are executed three times at the tf32 rate (half the bf16 rate the peak was measured at): the
        # same number against peak / 6 is the fraction of what a 3xTF32 GEMM could reach on this machine
        res["step_frac_of_3xtf32_sustained"] = 6.0 * res["step_frac_of_sustained"]
        res["note"] = "3 error-compensated tf32 passes: tensor ceiling = the measured bf16 sustained peak / 6"
    if rank == 0:
        emb, feats = model.extract_from_wav(wavs[0], return_feats=True)   # the timed batch (full B: same kernels / tiles)
        sel = [int(round(j * (B - 1) / max(1, parity_n - 1))) for j in range(parity_n)]
        res["parity_rel_l2"] = _parity(model_name, [emb[j] for j in sel], [feats[j] for j in sel])
        res["parity_bar"] = PARITY_BAR[prec]
        res["parity_utts"] = sel
    del model
    torch.cuda.empty_cache()
    return res


def varlen_leg(steps, warmup, dev, rank, world, parallel, peaks, sampler, n_utts=256, parity_n=4):
    """BASELINE.json configs[3]: CAM++ bf16 on utterances of 1..10 s (durations U{1..10} s, seed 2), bucketed by length."""
    from wespeaker_b200.models import from_synthetic
    from wespeaker_b200 import synthetic as syn
    model_name, prec = "CAMPPlus", "bf16"
    model = from_synthetic(model_name, 0, precision=prec).to(dev)
    rng = np.random.default_rng(2 + 1000 * rank)
    secs = rng.integers(1, 11, n_utts)
    pool = syn.make_wavs(16, 160000, seed=500 + rank)
    wavs = [torch.from_numpy(pool[i % 16, : int(s) * 16000].copy()).to(dev) for i, s in enumerate(secs)]
    frames = [1 + (int(s) * 16000 - 400) // 160 for s in secs]
    gflop = sum(2.252 * f / 200.0 for f in frames)       # conv+linear FLOPs scale with T (2.252 GFLOP at T=200)
    for _ in range(max(2, min(warmup, 3))):
        model.extract_from_wav_list(wavs, max_batch=128, device=dev)
    nrep = max(1, steps // 10)
    ms, emb = _timed(lambda: [model.extract_from_wav_list(wavs, max_batch=128, device=dev) for _ in range(nrep)][-1],
                     dev, parallel, world)
    value = world * n_utts * nrep / (ms * 1e-3)
    res = {"workload": "campplus_bf16_varlen_1to10s", "model": model_name, "precision": prec, "utts_per_gpu": n_utts,
           "durations": "U{1..10} s, seed 2 (+1000*rank), bucketed by exact frame count (<= 128 per launch), buckets overlapped on the engine's streams",
           "value": value, "unit": "utt/s", "audio_s_per_s": world * float(secs.sum()) * nrep / (ms * 1e-3),
           "ms_per_pass": ms / nrep, "passes": nrep,
           "step_tflops_per_gpu": gflop * nrep / (ms * 1e-3) / 1e3,
           "step_frac_of_sustained": gflop * nrep / (ms * 1e-3) / 1e3 / peaks["tf_sustained"]}
    # the same job with CONTINUOUS durations (U[1, 10) s, arbitrary sample counts): exact-length bucketing would need one plan
    # per utterance; the ragged / length-masked path runs it through the frame grid's bounded set of plans
    nsamp = rng.integers(16000, 160000, n_utts)
    cwavs = [torch.from_numpy(pool[i % 16, : int(n)].copy()).to(dev) for i, n in enumerate(nsamp)]
    for _ in range(max(2, min(warmup, 3))):
        model.extract_from_wav_list_ragged(cwavs, max_batch=64, device=dev)
    cms, cemb = _timed(lambda: [model.extract_from_wav_list_ragged(cwavs, max_batch=64, device=dev) for _ in range(nrep)][-1],
                       dev, parallel, world)
    res["masked_continuous"] = {
        "durations": "U[1, 10) s with arbitrary sample counts, concatenated PCM + offsets (ws_engine_extract_wav_ragged_async), "
                     "length-masked buckets on the x1.15 frame grid, <= 64 per launch",
        "value": world * n_utts * nrep / (cms * 1e-3), "unit": "utt/s",
        "audio_s_per_s": world * float(nsamp.sum()) / 16000.0 * nrep / (cms * 1e-3), "ms_per_pass": cms / nrep}
    if rank == 0:
        from wespeaker_b200 import frontend
        csel = [int(np.argmin(nsamp)), int(np.argsort(nsamp)[n_utts // 2]), int(np.argmax(nsamp))]
        cfeats = [frontend.fbank_batch(cwavs[j][None], cmn=True)[0] for j in csel]
        res["masked_continuous"]["parity_rel_l2"] = _parity(model_name, [cemb[j] for j in csel], cfeats)
        res["masked_continuous"]["parity_bar"] = PARITY_BAR[prec]
        order = np.argsort(secs, kind="stable")
        sel = [int(order[int(round(j * (n_utts - 1) / max(1, parity_n - 1)))]) for j in range(parity_n)]
        feats = [frontend.fbank_batch(wavs[j][None], cmn=True)[0] for j in sel]
        res["parity_rel_l2"] = _parity(model_name, [emb[j] for j in sel], feats)
        res["parity_bar"] = PARITY_BAR[prec]
        res["parity_utts"] = [f"{int(secs[j])}s" for j in sel]
    del model
    torch.cuda.empty_cache()
    return res


def fp64_peak(dev, n=4096, iters=5):
    """Measured fp64 matmul rate of this GPU (torch.matmul = cuBLAS DGEMM, best of `iters`): the denominator of the PLDA
    roofline fraction, taken the same way MEASURED_PEAKS.json takes the bf16 peak."""
    a = torch.randn(n, n, dtype=torch.float64, device=dev)
    b = torch.randn(n, n, dtype=torch.float64, device=dev)
    torch.matmul(a, b)
    best = None
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); torch.matmul(a, b); e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        best = ms if best is None else min(best, ms)
    return 2.0 * n ** 3 / (best * 1e-3) / 1e12


def plda_leg(dev, rank, world, parallel, peaks, n_enroll=1_000_000, n_test=100_000, dim=256, tile=32768, cpu_loop=True):
    """BASELINE.json configs[4]: all 10^11 LLR scores of 10^6 enroll x 10^5 test embeddings (D = 256, n = 1), fp64
    arithmetic, fp32 scores.  The score matrix (400 GB) does not fit in HBM: enroll rows are processed in tiles into ONE
    reused 32768 x 100000 fp32 buffer; with several ranks the enroll rows are sharded (no output collective)."""
    from wespeaker_b200 import synthetic as syn
    from wespeaker_b200.plda import TwoCovPLDA
    from oracle import plda_np
    pm = syn.make_plda(dim, seed=3, normalize_length=True)
    p = TwoCovPLDA.from_arrays(**pm, device=dev.index)
    lo, hi = parallel.shard_rows(n_enroll, rank, world)
    g = torch.Generator(device=dev); g.manual_seed(3 + rank)
    e = torch.randn((hi - lo, dim), generator=g, device=dev, dtype=torch.float32)
    g.manual_seed(4)
    t = torch.randn((n_test, dim), generator=g, device=dev, dtype=torch.float32)
    e_t, t_t = p.transform_batch(e), p.transform_batch(t)
    out = torch.empty((min(tile, hi - lo), n_test), dtype=torch.float32, device=dev)
    p.score_matrix(e_t[:tile], t_t, 1, out=out[: min(tile, hi - lo)])
    first = out[:200, :100].double().cpu().numpy()

    def run():
        for r in range(0, hi - lo, tile):
            n = min(tile, hi - lo - r)
            p.score_matrix(e_t[r:r + n], t_t, 1, out=out[:n])
    ms, _ = _timed(run, dev, parallel, world)
    scores = float(n_enroll) * n_test
    res = {"workload": "plda_1Mx100k", "value": scores / (ms * 1e-3), "unit": "scores/s", "dtype": "f64", "enroll": n_enroll,
           "test": n_test, "dim": dim, "enroll_tile": tile, "ms_total": ms, "sharding": f"enroll rows over {world} rank(s)",
           "tflops_f64": scores * 2 * dim / (ms * 1e-3) / 1e12 / world, "out_gbs_per_gpu": scores * 4 / (ms * 1e-3) / 1e9 / world}
    if rank == 0:
        pk = fp64_peak(dev)
        res["roofline"] = {"bound": "fp64 matmul", "achieved": res["tflops_f64"], "peak": pk, "unit": "TFLOP/s",
                           "frac": res["tflops_f64"] / pk, "peak_source": "torch.matmul fp64 4096^3 on this GPU, best of 5",
                           "hbm_write_frac": res["out_gbs_per_gpu"] / peaks["hbm_gbs"]}
        ref = plda_np.llr_matrix(pm, e_t[:200].cpu().numpy(), t_t[:100].cpu().numpy(), 1)
        res["max_abs_err_vs_fp64_oracle"] = float(np.abs(first - ref).max())
        res["parity_bar"] = "1e-5 * max(1, |s|)"
        res["parity_ok"] = bool((np.abs(first - ref) <= 1e-5 * np.maximum(1.0, np.abs(ref))).all())
        if cpu_loop:   # the reference's per-trial Python loop (two_cov_plda.py:248-256), single thread, 20k-trial sample
            et, tt = e_t[:200].cpu().numpy(), t_t[:100].cpu().numpy()
            t0 = time.perf_counter()
            for i in range(200):
                for j in range(100):
                    plda_np.log_likelihood_ratio(pm, et[i], tt[j], 1)
            res["cpu_baseline"] = {"value": 20000 / (time.perf_counter() - t0), "unit": "scores/s", "cores": 1, "kind": "port",
                                   "sample": "20000 trials, per-trial log_likelihood_ratio loop as in eval_sv"}
    del out, e_t, t_t, e, t
    torch.cuda.empty_cache()
    return res


def time_dominant_kernel(model, prec, B, T, iters=10, tc_version=3):
    """Roofline leg: the dominant launch of the step — ECAPA's 1x1 conv 3C->1536 over B*T positions
    (ecapa_tdnn.py:200,218; 47-49% of the model's MACs) — timed live with CUDA events on the launching stream
    through ws_conv.  Algorithmic FLOPs per launch = 2 * B*T * 3C * 1536."""
    import ctypes as C
    from wespeaker_b200 import lib
    if not model.startswith("ECAPA") or prec not in ("fp32", "tf32", "bf16", "fp16"):
        return None
    Cc = 1024 if "1024" in model else 512
    cin, cout = 3 * Cc, 1536
    code, tdt = {"fp32": (0, torch.float32), "tf32": (0, torch.float32), "bf16": (1, torch.bfloat16),
                 "fp16": (2, torch.float16)}[prec]
    dev = torch.device("cuda", torch.cuda.current_device())
    # rotate over enough (x, out) pairs that every launch reads operands not left in L2 by the previous one
    per = B * T * (cin + cout) * (2 if code else 4)
    nbuf = max(2, int(2 * 126e6 // per) + 1)
    xs = [torch.randn(B, 1, T, cin, device=dev).to(tdt) for _ in range(nbuf)]
    outs = [torch.empty(B, 1, T, cout, device=dev, dtype=tdt) for _ in range(nbuf)]
    w = (torch.randn(cout, cin, device=dev) / cin ** 0.5).to(tdt)
    bias = torch.zeros(cout, device=dev)
    L = lib.load()
    descs = []
    for x, o in zip(xs, outs):
        d = lib.ConvDesc()
        d.x, d.B, d.F, d.T, d.Cin, d.x_ld = x.data_ptr(), B, 1, T, cin, cin
        d.w, d.Cout, d.kf, d.kt = w.data_ptr(), cout, 1, 1
        d.dil_f = d.dil_t = d.stride_f = d.stride_t = 1
        d.bias, d.act1, d.out, d.out_ld, d.dtype, d.use_tc = bias.data_ptr(), 1, o.data_ptr(), cout, code, (0 if prec == "fp32" else tc_version)
        descs.append(d)
    st = lib.cur_stream_ptr()
    for i in range(3):
        lib.check(L.ws_conv(C.byref(descs[i % nbuf]), st), "ws_conv")
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        lib.check(L.ws_conv(C.byref(descs[i % nbuf]), st), "ws_conv")
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    flops = 2.0 * B * T * cin * cout
    return dict(ms=ms, tflops=flops / (ms * 1e-3) / 1e12, flops=flops, nbuf=nbuf,
                kernel=f"ws_conv_gemm_tc{tc_version}_kernel 1x1 {cin}->{cout} over {B * T} positions")


def _quiet_nccl():
    """NCCL prints its version banner to STDOUT at level VERSION; the driver reads ONE JSON line from stdout."""
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"


def main():
    _quiet_nccl()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-plda", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-config legs (configs block)")
    ap.add_argument("--sustained-s", type=float, default=2.0, help="length of the seconds-long sustained leg (0 = skip)")
    ap.add_argument("--tc-version", type=int, default=0, help="override the engine's tcgen05 kernel generation (1,2,3)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the embeddings of the last timed step (rank 0's batch) to DIR/embeddings.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's embeddings; it cannot be combined with --impl reference")
    wl = args.workload
    if args.impl == "reference":
        run_reference(args, wl)
        return
    model_name, prec, B, nsamples, gflop_utt = WORKLOADS[wl]
    torch.set_num_threads(2)  # the GPU arm needs no host parallelism; idle-spinning worker pools only add scheduler noise

    from wespeaker_b200 import parallel
    from wespeaker_b200.models import from_synthetic
    from wespeaker_b200 import synthetic as syn
    rank, world, local = parallel.init_from_env("nccl")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world != args.gpus and rank == 0:
        print(f"warning: --gpus {args.gpus} but WORLD_SIZE={world}", file=sys.stderr)
    peaks = measured_peaks()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()          # NVML init happens here, far from any timed window

    model = from_synthetic(model_name, 0, precision=prec).to(dev)
    if args.tc_version:
        model.set_option("tc_version", args.tc_version)
    L_frames = 1 + (nsamples - 400) // 160
    # rotate over distinct input batches; the per-step working set (activations) is >> the 126 MB L2 anyway
    nrot = 4
    base = syn.make_wavs(B, nsamples, seed=100 + rank)
    wav_dev = [torch.from_numpy(np.roll(base, i, axis=0)).to(dev) for i in range(nrot)]
    wav_pin = [torch.from_numpy(np.roll(base, i, axis=0).astype(np.int16)).pin_memory() for i in range(nrot)]
    emb = None
    for i in range(max(3, args.warmup)):
        emb = model.extract_from_wav(wav_dev[i % nrot])
    # warm the communicator with the SHAPE the timed gather uses (first NCCL collective pays lazy init per shape class)
    parallel.gather_embeddings(torch.cat([emb] * args.steps, 0), args.steps * B * world)
    torch.cuda.synchronize()
    launches_per_step = model.last_launches()
    embed_dim = model.embed_dim

    # ---------------- device-resident throughput (`value`): K steps + the one all-gather, best of 3 windows
    last_step = []

    def value_run():
        local_embs = [model.extract_from_wav(wav_dev[i % nrot]) for i in range(args.steps)]
        last_step[:] = local_embs[-1:]
        allemb = torch.cat(local_embs, 0)
        return parallel.gather_embeddings(allemb, allemb.shape[0] * world)  # the one NCCL all-gather of the job
    if sampler:
        sampler.mark(True)
    ms_total, gathered = _timed(value_run, dev, parallel, world, reps=3)
    clocks = None
    if sampler:
        sampler.mark(False)
        clocks = sampler.read() if sampler.nvml is not None else None
    assert gathered.shape[0] == args.steps * B * world and torch.isfinite(gathered).all()
    value = world * B * args.steps / (ms_total * 1e-3)
    if args.dump_outputs and rank == 0:
        # inputs and weights are seeded (make_wavs seed 100 + rank, from_synthetic seed 0): two builds of the project run
        # with the same arguments can be compared output for output
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "embeddings.npy"), last_step[0].float().cpu().numpy())

    # ---------------- end-to-end through the public host-buffer API (`e2e`)
    # B200SpeakerModel.extract_stream: every step copies that step's pinned int16 PCM batch H2D, runs fbank+CMN+forward
    # and copies the embeddings back D2H; the copy of batch i+1 overlaps the kernels of batch i (4 staging slots).
    # Warm-up stream first (allocations, pinned pools), then time K complete steps: the clock starts before the first
    # timed batch is submitted (its H2D copy is NOT hidden) and stops when the K-th batch's embeddings are in host memory.
    for out_h in model.extract_stream(wav_pin[i % nrot] for i in range(max(4, args.warmup))):
        pass
    best_dt = None
    for rep in range(3):   # best of 3 windows, the same estimator as `value`
        parallel.barrier(); torch.cuda.synchronize()
        t0, nout = time.perf_counter(), 0
        for out_h in model.extract_stream(wav_pin[i % nrot] for i in range(args.steps)):
            nout += out_h.shape[0]
        dt_rep = parallel.max_over_ranks(time.perf_counter() - t0, dev)
        best_dt = dt_rep if best_dt is None else min(best_dt, dt_rep)
    dt = best_dt
    torch.cuda.synchronize()
    parallel.barrier()
    e2e_value = world * B * args.steps / dt
    assert nout == B * args.steps and torch.isfinite(out_h).all()
    assert torch.equal(out_h.to(dev), model.extract_from_wav(wav_dev[(args.steps - 1) % nrot]))

    # ---------------- seconds-long sustained run (clocks settle under load; MEASURED_PEAKS' sustained figure is its peer)
    sustained = None
    if args.sustained_s > 0:
        n_sus = max(args.steps, int(args.sustained_s * 1e3 / (ms_total / args.steps)))
        if sampler:
            sampler.mark(True)
        ms_sus, _ = _timed(lambda: [model.extract_from_wav(wav_dev[i % nrot]) for i in range(n_sus)][-1], dev, parallel, world)
        v_sus = world * B * n_sus / (ms_sus * 1e-3)
        sustained = {"value": v_sus, "unit": "utt/s", "steps": n_sus, "seconds": ms_sus * 1e-3,
                     "step_frac_of_sustained": v_sus / world * gflop_utt / 1e3 / peaks["tf_sustained"]}
        if sampler:
            sampler.mark(False)
            sustained["clocks"] = sampler.read() if sampler.nvml is not None else None

    # ---------------- parity of the TIMED configuration (full batch: the cta_group::2 kernels at bench size)
    parity = None
    if rank == 0:
        emb_b, feats_b = model.extract_from_wav(wav_dev[0], return_feats=True)
        sel = [0, B // 3, (2 * B) // 3, B - 1]
        parity = {"parity_rel_l2": _parity(model_name, [emb_b[j] for j in sel], [feats_b[j] for j in sel]),
                  "parity_bar": PARITY_BAR[prec], "parity_utts": sel,
                  "against": "oracle.models_torch (CPU fp32) on the identical GPU fbank+CMN features of the timed batch"}
    del model
    torch.cuda.empty_cache()

    # ---------------- the other BASELINE.json configs, one short leg each (all ranks take part; rank 0 reports)
    configs = None
    if not args.no_configs:
        configs = {}
        for name in ("ecapa512_tf32x3_b256", "ecapa512_bf16_b256", "resnet34_fp16_b64"):
            m, pr, b, ns, gf = WORKLOADS[name]
            configs[name] = model_leg(name, m, pr, b, ns, gf, args.steps, args.warmup, dev, rank, world, parallel, peaks, sampler)
        configs["resnet34_fp16_b64"]["note"] = "BASELINE configs[2] is batch 512 sharded 64/GPU over 8 ranks: this leg IS that job when n_gpus == 8"
        configs["campplus_bf16_varlen"] = varlen_leg(args.steps, args.warmup, dev, rank, world, parallel, peaks, sampler)
        if not args.no_plda:
            configs["plda_1Mx100k"] = plda_leg(dev, rank, world, parallel, peaks)
    extras = None
    if not args.no_configs and world == 1:
        extras = {}
        for name, (m, pr, b, ns) in EXTRA_WORKLOADS.items():
            try:   # an extra must never cost the line its contract fields
                r = model_leg(name, m, pr, b, ns, 0.0, args.steps, args.warmup, dev, rank, world, parallel, peaks, sampler, parity_n=min(2, b))
                for k in ("step_tflops_per_gpu", "step_frac_of_sustained", "step_frac_of_3xtf32_sustained", "note"):
                    r.pop(k, None)
                if b == 1:
                    r["latency_ms_per_utt"] = r["ms_per_step"]
                extras[name] = r
            except Exception as ex:
                extras[name] = {"workload": name, "error": repr(ex)[:300]}
    if sampler:
        last = sampler.stop()
        if clocks is None:     # nvidia-smi fallback: one window over the whole run
            clocks = last

    if rank != 0:
        return
    # ---------------- roofline for the dominant kernel + whole-step tensor utilisation
    dom = time_dominant_kernel(model_name, prec, B, L_frames, tc_version=args.tc_version or 3)
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")
    if os.path.exists(tpath) and wl == DEFAULT_WORKLOAD:   # DRAM bytes per launch of this kernel from the committed ncu capture
        traffic = json.load(open(tpath))["traffic_bytes_per_launch"]
    step_tf = value / world * gflop_utt / 1e3  # TFLOP/s per GPU, algorithmic
    if dom is not None:
        roof = {"bound": "tensor", "achieved": dom["tflops"], "peak": peaks["tf_burst"], "unit": "TFLOP/s",
                "frac": dom["tflops"] / peaks["tf_burst"], "traffic": traffic, "kernel": dom["kernel"],
                "kernel_ms": dom["ms"], "flops_per_launch": dom["flops"], "peak_source": peaks["src"] + " (burst, kernel timed alone)",
                "step_tflops_per_gpu": step_tf, "step_frac_of_sustained": step_tf / peaks["tf_sustained"]}
    else:
        roof = {"bound": "tensor", "achieved": step_tf, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                "frac": step_tf / peaks["tf_sustained"], "traffic": None, "kernel": "whole step (conv GEMMs)",
                "peak_source": peaks["src"] + " (sustained, whole step)"}
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        pool = CpuPool(model_name, nsamples)
        pool.calibrate()
        nst, cdt = 0, 0.0
        while cdt < 10.0 and nst < 50:
            cdt += pool.run(1); nst += 1
        cpu = {"value": nst * pool.utts_per_step / cdt, "unit": "utt/s", "cores": pool.active * pool.threads, "kind": "port",
               "sample": f"{nst} pool steps in {cdt:.1f} s; " + pool.describe(nsamples)}
        pool.close()
        try:
            # the reference-faithful mode: one whole utterance per forward, as the reference extracts every test set
            # (examples/voxceleb/v2/local/extract_vox.sh:31: batch size 1); one process, 8 torch threads, ~3 s
            th0 = torch.get_num_threads()
            torch.set_num_threads(min(8, os.cpu_count() or 1))
            one = _cpu_path(model_name, nsamples, 1)
            one()
            n1, t1 = 0, time.perf_counter()
            while time.perf_counter() - t1 < 3.0:
                one(); n1 += 1
            d1 = time.perf_counter() - t1
            torch.set_num_threads(th0)
            cpu["batch1"] = {"value": n1 / d1, "unit": "utt/s", "latency_ms_per_utt": 1e3 * d1 / n1, "cores": min(8, os.cpu_count() or 1),
                             "sample": f"{n1} utterances one at a time in {d1:.1f} s, one process"}
        except Exception as ex:
            cpu["batch1"] = {"error": repr(ex)[:200]}
    act_mb = B * L_frames * (1536 * 2 + 128 + (1024 if '1024' in model_name else 512) * 7) * (4 if prec in ("fp32", "tf32", "tf32x3") else 2) / 1e6
    line = {
        "metric": METRIC, "value": value, "unit": "utt/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": DTYPE_NAME[prec], "data": "synthetic",
        "config": {"workload": wl, "model": model_name, "batch_per_gpu": B, "samples_per_utt": nsamples,
                   "frames": L_frames, "precision": prec, "gflop_per_utt": gflop_utt,
                   "l2": f"inputs rotate over {nrot} batches; per-step activation working set ~{act_mb:.0f} MB > 126 MB L2",
                   "estimator": "best of 3 windows of K steps for both value and e2e; device events, max over ranks",
                   "collective": "one all_gather_into_tensor of embeddings at job end (inside timed region)" if world > 1 else "none"},
        "e2e": {"value": e2e_value, "unit": "utt/s", "h2d_bytes_per_step": B * nsamples * 2, "d2h_bytes_per_step": B * embed_dim * 4,
                "api": "B200SpeakerModel.extract_stream(pinned int16 PCM host batches): H2D + fbank + CMN + forward + D2H per step, copy/compute overlapped over 4 slots; best of 3 windows of K steps"},
        "gpu_launches": int(launches_per_step * args.steps),
        "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "parity": parity, "sustained": sustained, "configs": configs, "extras": extras,
    }
    if configs and "plda_1Mx100k" in configs:
        line["plda"] = configs["plda_1Mx100k"]
    print(json.dumps(line))


if __name__ == "__main__":
    main()
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        torch.distributed.destroy_process_group()
