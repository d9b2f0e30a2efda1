#!/usr/bin/env python
"""bench.py - clips/s of the NISQA predict hot path (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|reference-gpu] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[1]): predict_dir bs=64, synthetic 10 s 48 kHz PCM16 clips,
weights/nisqa.tar.  One "step" = one pass of the hot path (PCM -> 5 scores) over one batch of 64
clips per GPU; for N > 1 each rank has its own batch (weak scaling) and a step ends with the
path's single exchange step, one NCCL all-gather of the score rows.

Printed JSON line (rank 0): `value` = whole-job clips/s with the PCM already resident in HBM,
`e2e` = the same through the C-ABI call with pinned HOST buffers (H2D of the PCM and D2H of the
scores inside the timed region), `roofline` for the dominant kernel (CUDA-event timed on the
engine stream), `cpu_baseline` = the oracle port on the host cores on a bounded sample.
`--impl reference` times the reference's CPU implementation of the path (the oracle port run
clip-parallel on all host cores) and prints the same line with "impl": "reference".
`--impl reference-gpu` (and the `reference_gpu` key of the default line at N=1) times the UNMODIFIED
reference torch modules in PyTorch eager on this GPU (tools/reference_gpu.py; SURVEY.md 8d's "honest thing to
beat"), when the reference package was installed under baseline/_ref by `tools/reference_gpu.py --install SRC`.
`--dump-outputs DIR` (default impl): after the timed steps, rank 0 writes what the last timed step returned to its
caller as DIR/<name>.npy (float32 scores, n_segments and status as float64; with N > 1 also the gathered rows).
The inputs depend only on the arguments, so two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "clips/sec (48 kHz, 10 s) NISQA v2.0 predict"
UNIT = "clips/s"
BS, SECONDS, SR = 64, 10.0, 48000
N_ROT = 4                      # rotating batches: 4 x 61 MB PCM16 = 245 MB > 126 MB L2
CKPT = os.path.join(ROOT, "weights", "nisqa.tar")

# algorithmic FLOPs per segment of each conv layer (SURVEY.md 8a row a10 / BASELINE.md section 3)
CONV_FLOP_PER_SEG = {"conv1": 207360, "conv2": 1548288, "conv3": 2211840, "conv4": 4423680,
                     "conv5": 1327104, "conv6": 442368, "conv12": 207360 + 1548288}
SEGS_PER_CLIP = 247
FLOP_PER_CLIP = 2.735e9


# algorithmic FLOPs per clip of the self-attention layers (SURVEY.md 8a rows a11/a12 at S = 247, 2 layers):
# QK^T + PV = 31.2 M (the "attention-FLOP roofline" of 8d), out-proj + FFN = 24.4 M
ATT_FLOP_PER_CLIP = 31.2e6
SA_LAYER_FLOP_PER_CLIP = 55.6e6


def build_rooflines(kernel_ms, peaks, sm_max_mhz, traffic_tab, n_samples):
    """Per-kernel rooflines from CUDA-event kernel times (ms per 64-clip step).  Returns (all, dominant):
    `dominant` is the kernel with the largest share of the step.  Pure function (tests/test_host_logic.py
    replays a recorded bench line through it)."""
    n_seg_step = BS * SEGS_PER_CLIP
    fp32_peak = 148 * 128 * 2 * (sm_max_mhz or 1965.0) * 1e6 / 1e12
    tc_layers = ("conv12", "conv2", "conv3", "conv4", "conv5", "conv6")
    roofs = {}
    for k in ("conv1",) + tc_layers:
        if kernel_ms.get(k, 0) <= 0:
            continue
        flop = CONV_FLOP_PER_SEG[k] * n_seg_step
        ach = flop / (kernel_ms[k] / 1e3) / 1e12
        r = {"kernel": k, "bound": "tensor", "achieved": ach, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
             "frac": ach / peaks["bf16_tflops_sustained"], "traffic": traffic_tab.get(k),
             "peak_source": peaks["source"] + ", sustained 16-bit dense (kernel timed inside a long step)",
             "kernel_ms": kernel_ms[k], "algorithmic_flop_per_launch": flop}
        if k in tc_layers:
            r["note"] = ("tcgen05 kind::f16 implicit GEMM with a two-term fp16 split: 3 MMAs per algorithmic MAC "
                         "(parity: plain 16-bit operands move MOS by >1e-3), so the tensor pipe executes 3x `achieved`")
            r["executed_tflops"] = 3 * ach
            r["frac_executed"] = 3 * ach / peaks["bf16_tflops_sustained"]
            if k == "conv12":
                r["note"] = ("conv1 + pool1 (fp32 FFMA, producer warps) fused with conv2 + pool2 (tcgen05, fp16 two-term split) in one "
                             "persistent kernel: the pool1 activations never reach HBM; algorithmic FLOPs of both layers")
        else:
            r["note"] = "conv1 (C_in=1, K=9) is direct fp32 FFMA; fraction of the fp32 FFMA peak in frac_fp32"
            r["fp32_peak_tflops"] = fp32_peak
            r["frac_fp32"] = ach / fp32_peak
        roofs[k] = r
    byts = BS * (n_samples * 2 + 1001 * 48 * 4)
    hbm = byts / (kernel_ms["frontend"] / 1e3) / 1e9
    fft_tf = 136.7e6 * BS / (kernel_ms["frontend"] / 1e3) / 1e12
    # The front-end moves 1.2 MB per clip but executes 137 MFLOP of radix-32 butterflies + mel on the FFMA pipe: it
    # is bound by fp32 instruction issue, so `frac` is the fraction of the fp32 FFMA peak (the HBM view of SURVEY
    # 8d's "STFT-bandwidth roofline" is kept beside it: hbm_gbs / hbm_frac say how far it is from being a copy)
    roofs["frontend"] = {"kernel": "frontend", "bound": "fp32-issue", "achieved": fft_tf, "peak": fp32_peak, "unit": "TFLOP/s",
                         "frac": fft_tf / fp32_peak, "traffic": traffic_tab.get("frontend"),
                         "peak_source": "fp32 FFMA peak 148 SM x 128 lanes x 2 x SM clock", "kernel_ms": kernel_ms["frontend"],
                         "algorithmic_flop_per_launch": 136.7e6 * BS, "algorithmic_bytes_per_launch": byts,
                         "hbm_gbs": hbm, "hbm_peak_gbs": peaks["hbm_gbs"], "hbm_frac": hbm / peaks["hbm_gbs"],
                         "hbm_peak_source": peaks["source"],
                         "note": "123 MFLOP/clip of FFT butterflies + 13.7 MFLOP magnitude / mel / log (BASELINE.md section 3), "
                                 "PCM16 in + mel out = algorithmic_bytes_per_launch"}
    if kernel_ms.get("sa_layer", 0) > 0:
        # the two self-attention layer launches (flash-style softmax(QK^T)V + out-proj + FFN + 2 LayerNorms), fp32 FFMA
        ms = kernel_ms["sa_layer"]
        att = ATT_FLOP_PER_CLIP * BS / (ms / 1e3) / 1e12
        roofs["sa_layer"] = {"kernel": "sa_layer", "bound": "tensor", "achieved": att, "peak": fp32_peak, "unit": "TFLOP/s",
                             "frac": att / fp32_peak, "traffic": traffic_tab.get("sa_layer"),
                             "peak_source": "fp32 FFMA peak 148 SM x 128 lanes x 2 x SM clock (the kernel runs on the FFMA pipe, "
                                            "no tensor cores: fp32 parity)",
                             "kernel_ms": ms, "algorithmic_flop_per_launch": ATT_FLOP_PER_CLIP * BS,
                             "note": "attention-FLOP roofline of SURVEY 8d(iii): QK^T + PV only; with out-proj + FFN the same "
                                     "launches do %.1f TFLOP/s" % (SA_LAYER_FLOP_PER_CLIP * BS / (ms / 1e3) / 1e12)}
    dom = max(roofs, key=lambda k: kernel_ms[k])
    return roofs, roofs[dom]


def make_clips(n, seed0=0):
    """n distinct 10-s PCM16 clips: a few synthesised bases, circularly shifted (np.roll)."""
    from nisqa_b200 import synth
    n_base = min(n, 16)
    bases = [synth.synth_speech_pcm16(seed0 + i, SECONDS, SR) for i in range(n_base)]
    rng = np.random.default_rng(seed0 + 999)
    out = []
    for i in range(n):
        b = bases[i % n_base]
        out.append(b if i < n_base else np.roll(b, int(rng.integers(1, len(b) - 1))))
    return out


class ClockSampler(object):
    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def mark(self):
        return len(self.rows)

    def stop(self, lo=0, hi=None):
        if self.proc is not None:
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = self.rows[lo:hi] if len(self.rows[lo:hi]) >= 2 else self.rows[max(0, lo - 3):]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
                for nm, v in zip(names, f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0,
            "source": "fallback (B200_PROFILING.md)"}


class CpuPool(object):
    """Oracle port on the host cores, clip-parallel: `procs` worker processes with one torch
    thread each - per-clip parallelism is the reference's own way to use cores (DataLoader
    workers, reference lib:1425-1430)."""

    def __init__(self, procs):
        self.procs = procs
        self.pool = None
        # one compute thread per worker process: BLAS / OpenMP pools must not oversubscribe
        for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
            os.environ[k] = "1"
        if procs > 1:
            import torch.multiprocessing as mp
            self.pool = mp.get_context("spawn").Pool(procs, initializer=_cpu_worker_init)
            self.pool.map(_cpu_worker, list(range(4000, 4000 + procs)))   # spin-up + imports, untimed
        else:
            _cpu_worker_init()
            _cpu_worker(4000)

    def run(self, n_clips, seed0=5000):
        seeds = list(range(seed0, seed0 + n_clips))
        t0 = time.perf_counter()
        if self.pool is None:
            res = [_cpu_worker(s) for s in seeds]
        else:
            res = self.pool.map(_cpu_worker, seeds, chunksize=1)
        dt = time.perf_counter() - t0
        return n_clips / dt, dt, res

    def close(self):
        if self.pool is not None:
            self.pool.close()
            self.pool.join()


_CPU = {}


def host_cores():
    """Cores the CPU arm may really use: affinity mask capped by the cgroup CPU quota (tools/reference_gpu.py)."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import reference_gpu
    return reference_gpu.effective_cores()


def _cpu_worker_init():
    import torch
    torch.set_num_threads(1)
    try:
        from threadpoolctl import threadpool_limits
        _CPU["tpl"] = threadpool_limits(limits=1)
    except Exception:
        pass
    from oracle import nisqa_oracle as O
    _CPU["O"] = O
    _CPU["ck"] = O.load_checkpoint(CKPT)


def _cpu_worker(seed):
    from nisqa_b200 import synth
    O = _CPU["O"]
    args, sd = _CPU["ck"]
    rng = np.random.default_rng(seed)
    y = (rng.standard_normal(int(SECONDS * SR)) * 0.05).astype(np.float32)   # cheap synthetic input
    sc, _, _ = O.predict_pcm(args, sd, y, SR)
    return float(sc[0])


def _host_info():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import reference_gpu
    return reference_gpu.host_info()


def load_traffic_table():
    """Per-launch DRAM traffic (ncu dram__bytes_read + write) of the kernels, measured by tools/profile_round.sh and
    stamped with the digest of the kernel sources it was measured on (nisqa_b200/build.py _digest).  ncu cannot run
    inside the bench, so a table taken on OTHER sources is refused: traffic is then null, never stale."""
    tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if not os.path.exists(tp):
        return {}, "no profiles/roofline_traffic.json"
    tab = json.load(open(tp))
    from nisqa_b200 import build as nb_build
    have, want = tab.get("_source_digest"), nb_build.kernel_digest()
    if have != want:
        return {}, "profiles/roofline_traffic.json was measured on other kernel sources (digest %s..., library %s...): traffic = null" % (
            str(have)[:12], want[:12])
    if "td_sa_kernel" in tab and "sa_layer" not in tab:
        tab["sa_layer"] = 2 * tab["td_sa_kernel"]          # the group "sa_layer" = the two encoder-layer launches of a step
    return tab, "profiles/roofline_traffic.json (%s), same kernel sources as this library" % tab.get("_note", "")


def cpu_baseline_leg(target_s=6.0, repeats=3):
    """Oracle port on every host core, clip-parallel; `repeats` bounded samples, median reported, host described
    (the same port printed 87 and 420-460 clips/s on two '128 core' boxes in round 1: the box matters)."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import reference_gpu
    cores = host_cores()
    pool = CpuPool(cores)
    _, dt1, _ = pool.run(cores)
    n_cpu = int(min(max(cores, cores * target_s / max(dt1, 1e-3)), 64 * cores))
    runs = [pool.run(n_cpu, seed0=7000 + 100 * r) for r in range(repeats)]
    pool.close()
    vals = sorted(v for v, _, _ in runs)
    return {"value": float(np.median(vals)), "unit": UNIT, "cores": cores, "kind": "port",
            "repeats": [float(v) for v, _, _ in runs], "host": reference_gpu.host_info(),
            "sample": "median of %d runs of %d x 10 s 48 kHz white-noise clips (cost is data independent), %d worker "
                      "processes x 1 torch thread, %.1f s of wall time each; oracle port of the reference "
                      "CPU path (NumPy librosa restatement + torch CPU)" % (repeats, n_cpu, cores, float(np.median([d for _, d, _ in runs])))}


def reference_gpu_leg(eng=None):
    """The unmodified reference modules in PyTorch eager on this GPU (tools/reference_gpu.py)."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import reference_gpu
    ours = None
    if eng is not None:
        def ours(paths):
            from nisqa_b200 import wav
            pcm = [wav.read_wav(p)[0] for p in paths]
            return eng.predict_pcm(pcm, [SR] * len(pcm))[0]
    try:
        return reference_gpu.measure(n_clips=BS, bs=BS, seconds=SECONDS, sr=SR, ckpt=CKPT, ours=ours)
    except Exception as exc:       # the extra arm must never take the bench line down
        return {"unavailable": "reference-gpu arm failed: %r" % (exc,)}


def run_reference_gpu(a, rank, world):
    if rank != 0:
        return
    r = reference_gpu_leg(None)
    if "unavailable" in r:
        print(json.dumps({"impl": "reference-gpu", "unavailable": r["unavailable"]}), flush=True)
        return
    v = r["predict_dir"]["clips_per_s"]
    line = {"impl": "reference-gpu", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": 1, "steps": 3, "warmup": 1,
            "ms_per_step": r["predict_dir"]["wall_s"] * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "predict_dir bs=64, synthetic 10 s 48 kHz clips, nisqa.tar (configs[1]); unmodified "
                                   "reference package, PyTorch eager on cuda:0, %d DataLoader workers" % r["num_workers"]},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": int(BS * 1300 * 48 * 15 * 4), "d2h_bytes_per_step": BS * 5 * 4},
            "reference_gpu": r}
    print(json.dumps(line), flush=True)


def run_reference(a, rank, world):
    if rank != 0:
        return
    cores = host_cores()
    procs = max(1, cores)
    per_step = max(procs, 8)
    pool = CpuPool(procs)
    vals = []
    for s in range(a.warmup + a.steps):
        v, dt, _ = pool.run(per_step, seed0=5000 + 1000 * s)
        if s >= a.warmup:
            vals.append((v, dt))
        if s == 0 and dt * (a.warmup + a.steps) > 240:      # keep the run within a few minutes
            per_step = max(procs, int(per_step * 240 / (dt * (a.warmup + a.steps))))
    pool.close()
    value = float(np.mean([v for v, _ in vals]))
    ms = float(np.mean([dt for _, dt in vals]) * 1e3)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "predict_dir bs=64, synthetic 10 s 48 kHz clips, nisqa.tar (configs[1])",
                       "sample": "%d clips per step" % per_step},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": procs, "kind": "port", "host": _host_info(),
                             "sample": "%d x 10 s 48 kHz clips per step, %d worker processes x 1 torch thread, "
                                       "oracle port of the reference CPU path (NumPy librosa restatement + torch CPU)"
                                       % (per_step, procs)},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def sharded_predict_csv_check(eng, rank, world, local):
    """BASELINE configs[4] in miniature on the real ranks: `nisqaModel(mode=predict_csv).predict()` (the product
    surface: _loadDatasetsCSVpredict -> predict_dim -> rows sharded over the ranks -> ONE ncclAllGather through the
    engine) over 16 clips per rank, compared on rank 0 with the same rows computed by ONE engine in one process (must
    be bit-identical: clips are independent) and with the oracle on two of them."""
    import shutil
    import tempfile
    import torch.distributed as dist
    import pandas as pd
    from nisqa_b200 import synth, wav
    from nisqa_b200.NISQA_model import nisqaModel
    n = 16 * world
    box = [tempfile.mkdtemp(prefix="nisqa_cfg5_") if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    td = box[0]
    specs = [(3000 + i, 1.0 + 0.25 * (i % 9), (48000, 16000, 44100)[i % 3]) for i in range(n)]
    try:
        if rank == 0:
            for seed, sec, sr in specs:
                wav.write_wav_pcm16(os.path.join(td, "c%04d.wav" % seed), synth.synth_speech_pcm16(seed, sec, sr), sr)
            pd.DataFrame({"deg": ["c%04d.wav" % s for s, _, _ in specs]}).to_csv(os.path.join(td, "files.csv"), index=False)
        dist.barrier()
        import contextlib
        import io
        with contextlib.redirect_stdout(io.StringIO()):
            m = nisqaModel({"mode": "predict_csv", "pretrained_model": CKPT, "data_dir": td, "csv_file": "files.csv",
                            "csv_deg": "deg", "output_dir": None, "tr_bs_val": 8, "tr_num_workers": 2, "ms_channel": None})
            df = m.predict()
        m.model.close()
        dist.barrier()
        if rank != 0:
            return None
        cols = ["mos_pred", "noi_pred", "dis_pred", "col_pred", "loud_pred"]
        got = df[cols].to_numpy(dtype=np.float32)
        pcm = [wav.read_wav(os.path.join(td, "c%04d.wav" % s))[0] for s, _, _ in specs]
        single = eng.predict_pcm(pcm, [sr for _, _, sr in specs])[0]
        from oracle import nisqa_oracle as O
        args, sd = O.load_checkpoint(CKPT)
        worst = 0.0
        for i in (0, n - 1):
            ref = O.predict_pcm(args, sd, pcm[i].astype(np.float32) / 32768.0, specs[i][2])[0]
            worst = max(worst, float(np.abs(got[i] - ref).max()))
        return {"rows": n, "ranks": world, "api": "nisqaModel(mode='predict_csv').predict() under torchrun, rows sharded, one ncclAllGather",
                "bit_identical_to_single_process": bool(np.array_equal(got, single)), "max_abs_vs_oracle": worst}
    finally:
        if rank == 0:
            shutil.rmtree(td, ignore_errors=True)


def run_ours(a, rank, world, local):
    import torch
    from nisqa_b200 import engine as E
    import torch.distributed as dist

    torch.cuda.set_device(local)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()               # nvidia-smi needs a second or two to come up
    from nisqa_b200 import dist as nb_dist
    all_cpus = os.sched_getaffinity(0)
    numa_node = nb_dist.bind_to_gpu_numa(local)      # pinned PCM buffers next to the GPU's PCIe root
    ck = torch.load(CKPT, map_location="cpu", weights_only=False)     # as nisqaModel._loadModel does (model:938-942)
    args, sd = ck["args"], ck["model_state_dict"]
    eng = E.Engine(E.config_from_args(args), local)
    eng.load_state_dict(sd)
    n_out = eng.n_out

    clips = make_clips(BS * N_ROT, seed0=1000 * (rank + 1))
    n_s = np.array([len(c) for c in clips[:BS]], dtype=np.int64)
    srs = np.full(BS, SR, dtype=np.int32)
    stride = (int(n_s[0]) + 15) // 16 * 16
    offs = np.arange(BS, dtype=np.int64) * stride
    dev_batches, pin_batches, ptr_arrays = [], [], []
    import ctypes as C
    for r in range(N_ROT):
        host = torch.zeros(BS * stride, dtype=torch.int16).pin_memory()
        hv = host.numpy()
        for i in range(BS):
            hv[i * stride:i * stride + n_s[i]] = clips[r * BS + i]
        pin_batches.append(host)
        dev_batches.append(host.cuda(non_blocking=False))
        ptr_arrays.append((C.c_void_p * BS)(*[host.data_ptr() + 2 * i * stride for i in range(BS)]))
    scores_dev = torch.empty((BS, n_out), dtype=torch.float32, device="cuda")
    scores_ring = [torch.empty((BS, n_out), dtype=torch.float32, device="cuda") for _ in range(3)]
    scores_host = np.empty((BS, n_out), dtype=np.float32)
    stream = torch.cuda.ExternalStream(eng.stream())

    gather = None
    if world > 1:
        uid = [eng.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        eng.nccl_init(world, rank, uid[0])
        glob = torch.empty((world, BS, n_out), dtype=torch.float32, device="cuda")
        # the exchange step rides on every call's own compute lane (nisqa_set_gather_target)
        eng.set_gather_target(glob.data_ptr(), BS)
        gather = True

    last_dev = {}                                # the latest step: (index, n_segments, status)

    def step_dev(i, sync=False):
        last_dev["out"] = (i,) + eng.predict_pcm_device(dev_batches[i % N_ROT].data_ptr(), offs, n_s, srs, E.FMT_S16,
                                                        scores_ring[i % 3].data_ptr(), sync=sync)

    # e2e: the public streaming API - submit batch i (pinned host PCM16 -> H2D -> kernels -> D2H of the
    # scores), then collect batch i-1; two batches in flight, every step's copies inside the timed region
    NF = 5                                       # submissions in flight (the engine has 6 staging slots)
    e2e_scores = [np.empty((BS, n_out), dtype=np.float32) for _ in range(NF)]
    e2e_aux = [(np.empty(BS, np.int32), np.empty(BS, np.int32)) for _ in range(NF)]
    tickets = [None] * NF

    def collect(k):
        if tickets[k] is not None:
            eng.wait_ticket(tickets[k]); tickets[k] = None       # (N > 1: the all-gather ran on the lane)

    def step_e2e(i):
        k = i % NF
        collect(k)                                # the oldest submission (i - NF) is collected first
        tickets[k] = eng.submit_pcm_ptrs(ptr_arrays[i % N_ROT], n_s, srs, E.FMT_S16, e2e_scores[k], e2e_aux[k][0], e2e_aux[k][1])

    def drain_e2e():
        for k in range(NF):
            collect(k)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, drain=None):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(stream)
        for i in range(steps):
            fn(i)
        if drain is not None:
            drain()
        eng.join()                 # lane 0 waits for the other compute lanes: e1 covers all of them
        e1.record(stream)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        ms = max(e0.elapsed_time(e1), 0.0)
        if world > 1:
            t = torch.tensor([ms, wall * 1e3], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, wall = float(t[0]), float(t[1]) / 1e3
        barrier()
        return ms, wall

    # ---- parity spot check of what is being timed (rank 0, first clip of batch 0)
    step_dev(0, sync=True)
    torch.cuda.synchronize()
    got = scores_ring[0][0].cpu().numpy()

    # warm-up: W steps, then as many more as ~warmup_seconds needs (clocks take ~1 s to ramp).  The
    # step count is agreed across ranks (every step holds a collective when N > 1).
    t_w = time.perf_counter()
    for i in range(a.warmup):
        step_dev(i)
    torch.cuda.synchronize()
    per_step = max((time.perf_counter() - t_w) / max(a.warmup, 1), 1e-4)
    n_extra = int(min(max(a.warmup_seconds / per_step, 0), 5000))
    if world > 1:
        t = torch.tensor([n_extra], dtype=torch.int64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        n_extra = int(t[0])
    for i in range(n_extra):
        step_dev(a.warmup + i)
        if i % 8 == 7:
            torch.cuda.synchronize()
    torch.cuda.synchronize()
    l0 = eng.kernel_launches()
    mark0 = sampler.mark()
    ms_dev, _ = timed(step_dev, a.steps)
    launches = eng.kernel_launches() - l0
    dump = None
    if a.dump_outputs and rank == 0:
        i_last, nseg_last, status_last = last_dev["out"]
        dump = {"scores": scores_ring[i_last % 3].cpu().numpy(),
                "n_segments": nseg_last.astype(np.float64), "status": status_last.astype(np.float64)}
        if world > 1:
            dump["scores_all_ranks"] = glob.cpu().numpy()
    for i in range(max(a.warmup, 4)):
        step_e2e(i)
    drain_e2e()
    ms_e2e, wall_e2e = timed(step_e2e, a.steps, drain_e2e)
    clocks = sampler.stop(mark0, sampler.mark()) if rank == 0 else None

    # ---- per-kernel durations (CUDA events on the engine stream), same workload
    eng.set_profiling(True)
    names = ["frontend", "conv12", "conv1", "conv2", "conv3", "conv4", "conv5", "conv6", "lin_ln", "qkv",
             "sa_layer", "pool", "seg_table"]
    acc = dict((k, 0.0) for k in names)
    prof_steps = max(3, min(a.steps, 10))
    for i in range(prof_steps):
        eng.predict_pcm_device(dev_batches[i % N_ROT].data_ptr(), offs, n_s, srs, E.FMT_S16,
                               scores_ring[0].data_ptr(), sync=True)
        for k in names:
            v = eng.group_ms(k)
            if v > 0:
                acc[k] += v
    eng.set_profiling(False)
    kernel_ms = dict((k, v / prof_steps) for k, v in acc.items())
    sharded = None
    if world > 1:
        try:
            eng.set_gather_target(0, 0)
            sharded = sharded_predict_csv_check(eng, rank, world, local)
        except Exception as exc:                 # never takes the bench line down; reported instead
            sharded = {"error": repr(exc)}

    if rank != 0:
        return
    peaks = measured_peaks()
    total_clips = BS * world * a.steps
    value = total_clips / (ms_dev / 1e3)
    e2e_wall = total_clips / max(wall_e2e, 1e-9)
    e2e_value = min(total_clips / (max(ms_e2e / 1e3, 1e-9)), e2e_wall)
    # ---- rooflines: every heavy kernel, `roofline` = the dominant one (largest share of the step)
    traffic_tab, traffic_note = load_traffic_table()
    roofs, roof = build_rooflines(kernel_ms, peaks, (clocks or {}).get("sm_max_mhz"), traffic_tab, int(n_s[0]))
    cnn_ms = sum(kernel_ms[k] for k in ("conv12", "conv1", "conv2", "conv3", "conv4", "conv5", "conv6"))
    # ---- checker legs (the only place this arm touches oracle/): parity of what was timed, then the CPU baseline
    from oracle import nisqa_oracle as O
    ref, _, _ = O.predict_pcm(args, sd, clips[0].astype(np.float32) / 32768.0, SR)
    parity = float(np.abs(got - ref).max())
    cpu_base = None
    os.sched_setaffinity(0, all_cpus)               # the CPU baseline may use every host core again
    if world == 1 and not a.skip_cpu:
        cpu_base = cpu_baseline_leg()
    ref_gpu = None
    if world == 1 and not a.skip_cpu and not a.skip_reference_gpu:
        ref_gpu = reference_gpu_leg(eng)
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": ms_dev / a.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "predict_dir bs=64, synthetic 10 s 48 kHz PCM16 clips, weights/nisqa.tar "
                                   "(BASELINE.json configs[1]); one step = 64 clips per GPU",
                       "clips_per_step_per_gpu": BS, "segments_per_clip": SEGS_PER_CLIP,
                       "l2": "inputs rotate over %d resident batches (%.0f MB PCM16 > 126 MB L2); per-step "
                             "activations ~730 MB stream through L2" % (N_ROT, N_ROT * BS * stride * 2 / 1e6),
                       "exchange": "1 ncclAllGather of [64,5] rows per step" if world > 1 else "none (N=1)"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(BS * int(n_s[0]) * 2),
                    "d2h_bytes_per_step": int(BS * n_out * 4), "wall_clock_value": e2e_wall,
                    "api": "nisqa_submit_pcm / nisqa_wait (C-ABI, five batches in flight) on pinned host PCM16; value is wall-clock based", "numa_node": numa_node},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "roofline_kernels": roofs,
            "roofline_traffic_source": traffic_note,
            "kernel_ms_per_step": kernel_ms, "cnn_ms_per_step": cnn_ms,
            "achieved_tflops_whole_step": FLOP_PER_CLIP * BS / (ms_dev / a.steps / 1e3) / 1e12,
            "parity_max_abs_vs_oracle": parity,
            "cpu_baseline": cpu_base, "reference_gpu": ref_gpu, "sharded_predict_csv": sharded}
    if dump is not None:
        os.makedirs(a.dump_outputs, exist_ok=True)
        for name, arr in dump.items():
            np.save(os.path.join(a.dump_outputs, name + ".npy"), arr)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default: 200, or 20 for --impl reference)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu"])
    ap.add_argument("--skip-reference-gpu", dest="skip_reference_gpu", action="store_true",
                    help="omit the reference_gpu key (the reference torch modules in eager mode on this GPU)")
    ap.add_argument("--warmup-seconds", dest="warmup_seconds", type=float, default=1.5,
                    help="minimum duration of the untimed warm-up (in addition to --warmup steps)")
    ap.add_argument("--skip-cpu", dest="skip_cpu", action="store_true", help="omit the cpu_baseline leg (profiling runs)")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (--impl ours)")
    a = ap.parse_args()
    if a.steps is None:
        a.steps = 200 if a.impl == "ours" else 20
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    a.warmup = max(a.warmup, 3) if a.impl == "ours" else max(a.warmup, 0)
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    if a.impl == "reference":
        run_reference(a, rank, world)
        return
    if a.impl == "reference-gpu":
        run_reference_gpu(a, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group(backend="nccl", rank=rank, world_size=world)
    try:
        run_ours(a, rank, world, local)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
