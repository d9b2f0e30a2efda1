"""The reference's OWN torch modules on the B200 (PyTorch eager, ``dev=cuda``) - SURVEY.md 8(d)'s "reference on
this GPU" row, the honest thing the hand-written engine has to beat.

    python tools/reference_gpu.py [--clips 64] [--workers N]        (prints one JSON object)
    python bench.py --impl reference-gpu                            (same numbers in the bench line format)

What runs is the UNMODIFIED reference package (``nisqa/NISQA_model.py`` + ``nisqa/NISQA_lib.py``) through its own
public API ``nisqaModel(args).predict()`` -> ``NL.predict_dim(model, ds, bs, dev, num_workers)`` (reference
lib:1441-1467) with the device it picks itself (CUDA when available, model:1036-1045).  The package is not part of
this repository: ``python tools/reference_gpu.py --install SRC`` copies ``SRC/nisqa`` of a NISQA checkout under
``baseline/_ref/`` (git-ignored); without it this module reports ``{"unavailable": ...}``.  ``librosa`` is not
installable offline, so the reference's ``lb.load / melspectrogram / amplitude_to_db`` calls land in
``oracle/librosa_compat.py`` (NumPy restatement of librosa 0.8.1) - stated in the output.  Nothing of the product (engine, kernels, native wav reader) is on this path.

Two figures:
  * ``predict_dir``: wall time of ``nisqaModel.predict()`` over a directory of synthetic 10 s 48 kHz wavs, bs=64,
    DataLoader workers = half the host cores (the reference computes mel spectrograms in the workers on the CPU,
    pads every clip to [1300,1,48,15] and runs the torch model on the GPU);
  * ``model_only``: the reference model's forward on ONE resident padded batch (``model(xb, n_wins)``), CUDA
    events - the model half alone, no front-end, no DataLoader.
"""
import contextlib
import io
import json
import os
import shutil
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(ROOT, "baseline", "_ref")
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def install_reference(src):
    """Copy of the reference package from the NISQA checkout `src` (pure Python, no build metadata: `pip install
    --target` has nothing to build, the package directory IS the install).  No-op without the source tree."""
    pkg = os.path.join(src, "nisqa")
    if not os.path.isdir(pkg):
        return False
    dst = os.path.join(REF_DIR, "nisqa")
    os.makedirs(REF_DIR, exist_ok=True)
    if os.path.isdir(dst):
        shutil.rmtree(dst)
    shutil.copytree(pkg, dst)          # as it lies: a namespace package (no __init__.py), nothing added or edited
    return True


def available():
    return os.path.isfile(os.path.join(REF_DIR, "nisqa", "NISQA_model.py"))


def _import_reference():
    from oracle import librosa_compat
    librosa_compat.install()
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    from nisqa.NISQA_model import nisqaModel
    import nisqa.NISQA_lib as NL
    return nisqaModel, NL


def host_info():
    info = {"nproc": os.cpu_count()}
    try:
        info["affinity"] = len(os.sched_getaffinity(0))
    except Exception:
        pass
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                info["cpu_model"] = line.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    for p in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            info["cpu_max"] = open(p).read().strip()
            break
        except Exception:
            pass
    try:
        info["loadavg_1m"] = float(open("/proc/loadavg").read().split()[0])
    except Exception:
        pass
    return info


def effective_cores():
    """Host cores this process can really use: the affinity mask, cut down to the cgroup CPU quota (the GPU boxes show
    128 cores but run under `cpu.max = 1600000 100000`, i.e. 16 CPUs - the reason the same CPU baseline printed 87 and
    420-460 clips/s on two "128 core" boxes in round 1)."""
    info = host_info()
    cores = info.get("affinity") or info.get("nproc") or 1
    try:
        quota, period = info.get("cpu_max", "max").split()[:2]
        if quota != "max" and int(quota) > 0:
            cores = max(1, min(cores, -(-int(quota) // int(period))))
    except Exception:
        pass
    return cores


def measure(n_clips=64, bs=64, seconds=10.0, sr=48000, workers=None, ckpt=None, model_iters=10, ours=None,
            allow_cpu=False):
    """-> dict (see module docstring).  ``ours``: optional callable(list of wav paths) -> [n, 5] scores of the
    engine on the same files, for the |delta| column."""
    if not available():
        return {"unavailable": "baseline/_ref/nisqa is absent (install it with tools/reference_gpu.py --install SRC)"}
    import torch
    cuda = torch.cuda.is_available()
    if not cuda and not allow_cpu:           # allow_cpu: plumbing test of this module in the build container
        return {"unavailable": "no CUDA device"}
    sync = torch.cuda.synchronize if cuda else (lambda: None)
    from nisqa_b200 import synth, wav
    nisqaModel, NL = _import_reference()
    ckpt = ckpt or os.path.join(ROOT, "weights", "nisqa.tar")
    cores = effective_cores()
    if workers is None:
        workers = max(1, min(cores, 32))
    out = {"impl": "unmodified reference nisqa/ package, PyTorch %s eager, device cuda" % torch.__version__,
           "front_end": "oracle/librosa_compat.py (NumPy restatement of librosa 0.8.1; real librosa is not installable offline)",
           "clips": n_clips, "bs": bs, "num_workers": workers, "host": host_info()}
    td = tempfile.mkdtemp(prefix="nisqa_refgpu_")
    try:
        n_base = min(n_clips, 8)
        bases = [synth.synth_speech_pcm16(9000 + i, seconds, sr) for i in range(n_base)]
        rng = np.random.default_rng(9)
        names = []
        for i in range(n_clips):
            pcm = bases[i % n_base] if i < n_base else np.roll(bases[i % n_base], int(rng.integers(1, len(bases[0]) - 1)))
            names.append("r%04d.wav" % i)
            wav.write_wav_pcm16(os.path.join(td, names[-1]), pcm, sr)
        args = {"mode": "predict_dir", "pretrained_model": ckpt, "data_dir": td, "output_dir": None,
                "num_workers": workers, "bs": bs, "ms_channel": None, "tr_bs_val": bs, "tr_num_workers": workers}
        sink = io.StringIO()
        with contextlib.redirect_stdout(sink):
            m = nisqaModel(dict(args))
            m.predict()                                   # warm-up: cuDNN heuristics, worker start-up, allocator
            sync()
            walls = []
            for _ in range(3):
                t0 = time.perf_counter()
                df = m.predict()
                sync()
                walls.append(time.perf_counter() - t0)
        wall = float(np.median(walls))
        out["predict_dir"] = {"clips_per_s": n_clips / wall, "wall_s": wall, "repeats": walls, "device": str(m.dev)}
        cols = ["mos_pred", "noi_pred", "dis_pred", "col_pred", "loud_pred"]
        ref_scores = df.set_index("deg").loc[names, cols].to_numpy(dtype=np.float64)
        # ---- model half alone on one resident padded batch
        from torch.utils.data import DataLoader
        dl = DataLoader(m.ds_val, batch_size=bs, shuffle=False, num_workers=workers)
        xb, yb, (idx, n_wins) = next(iter(dl))
        xb, n_wins = xb.to(m.dev), n_wins.to(m.dev)
        m.model.to(m.dev).eval()
        with torch.no_grad():
            for _ in range(3):
                m.model(xb, n_wins)
            sync()
            if cuda:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
            t0 = time.perf_counter()
            for _ in range(model_iters):
                m.model(xb, n_wins)
            if cuda:
                e1.record()
            sync()
        ms = (e0.elapsed_time(e1) if cuda else (time.perf_counter() - t0) * 1e3) / model_iters
        out["model_only"] = {"clips_per_s": xb.shape[0] / (ms / 1e3), "ms_per_batch": ms, "batch": int(xb.shape[0]),
                             "input": "resident padded segments %s fp32 (%.0f MB)" % (list(xb.shape), xb.numel() * 4 / 1e6),
                             "tf32": "PyTorch defaults: cuDNN convolutions may use TF32 (torch.backends.cudnn.allow_tf32 = %s)"
                                     % torch.backends.cudnn.allow_tf32}
        # the same forward with TF32 switched off: the reference's fp32 arithmetic on this GPU (what its CPU path and
        # the 1e-4 parity target mean); scores of the first batch against the default (TF32) run
        if cuda:
            with torch.no_grad():
                y_tf32 = m.model(xb, n_wins).float().cpu().numpy()
                old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
                torch.backends.cudnn.allow_tf32 = False
                torch.backends.cuda.matmul.allow_tf32 = False
                try:
                    for _ in range(3):
                        y_fp32 = m.model(xb, n_wins)
                    sync()
                    e0.record()
                    for _ in range(model_iters):
                        m.model(xb, n_wins)
                    e1.record()
                    sync()
                finally:
                    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
            ms32 = e0.elapsed_time(e1) / model_iters
            y_fp32 = y_fp32.float().cpu().numpy()
            out["model_only_fp32"] = {"clips_per_s": xb.shape[0] / (ms32 / 1e3), "ms_per_batch": ms32,
                                      "max_abs_diff_vs_default_tf32_run": float(np.abs(y_fp32 - y_tf32).max())}
        if ours is not None:
            got = np.asarray(ours([os.path.join(td, f) for f in names]), dtype=np.float64)
            out["max_abs_diff_engine_vs_reference_gpu"] = float(np.abs(got - ref_scores).max())
            if cuda:
                first = [names.index(df["deg"].iloc[int(i)]) for i in idx.numpy()] if hasattr(idx, "numpy") else list(range(xb.shape[0]))
                out["max_abs_diff_engine_vs_reference_gpu_fp32"] = float(np.abs(got[first] - y_fp32.astype(np.float64)).max())
    finally:
        shutil.rmtree(td, ignore_errors=True)
    return out


def main():
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("--clips", type=int, default=64)
    ap.add_argument("--workers", type=int, default=None)
    ap.add_argument("--install", metavar="SRC", default=None,
                    help="copy SRC/nisqa of a NISQA checkout to baseline/_ref and exit")
    a = ap.parse_args()
    if a.install:
        print(json.dumps({"installed": install_reference(a.install)}))
        return
    print(json.dumps(measure(n_clips=a.clips, workers=a.workers)))


if __name__ == "__main__":
    main()
