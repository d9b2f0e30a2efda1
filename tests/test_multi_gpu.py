"""BASELINE configs[4] through the product surface on real GPUs: ``run_predict.py --mode predict_csv`` under
``torchrun`` - ``nisqaModel._loadDatasetsCSVpredict`` (reference model:811-847) -> ``NL.predict_dim`` (reference
lib:1441-1467) with the rows sharded over the ranks (``dist.shard_rows``) and ONE ``ncclAllGather`` of the score
rows through the engine (``_predict_all`` -> ``dist.all_gather_scores`` -> ``nisqa_gather_nccl``).

The gathered table must be BIT-identical to the single-process run (clips are independent units; sharding only
changes which GPU computes a row) and within 1e-4 of the oracle.  Needs >= 2 GPUs on the machine and skips
otherwise; the world_size-2 ``gloo`` twin of the host logic runs on the CPU in tests/test_host_logic.py.
"""
import os
import subprocess
import sys

import numpy as np
import pandas as pd
import pytest

from conftest import ROOT, WEIGHTS
from nisqa_b200 import synth, wav

pytestmark = pytest.mark.gpu

COLS = ["mos_pred", "noi_pred", "dis_pred", "col_pred", "loud_pred"]


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _run(cmd, timeout=150):       # (a hang must fail fast: GPU-box minutes are charged per GPU)
    env = dict(os.environ, PYTHONPATH=ROOT)
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, cwd=ROOT, env=env)
    assert r.returncode == 0, (" ".join(cmd), r.stdout[-3000:], r.stderr[-3000:])
    return r


@pytest.mark.skipif(_n_gpus() < 2, reason="needs two GPUs on the machine")
def test_predict_csv_sharded_equals_single_rank(tmp_path, built_lib):
    from oracle import nisqa_oracle as O
    rng = np.random.default_rng(3)
    specs = []
    for i in range(64):                                  # mixed lengths and sample rates: uneven shards, ragged batches
        # (short clips: the synthesiser runs on the host)
        sr = int(rng.choice([48000, 48000, 16000, 44100]))
        specs.append((1200 + i, float(rng.uniform(0.6, 2.5)), sr))
    data = tmp_path / "data"
    data.mkdir()
    for seed, sec, sr in specs:
        wav.write_wav_pcm16(str(data / ("c%04d.wav" % seed)), synth.synth_speech_pcm16(seed, sec, sr), sr)
    pd.DataFrame({"deg": ["c%04d.wav" % s for s, _, _ in specs], "con": np.arange(64) % 4}).to_csv(str(data / "files.csv"), index=False)
    common = ["--mode", "predict_csv", "--pretrained_model", os.path.join(WEIGHTS, "nisqa.tar"), "--data_dir", str(data),
              "--csv_file", "files.csv", "--csv_deg", "deg", "--bs", "8", "--num_workers", "2"]
    out1, out2 = tmp_path / "out1", tmp_path / "out2"
    out1.mkdir(); out2.mkdir()
    _run([sys.executable, os.path.join(ROOT, "run_predict.py")] + common + ["--output_dir", str(out1)])
    port = 29600 + (os.getpid() % 1500)
    _run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
          "--master-port", str(port), os.path.join(ROOT, "run_predict.py")] + common + ["--output_dir", str(out2)])
    a = pd.read_csv(str(out1 / "NISQA_results.csv"))
    b = pd.read_csv(str(out2 / "NISQA_results.csv"))
    assert list(a.columns) == list(b.columns) == ["deg", "con"] + COLS + ["model"]
    assert list(a["deg"]) == list(b["deg"]) == ["c%04d.wav" % s for s, _, _ in specs]        # csv row order kept
    # same text in both files: the float32 scores were produced by the same kernels, whichever rank ran them
    assert open(str(out1 / "NISQA_results.csv")).read() == open(str(out2 / "NISQA_results.csv")).read()
    args, sd = O.load_checkpoint(os.path.join(WEIGHTS, "nisqa.tar"))
    for i in (0, 7, 21, 40, 63):
        ref = O.predict_file(args, sd, str(data / a["deg"].iloc[i]))[0]
        assert np.abs(b[COLS].iloc[i].to_numpy(dtype=np.float64) - ref).max() <= 1e-4, i
