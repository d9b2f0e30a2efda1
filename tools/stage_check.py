"""GPU-box diagnostic: every stage of the CUDA path against the oracle taps, all errors printed
(does not stop at the first mismatch).  python tools/stage_check.py"""
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from nisqa_b200 import engine as E, synth  # noqa: E402
from oracle import nisqa_oracle as O       # noqa: E402


def check(ckpt, clips):
    args, sd = O.load_checkpoint(os.path.join(ROOT, "weights", ckpt))
    cfg = E.config_from_args(args)
    eng = E.Engine(cfg, 0)
    eng.load_state_dict(sd)
    std = args["cnn_model"] == "standard"
    pcm = [synth.synth_speech_pcm16(s, sec, sr) for (s, sec, sr) in clips]
    srs = [c[2] for c in clips]
    eng.set_option("keep_pool1", 1)       # pool1 is only written to HBM for the dump
    t0 = time.time()
    scores, nseg, status = eng.predict_pcm(pcm, srs)
    print("== %s: predict %.3fs  status=%s nseg=%s launches=%d" % (ckpt, time.time() - t0, status.tolist(), nseg.tolist(), eng.kernel_launches()))
    dumps = {k: eng.stage_dump(v) for k, v in dict(mel=E.STAGE_MEL_DB, pool1=E.STAGE_POOL1, pool2=E.STAGE_POOL2,
             conv3=E.STAGE_CONV3, pool3=E.STAGE_POOL3, conv5=E.STAGE_CONV5, feat=E.STAGE_CNN_FEAT,
             td_out=E.STAGE_TD_OUT).items()}
    if not std:
        dumps["td_in"] = eng.stage_dump(E.STAGE_TD_IN)
    off = dict((k, 0) for k in dumps)
    worst = 0.0
    for i, (p, sr) in enumerate(zip(pcm, srs)):
        taps = {}
        y = p.astype(np.float32) / 32768.0
        sc, ns, st = O.predict_pcm(args, sd, y, sr, taps)
        line = "clip %d sr=%d n=%d nseg=%d/%d" % (i, sr, len(p), nseg[i], ns)
        if st != 0:
            print(line, "status", st, status[i]); continue
        def cmp(name, ref):
            ref = np.asarray(ref, dtype=np.float32).reshape(-1)
            got = dumps[name][off[name]:off[name] + ref.size]
            off[name] += ref.size
            d = np.abs(got - ref)
            return "%s=%.2e" % (name, d.max() if d.size else 0.0)
        parts = [cmp("mel", taps["mel_db"]), cmp("pool1", taps["pool1"].numpy()), cmp("pool2", taps["pool2"].numpy()),
                 cmp("conv3", taps["conv3"].numpy()), cmp("pool3", taps["pool3"].numpy()), cmp("conv5", taps["conv5"].numpy()),
                 cmp("feat", taps["cnn_feat"].numpy())]
        if not std:
            parts.append(cmp("td_in", taps["sa_in"].numpy()))
        parts.append(cmp("td_out", taps["td_out"].numpy()))
        ds = np.abs(scores[i] - sc).max()
        worst = max(worst, ds)
        print(line, " ".join(parts), "dscore=%.2e" % ds, "scores", scores[i].tolist())
    print("worst |dscore| = %.3e" % worst)
    fb = eng.mel_filterbank(48000)
    from oracle import librosa_compat as lb
    ref = lb.mel(48000, 4096, n_mels=48, fmin=0.0, fmax=args["ms_fmax"], htk=False, norm="slaney")
    print("fbank max abs diff", np.abs(fb - ref).max(), "nnz", (fb != 0).sum(), (ref != 0).sum())
    eng.close()
    return worst


if __name__ == "__main__":
    w = 0.0
    w = max(w, check("nisqa.tar", [(1, 3.0, 48000), (2, 1.37, 48000), (3, 2.0, 16000), (4, 2.5, 44100),
                                  (5, 0.1875, 8000), (6, 1.0, 22050), (0, 10.0, 48000), (13, 0.05, 48000)]))
    w = max(w, check("nisqa_mos_only.tar", [(8, 2.2, 48000), (9, 1.0, 32000)]))
    w = max(w, check("nisqa_tts.tar", [(10, 2.0, 16000), (11, 1.3, 48000), (12, 0.9, 22050)]))
    print("OVERALL worst |dscore| = %.3e" % w)
