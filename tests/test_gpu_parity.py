"""Parity tests proper (run on a B200): the CUDA path, called through the C-ABI, against the
oracle on the same seeded inputs, against the committed reference goldens, and - at
BASELINE.json's full sizes - through size-independent properties.

Tolerances (north_star): every predicted dimension within 1e-4 of the reference path in fp32,
segment counts bit-exact.  Intermediate tolerances are stated next to each check.
"""
import os

import numpy as np
import pandas as pd
import pytest

from conftest import GOLDEN, ROOT, WEIGHTS
from nisqa_b200 import engine as E
from nisqa_b200 import synth, wav
from oracle import nisqa_oracle as O

pytestmark = pytest.mark.gpu

SCORE_TOL = 1e-4          # north_star: all five dimensions within +-1e-4
MEL_TOL_DB = 1e-3         # SURVEY.md 0.8: front-end must hold <~1e-3 dB
ACT_TOL = 2e-4            # CNN / time-dependency activations (values are O(1..10))


@pytest.fixture(scope="module")
def engines(built_lib):
    out = {}
    for ck in ("nisqa.tar", "nisqa_mos_only.tar", "nisqa_tts.tar"):
        args, sd = O.load_checkpoint(os.path.join(WEIGHTS, ck))
        eng = E.Engine(E.config_from_args(args), 0)
        eng.load_state_dict(sd)
        out[ck] = (eng, args, sd)
    yield out
    for eng, _, _ in out.values():
        eng.close()


def _f32(pcm):
    return pcm.astype(np.float32) / np.float32(32768.0)


STAGES = [("mel_db", E.STAGE_MEL_DB, MEL_TOL_DB), ("pool1", E.STAGE_POOL1, ACT_TOL), ("pool2", E.STAGE_POOL2, ACT_TOL),
          ("conv3", E.STAGE_CONV3, ACT_TOL), ("pool3", E.STAGE_POOL3, ACT_TOL), ("conv5", E.STAGE_CONV5, ACT_TOL),
          ("cnn_feat", E.STAGE_CNN_FEAT, ACT_TOL), ("td_out", E.STAGE_TD_OUT, ACT_TOL)]


@pytest.mark.parametrize("ckpt,clips", [
    ("nisqa.tar", [(1, 3.0, 48000), (2, 1.37, 48000), (3, 2.0, 16000), (4, 2.5, 44100), (5, 0.1875, 8000),
                   (6, 1.0, 22050), (21, 0.5, 96000)]),
    ("nisqa_mos_only.tar", [(8, 2.2, 48000), (9, 1.0, 32000)]),
    ("nisqa_tts.tar", [(10, 2.0, 16000), (11, 1.3, 48000), (12, 0.9, 22050)]),
])
def test_stage_dumps_match_oracle(engines, ckpt, clips):
    eng, args, sd = engines[ckpt]
    pcm = [synth.synth_speech_pcm16(s, sec, sr) for s, sec, sr in clips]
    srs = [c[2] for c in clips]
    eng.set_option("keep_td_out", 1)              # BiLSTM: per-step outputs are only stored for the dump
    eng.set_option("keep_pool1", 1)               # pool1 is only written to HBM for the dump
    try:
        scores, nseg, status = eng.predict_pcm(pcm, srs)
    finally:
        eng.set_option("keep_td_out", 0)
        eng.set_option("keep_pool1", 0)
    assert np.all(status == E.CLIP_OK)
    dumps = {name: eng.stage_dump(st) for name, st, _ in STAGES}
    off = {name: 0 for name, _, _ in STAGES}
    for i, (p, sr) in enumerate(zip(pcm, srs)):
        taps = {}
        ref, ns, st = O.predict_pcm(args, sd, _f32(p), sr, taps)
        assert st == O.STATUS_OK and int(nseg[i]) == ns            # bit-exact segment count
        for name, _, tol in STAGES:
            r = np.asarray(taps[name].numpy() if hasattr(taps[name], "numpy") else taps[name], dtype=np.float32).reshape(-1)
            g = dumps[name][off[name]:off[name] + r.size]
            off[name] += r.size
            assert g.size == r.size
            assert np.abs(g - r).max() <= tol, (ckpt, i, name, float(np.abs(g - r).max()))
        assert np.abs(scores[i] - ref).max() <= SCORE_TOL
    for name, _, _ in STAGES:
        assert off[name] == dumps[name].size                        # no extra rows anywhere


@pytest.mark.parametrize("name,ckpt", [("nisqa_48k_3s", "nisqa.tar"), ("nisqa_mixed", "nisqa.tar"),
                                       ("nisqa_48k_10s", "nisqa.tar"), ("mos_only_48k", "nisqa_mos_only.tar"),
                                       ("tts_16k", "nisqa_tts.tar")])
def test_scores_match_reference_goldens(engines, name, ckpt):
    """tests/golden/*.npz hold the outputs of the unmodified reference (oracle/make_golden.py)."""
    eng, _, _ = engines[ckpt]
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    pcm = [synth.synth_speech_pcm16(int(s), float(sec), int(sr)) for s, sec, sr in zip(g["seeds"], g["seconds"], g["sr"])]
    scores, nseg, status = eng.predict_pcm(pcm, [int(x) for x in g["sr"]])
    assert np.all(status == 0)
    np.testing.assert_array_equal(nseg, g["n_segments"].astype(np.int32))
    assert np.abs(scores - g["scores"]).max() <= SCORE_TOL


def test_filterbank_matches_oracle(engines):
    from oracle import librosa_compat as lb
    for ck, fmax in (("nisqa.tar", 20000), ("nisqa_tts.tar", 8000)):
        eng = engines[ck][0]
        for sr in (48000, 44100, 16000, 8000):
            ref = lb.mel(sr, 4096, n_mels=48, fmin=0.0, fmax=fmax, htk=False, norm="slaney")
            np.testing.assert_allclose(eng.mel_filterbank(sr), ref, rtol=0, atol=1e-7)


def test_edge_inputs(engines):
    eng, args, sd = engines["nisqa.tar"]
    sr = 48000
    silence = np.zeros(48000, np.int16)                            # every band at the -80 dB floor
    full = (np.sign(np.sin(np.arange(96000) * 0.05)) * 32767).astype(np.int16)   # full-scale square
    shortest = synth.synth_speech_pcm16(31, 14 * 480 / sr, sr)     # exactly 15 frames -> 1 segment
    too_short = shortest[:-1]                                       # 14 frames
    f32clip = synth.synth_speech_f32(32, 1.0, sr)
    scores, nseg, status = eng.predict_pcm([_f32(silence), _f32(full), _f32(shortest), _f32(too_short), f32clip], [sr] * 5)
    assert status.tolist() == [0, 0, 0, E.CLIP_TOO_SHORT, 0]
    assert nseg.tolist()[:3] == [22, 47, 1] and nseg[3] == 0
    assert np.all(np.isnan(scores[3]))
    for i, y in ((0, _f32(silence)), (1, _f32(full)), (2, _f32(shortest)), (4, f32clip)):
        ref, ns, st = O.predict_pcm(args, sd, y, sr)
        assert ns == nseg[i] and np.abs(scores[i] - ref).max() <= SCORE_TOL, i
    mel = eng.stage_dump(E.STAGE_MEL_DB)
    assert np.all(mel[:48 * 101] == -80.0)                          # digital silence: floor everywhere


def test_max_length_and_too_long(engines):
    eng, args, sd = engines["nisqa.tar"]
    sr = 16000                                                      # 52 s at 16 kHz keeps the oracle quick
    ok = synth.synth_speech_pcm16(41, 52.0, sr)
    long_ = synth.synth_speech_pcm16(42, 52.2, sr)
    scores, nseg, status = eng.predict_pcm([ok, long_], [sr, sr])
    assert status.tolist() == [0, E.CLIP_TOO_LONG] and nseg.tolist() == [1297, 1302]
    ref, ns, st = O.predict_pcm(args, sd, _f32(ok), sr)
    assert ns == 1297 and np.abs(scores[0] - ref).max() <= SCORE_TOL
    assert np.all(np.isnan(scores[1]))


def test_ragged_batch_config3(engines):
    """configs[2]: mixed 2-30 s clips in one call (ragged path, no padding anywhere)."""
    eng, args, sd = engines["nisqa.tar"]
    durs = synth.ragged_durations(24, 2.0, 30.0, seed=7)
    pcm = [synth.synth_speech_pcm16(200 + i, float(d), 48000) for i, d in enumerate(durs)]
    scores, nseg, status = eng.predict_pcm(pcm, [48000] * len(pcm))
    assert np.all(status == 0)
    for i in (0, 5, 11, 17, 23, int(np.argmax(durs)), int(np.argmin(durs))):
        ref, ns, st = O.predict_pcm(args, sd, _f32(pcm[i]), 48000)
        assert ns == nseg[i] and np.abs(scores[i] - ref).max() <= SCORE_TOL, i


def test_tts_config4_full_length(engines):
    """configs[3]: nisqa_tts.tar on 10 s 16 kHz clips (987 segments, 987 serial LSTM steps)."""
    eng, args, sd = engines["nisqa_tts.tar"]
    pcm = [synth.synth_speech_pcm16(300 + i, 10.0, 16000) for i in range(3)]
    scores, nseg, status = eng.predict_pcm(pcm, [16000] * 3)
    assert nseg.tolist() == [987] * 3 and np.all(status == 0)
    ref, ns, st = O.predict_pcm(args, sd, _f32(pcm[1]), 16000)
    assert np.abs(scores[1] - ref).max() <= SCORE_TOL


def test_full_size_properties_config2(engines):
    """BASELINE configs[1] at full size (64 x 10 s x 48 kHz): size-independent properties.
    Per-clip arithmetic does not depend on batch composition, position or pass splitting, so
    these must hold BIT-EXACTLY; one clip is also checked against the reference golden."""
    eng, args, sd = engines["nisqa.tar"]
    base = [synth.synth_speech_pcm16(400 + i, 10.0, 48000) for i in range(8)]
    rng = np.random.default_rng(0)
    clips = [base[i % 8] if i < 8 else np.roll(base[i % 8], int(rng.integers(1, 400000))) for i in range(62)]
    clips += [synth.synth_speech_pcm16(0, 10.0, 48000), base[3]]      # golden clip + a duplicate
    srs = [48000] * 64
    s1, n1, st1 = eng.predict_pcm(clips, srs)
    assert np.all(st1 == 0) and np.all(n1 == 247)
    g = np.load(os.path.join(GOLDEN, "nisqa_48k_10s.npz"))
    assert np.abs(s1[62] - g["scores"][0]).max() <= SCORE_TOL           # vs the reference itself
    np.testing.assert_array_equal(s1[63], s1[3])                        # duplicates -> identical rows
    perm = rng.permutation(64)
    s2, _, _ = eng.predict_pcm([clips[j] for j in perm], srs)
    np.testing.assert_array_equal(s2, s1[perm])                         # permutation equivariance
    s3, _, _ = eng.predict_pcm([clips[62]], [48000])
    np.testing.assert_array_equal(s3[0], s1[62])                        # alone == inside the batch
    # multi-pass engine (4000 segments per pass -> 4 passes) == single pass
    cfg = E.config_from_args(args, max_chunk_segments=4000)
    e2 = E.Engine(cfg, 0)
    e2.load_state_dict(sd)
    s4, n4, _ = e2.predict_pcm(clips, srs)
    e2.close()
    np.testing.assert_array_equal(s4, s1)
    assert np.all(np.isfinite(s1)) and s1.min() > 0.0 and s1.max() < 6.0



def _sliced_clips(durations, sr, seed):
    """Distinct clips of the given durations cut out of a few 30-s synthetic bases (synthesis cost stays bounded)."""
    bases = [synth.synth_speech_pcm16(900 + i, 30.0, sr) for i in range(8)]
    rng = np.random.default_rng(seed)
    clips = []
    for i, d in enumerate(durations):
        n = int(round(float(d) * sr))
        st = int(rng.integers(0, len(bases[0]) - n + 1))
        clips.append(bases[i % 8][st:st + n])
    return clips


def _check_full_size(eng, args, sd, clips, sr, sample_idx):
    cfg = E.config_from_args(args)
    srs = [sr] * len(clips)
    scores, nseg, status = eng.predict_pcm(clips, srs)
    assert np.all(status == E.CLIP_OK) and np.all(np.isfinite(scores))
    want = np.array([E.segment_counts(cfg, len(c), sr)[1] for c in clips], np.int32)
    np.testing.assert_array_equal(nseg, want)                          # every segment count, exactly
    worst = 0.0
    for i in sample_idx:
        ref, ns, st = O.predict_pcm(args, sd, _f32(clips[i]), sr)
        assert st == O.STATUS_OK and ns == nseg[i]
        worst = max(worst, float(np.abs(scores[i] - ref).max()))
        assert worst <= SCORE_TOL, (i, worst)
    return scores, nseg, worst


def test_config3_full_size_ragged_bs512(engines):
    """BASELINE configs[2] at FULL size: 512 clips of U(2,30) s at 48 kHz in ONE call = 7 internal passes of
    <= 32768 segments, the last one smaller than the others (the shape that exposed the lo-plane offset bug of
    round 1).  Eight sampled clips against the oracle (<= 1e-4), all 512 segment counts exact, and the
    pass-splitting properties bit-exact: a clip alone == inside the batch, and the reversed batch (different
    pass boundaries, different plane rows) == the same rows."""
    _, args, sd = engines["nisqa.tar"]
    eng = E.Engine(E.config_from_args(args, max_chunk_segments=32768), 0)      # 7 passes (the default pass is 131072 segments)
    eng.load_state_dict(sd)
    durs = synth.ragged_durations(512, 2.0, 30.0, seed=11)
    clips = _sliced_clips(durs, 48000, seed=5)
    order = np.argsort(durs)
    sample = [int(order[0]), int(order[3]), int(order[-1]), 0, 100, 255, 400, 511]     # shortest, longest, spread over the passes
    scores, nseg, worst = _check_full_size(eng, args, sd, clips, 48000, sample)
    assert int(nseg.sum()) > 6 * 32768                                  # really a multi-pass call
    for i in (sample[0], sample[2], 511):
        alone, _, _ = eng.predict_pcm([clips[i]], [48000])
        np.testing.assert_array_equal(alone[0], scores[i])
    rev, nrev, _ = eng.predict_pcm(clips[::-1], [48000] * 512)
    np.testing.assert_array_equal(rev[::-1], scores)
    eng.close()
    big, nbig, _ = engines["nisqa.tar"][0].predict_pcm(clips, [48000] * 512)     # default pass size: 2 passes
    np.testing.assert_array_equal(big, scores)
    print("configs[2] full size: max |d| vs oracle over %d sampled clips = %.2e, %d segments" % (len(sample), worst, int(nseg.sum())))


def test_config4_full_size_tts_bs256(engines):
    """BASELINE configs[3] at FULL size: nisqa_tts.tar, 256 clips of 10 s at 16 kHz (987 segments each) in one
    call = 8 passes.  Eight sampled clips against the oracle, all segment counts exact, alone == in-batch."""
    _, args, sd = engines["nisqa_tts.tar"]
    eng = E.Engine(E.config_from_args(args, max_chunk_segments=32768), 0)      # 8 passes of 33 clips (the last one: 25)
    eng.load_state_dict(sd)
    clips = _sliced_clips([10.0] * 256, 16000, seed=6)
    sample = [0, 33, 66, 99, 132, 200, 254, 255]
    scores, nseg, worst = _check_full_size(eng, args, sd, clips, 16000, sample)
    assert np.all(nseg == 987) and int(nseg.sum()) > 7 * 32768
    for i in (0, 132, 255):
        alone, _, _ = eng.predict_pcm([clips[i]], [16000])
        np.testing.assert_array_equal(alone[0], scores[i])
    eng.close()
    big, _, _ = engines["nisqa_tts.tar"][0].predict_pcm(clips, [16000] * 256)     # default pass size: 2 passes of 128 clips
    np.testing.assert_array_equal(big, scores)
    print("configs[3] full size: max |d| vs oracle over %d sampled clips = %.2e" % (len(sample), worst))

@pytest.mark.parametrize("ckpt,clips", [
    ("nisqa.tar", [(31, 10.0, 48000), (32, 2.3, 48000), (33, 4.0, 16000), (34, 0.1875, 8000)]),
    ("nisqa_tts.tar", [(35, 3.0, 16000), (36, 1.1, 48000)]),
])
def test_keep_pool1_and_plane_reuse(engines, ckpt, clips):
    """keep_pool1 only adds a store of pool1 for the stage dump: scores and the pool2 / pool3 / CNN-feature dumps are
    BIT-identical with it on and off.  Growing / shrinking batches reuse the zero-padded planes (stale rows of earlier,
    larger passes must not leak)."""
    eng, args, sd = engines[ckpt]
    pcm = [synth.synth_speech_pcm16(s, sec, sr) for s, sec, sr in clips]
    srs = [c[2] for c in clips]
    out = {}
    try:
        for keep in (0, 1):
            eng.set_option("keep_pool1", keep)
            sc, nseg, st = eng.predict_pcm(pcm, srs)
            out[keep] = (sc.copy(), eng.stage_dump(E.STAGE_CNN_FEAT), eng.stage_dump(E.STAGE_POOL3), eng.stage_dump(E.STAGE_POOL2))
        eng.set_option("keep_pool1", 0)
        for i in range(4):
            np.testing.assert_array_equal(out[0][i], out[1][i])
        # shrink, then grow again: same rows as in the first call
        s_small, _, _ = eng.predict_pcm(pcm[1:2], srs[1:2])
        np.testing.assert_array_equal(s_small[0], out[0][0][1])
        s_again, _, _ = eng.predict_pcm(pcm[::-1], srs[::-1])
        np.testing.assert_array_equal(s_again[::-1], out[0][0])
    finally:
        eng.set_option("keep_pool1", 0)


def test_removed_kernel_switches_are_rejected(engines):
    """Each stage has one implementation: the former A/B switches are unknown options, not silent no-ops."""
    eng = engines["nisqa.tar"][0]
    for name in ("conv_tc", "conv_split", "conv_pipe", "conv12", "lstm_batched", "td_tiled"):
        with pytest.raises(E.EngineError, match="unknown option"):
            eng.set_option(name, 1)


def test_batched_lstm_matches_oracle(engines):
    """Batched BiLSTM (NB clips of one direction per CTA, sorted by length) against the oracle: ragged lengths inside a
    group, a too-short clip (no segments) and batch sizes that select the NB = 1, 2 and 4 variants."""
    eng, args, sd = engines["nisqa_tts.tar"]
    spec = [(61, 10.0, 16000), (62, 0.5, 16000), (63, 3.3, 48000), (64, 0.01, 16000), (65, 6.1, 22050), (66, 2.0, 16000), (67, 1.1, 8000)]
    base = [synth.synth_speech_pcm16(s, sec, sr) for s, sec, sr in spec]
    ref = [O.predict_pcm(args, sd, _f32(p), sr)[0] for p, (_, _, sr) in zip(base, spec)]     # once per distinct clip
    for reps in (1, 25, 50):                      # 7, 175, 350 clips -> 14, 350, 700 sequences: NB = 1, 4 (> 296) / 2
        pcm = base * reps
        srs = [c[2] for c in spec] * reps
        s1, n1, st1 = eng.predict_pcm(pcm, srs)
        ok = st1 == E.CLIP_OK
        assert np.all(np.isnan(s1[~ok]))
        for i in np.nonzero(ok)[0]:
            assert np.abs(s1[i] - ref[i % 7]).max() <= SCORE_TOL, (reps, int(i), float(np.abs(s1[i] - ref[i % 7]).max()))
        assert st1[3] == E.CLIP_TOO_SHORT and np.isnan(s1[3, 0])
        np.testing.assert_array_equal(s1[:7], s1[7 * (reps - 1):])     # the same clip scores the same in any group
    pcm = base[:5] * 30                              # 150 clips -> 300 sequences: NB = 4
    s, _, _ = eng.predict_pcm(pcm, [c[2] for c in spec][:5] * 30)
    np.testing.assert_array_equal(s[:5], s[145:])


def test_architecture_variants(built_lib):
    """SURVEY.md 8f.4: PoolAtt / PoolAvg / PoolMax / PoolLastStep after self-attention and after the BiLSTM, and the
    positional encoding - against the oracle AND against the scores of the unmodified reference modules
    (tests/golden/variants.npz), in one batch and alone."""
    from oracle import variants as V
    g = np.load(os.path.join(GOLDEN, "variants.npz"))
    pcm = [synth.synth_speech_pcm16(s, sec, sr) for s, sec, sr in V.CLIPS]
    srs = [c[2] for c in V.CLIPS]
    for name, (base, _) in V.VARIANTS.items():
        bargs, bsd = O.load_checkpoint(os.path.join(WEIGHTS, base))
        args, sd = V.variant_checkpoint(name, bargs, bsd)
        eng = E.Engine(E.config_from_args(args), 0)
        eng.load_state_dict(sd)
        scores, nseg, status = eng.predict_pcm(pcm, srs)
        assert np.all(status == E.CLIP_OK), name
        assert np.abs(scores - g[name]).max() <= SCORE_TOL, (name, float(np.abs(scores - g[name]).max()))
        for i, (p, sr) in enumerate(zip(pcm, srs)):
            ref, ns, st = O.predict_pcm(args, sd, _f32(p), sr)
            assert ns == nseg[i] and np.abs(scores[i] - ref).max() <= SCORE_TOL, (name, i)
        alone, _, _ = eng.predict_pcm(pcm[1:2], srs[1:2])
        np.testing.assert_array_equal(alone[0], scores[1])
        eng.close()


def test_double_ended_model(built_lib, tmp_path):
    """SURVEY.md 8f.4: NISQA_DE through the C-ABI (clips in (degraded, reference) pairs) against the scores of the
    unmodified reference model (tests/golden/variants_de.npz) and the oracle; pair alone == pair in the batch; a
    too-short reference makes the pair NaN with the status on the right clip; and the product surface:
    nisqaModel(mode='predict_csv', csv_ref=...) on a checkpoint file."""
    import pandas as pd
    import torch
    from oracle import variants as V
    from nisqa_b200 import wav
    from nisqa_b200.NISQA_model import nisqaModel
    g = np.load(os.path.join(GOLDEN, "variants_de.npz"))
    bargs, bsd = O.load_checkpoint(os.path.join(WEIGHTS, "nisqa_mos_only.tar"))
    pairs = [V.de_pair_pcm(p) for p in V.DE_PAIRS]
    clips, srs = [], []
    for deg, srd, ref, srr in pairs:
        clips += [deg, ref]; srs += [srd, srr]
    for name in V.DE_VARIANTS:
        args, sd = V.de_checkpoint(name, bargs, bsd)
        eng = E.Engine(E.config_from_args(args), 0)
        eng.load_state_dict(sd)
        scores, nseg, status = eng.predict_pcm(clips, srs)
        assert np.all(status == E.CLIP_OK), name
        assert np.all(np.isnan(scores[1::2])), name                       # reference rows carry no score
        got = scores[0::2, 0]
        # hard alignment picks ONE reference step per degraded step: a near-tie decided differently moves the score by
        # more than rounding, so the hard variants get a looser bound than the soft ones (same budget as everywhere)
        tol = SCORE_TOL if args["de_align_apply"] == "soft" else 5 * SCORE_TOL
        assert np.abs(got - g[name][:, 0]).max() <= tol, (name, got, g[name][:, 0])
        for i, (deg, srd, ref, srr) in enumerate(pairs):
            sc, ns, st = O.predict_pcm_de(args, sd, _f32(deg), srd, _f32(ref), srr)
            assert (nseg[2 * i], nseg[2 * i + 1]) == ns and abs(got[i] - sc[0]) <= tol, (name, i)
        alone, _, _ = eng.predict_pcm(clips[2:4], srs[2:4])
        np.testing.assert_array_equal(alone[0], scores[2])
        short = np.zeros(100, np.int16)
        s2, _, st2 = eng.predict_pcm([clips[0], short, clips[2], clips[3]], [srs[0], 48000, srs[2], srs[3]])
        assert st2[1] == E.CLIP_TOO_SHORT and st2[0] == E.CLIP_OK and np.isnan(s2[0, 0])
        np.testing.assert_array_equal(s2[2], scores[2])
        with pytest.raises(E.EngineError):
            eng.predict_pcm(clips[:3], srs[:3])                            # odd number of clips
        eng.close()
    # product surface
    name = "de_cosine_hard"
    args, sd = V.de_checkpoint(name, bargs, bsd)
    rows = []
    for i, (deg, srd, ref, srr) in enumerate(pairs):
        wav.write_wav_pcm16(str(tmp_path / ("deg%d.wav" % i)), deg, srd)
        wav.write_wav_pcm16(str(tmp_path / ("ref%d.wav" % i)), ref, srr)
        rows.append(("deg%d.wav" % i, "ref%d.wav" % i))
    pd.DataFrame(rows, columns=["deg", "ref"]).to_csv(tmp_path / "files.csv", index=False)
    torch.save({"args": args, "model_state_dict": sd}, tmp_path / "de.tar")
    m = nisqaModel({"mode": "predict_csv", "pretrained_model": str(tmp_path / "de.tar"), "csv_file": "files.csv",
                    "csv_deg": "deg", "csv_ref": "ref", "data_dir": str(tmp_path), "output_dir": None, "ms_channel": None,
                    "tr_bs_val": 2, "tr_num_workers": 0})
    df = m.predict()
    assert df["mos_pred"].dtype == np.float64
    assert np.abs(df["mos_pred"].to_numpy() - g[name][:, 0]).max() <= 5 * SCORE_TOL
    m.model.close()


def test_device_resident_entry_point_equals_host_entry_point(engines):
    import torch
    eng, args, sd = engines["nisqa.tar"]
    clips = [synth.synth_speech_pcm16(500 + i, 2.0 + 0.37 * i, 48000) for i in range(5)]
    s_host, n_host, _ = eng.predict_pcm(clips, [48000] * 5)
    offs, tot = [], 0
    for c in clips:
        offs.append(tot); tot += (len(c) + 15) // 16 * 16
    buf = np.zeros(tot, np.int16)
    for o, c in zip(offs, clips):
        buf[o:o + len(c)] = c
    d = torch.from_numpy(buf).cuda()
    out = torch.empty((5, 5), dtype=torch.float32, device="cuda")
    nseg, status = eng.predict_pcm_device(d.data_ptr(), offs, [len(c) for c in clips], [48000] * 5, E.FMT_S16, out.data_ptr(), sync=True)
    np.testing.assert_array_equal(out.cpu().numpy(), s_host)
    np.testing.assert_array_equal(nseg, n_host)
    assert eng.kernel_launches() > 0


def test_single_rank_nccl_gather(engines):
    import torch
    eng = engines["nisqa.tar"][0]
    eng.nccl_init(1, 0, eng.nccl_unique_id())
    loc = torch.arange(15, dtype=torch.float32, device="cuda").reshape(3, 5)
    glob = torch.zeros((1, 3, 5), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    eng.gather_nccl(loc.data_ptr(), 3, glob.data_ptr())
    np.testing.assert_array_equal(glob[0].cpu().numpy(), loc.cpu().numpy())


# ------------------------------------------------------------------ the reference-facing surface
@pytest.fixture(scope="module")
def wav_dir(tmp_path_factory):
    d = tmp_path_factory.mktemp("wavs")
    specs = [(601, 2.0, 48000), (602, 3.1, 16000), (603, 1.2, 44100), (604, 4.0, 48000)]
    for seed, sec, sr in specs:
        wav.write_wav_pcm16(str(d / ("c%d.wav" % seed)), synth.synth_speech_pcm16(seed, sec, sr), sr)
    st = np.stack([synth.synth_speech_pcm16(605, 1.5, 48000), synth.synth_speech_pcm16(606, 1.5, 48000)], axis=1)
    os.makedirs(str(d / "stereo"))
    wav.write_wav_pcm16(str(d / "stereo" / "s.wav"), st, 48000)
    wav.write_wav_f32(str(d / "stereo" / "f.wav"), synth.synth_speech_f32(607, 1.0, 32000), 32000)
    pd.DataFrame({"deg": ["c%d.wav" % s for s, _, _ in specs], "con": [1, 1, 2, 2]}).to_csv(str(d / "files.csv"), index=False)
    return d


def _oracle_file(ckpt, path, ms_channel=None):
    args, sd = O.load_checkpoint(os.path.join(WEIGHTS, ckpt))
    return O.predict_file(args, sd, path, ms_channel)[0]


def test_predict_dir_csv_file_modes(wav_dir, built_lib, capsys):
    from nisqa_b200.NISQA_model import nisqaModel
    import run_predict
    out_dir = str(wav_dir / "out"); os.makedirs(out_dir, exist_ok=True)
    a = run_predict.parse_args(["--mode", "predict_dir", "--pretrained_model", os.path.join(WEIGHTS, "nisqa.tar"),
                                "--data_dir", str(wav_dir), "--bs", "3", "--num_workers", "2", "--output_dir", out_dir])
    df = nisqaModel(a).predict()
    assert list(df.columns) == ["deg", "mos_pred", "noi_pred", "dis_pred", "col_pred", "loud_pred", "model"]
    assert sorted(df["deg"]) == ["c601.wav", "c602.wav", "c603.wav", "c604.wav"] and set(df["model"]) == {"NISQAv2"}
    assert df["mos_pred"].dtype == np.float32
    csv = pd.read_csv(os.path.join(out_dir, "NISQA_results.csv"))
    assert list(csv.columns) == list(df.columns)
    for _, row in df.iterrows():                                        # join on 'deg' (glob order is arbitrary)
        ref = _oracle_file("nisqa.tar", str(wav_dir / row["deg"]))
        got = row[["mos_pred", "noi_pred", "dis_pred", "col_pred", "loud_pred"]].to_numpy(dtype=np.float64)
        assert np.abs(got - ref).max() <= SCORE_TOL
    assert "---> Predicting ..." in capsys.readouterr().out
    # predict_csv with the mos-only checkpoint: float64 column, no 'model' column without output_dir
    a = run_predict.parse_args(["--mode", "predict_csv", "--pretrained_model", os.path.join(WEIGHTS, "nisqa_mos_only.tar"),
                                "--data_dir", str(wav_dir), "--csv_file", "files.csv", "--csv_deg", "deg", "--bs", "8"])
    df = nisqaModel(a).predict()
    assert list(df.columns) == ["deg", "con", "mos_pred"] and df["mos_pred"].dtype == np.float64
    for _, row in df.iterrows():
        assert abs(row["mos_pred"] - _oracle_file("nisqa_mos_only.tar", str(wav_dir / row["deg"]))[0]) <= SCORE_TOL
    # predict_file with the TTS checkpoint
    a = run_predict.parse_args(["--mode", "predict_file", "--pretrained_model", os.path.join(WEIGHTS, "nisqa_tts.tar"),
                                "--deg", str(wav_dir / "c602.wav")])
    df = nisqaModel(a).predict()
    assert len(df) == 1 and abs(df["mos_pred"].iloc[0] - _oracle_file("nisqa_tts.tar", str(wav_dir / "c602.wav"))[0]) <= SCORE_TOL


def test_stereo_channel_pick_and_float_wav(wav_dir, built_lib):
    from nisqa_b200.NISQA_model import nisqaModel
    base = {"mode": "predict_dir", "pretrained_model": os.path.join(WEIGHTS, "nisqa.tar"), "data_dir": str(wav_dir / "stereo"),
            "output_dir": None, "tr_bs_val": 4, "tr_num_workers": 0}
    for ch in (None, 0, 1):
        df = nisqaModel(dict(base, ms_channel=ch)).predict()
        for _, row in df.iterrows():
            ref = _oracle_file("nisqa.tar", str(wav_dir / "stereo" / row["deg"]), ch)
            got = row[["mos_pred", "noi_pred", "dis_pred", "col_pred", "loud_pred"]].to_numpy(dtype=np.float64)
            assert np.abs(got - ref).max() <= SCORE_TOL, (ch, row["deg"])


def test_ms_sr_checkpoint_resamples_on_ingest(wav_dir, built_lib):
    """A checkpoint whose args carry ms_sr (here: forced through the caller's dict, model:941-942): every file
    is converted to that rate before the engine sees it, like lb.load(path, sr=ms_sr) at lib:2300-2304."""
    from nisqa_b200.NISQA_model import nisqaModel
    df = nisqaModel({"mode": "predict_dir", "pretrained_model": os.path.join(WEIGHTS, "nisqa.tar"), "data_dir": str(wav_dir),
                     "output_dir": None, "tr_bs_val": 3, "tr_num_workers": 2, "ms_sr": 16000}).predict()
    args, sd = O.load_checkpoint(os.path.join(WEIGHTS, "nisqa.tar"))
    args = dict(args, ms_sr=16000)
    for _, row in df.iterrows():
        ref = O.predict_file(args, sd, str(wav_dir / row["deg"]))[0]
        got = row[["mos_pred", "noi_pred", "dis_pred", "col_pred", "loud_pred"]].to_numpy(dtype=np.float64)
        assert np.abs(got - ref).max() <= SCORE_TOL, row["deg"]


def test_device_resampler_is_bit_identical_to_the_host_resampler(engines, wav_dir, monkeypatch):
    """SURVEY.md 8f.2: csrc/resample_gpu.cu against csrc/resample.cpp (itself bit-identical to the oracle's restatement
    of resampy 'kaiser_best', tests/test_resample.py): up- and down-sampling, rational and awkward ratios, PCM16 and
    float input, lengths around the 256-sample chunks; then the product surface with the host path selected."""
    from nisqa_b200 import resample as RS
    from nisqa_b200.NISQA_model import nisqaModel
    eng = engines["nisqa.tar"][0]
    cases = [(48000, 16000, 1.3), (16000, 48000, 0.7), (44100, 48000, 1.0), (48000, 44100, 0.9), (8000, 22050, 0.5),
             (32000, 32000, 0.4), (48000, 8000, 0.31), (22050, 16000, 0.77)]
    for sr0, sr1, sec in cases:
        x = synth.synth_speech_pcm16(900 + sr0 // 1000, sec, sr0)
        for xin in (x, synth.synth_speech_f32(901 + sr1 // 1000, sec, sr0)[:len(x) - 3]):
            host = RS.resample(xin, sr0, sr1)
            dev = eng.resample_device(xin, sr0, sr1)
            assert dev.shape == host.shape, (sr0, sr1)
            np.testing.assert_array_equal(dev, host, err_msg="%d -> %d" % (sr0, sr1))
    a = {"mode": "predict_dir", "pretrained_model": os.path.join(WEIGHTS, "nisqa.tar"), "data_dir": str(wav_dir),
         "output_dir": None, "tr_bs_val": 3, "tr_num_workers": 2, "ms_sr": 16000}
    dev = nisqaModel(dict(a)).predict().sort_values("deg")
    monkeypatch.setenv("NISQA_RESAMPLE", "host")
    host = nisqaModel(dict(a)).predict().sort_values("deg")
    cols = ["mos_pred", "noi_pred", "dis_pred", "col_pred", "loud_pred"]
    np.testing.assert_array_equal(dev[cols].to_numpy(), host[cols].to_numpy())


def test_run_evaluate_end_to_end(tmp_path, built_lib, capsys):
    """SURVEY.md 8f.3: run_evaluate.py's flow (predict_csv on a labelled per-file table + per-condition table, then
    evaluate()) on the GPU engine: the printed report and the statistics equal nisqa_b200.evaluate applied to the
    ORACLE's scores of the same files (the statistics themselves are pinned to the reference's functions by
    tests/golden/eval_golden.json, tests/test_evaluate.py)."""
    import run_evaluate
    from nisqa_b200 import evaluate as EV
    from nisqa_b200.NISQA_model import nisqaModel
    rng = np.random.default_rng(11)
    args, sd = O.load_checkpoint(os.path.join(WEIGHTS, "nisqa.tar"))
    rows = []
    for i in range(12):
        seed, sec, sr = 700 + i, 1.0 + 0.2 * (i % 5), (48000, 16000, 32000)[i % 3]
        pcm = synth.synth_speech_pcm16(seed, sec, sr)
        if i % 4 == 3:
            pcm = np.clip(pcm.astype(np.int32) * 6, -32768, 32767).astype(np.int16)      # a distorted condition
        wav.write_wav_pcm16(str(tmp_path / ("e%02d.wav" % i)), pcm, sr)
        ref = O.predict_pcm(args, sd, _f32(pcm), sr)[0]
        rows.append(dict(deg="e%02d.wav" % i, db="db%d" % (i // 6), con=1 + (i % 6) // 2, oracle=ref,
                         **{k: float(np.clip(v + rng.normal(0, 0.15), 1, 5)) for k, v in zip(("mos", "noi", "dis", "col", "loud"), ref)}))
    dfile = pd.DataFrame(rows)
    dcon = dfile.groupby(["db", "con"], as_index=False)[["mos", "noi", "dis", "col", "loud"]].mean()
    for k in ("mos", "noi", "dis", "col", "loud"):
        dcon[k + "_ci"] = 0.2
    dfile.drop(columns=["oracle"]).to_csv(tmp_path / "file.csv", index=False)
    dcon.to_csv(tmp_path / "con.csv", index=False)
    a = run_evaluate.parse_args(["--pretrained_model", os.path.join(WEIGHTS, "nisqa.tar"), "--data_dir", str(tmp_path),
                                 "--csv_file", "file.csv", "--csv_con", "con.csv", "--csv_deg", "deg", "--bs", "5", "--num_workers", "2"])
    mapping = a.pop("mapping"); a.pop("plot")
    m = nisqaModel(a)
    df = m.predict()
    capsys.readouterr()
    m.evaluate(mapping=mapping, do_print=True, do_plot=False)
    out = capsys.readouterr().out
    assert "--> MOS:" in out and "--> LOUD:" in out and "Average over MOS and dimensions" in out
    got = df[["mos_pred", "noi_pred", "dis_pred", "col_pred", "loud_pred"]].to_numpy()
    want = np.stack(dfile["oracle"].to_numpy())
    assert np.abs(got - want).max() <= SCORE_TOL
    # the statistics of the engine's table == the statistics of the oracle's table (same labels) to the score tolerance
    dref = dfile.drop(columns=["oracle"]).copy()
    for j, k in enumerate(("mos", "noi", "dis", "col", "loud")):
        dref[k + "_pred"] = want[:, j]
    _, r_ref = EV.eval_results(dref, dcon=dcon, target_mos="mos", target_ci="mos_ci", pred="mos_pred", mapping="first_order")
    for key in ("r_p_mean_file", "rmse_mean_file", "r_p_mean_con", "rmse_mean_con", "rmse_star_map_mean_con"):
        assert abs(m.r[key] - r_ref[key]) <= 2e-3, (key, m.r[key], r_ref[key])
    m.model.close()


def test_flac_files_score_like_their_wav_twins(tmp_path, built_lib):
    """SURVEY.md 8f.1: a FLAC file (native reader csrc/flac.cpp; test encoder tests/flac_enc.py) goes through predict_csv
    like a wav file and scores bit-identically to the wav holding the same samples (mono 16-bit stays int16 on the way to the
    GPU; the 24-bit stereo file takes the float32 mono-mix path in both containers)."""
    import flac_enc as FE
    from nisqa_b200.NISQA_model import nisqaModel
    a = synth.synth_speech_pcm16(801, 1.4, 48000)
    wav.write_wav_pcm16(str(tmp_path / "a.wav"), a, 48000)
    open(str(tmp_path / "a.flac"), "wb").write(FE.encode(a, 48000, 16))
    st = np.stack([synth.synth_speech_pcm16(802, 1.1, 16000), synth.synth_speech_pcm16(803, 1.1, 16000)], axis=1)
    wav.write_wav_pcm16(str(tmp_path / "s.wav"), st, 16000)
    open(str(tmp_path / "s.flac"), "wb").write(FE.encode(st, 16000, 16, blocksize=1152, plan=lambda f, c: ("ms", "ls", "rs", "indep")[f % 4] if c is None else {"kind": "auto"}))
    pd.DataFrame({"deg": ["a.wav", "a.flac", "s.wav", "s.flac"]}).to_csv(str(tmp_path / "f.csv"), index=False)
    df = nisqaModel({"mode": "predict_csv", "pretrained_model": os.path.join(WEIGHTS, "nisqa.tar"), "data_dir": str(tmp_path),
                     "csv_file": "f.csv", "csv_deg": "deg", "output_dir": None, "tr_bs_val": 4, "tr_num_workers": 2}).predict()
    cols = ["mos_pred", "noi_pred", "dis_pred", "col_pred", "loud_pred"]
    v = df[cols].to_numpy()
    np.testing.assert_array_equal(v[0], v[1])
    np.testing.assert_array_equal(v[2], v[3])
    ref = _oracle_file("nisqa.tar", str(tmp_path / "a.wav"))
    assert np.abs(v[1] - ref).max() <= SCORE_TOL


def test_reference_error_behaviour(tmp_path, built_lib):
    from nisqa_b200.NISQA_model import nisqaModel
    ck = os.path.join(WEIGHTS, "nisqa.tar")
    base = {"pretrained_model": ck, "output_dir": None, "tr_bs_val": 2, "tr_num_workers": 0, "ms_channel": None}
    wav.write_wav_pcm16(str(tmp_path / "short.wav"), synth.synth_speech_pcm16(1, 0.1, 48000), 48000)
    with pytest.raises(ValueError, match="Sample too short"):
        nisqaModel(dict(base, mode="predict_file", deg=str(tmp_path / "short.wav"))).predict()
    wav.write_wav_pcm16(str(tmp_path / "long.wav"), np.zeros(8000 * 53, np.int16), 8000)
    with pytest.raises(ValueError, match="Increase max window length ms_max_segments"):
        nisqaModel(dict(base, mode="predict_file", deg=str(tmp_path / "long.wav"))).predict()
    (tmp_path / "bad.wav").write_bytes(b"RIFFxxxxWAVEjunk")
    with pytest.raises(ValueError, match="Could not load file"):
        nisqaModel(dict(base, mode="predict_file", deg=str(tmp_path / "bad.wav"))).predict()
    empty = tmp_path / "empty"; empty.mkdir()
    with pytest.raises(ValueError, match="No wav files found"):
        nisqaModel(dict(base, mode="predict_dir", data_dir=str(empty)))
    with pytest.raises(NotImplementedError):
        nisqaModel(dict(base, mode="predict_nothing"))


def test_async_submit_wait_equals_sync(engines):
    """nisqa_submit_pcm / nisqa_wait (two batches in flight) return exactly what the synchronous
    entry point returns, in submission order, also when collected late or out of order."""
    eng, args, sd = engines["nisqa.tar"]
    batches = [[synth.synth_speech_pcm16(700 + 10 * b + i, 1.0 + 0.3 * i + 0.1 * b, 48000) for i in range(4)] for b in range(5)]
    ref = [eng.predict_pcm(bt, [48000] * 4) for bt in batches]
    handles = []
    got = {}
    for b, bt in enumerate(batches):
        handles.append(eng.submit_pcm(bt, [48000] * 4))       # third submit waits for the oldest internally
        if b >= 2:
            got[b - 2] = eng.wait(handles[b - 2])
    got[4] = eng.wait(handles[4])                               # newest first ...
    got[3] = eng.wait(handles[3])                               # ... then an already finished one
    for b in range(5):
        np.testing.assert_array_equal(got[b][0], ref[b][0])
        np.testing.assert_array_equal(got[b][1], ref[b][1])
    s, n, st = eng.predict_pcm(batches[0], [48000] * 4)         # sync call after async traffic
    np.testing.assert_array_equal(s, ref[0][0])
