"""Each CUDA kernel of the framewise CNN, the self-attention stack, the BiLSTM and the pooling heads held to a float64
restatement of its OWN layer (the per-layer entry points of oracle/nisqa_oracle.py, checkpoint tensors cast to float64
before any folding), fed the kernel's own input: the stage dump of the previous kernel, as the kernel read it (the
plane dumps are hi + lo, exactly the operand the tensor cores see).  tests/test_gpu_parity.py compares every stage with
the float32 oracle run end to end, so each of its checks carries the error of every stage before it; here one layer's
error stands alone and a kernel that is slightly wrong in part of its arithmetic shows up.

Metrics (oracle/precision.py):
  * convolutions: |got - ref| <= GAMMA * N per element, N = maxpool(conv(|x|, |W folded|) + |b folded|);
    tests/test_split_precision.py shows on the CPU that a kernel missing one cross term of its fp16 split for a single
    tap, K chunk or half of its output channels exceeds GAMMA by more than 10x;
  * Linear + LayerNorm, attention, BiLSTM, pooling heads: max |got - ref| <= R * (max error of the same torch op in
    float32 on the same input) + a floor of a few fp32 ulps.
Every check prints its error, its bound and their ratio.

Shapes are chosen by tile geometry: segment totals whose tile count per persistent CTA grid is 1, 2, SMs - 1, SMs,
SMs + 1, 2 SMs and 2 SMs + 1 (1, 2 and 3 tiles per CTA) for every tile height G of the CNN (1: conv1 / conv12,
3: conv3 / conv4, 9 or 12: conv5 / conv6), with the last tile full when the tile count is even and holding one segment
when it is odd; attention over clips whose lengths end on and off the 64-row tiles; the BiLSTM over 1..987 steps at
the group sizes that select NB = 1, 2 and 4 clips per CTA.

Not held here (score level in tests/test_gpu_parity.py): de_align_kernel, linear_tile_kernel and seg_feats_kernel
(NISQA_DE, SkipCNN, DFF), the front end and the resampler (bit-exact against the host one).
"""
import os

import numpy as np
import pytest
import torch

from conftest import WEIGHTS
from nisqa_b200 import engine as E
from nisqa_b200 import synth
from oracle import nisqa_oracle as O
from oracle import precision as PR
from oracle import variants as V

pytestmark = pytest.mark.gpu

SR, HOP = 16000, 160                   # 10 ms hop at 16 kHz
F64 = torch.float64


def _model(name):
    """(args, float32 sd, float64 sd) of a shipped checkpoint or a variant of oracle/variants.py."""
    if name in V.VARIANTS:
        bargs, bsd = O.load_checkpoint(os.path.join(WEIGHTS, V.VARIANTS[name][0]))
        args, sd = V.variant_checkpoint(name, bargs, bsd)
    else:
        args, sd = O.load_checkpoint(os.path.join(WEIGHTS, name))
    return args, sd, O.state_dict_as(sd, F64)


@pytest.fixture(scope="module")
def models(built_lib):
    out = {}
    for name in ("nisqa.tar", "nisqa_mos_only.tar", "nisqa_tts.tar", "dim_pos_enc"):
        args, sd, sd64 = _model(name)
        eng = E.Engine(E.config_from_args(args), 0)
        eng.load_state_dict(sd)
        out[name] = (eng, args, sd, sd64)
    yield out
    for eng, _, _, _ in out.values():
        eng.close()


_BASES = []


def _clips(eng, args, counts, seed):
    """16 kHz clips with exactly the given segment counts, cut out of four 60 s synthetic bases."""
    if not _BASES:
        _BASES.extend(synth.synth_speech_pcm16(950 + i, 60.0, SR) for i in range(4))
    rng = np.random.default_rng(seed)
    out = []
    for j, k in enumerate(counts):
        n = ((k - 1) * args["ms_seg_hop_length"] + args["ms_seg_length"] - 1) * HOP      # (k-1) hop + 15 frames
        assert E.segment_counts(eng.cfg, n, SR)[1:] == (k, E.CLIP_OK)
        st = int(rng.integers(0, len(_BASES[0]) - n + 1))
        out.append(_BASES[j % 4][st:st + n])
    return out


def _split(total):
    """A segment total as clips of <= 997 segments of varied lengths."""
    sizes, out = (997, 401, 730, 64, 883, 129), []
    while total > 0:
        out.append(min(total, sizes[len(out) % len(sizes)]))
        total -= out[-1]
    return out


def _run(eng, args, clips):
    """One predict call (one pass) with pool1 and the per-step outputs kept -> (scores, per-clip rows, dumps)."""
    std = args["cnn_model"] == "standard"
    eng.set_option("keep_pool1", 1)
    eng.set_option("keep_td_out", 1)
    try:
        scores, nseg, status = eng.predict_pcm(clips, [SR] * len(clips))
    finally:
        eng.set_option("keep_pool1", 0)
        eng.set_option("keep_td_out", 0)
    assert np.all(status == E.CLIP_OK)
    W1, W2, W3 = (8, 4, 2) if std else (7, 5, 3)
    shapes = {"pool1": (E.STAGE_POOL1, (16, 24, W1)), "pool2": (E.STAGE_POOL2, (32, 12, W2)),
              "conv3": (E.STAGE_CONV3, (64, 12, W2)), "pool3": (E.STAGE_POOL3, (64, 6, W3)),
              "conv5": (E.STAGE_CONV5, (64, 6, W3)), "cnn_feat": (E.STAGE_CNN_FEAT, (20 if std else 384,)),
              "td_out": (E.STAGE_TD_OUT, (256 if std else 64,))}
    if not std:
        shapes["td_in"] = (E.STAGE_TD_IN, (64,))
    d = {k: torch.from_numpy(eng.stage_dump(st).reshape((-1,) + shp)).to(F64) for k, (st, shp) in shapes.items()}
    mel = eng.stage_dump(E.STAGE_MEL_DB)
    segs, off = [], 0
    for c in clips:
        nf = E.segment_counts(eng.cfg, len(c), SR)[0]
        segs.append(O.segments(mel[off:off + 48 * nf].reshape(48, nf), args, F64))      # clamped as the engine reads it
        off += 48 * nf
    assert off == mel.size
    d["mel"] = torch.cat(segs)
    rows = np.concatenate([[0], np.cumsum(nseg)])
    assert all(v.shape[0] == rows[-1] for v in d.values())
    return scores, rows, d


def _report(what, err, bound):
    print("%-62s err %.3e  bound %.3e  ratio %.3f" % (what, err, bound, err / bound))
    return err <= bound


# ------------------------------------------------------------------------------------------------------ CNN
def _tile_heights(args):
    """Segments per tile: 1 (conv1_pool1_kernel, conv12_kernel), then 256 // BLK of conv3 / conv4 and of conv5 / conv6
    (BLK = (H + 1)(W + 1) padded rows per segment, csrc/conv_split.cuh)."""
    W2, W3 = (4, 2) if args["cnn_model"] == "standard" else (5, 3)
    return 1, 256 // (13 * (W2 + 1)), 256 // (7 * (W3 + 1))


def _segment_totals(args, n_sm):
    out = set()
    for G in _tile_heights(args):
        for T in (1, 2, n_sm - 1, n_sm, n_sm + 1, 2 * n_sm, 2 * n_sm + 1):
            out.add(G * T - (G - 1) * (T & 1))          # even T: full last tile; odd T: one segment in the last tile
    return sorted(out)


def _selection(args, N, n_sm, rng):
    """The segments of the first and last tile, of the last CTA's first tile and of CTA 0's second and third tiles,
    for every tile height, and a few random ones."""
    sel = set(int(s) for s in rng.choice(N, min(N, 6), replace=False))
    for G in _tile_heights(args):
        T = -(-N // G)
        for t in {0, T - 1, n_sm - 1, n_sm, 2 * n_sm}:
            if t < T:
                sel.update(range(t * G, min(N, t * G + G)))
    return torch.tensor(sorted(sel))


def _conv_checks(tag, args, sd64, d, sel):
    ok = True
    x = {k: d[k][sel] for k in ("mel", "pool1", "pool2", "conv3", "pool3", "conv5", "cnn_feat")}
    for kern, i, src, dst in (("conv1_pool1_kernel", 1, "mel", "pool1"), ("conv12_kernel conv2+pool2", 2, "pool1", "pool2"),
                              ("conv_pipe_kernel conv3", 3, "pool2", "conv3"), ("conv_pipe_kernel conv4+pool3", 4, "conv3", "pool3"),
                              ("conv_pipe_kernel conv5", 5, "pool3", "conv5")):
        ref = O.conv_layer(sd64, i, x[src], args)
        cond = PR.conv_condition(args, sd64, i, x[src])
        ok &= _report("%s %s %s -> %s" % (tag, kern, src, dst), PR.normalised_error(x[dst], ref, cond), PR.GAMMA)
    # conv12_kernel from the mel: conv1's result (pool1) never leaves the chip, so its error (<= GAMMA N1) enters conv2
    r1 = O.conv_layer(sd64, 1, x["mel"], args)
    n1 = PR.conv_condition(args, sd64, 1, x["mel"])
    ref = O.conv_layer(sd64, 2, r1, args)
    cond = PR.conv_condition(args, sd64, 2, r1.abs() + n1)
    ok &= _report("%s conv12_kernel conv1..pool2 mel -> pool2" % tag, PR.normalised_error(x["pool2"], ref, cond), PR.GAMMA)
    # conv6 (+ the Linear behind it): the Linear's own rounding counts against |W_fc| |conv6| + |b_fc|
    r6 = O.conv_layer(sd64, 6, x["conv5"], args)
    n6 = PR.conv_condition(args, sd64, 6, x["conv5"])
    head = {k: v.abs() for k, v in sd64.items() if k.startswith("cnn.model.fc")}
    ref = O.cnn_head(sd64, r6, args)
    cond = O.cnn_head(head, n6 + r6.abs() if head else n6, args)
    ok &= _report("%s conv_pipe_kernel conv6%s conv5 -> cnn_feat" % (tag, " + fc_out" if head else ""),
                  PR.normalised_error(x["cnn_feat"], ref, cond), PR.GAMMA)
    return ok


def _cpu32_check(what, got, ref, cpu32):
    return _report(what, PR.max_abs_error(got, ref), PR.cpu32_bound(PR.max_abs_error(cpu32, ref), ref))


def _td_in_check(tag, args, sd, sd64, d, rows):
    """td_in_kernel: CNN features -> Linear + LayerNorm (+ positional encoding) -> td_in, every row of the pass."""
    pe = bool(args.get("td_sa_pos_enc"))
    ref, cpu = [], []
    for a, b in zip(rows[:-1], rows[1:]):
        f = d["cnn_feat"][a:b]
        ref.append(O.sa_input(sd64, f, pe))
        cpu.append(O.sa_input(sd, f.float(), pe).to(F64))
    return _cpu32_check("%s td_in_kernel cnn_feat -> td_in%s" % (tag, " (+pos. enc.)" if pe else ""),
                        d["td_in"], torch.cat(ref), torch.cat(cpu))


@pytest.mark.parametrize("name", ["nisqa.tar", "nisqa_mos_only.tar", "nisqa_tts.tar"])
def test_cnn_kernels_against_float64(models, name):
    eng, args, sd, sd64 = models[name]
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    rng = np.random.default_rng(17)
    ok = True
    with torch.no_grad():
        for N in _segment_totals(args, n_sm):
            clips = _clips(eng, args, _split(N), seed=N)
            _, rows, d = _run(eng, args, clips)
            assert rows[-1] == N
            sel = _selection(args, N, n_sm, rng)
            tag = "%s N=%d (%d checked)" % (name, N, len(sel))
            ok &= _conv_checks(tag, args, sd64, d, sel)
            if args["td"] == "self_att":
                ok &= _td_in_check(tag, args, sd, sd64, d, rows)
    assert ok


# ------------------------------------------------------------------------------------------- self-attention
@pytest.mark.parametrize("name", ["nisqa.tar", "nisqa_mos_only.tar", "dim_pos_enc"])
def test_self_attention_kernels_against_float64(models, name):
    """Clip lengths around the 64-row query tiles and key blocks in one batch: the tiles of td_in_kernel run over the
    whole pass and cross clips, td_sa_kernel walks qtile_prefix across them."""
    eng, args, sd, sd64 = models[name]
    counts = [1, 2, 63, 64, 65, 128, 129, 247]
    scores, rows, d = _run(eng, args, _clips(eng, args, counts, seed=3))
    ok = True
    with torch.no_grad():
        ok &= _td_in_check(name, args, sd, sd64, d, rows)
        ref, cpu, sref, scpu = [], [], [], []
        for a, b in zip(rows[:-1], rows[1:]):
            x = d["td_in"][a:b]
            y64, y32 = x, x.float()
            for l in range(O.sa_layers(sd)):
                y64, y32 = O.sa_layer(sd64, l, y64), O.sa_layer(sd, l, y32)
            ref.append(y64)
            cpu.append(y32.to(F64))
            t = d["td_out"][a:b]
            sref.append(O.pool_heads(args, sd64, t))
            scpu.append(O.pool_heads(args, sd, t.float()).to(F64))
        ok &= _cpu32_check("%s td_sa_kernel x%d td_in -> td_out (S = %s)" % (name, O.sa_layers(sd), counts),
                           d["td_out"], torch.cat(ref), torch.cat(cpu))
        ok &= _cpu32_check("%s pool_final_kernel td_out -> scores" % name, torch.from_numpy(scores).reshape(-1),
                           torch.cat(sref), torch.cat(scpu))
    assert ok


# ------------------------------------------------------------------------------------------------- BiLSTM
def test_bilstm_kernels_against_float64(models):
    """lstm_batched_kernel and lastbi_final_kernel (nisqa_tts.tar): sequences of 1..987 steps, ragged inside a group,
    at batch sizes that select NB = 1 (7 clips), 2 (98) and 4 (175) clips per CTA.  Copies of a clip have identical
    inputs, so each distinct clip is restated once."""
    eng, args, sd, sd64 = models["nisqa_tts.tar"]
    counts = [987, 1, 2, 63, 300, 640, 986]
    base = _clips(eng, args, counts, seed=5)
    ok, restated = True, {}
    with torch.no_grad():
        for reps in (1, 14, 25):
            scores, rows, d = _run(eng, args, base * reps)
            ref, cpu, sref, scpu, got, sgot = [], [], [], [], [], []
            for j in range(len(counts)):
                f = d["cnn_feat"][rows[j]:rows[j + 1]]
                if j not in restated:
                    restated[j] = (f, O.bilstm(sd64, f), O.bilstm(sd, f.float()).to(F64))
                f0, r64, r32 = restated[j]
                for c in range(j, len(base) * reps, len(counts)):
                    a, b = rows[c], rows[c + 1]
                    assert torch.equal(d["cnn_feat"][a:b], f0)
                    ref.append(r64); cpu.append(r32); got.append(d["td_out"][a:b])
                    sref.append(O.pool_heads(args, sd64, d["td_out"][a:b]))
                    scpu.append(O.pool_heads(args, sd, d["td_out"][a:b].float()).to(F64))
                    sgot.append(torch.from_numpy(scores[c]).to(F64))
            tag = "nisqa_tts.tar %d clips" % (len(base) * reps)
            ok &= _cpu32_check("%s lstm_batched_kernel cnn_feat -> td_out (S = 1..987)" % tag,
                               torch.cat(got), torch.cat(ref), torch.cat(cpu))
            ok &= _cpu32_check("%s lastbi_final_kernel td_out -> scores" % tag, torch.cat(sgot), torch.cat(sref), torch.cat(scpu))
    assert ok
