"""The conv bound of tests/test_kernel_precision.py has teeth: a CPU emulation of the arithmetic of conv12_kernel /
conv_pipe_kernel (csrc/conv12.cu, csrc/conv_split.cu) passes it, and the same emulation with one cross term missing
for part of the work fails it by more than 10x.

The emulation follows the kernels step by step:
  * weights: BatchNorm folded in double and rounded to float, pre-scaled by 2^S with S the largest value <= 14 such
    that max|w| 2^S <= 1024 (pack_weights, csrc/engine.cu), split into fp16 hi + lo;
  * activations: split8 (csrc/tc_ptx.cuh): min(x, 60000), hi = fp16(x), lo = fp16(x - hi);
  * per tap and 16-channel K step: two accumulators in fp32, [hi*hi] and [hi*lo + lo*hi] (products exact, the sum of
    16 products rounded once per step);
  * epilogue: relu(fmaf(acc_a + acc_b, 2^-S, bias)), the layer's max-pool, split8 of the result.
Inputs are the float32 oracle activations of a seeded clip, through split8, as the kernels read them.
"""
import os

import numpy as np
import pytest
import torch

from conftest import WEIGHTS
from nisqa_b200 import synth
from oracle import nisqa_oracle as O
from oracle import precision as PR

LAYERS = [(3, "pool2"), (4, "conv3"), (5, "pool3")]          # conv i and the tap that feeds it


def split8(x):
    """fp32 x >= 0 -> (hi, lo) as float64 tensors holding fp16 values."""
    x = torch.minimum(x.float(), torch.tensor(60000.0))
    hi = x.half().float()
    lo = (x - hi).half()
    return hi.double(), lo.double()


def packed_weights(sd, i, prescale=True):
    """pack_weights of csrc/engine.cu for conv i: (w_hi, w_lo, 2^-S, bias), float64 tensors of fp16 / fp32 values."""
    w, b = PR.folded_conv(O.state_dict_as(sd, torch.float64), i)
    wf = w.float()
    S = 0
    while prescale and S < 14 and float(wf.abs().max()) * 2.0 ** (S + 1) <= 1024.0:
        S += 1
    ws = wf * 2.0 ** S
    hi = ws.half().float()
    lo = (ws - hi).half()
    return hi.double(), lo.double(), 2.0 ** -S, b.float().double()


def emulate(args, sd, i, x_hi, x_lo, prescale=True, drop_lohi_tap=None, drop_lohi_chunk=None, drop_hilo_half=False):
    """conv i (+ its pool) as the tcgen05 kernels compute it; the drop_* arguments remove a cross term from part of the
    arithmetic (the defects the bound must catch)."""
    w_hi, w_lo, scale, bias = packed_weights(sd, i, prescale)
    ph, pw = O.conv_padding(i, args)
    pad = lambda t: torch.nn.functional.pad(t, (pw, pw, ph, ph))
    xh, xl = pad(x_hi), pad(x_lo)
    n, cin, H, W = x_hi.shape
    Ho, Wo = H + 2 * ph - 2, W + 2 * pw - 2
    cout = w_hi.shape[0]
    acc_a = torch.zeros(n, cout, Ho, Wo, dtype=torch.float32)
    acc_b = torch.zeros(n, cout, Ho, Wo, dtype=torch.float32)
    keep_hilo = torch.ones(cout, dtype=torch.float64)
    if drop_hilo_half:
        keep_hilo[cout // 2:] = 0.0
    for t in range(9):
        ky, kx = t // 3, t % 3
        for ks in range(cin // 16):
            c = slice(16 * ks, 16 * ks + 16)
            ah, al = xh[:, c, ky:ky + Ho, kx:kx + Wo], xl[:, c, ky:ky + Ho, kx:kx + Wo]
            mm = lambda a, wt: torch.einsum("nchw,oc->nohw", a, wt[:, c, ky, kx])      # exact: 16 products of 11 x 11 bits
            acc_a = (acc_a.double() + mm(ah, w_hi)).float()
            acc_b = (acc_b.double() + mm(ah, w_lo) * keep_hilo[None, :, None, None]).float()
            if t != drop_lohi_tap and ks != drop_lohi_chunk:
                acc_b = (acc_b.double() + mm(al, w_hi)).float()
    y = ((acc_a.double() + acc_b.double()).float().double() * scale + bias[None, :, None, None]).float()
    y = O.cnn_pool(i, torch.relu(y), args)
    hi, lo = split8(y)
    return hi + lo


MUTANTS = {
    "lo*hi missing for one tap of nine": dict(drop_lohi_tap=4),
    "lo*hi missing for one 16-channel K chunk": dict(drop_lohi_chunk=1),
    "hi*lo missing for half of the output channels": dict(drop_hilo_half=True),
}


@pytest.fixture(scope="module")
def model():
    """nisqa.tar and the float32 oracle activations of a seeded 3 s 48 kHz clip (72 segments)."""
    args, sd = O.load_checkpoint(os.path.join(WEIGHTS, "nisqa.tar"))
    pcm = synth.synth_speech_pcm16(1, 3.0, 48000)
    taps = {}
    O.predict_pcm(args, sd, pcm.astype(np.float32) / np.float32(32768.0), 48000, taps)
    return args, sd, O.state_dict_as(sd, torch.float64), taps


def _layer(model, i, tap, w_scale=1.0):
    args, sd, sd64, taps = model
    if w_scale != 1.0:                                                # conv i's weights and bias scaled by w_scale
        p = "cnn.model.conv%d." % i
        sd = dict(sd, **{p + "weight": sd[p + "weight"] * w_scale, p + "bias": sd[p + "bias"] * w_scale})
        sd64 = O.state_dict_as(sd, torch.float64)
    x_hi, x_lo = split8(taps[tap])
    x = x_hi + x_lo                                                   # what the kernel reads (the stage dumps' hi + lo)
    with torch.no_grad():
        ref = O.conv_layer(sd64, i, x, args)
        cond = PR.conv_condition(args, sd64, i, x)
    return args, sd, x_hi, x_lo, x, ref, cond


@pytest.mark.parametrize("i,tap", LAYERS)
def test_split_arithmetic_meets_the_bound(model, i, tap):
    args, sd, x_hi, x_lo, x, ref, cond = _layer(model, i, tap)
    with torch.no_grad():
        err = PR.normalised_error(emulate(args, sd, i, x_hi, x_lo), ref, cond)
        err32 = PR.normalised_error(O.conv_layer(sd, i, x.float(), args), ref, cond)
    print("conv%d: split emulation %.2e, torch fp32 %.2e, gamma %.1e" % (i, err, err32, PR.GAMMA))
    assert err <= PR.GAMMA and err32 <= PR.GAMMA


@pytest.mark.parametrize("i,tap", LAYERS)
@pytest.mark.parametrize("mutant", sorted(MUTANTS))
def test_a_missing_cross_term_fails_by_more_than_10x(model, i, tap, mutant):
    args, sd, x_hi, x_lo, x, ref, cond = _layer(model, i, tap)
    with torch.no_grad():
        err = PR.normalised_error(emulate(args, sd, i, x_hi, x_lo, **MUTANTS[mutant]), ref, cond)
    print("conv%d, %s: %.2e = %.0f x gamma" % (i, mutant, err, err / PR.GAMMA))
    assert err >= 10 * PR.GAMMA


@pytest.mark.parametrize("i,tap", LAYERS)
def test_weights_split_without_the_prescale_fail(model, i, tap):
    """Without the 2^S pre-scale, w_lo lands in the fp16 subnormals (spacing 2^-24) and loses bits.  With the shipped
    weights (folded max|w| ~0.45, median ~0.05) that costs little: the normalised error goes from ~1.3e-7 to <= 2.1e-7,
    which no bound at the level of the correct kernel's own rounding can tell apart.  The pre-scale matters for a
    checkpoint with smaller weights: with conv i's weights and bias scaled by 2^-6 the split without it exceeds gamma,
    while the pre-scaled split still meets it."""
    args, sd, x_hi, x_lo, x, ref, cond = _layer(model, i, tap, w_scale=2.0 ** -6)
    with torch.no_grad():
        ok = PR.normalised_error(emulate(args, sd, i, x_hi, x_lo), ref, cond)
        err = PR.normalised_error(emulate(args, sd, i, x_hi, x_lo, prescale=False), ref, cond)
    print("conv%d, weights x 2^-6: pre-scaled split %.2e, split without the pre-scale %.2e = %.1f x gamma"
          % (i, ok, err, err / PR.GAMMA))
    assert ok <= PR.GAMMA < err
