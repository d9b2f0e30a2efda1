"""Error metrics that hold one kernel to a float64 restatement of its own layer (TEST INFRASTRUCTURE ONLY, like the rest
of oracle/).  tests/test_kernel_precision.py applies them to the CUDA kernels on a B200; tests/test_split_precision.py
applies the same functions and constants to a CPU emulation of the two-term fp16 split arithmetic, with and without
deliberate defects, which shows that the bounds are tight enough to catch a partly wrong kernel.

Convolutions.  For every output element the error is measured against a condition number of that element,
    N = maxpool( conv(|x|, |W|) + |b| )        (W, b: the BatchNorm-folded float64 weights; the layer's own pooling),
an upper bound of the sum of |terms| that feeds the element.  ReLU and max are 1-Lipschitz, so an arithmetic that
rounds each term (and each partial sum) to a relative u has |got - ref| <= c u N.  The kernels must reach
|got - ref| <= GAMMA * N everywhere.

Everything else (Linear + LayerNorm, attention, the BiLSTM, the pooling heads): the kernel's error against float64 must
stay within R times the error of the same torch operation run in float32 on the same input, plus a floor of a few fp32
ulps of the layer's largest value.
"""
import torch

from . import nisqa_oracle as O

# Normalised conv error.  A CPU emulation of the split arithmetic (tests/test_split_precision.py) measures <= 1e-7 for
# the correct kernel and >= 5e-5 when one of its cross terms is missing for a single tap, K chunk or half of the output
# channels; torch's own fp32 convolution measures <= 3e-7.
GAMMA = 2e-6

R_CPU32 = 8.0                  # err_gpu <= R_CPU32 * err_cpu32 + floor
FLOOR_ULPS = 4.0               # floor = FLOOR_ULPS fp32 ulps (2^-23 relative) of the layer's largest |value|


def folded_conv(sd, i):
    """conv i with its eval-mode BatchNorm (eps 1e-5) folded in, in the dtype of ``sd``: (weight, bias)."""
    p = "cnn.model."
    s = sd[p + "bn%d.weight" % i] / torch.sqrt(sd[p + "bn%d.running_var" % i] + 1e-5)
    w = sd[p + "conv%d.weight" % i] * s[:, None, None, None]
    b = (sd[p + "conv%d.bias" % i] - sd[p + "bn%d.running_mean" % i]) * s + sd[p + "bn%d.bias" % i]
    return w, b


def conv_condition(args, sd64, i, x):
    """N of conv layer i (+ its pool) for the float64 input x: the oracle's own conv_layer() applied to |x| with the
    folded |W|, |b| and an identity BatchNorm (within one ulp)."""
    w, b = folded_conv(sd64, i)
    one = torch.ones_like(b)
    p = "cnn.model."
    sd_abs = {p + "conv%d.weight" % i: w.abs(), p + "conv%d.bias" % i: b.abs(),
              p + "bn%d.running_mean" % i: torch.zeros_like(b), p + "bn%d.running_var" % i: one,
              p + "bn%d.weight" % i: torch.sqrt(one + 1e-5), p + "bn%d.bias" % i: torch.zeros_like(b)}
    return O.conv_layer(sd_abs, i, x.abs(), args)


def normalised_error(got, ref, cond):
    """max |got - ref| / N over all elements (an element with N == 0 must be exact)."""
    d = (torch.as_tensor(got, dtype=torch.float64) - ref).abs()
    if bool((d[cond == 0] > 0).any()):
        return float("inf")
    return float((d / cond.clamp_min(1e-300)).max()) if d.numel() else 0.0


def max_abs_error(got, ref):
    return float((torch.as_tensor(got, dtype=torch.float64) - ref).abs().max())


def cpu32_bound(err_cpu32, ref):
    """R_CPU32 * err_cpu32 + FLOOR_ULPS ulps of max |ref|."""
    return R_CPU32 * err_cpu32 + FLOOR_ULPS * 2.0 ** -23 * float(ref.abs().max())
