"""CPU oracle for the NISQA predict hot path (wav samples -> MOS / dimension scores).

TEST INFRASTRUCTURE ONLY.  Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
CPU-baseline / ``--impl reference`` legs may import this module, and only as the checker or
as the CPU baseline being timed.  The product path (``nisqa_b200/``) never imports it.

What it is: a per-clip, unpadded restatement of the reference's predict path in NumPy +
torch-CPU functional ops (the same arithmetic library the reference uses on the CPU), each
function citing the reference ``file:line`` it follows (``lib`` = nisqa/NISQA_lib.py).
The model half follows the dtype of its inputs: float32 by default (the reference's own
arithmetic), float64 with ``state_dict_as(sd, torch.float64)`` and float64 inputs.  Its
per-layer entry points (``conv_layer``, ``cnn_head``, ``sa_input``, ``sa_layer``, ``bilstm``,
``pool_heads``) are what the whole-model functions are built from, so a single kernel can be
held to a restatement of exactly its own layer (tests/test_kernel_precision.py).

Pinning status
  * model half (segments -> scores): PINNED against the unmodified reference modules imported
    from ``/root/reference`` (``oracle/make_golden.py`` -> ``tests/golden/*.npz``,
    checked by ``tests/test_oracle_golden.py``).
  * front-end half (samples -> mel dB): PARITY UNPINNED - see ``oracle/librosa_compat.py``.

The reference pads every clip to ``ms_max_segments`` and masks; per-clip results do not depend
on the batch composition (SURVEY.md section 0.7, re-checked by ``tests/test_oracle_golden.py``),
so the oracle processes one clip at a time with no padding.
"""
import math
import os

import numpy as np
import torch
import torch.nn.functional as F

from . import librosa_compat as lb

STATUS_OK, STATUS_TOO_SHORT, STATUS_TOO_LONG = 0, 1, 2


def load_checkpoint(path):
    """reference model:938-942 - ``torch.load`` of {'args', 'model_state_dict'}."""
    ck = torch.load(path, map_location="cpu", weights_only=False)
    sd = {k: v.detach().clone() for k, v in ck["model_state_dict"].items()}
    return dict(ck["args"]), sd


def state_dict_as(sd, dtype):
    """The floating-point tensors of a state_dict cast to ``dtype`` (unfolded, as stored in the checkpoint): the model
    half is dtype-generic, so ``state_dict_as(sd, torch.float64)`` with float64 inputs restates it in float64."""
    return {k: (v.to(dtype) if v.is_floating_point() else v) for k, v in sd.items()}


# ------------------------------------------------------------------ front-end (a1-a6)
def hop_win(sr, args):
    """lib:2308-2309: int() truncation of sr * seconds (double arithmetic)."""
    return int(sr * args["ms_hop_length"]), int(sr * args["ms_win_length"])


def mel_db(y, sr, args):
    """lib:2311-2330 - melspectrogram(power=1) then amplitude_to_db(amin=1e-4, top_db=80)."""
    hop, win = hop_win(sr, args)
    S = lb.melspectrogram(y=y, sr=sr, S=None, n_fft=args["ms_n_fft"], hop_length=hop,
                          win_length=win, window="hann", center=True, pad_mode="reflect",
                          power=1.0, n_mels=args["ms_n_mels"], fmin=0.0,
                          fmax=args["ms_fmax"], htk=False, norm="slaney")
    return lb.amplitude_to_db(S, ref=1.0, amin=1e-4, top_db=80.0)


def segment_counts(n_samples, sr, args):
    """Exact integer bookkeeping of lib:2308 + librosa frame count + lib:2257-2277.

    Returns (n_frames, n_segments, status)."""
    hop, _ = hop_win(sr, args)
    n_frames = 1 + n_samples // hop
    seg_len, seg_hop = args["ms_seg_length"], args["ms_seg_hop_length"]
    n_wins = n_frames - (seg_len - 1)
    if n_wins < 1:
        return n_frames, 0, STATUS_TOO_SHORT
    n_seg = int(math.ceil(n_wins / seg_hop)) if seg_hop > 1 else n_wins
    if args["ms_max_segments"] is not None and n_seg > args["ms_max_segments"]:
        return n_frames, n_seg, STATUS_TOO_LONG
    return n_frames, n_seg, STATUS_OK


def segments(spec, args, dtype=torch.float32):
    """lib:2239-2273 without the zero-padding tail: x[i,0,m,t] = spec[m, i*seg_hop + t]."""
    seg_len, seg_hop = args["ms_seg_length"], args["ms_seg_hop_length"]
    spec = torch.as_tensor(np.ascontiguousarray(spec), dtype=dtype)
    n_wins = spec.shape[1] - (seg_len - 1)
    if n_wins < 1:
        raise ValueError("Sample too short")
    starts = torch.arange(0, n_wins, seg_hop)
    idx = starts[:, None] + torch.arange(seg_len)[None, :]          # [S, 15]
    x = spec[:, idx]                                                # [48, S, 15]
    return x.permute(1, 0, 2).unsqueeze(1).contiguous()             # [S, 1, 48, 15]


# ------------------------------------------------------------------------ CNN (a10/a15)
def _conv_bn_relu(sd, i, x, padding):
    p = "cnn.model."
    x = F.conv2d(x, sd[p + "conv%d.weight" % i], sd[p + "conv%d.bias" % i], padding=padding)
    x = F.batch_norm(x, sd[p + "bn%d.running_mean" % i], sd[p + "bn%d.running_var" % i],
                     sd[p + "bn%d.weight" % i], sd[p + "bn%d.bias" % i],
                     training=False, eps=1e-5)
    return F.relu(x)


def conv_layer(sd, i, x, args):
    """conv i + BN + ReLU, followed by the max-pool that belongs to that layer (pool1 / pool2 / pool3 behind conv 1 / 2
    / 4), of the AdaptCNN (lib:688-706, eval mode: Dropout2d is the identity) or the StandardCNN (lib:811-830: fixed
    MaxPool2d(2), the first one with padding (0,1))."""
    return cnn_pool(i, _conv_bn_relu(sd, i, x, conv_padding(i, args)), args)


def conv_padding(i, args):
    if args["cnn_model"] == "adapt" and i == 6:
        return (1, 0)                            # conv6: kernel (3, pool_3[1]) pad (1,0): W 3 -> 1
    return (1, 1)


def cnn_pool(i, x, args):
    """The max-pool behind conv i (the identity behind conv 3, 5 and 6)."""
    if args["cnn_model"] == "adapt":
        pool = {1: "cnn_pool_1", 2: "cnn_pool_2", 4: "cnn_pool_3"}.get(i)
        return F.adaptive_max_pool2d(x, output_size=tuple(args[pool])) if pool else x
    if i == 1:
        return F.max_pool2d(x, 2, stride=2, padding=(0, 1))
    return F.max_pool2d(x, 2, stride=2) if i in (2, 4) else x


def cnn_head(sd, x, args):
    """conv6's output -> the framewise features: flatten (lib:707, 831) and the optional Linear (AdaptCNN cnn_fc_out_h,
    lib:708-709; StandardCNN fc_out 768 -> 20, lib:832-834)."""
    if args["cnn_model"] == "adapt":
        x = x.reshape(-1, 64 * args["cnn_pool_3"][0])
        if "cnn.model.fc.weight" in sd:
            x = F.linear(x, sd["cnn.model.fc.weight"], sd["cnn.model.fc.bias"])
        return x
    x = x.reshape(-1, 64 * 6 * 2)
    if "cnn.model.fc_out.weight" in sd:
        x = F.linear(x, sd["cnn.model.fc_out.weight"], sd["cnn.model.fc_out.bias"])
    return x


_CNN_TAPS = {1: "pool1", 2: "pool2", 3: "conv3", 4: "pool3", 5: "conv5"}


def conv_cnn(sd, x, args, taps=None):
    """AdaptCNN (lib:688-710) or StandardCNN (lib:811-836): six conv_layer()s and cnn_head()."""
    for i in range(1, 7):
        x = conv_layer(sd, i, x, args)
        if taps is not None and i in _CNN_TAPS: taps[_CNN_TAPS[i]] = x
    return cnn_head(sd, x, args)


def skip_cnn(sd, x):
    """SkipCNN.forward (lib:529-533): BatchNorm2d(1) (eval) -> view(-1, 720) -> Linear or Identity."""
    p = "cnn.model."
    x = F.batch_norm(x, sd[p + "bn.running_mean"], sd[p + "bn.running_var"], sd[p + "bn.weight"], sd[p + "bn.bias"], training=False, eps=1e-5)
    x = x.reshape(-1, x.shape[2] * x.shape[3])
    if p + "linear.weight" in sd:
        x = F.linear(x, sd[p + "linear.weight"], sd[p + "linear.bias"])
    return x


def dff(sd, x):
    """DFF.forward (lib:569-583, eval: dropout is the identity): BN2d(1), then 4 x (Linear, BatchNorm1d, ReLU)."""
    p = "cnn.model."
    x = F.batch_norm(x, sd[p + "bn1.running_mean"], sd[p + "bn1.running_var"], sd[p + "bn1.weight"], sd[p + "bn1.bias"], training=False, eps=1e-5)
    x = x.reshape(-1, x.shape[2] * x.shape[3])
    for i in range(1, 5):
        x = F.linear(x, sd[p + "lin%d.weight" % i], sd[p + "lin%d.bias" % i])
        b = p + "bn%d." % (i + 1)
        x = F.relu(F.batch_norm(x, sd[b + "running_mean"], sd[b + "running_var"], sd[b + "weight"], sd[b + "bias"], training=False, eps=1e-5))
    return x


# --------------------------------------------------------- time dependency (a11/a12/a16)
def self_attention(sd, feats, taps=None, pos_enc=False):
    """lib:988-996 + lib:1025-1040 for ONE clip (so no key-padding mask is needed).

    nn.MultiheadAttention with one head: q,k,v = in_proj; q *= 1/sqrt(64); softmax(q k^T) v;
    out_proj; post-norm residual blocks."""
    x = sa_input(sd, feats, pos_enc, taps)
    for l in range(sa_layers(sd)):
        x = sa_layer(sd, l, x)
        if taps is not None: taps["sa_l%d" % l] = x
    return x


def sa_input(sd, feats, pos_enc=False, taps=None):
    """The input block of SelfAttention (lib:1025-1029) for ONE clip: Linear, LayerNorm, then the positional encoding
    (lib:1042-1062: x + pe[:S] with the registered buffer [max_len, 1, d]; eval: no dropout)."""
    p = "time_dependency.model."
    x = F.linear(feats, sd[p + "linear.weight"], sd[p + "linear.bias"])
    x = F.layer_norm(x, (x.shape[-1],), sd[p + "norm1.weight"], sd[p + "norm1.bias"], 1e-5)
    if taps is not None: taps["sa_in"] = x
    if pos_enc:
        x = x + sd[p + "pos_encoder.pe"][:x.shape[0], 0, :]
    return x


def sa_layers(sd):
    p = "time_dependency.model.layers."
    return len({k.split(".")[3] for k in sd if k.startswith(p)})


def sa_layer(sd, l, x):
    """Encoder layer l of SelfAttention (lib:988-996, 1030-1040) for ONE clip."""
    q = "time_dependency.model.layers.%d." % l
    d = x.shape[-1]
    qkv = F.linear(x, sd[q + "self_attn.in_proj_weight"], sd[q + "self_attn.in_proj_bias"])
    qq, kk, vv = qkv[:, :d], qkv[:, d:2 * d], qkv[:, 2 * d:]
    att = torch.softmax((qq * (1.0 / math.sqrt(d))) @ kk.t(), dim=-1)
    sa = F.linear(att @ vv, sd[q + "self_attn.out_proj.weight"], sd[q + "self_attn.out_proj.bias"])
    x = F.layer_norm(x + sa, (d,), sd[q + "norm1.weight"], sd[q + "norm1.bias"], 1e-5)
    ff = F.linear(F.relu(F.linear(x, sd[q + "linear1.weight"], sd[q + "linear1.bias"])),
                  sd[q + "linear2.weight"], sd[q + "linear2.bias"])
    return F.layer_norm(x + ff, (d,), sd[q + "norm2.weight"], sd[q + "norm2.bias"], 1e-5)


def bilstm(sd, feats):
    """lib:925-943: packed 1-layer BiLSTM for ONE clip. PyTorch gate order i,f,g,o;
    c = f*c + i*g; h = o*tanh(c); reverse direction starts at the clip's own last step."""
    p = "time_dependency.model.lstm."
    S = feats.shape[0]
    outs = []
    for suffix, order in (("", range(S)), ("_reverse", range(S - 1, -1, -1))):
        w_ih, w_hh = sd[p + "weight_ih_l0" + suffix], sd[p + "weight_hh_l0" + suffix]
        b = sd[p + "bias_ih_l0" + suffix] + sd[p + "bias_hh_l0" + suffix]
        H = w_hh.shape[1]
        gx = feats @ w_ih.t() + b
        h = torch.zeros(H, dtype=feats.dtype)
        c = torch.zeros(H, dtype=feats.dtype)
        out = torch.zeros(S, H, dtype=feats.dtype)
        for t in order:
            g = gx[t] + w_hh @ h
            i, f, gg, o = g[:H], g[H:2 * H], g[2 * H:3 * H], g[3 * H:]
            c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(gg)
            h = torch.sigmoid(o) * torch.tanh(c)
            out[t] = h
        outs.append(out)
    return torch.cat(outs, dim=1)                                   # [S, 2H] fwd || bwd


# ------------------------------------------------- double-ended model (SURVEY.md 8f.4)
def de_align(args, x, y, sd=None):
    """Alignment.forward (lib:1274-1285) for ONE pair: attention scores of every degraded step against the reference
    clip's own steps (no padding, so no mask), softmax over the reference steps, hard (argmax -> gather, lib:1359-1368)
    or soft (att @ y, lib:1370-1378) application.  x [Sx, d], y [Sy, d] -> y aligned to x [Sx, d]."""
    method = args["de_align"]
    if method == "dot":                                    # AttDot lib:1287-1296
        att = x @ y.t()
    elif method == "cosine":                               # AttCosine lib:1298-1308: nn.CosineSimilarity(dim=3), eps 1e-8
        att = F.cosine_similarity(x[:, None, :], y[None, :, :], dim=2, eps=1e-8)
    elif method == "distance":                             # AttDistance lib:1310-1323 with dist_norm = weight_norm = 1
        att = -(x[None, :, :] - y[:, None, :]).abs().pow(1).mean(dim=2).pow(1).t()
    elif method == "luong":                                # AttLuong lib:1344-1357: x . (W y + b)
        att = x @ F.linear(y, sd["align.att.W.weight"], sd["align.att.W.bias"]).t()
    elif method == "bahd":                                 # AttBahdanau lib:1325-1342: v . tanh(Wq x + Wy y) (+ bias)
        h = torch.tanh(F.linear(x, sd["align.att.Wq.weight"], sd["align.att.Wq.bias"])[None, :, :]
                       + F.linear(y, sd["align.att.Wy.weight"], sd["align.att.Wy.bias"])[:, None, :])
        att = F.linear(h, sd["align.att.v.weight"], sd["align.att.v.bias"]).squeeze(2).t()
    else:
        raise NotImplementedError(method)
    att = torch.softmax(att, dim=1)
    if args["de_align_apply"] == "hard":
        return y[att.argmax(1)]
    if args["de_align_apply"] == "soft":
        return att @ y
    raise NotImplementedError(args["de_align_apply"])


def de_fuse(args, x, y, sd=None):
    """Fusion.forward (lib:1402-1417) with the optional Linear (de_fuse_dim, lib:1399-1401)."""
    mode = args["de_fuse"]
    if mode == "x/y/-":
        f = torch.cat((x, y, x - y), 1)
    elif mode == "+/-":
        f = torch.cat((x + y, x - y), 1)
    elif mode == "x/y":
        f = torch.cat((x, y), 1)
    else:
        raise NotImplementedError(mode)
    if args.get("de_fuse_dim"):
        f = F.linear(f, sd["fuse.lin_fusion.weight"], sd["fuse.lin_fusion.bias"])
    return f


def forward_de_from_mel(args, sd, spec, spec_ref, taps=None):
    """NISQA_DE.forward (lib:404-424) for one (degraded, reference) pair of mel dB spectrograms -> score [1]."""
    if args["cnn_model"] != "adapt" or args["td"] != "self_att" or args.get("td_2") != "self_att":
        raise NotImplementedError("oracle: NISQA_DE with AdaptCNN + self-attention + td_2 self-attention")
    with torch.no_grad():
        outs = []
        for sp in (spec, spec_ref):
            feats = conv_cnn(sd, segments(sp, args), args)
            outs.append(self_attention(sd, feats, pos_enc=bool(args.get("td_sa_pos_enc"))))
        x, y = outs
        y_al = de_align(args, x, y, sd)
        if taps is not None: taps["de_x"], taps["de_y"], taps["de_y_aligned"] = x, y, y_al
        fused = de_fuse(args, x, y_al, sd)
        sd2 = {k.replace("time_dependency_2.", "time_dependency."): v for k, v in sd.items() if k.startswith("time_dependency_2.")}
        td2 = self_attention(sd2, fused, pos_enc=bool(args.get("td_2_sa_pos_enc")))
        if taps is not None: taps["td2_out"] = td2
        pf = "pool.model."
        if args["pool"] == "att":
            out = pool_attff(sd, pf, td2) if args.get("pool_att_h") else pool_att(sd, pf, td2)
        elif args["pool"] in ("avg", "max", "last_step"):
            out = {"avg": pool_avg, "max": pool_max, "last_step": pool_last_step}[args["pool"]](sd, pf, td2)
        else:
            raise NotImplementedError(args["pool"])
    return out.numpy()


def predict_pcm_de(args, sd, y_deg, sr_deg, y_ref, sr_ref, taps=None):
    """(degraded, reference) float32 mono samples -> (score [1], (n_seg_deg, n_seg_ref), status) - lib:2132-2214 +
    lib:1420-1439 for one double-ended row."""
    y_deg = np.ascontiguousarray(y_deg, dtype=np.float32)
    y_ref = np.ascontiguousarray(y_ref, dtype=np.float32)
    _, n1, st1 = segment_counts(y_deg.shape[0], sr_deg, args)
    _, n2, st2 = segment_counts(y_ref.shape[0], sr_ref, args)
    if st1 != STATUS_OK or st2 != STATUS_OK:
        return np.full(1, np.nan, dtype=np.float32), (n1, n2), (st1 if st1 != STATUS_OK else st2)
    score = forward_de_from_mel(args, sd, mel_db(y_deg, sr_deg, args), mel_db(y_ref, sr_ref, args), taps)
    return score.astype(np.float32), (n1, n2), STATUS_OK


# ---------------------------------------------------------------------- pooling (a13/a17)
def pool_attff(sd, prefix, x):
    """lib:1171-1183 for one clip: att = W2 relu(W1 x + b1) + b2; softmax over time;
    weighted sum of x; Linear 64 -> 1."""
    a = F.linear(F.relu(F.linear(x, sd[prefix + "linear1.weight"], sd[prefix + "linear1.bias"])),
                 sd[prefix + "linear2.weight"], sd[prefix + "linear2.bias"])      # [S,1]
    a = torch.softmax(a.t(), dim=1)                                                # [1,S]
    pooled = a @ x                                                                 # [1,64]
    return F.linear(pooled, sd[prefix + "linear3.weight"], sd[prefix + "linear3.bias"]).reshape(-1)


def pool_att(sd, prefix, x):
    """PoolAtt (lib:1131-1154) for one clip: att = linear1(x); softmax over time; weighted sum; linear2."""
    a = torch.softmax(F.linear(x, sd[prefix + "linear1.weight"], sd[prefix + "linear1.bias"]).t(), dim=1)     # [1,S]
    return F.linear(a @ x, sd[prefix + "linear2.weight"], sd[prefix + "linear2.bias"]).reshape(-1)


def pool_avg(sd, prefix, x):
    """PoolAvg (lib:1185-1204): sum over the valid steps / n_wins, Linear."""
    v = torch.div(x.sum(0, keepdim=True), float(x.shape[0]))
    return F.linear(v, sd[prefix + "linear.weight"], sd[prefix + "linear.bias"]).reshape(-1)


def pool_max(sd, prefix, x):
    """PoolMax (lib:1206-1225): max over the valid steps, Linear."""
    return F.linear(x.max(0, keepdim=True)[0], sd[prefix + "linear.weight"], sd[prefix + "linear.bias"]).reshape(-1)


def pool_last_step(sd, prefix, x):
    """PoolLastStep (lib:1117-1129): the last valid step, Linear."""
    return F.linear(x[-1:, :], sd[prefix + "linear.weight"], sd[prefix + "linear.bias"]).reshape(-1)


def pool_last_step_bi(sd, prefix, x):
    """lib:1107-1115: forward hidden at the last valid step || backward hidden at step 0."""
    H = x.shape[1] // 2
    v = torch.cat((x[-1, :H], x[0, H:]))[None, :]
    return F.linear(v, sd[prefix + "linear.weight"], sd[prefix + "linear.bias"]).reshape(-1)


# ------------------------------------------------------------------------- whole model
def forward_from_mel(args, sd, spec, taps=None):
    """mel dB [n_mels, F] -> scores [1] or [5] (order mos,noi,dis,col,loud; lib:255-266)."""
    x = segments(spec, args)
    if taps is not None: taps["n_segments"] = x.shape[0]
    with torch.no_grad():
        if args["cnn_model"] in ("adapt", "standard"):
            feats = conv_cnn(sd, x, args, taps)
        elif args["cnn_model"] in (None, "skip"):
            feats = skip_cnn(sd, x)
        elif args["cnn_model"] == "dff":
            feats = dff(sd, x)
        else:
            raise NotImplementedError(args["cnn_model"])
        if taps is not None: taps["cnn_feat"] = feats
        if args["td"] == "self_att":
            td = self_attention(sd, feats, taps, pos_enc=bool(args.get("td_sa_pos_enc")))
        elif args["td"] == "lstm":
            td = bilstm(sd, feats)
        else:
            raise NotImplementedError(args["td"])
        if args.get("td_2") == "self_att":
            # TimeDependency 2 (lib:114-141, 236-268): a second stack with the first one's output as its input
            sd2 = {k.replace("time_dependency_2.", "time_dependency."): v for k, v in sd.items() if k.startswith("time_dependency_2.")}
            td = self_attention(sd2, td, pos_enc=bool(args.get("td_2_sa_pos_enc")))
        elif args.get("td_2") not in (None, "skip"):
            raise NotImplementedError(args["td_2"])
        if taps is not None: taps["td_out"] = td
        return pool_heads(args, sd, td).numpy()


def pool_heads(args, sd, td):
    """The pooling module(s) of ONE clip (lib:255-266): five heads for NISQA_DIM (order mos,noi,dis,col,loud), one
    otherwise -> scores [5] or [1]."""
    if args["model"] == "NISQA_DIM":
        prefixes = ["pool_layers.%d.model." % i for i in range(5)]
    else:
        prefixes = ["pool.model."]
    outs = []
    for pf in prefixes:
        if args["pool"] == "att":
            outs.append(pool_attff(sd, pf, td) if args.get("pool_att_h") else pool_att(sd, pf, td))
        elif args["pool"] == "last_step_bi":
            outs.append(pool_last_step_bi(sd, pf, td))
        elif args["pool"] in ("avg", "max", "last_step"):
            outs.append({"avg": pool_avg, "max": pool_max, "last_step": pool_last_step}[args["pool"]](sd, pf, td))
        else:
            raise NotImplementedError(args["pool"])
    return torch.cat(outs)


def predict_pcm(args, sd, y, sr, taps=None):
    """float32 mono samples -> (scores, n_segments, status).  Mirrors lib:2162-2233 +
    lib:1441-1467 for one clip."""
    y = np.ascontiguousarray(y, dtype=np.float32)
    _, n_seg, status = segment_counts(y.shape[0], sr, args)
    n_out = 5 if args["model"] == "NISQA_DIM" else 1
    if status != STATUS_OK:
        return np.full(n_out, np.nan, dtype=np.float32), n_seg, status
    spec = mel_db(y, sr, args)
    if taps is not None: taps["mel_db"] = spec
    scores = forward_from_mel(args, sd, spec, taps)
    return scores.astype(np.float32), n_seg, STATUS_OK


def predict_file(args, sd, path, ms_channel=None, taps=None):
    """lib:2298-2306 + the rest of the path for one wav file."""
    if ms_channel is not None:
        y, sr = lb.load(path, sr=args.get("ms_sr"), mono=False)
        if y.ndim > 1:
            y = y[ms_channel, :]
    else:
        y, sr = lb.load(path, sr=args.get("ms_sr"))
    return predict_pcm(args, sd, y, sr, taps)


def default_weights_dir():
    return os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "weights")
