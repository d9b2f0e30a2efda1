#!/bin/bash
# GPU-box memory / race / init check of every kernel on the default path (SURVEY.md section 5: the reference has no
# sanitizer story; this is ours): compute-sanitizer memcheck over __graft_entry__.smoke() (nisqa.tar, two
# short clips at 48 / 16 kHz: front-end, conv1 + conv2 fused, the tcgen05 conv3..conv6 with their bulk copies /
# mbarriers / TMEM, self-attention, pooling) and over a short nisqa_tts.tar call (StandardCNN, BiLSTM).
#   gpurun --timeout 300 -- 'bash tools/sanitize.sh r01e'
TAG=${1:-rXX}
OUT=gpurun_out
mkdir -p $OUT
cat > /tmp/san_run.py <<'PY'
import os, sys
sys.path.insert(0, os.getcwd())
import numpy as np
import __graft_entry__ as g
g.smoke()
from nisqa_b200 import engine as E, synth
from oracle import nisqa_oracle as O
args, sd = O.load_checkpoint(os.path.join("weights", "nisqa_tts.tar"))
eng = E.Engine(E.config_from_args(args, max_chunk_segments=64), 0); eng.load_state_dict(sd)   # two passes: shrinking planes
sc, ns, st = eng.predict_pcm([synth.synth_speech_pcm16(7, 0.6, 16000), synth.synth_speech_pcm16(8, 0.3, 16000)], [16000, 16000])
ref, _, _ = O.predict_pcm(args, sd, synth.synth_speech_pcm16(7, 0.6, 16000).astype(np.float32) / 32768.0, 16000)
assert abs(float(sc[0, 0]) - float(ref[0])) <= 1e-4
print("tts ok", sc.tolist())
eng.close()
# round-2 kernels: double-ended model (de_align, td_in with 192 inputs, second stack), td_2 behind the first stack,
# device resampler (both directions), conv12 with the padded mel ring
from oracle import variants as V
bargs, bsd = O.load_checkpoint(os.path.join("weights", "nisqa_mos_only.tar"))
for name in ("de_cosine_hard", "de_distance_soft_xy"):
    a2, s2 = V.de_checkpoint(name, bargs, bsd)
    e2 = E.Engine(E.config_from_args(a2), 0); e2.load_state_dict(s2)
    d, srd, r, srr = V.de_pair_pcm(V.DE_PAIRS[1])
    got = e2.predict_pcm([d, r], [srd, srr])[0]
    ref = O.predict_pcm_de(a2, s2, d.astype(np.float32) / 32768.0, srd, r.astype(np.float32) / 32768.0, srr)[0]
    assert abs(float(got[0, 0]) - float(ref[0])) <= 5e-4, (name, got, ref)
    e2.close()
a3, s3 = V.variant_checkpoint("mos_td2_sa_pos_enc", bargs, bsd)
e3 = E.Engine(E.config_from_args(a3), 0); e3.load_state_dict(s3)
x = synth.synth_speech_pcm16(9, 0.8, 16000)
print("td2", e3.predict_pcm([x], [16000])[0].tolist())
from nisqa_b200 import resample as RS
for so, sn in ((48000, 16000), (16000, 44100)):
    xs = synth.synth_speech_pcm16(10, 0.25, so)
    assert np.array_equal(e3.resample_device(xs, so, sn), RS.resample(xs, so, sn))
print("resample ok", e3.predict_pcm_resampled([x, synth.synth_speech_pcm16(11, 0.5, 48000)], [16000, 48000], 16000)[0].tolist())
e3.close()
PY
timeout 280 compute-sanitizer --tool memcheck --error-exitcode 7 --log-file $OUT/${TAG}_memcheck.log python /tmp/san_run.py > $OUT/${TAG}_memcheck_stdout.log 2>&1
echo "memcheck exit $?"
tail -5 $OUT/${TAG}_memcheck.log; tail -3 $OUT/${TAG}_memcheck_stdout.log
# shared-memory hazards (racecheck) and uninitialised device reads (initcheck) of the same run (RACE=1)
[ -z "$RACE" ] && exit 0
timeout 400 compute-sanitizer --tool racecheck --error-exitcode 7 --log-file $OUT/${TAG}_racecheck.log python /tmp/san_run.py > $OUT/${TAG}_racecheck_stdout.log 2>&1
echo "racecheck exit $?"
tail -4 $OUT/${TAG}_racecheck.log
timeout 280 compute-sanitizer --tool initcheck --error-exitcode 7 --log-file $OUT/${TAG}_initcheck.log python /tmp/san_run.py > $OUT/${TAG}_initcheck_stdout.log 2>&1
echo "initcheck exit $?"
tail -4 $OUT/${TAG}_initcheck.log
