"""GPU box: where do the persistent conv CTAs (conv12_kernel, conv_pipe_kernel) spend their cycles?  Needs the
-DNISQA_TC_TIMING build (bash tools/tc_ab_build.sh -> nisqa_b200/exp/libnisqa_timing.so), in which every conv layer
accumulates into its own counter block.   python tools/pipe_timing.py"""
import ctypes as C, os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from nisqa_b200 import engine as E, synth
E._lib = E.load_library(os.path.join(ROOT, "nisqa_b200", "exp", "libnisqa_timing.so"))
import torch
ck = torch.load(os.path.join(ROOT, "weights", "nisqa.tar"), map_location="cpu", weights_only=False)
eng = E.Engine(E.config_from_args(ck["args"]), 0); eng.load_state_dict(ck["model_state_dict"])
lib = E._lib
lib.nisqa_debug_pipe_timing.argtypes = [C.POINTER(C.c_longlong), C.c_int, C.c_int]
lib.nisqa_debug_c12_timing.argtypes = [C.POINTER(C.c_longlong), C.c_int, C.c_int]
base = [synth.synth_speech_pcm16(i, 10.0, 48000) for i in range(8)]
clips = [np.roll(base[i % 8], 977 * i) for i in range(64)]
pipe = (C.c_longlong * (4 * 256 * 16))()         # [layer 3..6][CTA][slot]
c12 = (C.c_longlong * (256 * 16))()
eng.predict_pcm(clips, [48000] * 64)
lib.nisqa_debug_pipe_timing(pipe, len(pipe), 1)  # reset after warm-up
lib.nisqa_debug_c12_timing(c12, len(c12), 1)
eng.predict_pcm(clips, [48000] * 64)
lib.nisqa_debug_pipe_timing(pipe, len(pipe), 1)
lib.nisqa_debug_c12_timing(c12, len(c12), 1)
names = ["iss:wait_acc_free", "iss:wait_a_full", "iss:wait_b_full", "-", "iss:total", "epi:wait_acc_full", "epi:tmem->stage",
         "epi:part2(+bar)", "-", "prodA:wait_a_free", "-", "prodW:wait_b_empty", "-", "-", "-", "tiles"]
tp = np.array(pipe[:], dtype=np.float64).reshape(4, 256, 16)
for layer in (3, 4, 5, 6):
    t = tp[layer - 3, :148]
    tiles = t[:, 15].mean()
    print("conv%d  tiles/CTA %.1f  per tile (cycles, mean over CTAs): " % (layer, tiles) +
          "  ".join("%s %.0f" % (names[i], t[:, i].mean() / max(tiles, 1)) for i in (0, 1, 2, 4, 5, 6, 7, 9, 11)), flush=True)
t = np.array(c12[:], dtype=np.float64).reshape(256, 16)[:148]
tiles = t[:, 15].mean()
n12 = ["prod:wait_mel", "prod:conv1_cell", "prod:wait_a_free", "prod:split+store", "iss:wait_acc_free", "iss:wait_a_full",
       "iss:issue", "epi:wait_acc_full", "epi:tmem->stage", "epi:pool+store"]
print("conv12  tiles/CTA %.1f  per tile (cycles): " % tiles + "  ".join("%s %.0f" % (n12[i], t[:, i].mean() / max(tiles, 1)) for i in range(10)), flush=True)
eng.close()
