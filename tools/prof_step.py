"""Tiny driver for ncu captures: a few passes of ONE wave (default 8 clips x 30 s = 16 chunks)
through the bf16 path.  Usage (under gpurun):
  ncu --set full --clock-control none --import-source on --kernel-name-base demangled \
      -k regex:'attn_tc_kernel' -s 9 -c 3 -o gpurun_out/prof python tools/prof_step.py
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from beat_this_b200 import synthetic
from beat_this_b200.inference import Audio2Beats

n_clips = int(sys.argv[1]) if len(sys.argv) > 1 else 8
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 2
ckpt = synthetic.write_checkpoint(os.path.join(synthetic.cache_dir(), "final0_s0.ckpt"), "final0", 0)
a2b = Audio2Beats(ckpt, "cuda:0", float16=True)
a2b.model.engine.set_wave_chunks(2 * n_clips)
clips = [synthetic.synth_clip(2000 + (i % 4), 30.0).astype("float32") for i in range(n_clips)]
for _ in range(steps):
    out = a2b.batch(clips, 22050)
torch.cuda.synchronize()
print("done", len(out), a2b.model.engine.launches)
