"""Scratch timing of the hard-decision K=7 kernel only (65,536 frames of N=1024, BSC p=0.03 as in bench.py)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch
import helpers
from commpy_b200.channelcoding import viterbi_decode_batch
tr = helpers.k7()
rs = np.random.RandomState(0)
batch = int(os.environ.get("EXP_BATCH", "65536"))
mode = os.environ.get("EXP_MODE", "hard")
nbits = int(os.environ.get("EXP_NBITS", "1024"))
_, x = helpers.channel_frames(tr, rs, 2048, nbits, mode, "cont", flip=0.03, ebn0_db=4.0)
xt = torch.from_numpy(x.astype(np.uint8 if mode == "hard" else np.float32)).cuda().repeat(batch // 2048, 1).contiguous()
out = torch.empty((batch, nbits), dtype=torch.uint8, device="cuda")
reps = int(os.environ.get("EXP_REPS", "10"))
for _ in range(3):
    viterbi_decode_batch(xt, tr, None, mode, out=out)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(reps):
    viterbi_decode_batch(xt, tr, None, mode, out=out)
e1.record(); torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / reps
print("%s N=%d batch=%d: %.4f ms  %.3e cw/s" % (mode, nbits, batch, ms, batch / ms * 1e3), flush=True)
