"""Scratch: the 6-iteration turbo decode at the config-3 shape for the kernel / layout switches of cpb_set_option
(EXP_REF=1 also prints the decisions' difference from the round-1 form: per-step rescaling on frame-major arrays)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np, torch, helpers
from commpy_b200 import _lib
from commpy_b200.channelcoding import RandInterlv, turbo_decode_batch

def timeit(fn, reps=3, warm=2):
    for _ in range(warm): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps

rsc = helpers.rsc_k4(); N = 6144; il = RandInterlv(N, 1)
s2 = 1.0 / (2 * (1 / 3) * 10 ** (1.0 / 10))
modes = [("per-step, frame-major", 1, 1), ("block, frame-major", 0, 1), ("block, step-major", 0, 0)]
if not os.environ.get("EXP_REF"):
    modes = modes[1:]
for batch, wins in ((8192, (0,)), (1024, (128,))):
    g = torch.Generator(device="cuda"); g.manual_seed(5)
    y = [(-1 + s2 ** 0.5 * torch.randn(batch, N, device="cuda", generator=g)).float() for _ in range(3)]
    for win in wins:
        _lib.set_option(_lib.OPT_BCJR_WINDOW, win)
        ref = None
        for name, per_step, fm in modes:
            _lib.set_option(_lib.OPT_BCJR_PER_STEP_SCALING, per_step)
            _lib.set_option(_lib.OPT_TURBO_FRAME_MAJOR, fm)
            ms = timeit(lambda: turbo_decode_batch(y[0], y[1], y[2], rsc, s2, 6, il), reps=3, warm=1)
            out = turbo_decode_batch(y[0], y[1], y[2], rsc, s2, 6, il)
            if ref is None: ref = out.clone()
            print("batch %5d window %4d %-22s: turbo 6 it %.3f ms = %.3e cw/s, bits differing from the first row %d of %d" % (
                batch, win or 1024, name, ms, batch / ms * 1e3, int((out != ref).sum()), out.numel()), flush=True)
for o in (_lib.OPT_BCJR_WINDOW, _lib.OPT_BCJR_PER_STEP_SCALING, _lib.OPT_TURBO_FRAME_MAJOR):
    _lib.set_option(o, 0)
