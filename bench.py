#!/usr/bin/env python
"""bench.py -- the decoding hot path on N B200s: one JSON line with throughput, roofline, end-to-end and CPU-baseline
figures for one workload.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl reference] [--no-extras] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W [--workload NAME]

Workloads (BASELINE.json configs; the default is the headline metric's):
    viterbi_k7_n1024_hard   K=7 (0o133,0o171) rate-1/2 hard-decision Viterbi, N=1024           <- default
    viterbi_k7_n1024_soft   same code, soft decision
    viterbi_c2              config 2: soft decision, N=4096, 65,536 frames per launch
    turbo_c3                config 3: rate-1/3 turbo, two K=4 RSC, N=6144, 6 iterations, 8,192 codewords (split over the GPUs)
    ldpc_c4                 config 4: (64800, 32400) min-sum BP, 50 iterations, 128 frames per GPU
    link_c5                 config 5: 256-QAM soft demap + K=7 soft Viterbi link_performance, 5-point Eb/N0 sweep of 1e8 symbols

A "step" is one pass of the hot path over one batch of synthetic frames already resident in HBM (sized so that the
timed region of 20 steps is >= 100 ms): decode kernels + error count, the error counters accumulate on the device and
their all-reduce (the only collective) is issued asynchronously once per step.  Frames shard across ranks with no
data-path collective (weak scaling, except turbo_c3 and link_c5 whose fixed totals -- 8,192 codewords, 1e8 symbols per
point -- are split: strong).  `e2e` times the same
work through the public host-buffer API (pinned host memory, H2D and D2H inside the timed region).
`--impl reference` times the CPU restatement of the reference's algorithm (oracle/, fp64, all host threads) on the same
workload -- the Python reference itself cannot travel to the GPU box (BASELINE.md section 2: ~1.5 codewords/s/core).
`--dump-outputs DIR` writes, after the timed steps, what the last timed step computed as DIR/<name>.npy (float32 / float64,
<= 64 MB in all): the decoded bits (of a fixed seeded sample of frames where they are larger), the LDPC iteration counts or
the link's BER per point, and the step's error counters.  The inputs depend on the arguments only, so two builds run with
the same arguments can be compared output for output.  Keeping the sample is part of the last timed step (Viterbi: one
gather per launch), so time without the flag.
"""
import argparse
import json
import math
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

FALLBACK_HBM_GBS = 6650.0
HEADLINE_METRIC = "codewords/sec (K=7 rate-1/2 Viterbi, N=1024)"


# ------------------------------------------------------------------------------------------------ helpers
def usable_cores():
    """host threads this process may really use: CPU affinity, capped by the cgroup CPU quota when there is one"""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]) + 0.5)))
            else:
                q = int(txt[0])
                per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if q > 0:
                    n = min(n, max(1, int(q / per + 0.5)))
            break
        except Exception:
            continue
    return max(1, n)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst copy bandwidth)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel):
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(kernel)
        except Exception:
            return None
    return None


def bind_to_gpu_numa_node(local_rank):
    """Pin this rank's host threads (and therefore its pinned buffers, first touch) to the NUMA node of its GPU: the
    8-GPU box has GPUs 0-3 on node 0 and 4-7 on node 1, and a pinned buffer on the far node halves the PCIe rate."""
    try:
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(local_rank)
        node = None
        try:
            bus = nv.nvmlDeviceGetPciInfo(h).busId
            bus = bus.decode() if isinstance(bus, bytes) else bus
            path = "/sys/bus/pci/devices/%s/numa_node" % bus.lower()[-12:]
            node = int(open(path).read())
        except Exception:
            node = None
        if node is None or node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        return None
    return None


class ClockSampler:
    """SM clock and throttle reasons sampled through NVML on a host thread DURING the timed region."""

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.sm, self.reasons = [], set()
        self.mx = None
        self._stop = False
        self._t = None

    def _run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.gpu)
            self.mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                     "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                     "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                     "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
            while not self._stop:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                try:
                    fn = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
                    r = int(fn(h))
                    for k, bit in names.items():
                        if r & bit:
                            self.reasons.add(k)
                except Exception:
                    pass
                time.sleep(0.004)
        except Exception as e:          # NVML missing: report no samples rather than fail the bench
            self.err = repr(e)

    def start(self):
        import threading
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        time.sleep(0.05)

    def stop(self):
        self._stop = True
        if self._t is not None:
            self._t.join(timeout=2)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.mx, "reasons": [], "samples": 0, "error": getattr(self, "err", None)}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.mx, "reasons": sorted(self.reasons),
                "samples": len(self.sm)}


def count_errors(dec, msg, counters, torch):
    """cpb_count_errors: counters[0] += differing bits, counters[1] += frames with an error (device side, no sync)"""
    import ctypes as C
    from commpy_b200 import _lib
    L = msg.shape[1]
    rc = _lib.load().cpb_count_errors(_lib.ptr(dec), _lib.ptr(msg), C.c_int64(msg.shape[0]), C.c_int64(L),
                                      C.c_int64(dec.shape[1]), C.c_int64(L), _lib.ptr(counters), _lib.stream_ptr(torch))
    _lib.check(rc, "count_errors")


def dump_rows(n, k):
    """the frames --dump-outputs writes of an output too large to write whole: k of n, a fixed seeded sample, sorted"""
    return np.sort(np.random.RandomState(0).choice(n, min(n, k), replace=False))


# ------------------------------------------------------------------------------------------------ workloads
class Workload:
    """One BASELINE config.  Subclasses fill in: describe() (IDENTICAL in both arms), make(), step(), units, roofline data,
    e2e_*(), parity(), cpu_sample(), outputs()."""
    metric = HEADLINE_METRIC
    unit = "codewords/s"
    scaling = "weak"
    ncounters = 2
    capture = False             # set for the last timed step under --dump-outputs: step() then keeps what it computed

    def units_per_step(self, world):           # whole-job units processed by one step on `world` ranks
        raise NotImplementedError

    def finish(self, counters):
        return {}

    def outputs(self, torch):
        """what the captured step handed its caller, as float32 / float64 numpy arrays by name"""
        raise NotImplementedError


class ViterbiWorkload(Workload):
    """K=7 (0o133, 0o171) rate-1/2 'cont' frames through BSC (hard) or BPSK-AWGN (soft, LLR = 2y/sigma^2)."""

    def __init__(self, name, nbits, launch_frames, launches, mode, flip=0.03, ebn0_db=4.0, metric=None):
        self.name, self.nbits, self.batch, self.launches, self.mode = name, nbits, launch_frames, launches, mode
        self.flip, self.ebn0_db = flip, ebn0_db
        self.n_in = 2 * nbits
        self.dtype = "u8" if mode == "hard" else "int32 fixed-point metrics (f32 LLR in)"
        # SURVEY.md 8(d): coded values in + decoded bits out, u8 bits / f32 soft values
        self.alg_bytes = self.n_in * (1 if mode == "hard" else 4) + nbits
        self.kernel = "viterbi_fast_kernel_%s<FFCode<6,0133,0171>>" % ("hard" if mode == "hard" else "soft")
        if metric:
            self.metric = metric
        self.bound_note = ("add-compare-select issue bound, not HBM bound: 65,856 add-compare-selects per codeword; the "
                           "kernel issues ~0.6 instructions per cycle and scheduler at ~239 instructions per trellis "
                           "step and warp (DESIGN.md 4.1)")

    def describe(self):
        d = {"workload": self.name, "code": "K=7 (0o133,0o171) rate 1/2, 'cont'", "info_bits": self.nbits,
             "coded_values_per_frame": self.n_in, "decoding_type": self.mode, "tb_depth": 30,
             "frames_per_gpu": self.batch * self.launches, "frames_per_launch": self.batch,
             "alg_bytes_per_codeword": self.alg_bytes,
             "l2": "every step streams %d distinct device batches (%.0f MB of input per step, > 126 MB L2)" % (
                 self.launches, self.launches * self.batch * self.n_in * (1 if self.mode == "hard" else 4) / 1e6)}
        d["channel"] = ("BSC p=%.3g" % self.flip) if self.mode == "hard" else ("BPSK AWGN Eb/N0=%.1f dB" % self.ebn0_db)
        return d

    def units_per_step(self, world):
        return world * self.batch * self.launches

    def make(self, torch, rank, world):
        import helpers
        from commpy_b200.channelcoding import conv_encode
        self.trellis = helpers.k7()
        g = torch.Generator(device="cuda")
        g.manual_seed(1000 + rank)
        self.inputs, self.msgs = [], []
        taps = [[b for b in range(7) if (poly >> b) & 1] for poly in (0o133, 0o171)]
        for _ in range(self.launches):
            msg = torch.randint(0, 2, (self.batch, self.nbits), generator=g, device="cuda", dtype=torch.uint8)
            pad = torch.nn.functional.pad(msg, (6, 0))
            coded = torch.empty((self.batch, self.n_in), dtype=torch.uint8, device="cuda")
            for j, tp in enumerate(taps):
                acc = torch.zeros_like(msg)
                for b in tp:
                    acc ^= pad[:, 6 - b:6 - b + self.nbits]
                coded[:, j::2] = acc
            if not hasattr(self, "_checked"):
                ref = conv_encode(msg[0].cpu().numpy(), self.trellis, "cont")
                assert np.array_equal(ref, coded[0].cpu().numpy()), "device encoder disagrees with conv_encode"
                self._checked = True
            if self.mode == "hard":
                flips = (torch.rand(coded.shape, generator=g, device="cuda") < self.flip).to(torch.uint8)
                x = coded ^ flips
            else:
                sigma2 = 1.0 / (2.0 * 0.5 * 10 ** (self.ebn0_db / 10.0))
                y = (2.0 * coded.float() - 1.0) + (sigma2 ** 0.5) * torch.randn(coded.shape, generator=g, device="cuda")
                x = (2.0 / sigma2) * y if self.mode == "soft" else y
            self.inputs.append(x.contiguous())
            self.msgs.append(msg)
            del coded, pad
        self.out = torch.empty((self.batch, self.nbits), dtype=torch.uint8, device="cuda")
        self.dump_idx = torch.from_numpy(dump_rows(self.batch, 512)).cuda()
        self.kernel_launches_per_step = self.launches * (2 if self.mode == "hard" else 3)   # decode [+ frame scale] + count

    def step(self, torch, counters, ev=None):
        from commpy_b200.channelcoding import viterbi_decode_batch
        kept = [] if self.capture else None
        for i in range(self.launches):
            if ev is not None and i == 0:
                ev[0].record()
            viterbi_decode_batch(self.inputs[i], self.trellis, None, self.mode, out=self.out)
            if ev is not None and i == 0:
                ev[1].record()
            if kept is not None:                 # every launch overwrites self.out: keep the sampled frames of each
                kept.append(self.out.index_select(0, self.dump_idx))
            count_errors(self.out, self.msgs[i], counters, torch)
        if kept is not None:
            self.kept = kept

    def outputs(self, torch):
        """decoded bits of the same 512 sampled frames of every launch: (launches, 512, nbits)"""
        return {"decoded_bits": torch.stack(self.kept).float().cpu().numpy()}

    def kernel_units(self):                      # units the event-timed launch processes
        return self.batch

    def finish(self, counters, steps=1, world=1):
        bits = self.units_per_step(world) * steps * self.nbits
        return {"bit_errors": int(counters[0]), "frame_errors": int(counters[1]), "bits": int(bits),
                "ber": float(counters[0]) / max(bits, 1)}

    # ---- end to end: host buffers through the public API
    def e2e_setup(self, torch):
        """host copies of the WHOLE step's frames (all launches): one API call decodes them, chunked and pipelined inside"""
        from commpy_b200.channelcoding import viterbi_decode_batch
        frames = self.batch * self.launches
        info = {"frames_per_call": frames}
        x0 = self.inputs[0]
        if self.mode == "hard":
            self.h_pin = torch.empty((frames, self.n_in // 8), dtype=torch.uint8).pin_memory()
            for i, x in enumerate(self.inputs):
                self.h_pin[i * self.batch:(i + 1) * self.batch] = torch.from_numpy(np.packbits(x.cpu().numpy(), axis=1))
            self.h_pout = torch.empty((frames, self.nbits // 8), dtype=torch.uint8).pin_memory()
            # byte-per-bit comparison arm: a quarter of the step (pinning 3 GB only to show the PCIe bound is not worth it)
            q = max(1, self.launches // 4)
            self.h_in = torch.empty((q * self.batch, self.n_in), dtype=torch.uint8).pin_memory()
            for i in range(q):
                self.h_in[i * self.batch:(i + 1) * self.batch] = self.inputs[i].cpu()
            self.h_out = torch.empty((q * self.batch, self.nbits), dtype=torch.uint8).pin_memory()
            # the packed call must give the bits of the byte-per-bit call
            a = viterbi_decode_batch(self.h_pin, self.trellis, None, "hard", out=self.h_pout, packed=True)
            b = viterbi_decode_batch(self.h_in, self.trellis, None, "hard", out=self.h_out)
            assert np.array_equal(np.unpackbits(a[:len(b)].numpy(), axis=1), b.numpy()), "packed decode disagrees"
            info.update(api="commpy_b200.channelcoding.viterbi_decode_batch(pinned host array, packed=True) -> "
                            "cpb_viterbi_decode_host_packed (1 bit per coded / decoded bit, numpy.packbits order)",
                        h2d=self.h_pin.numel(), d2h=self.h_pout.numel())
        else:
            self.h_in = torch.empty((frames, self.n_in), dtype=x0.dtype).pin_memory()
            for i, x in enumerate(self.inputs):
                self.h_in[i * self.batch:(i + 1) * self.batch] = x.cpu()
            self.h_out = torch.empty((frames, self.nbits), dtype=torch.uint8).pin_memory()
            info.update(api="commpy_b200.channelcoding.viterbi_decode_batch(pinned host array) -> cpb_viterbi_decode_host",
                        h2d=self.h_in.numel() * self.h_in.element_size(), d2h=self.h_out.numel())
        return info

    def e2e_step(self):
        from commpy_b200.channelcoding import viterbi_decode_batch
        if self.mode == "hard":
            viterbi_decode_batch(self.h_pin, self.trellis, None, "hard", out=self.h_pout, packed=True)
        else:
            viterbi_decode_batch(self.h_in, self.trellis, None, self.mode, out=self.h_out)

    def e2e_alt(self):
        """hard decision only: the byte-per-bit host call (3 KB per codeword across PCIe), reported next to the packed one"""
        if self.mode != "hard":
            return None
        from commpy_b200.channelcoding import viterbi_decode_batch
        return (lambda: viterbi_decode_batch(self.h_in, self.trellis, None, "hard", out=self.h_out),
                {"api": "viterbi_decode_batch(pinned uint8 array, one byte per bit) -> cpb_viterbi_decode_host",
                 "frames_per_call": int(self.h_in.shape[0]),
                 "h2d_bytes_per_call": self.h_in.numel(), "d2h_bytes_per_call": self.h_out.numel()})

    def parity(self, torch, frames=48):
        """decode a few frames with the CPU oracle and compare (outside every timed region)"""
        from oracle import oracle
        from commpy_b200.channelcoding import viterbi_decode_batch
        viterbi_decode_batch(self.inputs[0], self.trellis, None, self.mode, out=self.out)
        torch.cuda.synchronize()
        x = self.inputs[0][:frames].cpu().numpy().astype(np.float64)
        want = oracle.viterbi_decode_batch(x, self.trellis, None, self.mode, threads=min(8, os.cpu_count() or 1))
        got = self.out[:frames].cpu().numpy()
        m = self.msgs[0][:frames].cpu().numpy()
        return {"frames_checked": frames, "bit_mismatches_vs_oracle": int((got != want).sum()),
                "oracle_bit_errors": int((want != m).sum()), "gpu_bit_errors": int((got != m).sum())}

    # ---- CPU restatement of the reference on the same recipe
    def cpu_make(self, frames, seed):
        import helpers
        rs = np.random.RandomState(seed)
        _, x = helpers.channel_frames(helpers.k7(), rs, frames, self.nbits, self.mode, "cont", flip=self.flip, ebn0_db=self.ebn0_db)
        return x

    def cpu_run(self, x, threads):
        import helpers
        from oracle import oracle
        oracle.viterbi_decode_batch(x, helpers.k7(), None, self.mode, threads=threads)
        return len(x)

    cpu_what = "oracle/commpy_oracle.c (fp64 restatement of convcode.py:561-749)"


class TurboWorkload(Workload):
    """Config 3: rate-1/3 turbo code, two K=4 RSC (8 states), RandInterlv(6144, 1), 6 iterations, Eb/N0 = 1 dB, all-zero
    codewords (-1 + noise); 8,192 codewords per step over all ranks."""
    metric = "codewords/sec (rate-1/3 turbo, 2x K=4 RSC, N=6144, 6 iterations)"
    scaling = "strong"

    def __init__(self):
        self.name, self.N, self.total, self.iters = "turbo_c3", 6144, 8192, 6
        self.dtype = "f32"
        self.alg_bytes = 3 * self.N * 4 + self.N             # SURVEY 8(d): compulsory
        self.kernel = "turbo iteration kernels (cpb_turbo_decode)"
        self.bound_note = "issue / latency bound in the MAP recursions; HBM fraction against the compulsory 79,872 B per codeword"

    def describe(self):
        return {"workload": self.name, "code": "rate-1/3 turbo, 2 x RSC K=4 (1, 15/13 octal), RandInterlv(6144, seed 1)",
                "info_bits": self.N, "iterations": self.iters, "codewords_per_step_all_gpus": self.total,
                "map_window": "commpy_b200.channelcoding.suggest_map_window(codewords per GPU, N): 1024 steps at 8,192 "
                              "codewords per GPU, 128 at 1,024 (CPB_OPT_BCJR_WINDOW; 96 warm-up steps either side always)",
                "channel": "BPSK AWGN Eb/N0=1.0 dB, all-zero codewords", "alg_bytes_per_codeword": self.alg_bytes,
                "l2": "inputs of one step (%.0f MB over all GPUs) exceed the 126 MB L2" % (3 * self.total * self.N * 4 / 1e6)}

    def units_per_step(self, world):
        return self.total

    def make(self, torch, rank, world):
        import helpers
        from commpy_b200 import parallel
        from commpy_b200.channelcoding import RandInterlv
        self.trellis = helpers.rsc_k4()
        self.il = RandInterlv(self.N, 1)
        lo, hi = parallel.shard_range(self.total, rank, world)
        self.batch = hi - lo
        from commpy_b200.channelcoding import set_map_window, suggest_map_window
        self.window = suggest_map_window(self.total // world, self.N)        # the same on every rank
        set_map_window(self.window)
        self.s2 = 1.0 / (2 * (1 / 3) * 10 ** (1.0 / 10))
        g = torch.Generator(device="cuda")
        g.manual_seed(2000 + rank)
        self.y = [(-1 + self.s2 ** 0.5 * torch.randn(self.batch, self.N, device="cuda", generator=g)).float() for _ in range(3)]
        self.zero = torch.zeros((self.batch, self.N), dtype=torch.uint8, device="cuda")
        self.kernel_launches_per_step = 2 * self.iters + 5      # 3 transposes in, 2 MAP passes per iteration, decisions out, error count

    def step(self, torch, counters, ev=None):
        from commpy_b200.channelcoding import turbo_decode_batch
        if ev is not None:
            ev[0].record()
        bits = turbo_decode_batch(self.y[0], self.y[1], self.y[2], self.trellis, self.s2, self.iters, self.il)
        if ev is not None:
            ev[1].record()
        count_errors(bits, self.zero, counters, torch)
        if self.capture:
            self.last_bits = bits

    def outputs(self, torch):
        """decoded bits of 1,024 sampled codewords of this rank: (1024, N)"""
        rows = torch.from_numpy(dump_rows(self.batch, 1024)).cuda()
        return {"decoded_bits": self.last_bits.index_select(0, rows).float().cpu().numpy()}

    def kernel_units(self):
        return self.batch

    def finish(self, counters, steps=1, world=1):
        bits = self.total * steps * self.N
        return {"bit_errors": int(counters[0]), "frame_errors": int(counters[1]), "bits": int(bits), "ber": float(counters[0]) / bits}

    def e2e_setup(self, torch):
        self.h = [t.cpu().pin_memory() for t in self.y]
        self.h_out = torch.empty((self.batch, self.N), dtype=torch.uint8).pin_memory()
        self.h_np = [t.numpy() for t in self.h]
        return {"frames_per_call": self.batch, "h2d": 3 * self.batch * self.N * 4, "d2h": self.batch * self.N,
                "api": "commpy_b200.channelcoding.turbo_decode_batch_host(pinned host arrays) -> cpb_turbo_decode_host"}

    def e2e_step(self):
        from commpy_b200.channelcoding import set_map_window, suggest_map_window, turbo_decode_batch_host
        set_map_window(suggest_map_window(min(self.batch, 2048), self.N))     # the host pipeline decodes chunks of <= 2,048 codewords
        self.e2e_bits = turbo_decode_batch_host(self.h_np[0], self.h_np[1], self.h_np[2], self.trellis, self.s2, self.iters, self.il,
                                                out=self.h_out)

    def e2e_alt(self):
        return None

    def parity(self, torch, frames=4):
        from oracle import oracle
        from commpy_b200.channelcoding import turbo_decode_batch
        got = turbo_decode_batch(self.y[0][:frames], self.y[1][:frames], self.y[2][:frames], self.trellis, self.s2, self.iters, self.il)
        want = oracle.turbo_decode_batch(*(t[:frames].cpu().numpy() for t in self.y), self.trellis, self.s2, self.iters, self.il, threads=4)
        return {"frames_checked": frames, "bit_mismatches_vs_oracle": int((got.cpu().numpy() != want).sum()), "bits": int(want.size)}

    def cpu_make(self, frames, seed):
        rs = np.random.RandomState(seed)
        s2 = 1.0 / (2 * (1 / 3) * 10 ** (1.0 / 10))
        return [-1 + np.sqrt(s2) * rs.randn(frames, self.N) for _ in range(3)]

    def cpu_run(self, x, threads):
        import helpers
        from oracle import oracle
        from commpy_b200.channelcoding import RandInterlv
        s2 = 1.0 / (2 * (1 / 3) * 10 ** (1.0 / 10))
        oracle.turbo_decode_batch(x[0], x[1], x[2], helpers.rsc_k4(), s2, self.iters, RandInterlv(self.N, 1), threads=threads)
        return len(x[0])

    cpu_what = "oracle/commpy_oracle.c (fp64 restatement of turbo.py:62-333)"


class LdpcWorkload(Workload):
    """Config 4: (64800, 32400) min-sum BP, 50 iterations, 128 frames per GPU (1,024 on 8), all-zero codeword at Eb/N0 = 1 dB
    (this graph does not converge there: all 50 iterations run)."""
    metric = "codewords/sec ((64800,32400) LDPC min-sum BP, 50 iterations)"

    def __init__(self):
        self.name, self.n, self.batch, self.iters = "ldpc_c4", 64800, 128, 50
        self.dtype = "f32"
        self.kernel = "bulk::cn_bulk_kernel + vn_kernel (per iteration)"
        self.bound_note = "HBM bound: 12 E + 8 n bytes per frame-iteration (SURVEY 8d)"

    def describe(self):
        return {"workload": self.name, "code": "(64800, 32400) DVB-S2-SHAPED surrogate matrix (tests/helpers.py::dvbs2_like_H), 226,799 edges",
                "algorithm": "MSA", "max_iterations": self.iters, "frames_per_gpu": self.batch,
                "channel": "BPSK AWGN Eb/N0=1.0 dB, all-zero codeword", "alg_bytes_per_frame_iteration": 12 * 226799 + 8 * 64800,
                "l2": "the messages of one step (%.0f MB) exceed the 126 MB L2" % (self.batch * 226799 * 4 / 1e6)}

    def units_per_step(self, world):
        return world * self.batch

    def make(self, torch, rank, world):
        import helpers
        self.H = helpers.dvbs2_like_H()
        self.params = {"n_vnodes": self.n, "n_cnodes": 32400, "parity_check_matrix": self.H.tocsc()}
        sigma = 1.0 / (2 * 0.5 * 10 ** (1.0 / 10)) ** 0.5
        g = torch.Generator(device="cuda")
        g.manual_seed(3000 + rank)
        self.llr = (2.0 * (1.0 + sigma * torch.randn(self.batch, self.n, device="cuda", generator=g)) / sigma ** 2).float()
        self.work = self.llr.clone()
        self.zero = torch.zeros((self.batch, self.n), dtype=torch.uint8, device="cuda")
        self.bytes_fi = 12 * self.H.nnz + 8 * self.n
        self.alg_bytes = self.iters * self.bytes_fi + 5 * self.n
        self.kernel_launches_per_step = 2 * self.iters + 4
        self.mean_it = None

    def step(self, torch, counters, ev=None):
        from commpy_b200.channelcoding import ldpc_bp_decode_batch
        self.work.copy_(self.llr)
        if ev is not None:
            ev[0].record()
        dec, it = ldpc_bp_decode_batch(self.work, self.params, self.iters, "fp32", return_llrs=False, return_iters=True)
        if ev is not None:
            ev[1].record()
        self.last_it = it
        count_errors(dec, self.zero, counters, torch)
        if self.capture:
            self.last_dec = dec

    def outputs(self, torch):
        """hard decisions of every frame (batch, n) and the iterations each frame ran (batch,)"""
        return {"decoded_bits": self.last_dec.float().cpu().numpy(), "iterations": self.last_it.float().cpu().numpy()}

    def kernel_units(self):
        return self.batch

    def finish(self, counters, steps=1, world=1):
        bits = self.units_per_step(world) * steps * self.n
        return {"bit_errors": int(counters[0]), "frame_errors": int(counters[1]), "bits": int(bits),
                "mean_iterations": float(self.last_it.float().mean())}

    def e2e_setup(self, torch):
        self.h_llr = self.llr.cpu().pin_memory()
        self.h_np = self.h_llr.numpy()
        self.h_dec = torch.empty((self.batch, self.n), dtype=torch.uint8).pin_memory()
        return {"frames_per_call": self.batch, "h2d": self.batch * self.n * 4, "d2h": self.batch * self.n,
                "api": "commpy_b200.channelcoding.ldpc_bp_decode_batch_host(pinned host array) -> cpb_ldpc_decode_host"}

    def e2e_step(self):
        from commpy_b200.channelcoding import ldpc_bp_decode_batch_host
        self.e2e_dec = ldpc_bp_decode_batch_host(self.h_np, self.params, self.iters, "fp32", return_llrs=False, out=self.h_dec)

    def e2e_alt(self):
        return None

    def parity(self, torch, frames=2):
        from oracle import oracle
        from commpy_b200.channelcoding import ldpc_bp_decode_batch
        x = self.llr[:frames].double()
        dec, it = ldpc_bp_decode_batch(x.clone(), self.params, 8, "fp64", return_llrs=False, return_iters=True)
        want, _, wit = oracle.ldpc_bp_decode(x.cpu().numpy().reshape(-1).copy(), self.params, "MSA", 8, return_iters=True, threads=2)
        want = want.reshape(self.n, frames).T if frames > 1 else want[None, :]
        return {"frames_checked": frames, "iterations": 8, "precision": "fp64 parity mode",
                "bit_mismatches_vs_oracle": int((dec.cpu().numpy() != want).sum())}

    def cpu_make(self, frames, seed):
        rs = np.random.RandomState(seed)
        sigma = 1.0 / (2 * 0.5 * 10 ** (1.0 / 10)) ** 0.5
        return 2.0 * (1.0 + sigma * rs.randn(frames, self.n)) / sigma ** 2

    def cpu_run(self, x, threads):
        import helpers
        from oracle import oracle
        if not hasattr(self, "_cpu_params"):
            self._cpu_params = {"n_vnodes": self.n, "n_cnodes": 32400, "parity_check_matrix": helpers.dvbs2_like_H().tocsc()}
        oracle.ldpc_bp_decode(x.reshape(-1).copy(), self._cpu_params, "MSA", self.iters, threads=threads)
        return len(x)

    cpu_what = "oracle/commpy_oracle.c (fp64 restatement of ldpc.py:144-254)"


class LinkWorkload(Workload):
    """Config 5: 256-QAM + K=7 rate-1/2 'cont' frames of 4096 bits (1024 symbols), soft demapper + soft Viterbi,
    link_performance over a 5-point Eb/N0 sweep, ~1e8 symbols per point over all ranks; one step = the whole sweep."""
    metric = "symbols/sec (256-QAM soft demap + K=7 soft Viterbi link_performance sweep)"
    unit = "symbols/s"
    scaling = "strong"
    ncounters = 3

    def __init__(self):
        self.name = "link_c5"
        self.frame_bits, self.frames_point = 4096, 98304          # 98,304 frames x 1024 symbols = 1.007e8 symbols
        self.ebn0 = [8.0, 10.0, 12.0, 14.0, 16.0]
        self.dtype = "f32 LLRs, int32 fixed-point Viterbi metrics"
        self.alg_bytes = 12.0                                      # per symbol: 8 B in + 4 decoded bits out (SURVEY 8d)
        self.kernel = "conv_link_tx -> demod_soft -> viterbi_fast_kernel_soft -> count_errors"
        self.bound_note = "symbols are generated on the device (no compulsory HBM input); fraction quoted against 12 B per symbol"

    def describe(self):
        return {"workload": self.name, "modem": "QAMModem(256), Es=170", "code": "K=7 (0o133,0o171) rate 1/2, 'cont', 4096-bit frames",
                "decoding_type": "soft", "tb_depth": 30, "ebn0_db": self.ebn0, "symbols_per_point_all_gpus": self.frames_point * 1024,
                "frames_per_batch_per_gpu": "frames_per_point / n_gpus (one batch per point)", "alg_bytes_per_symbol": self.alg_bytes,
                "l2": "one batch of symbols + LLRs is > 1 GB per GPU at N=1"}

    def units_per_step(self, world):
        return len(self.ebn0) * self.frames_point * 1024

    def make(self, torch, rank, world):
        import helpers
        from commpy_b200.links import ConvLinkGPU
        from commpy_b200.modulation import QAMModem
        self.world = world
        fpb = self.frames_point // world
        self.link = ConvLinkGPU(helpers.k7(), QAMModem(256), frame_bits=self.frame_bits, frames_per_batch=fpb, decoding_type="soft", seed=4)
        self.snrs = [e + 10 * math.log10(8) for e in self.ebn0]
        self.kernel_launches_per_step = len(self.ebn0) * 2 * 5 + len(self.ebn0) * 5
        self.bers = None

    def step(self, torch, counters, ev=None):
        if ev is not None:
            ev[0].record()
        send_max = self.frames_point * self.frame_bits
        self.bers, tot = self.link.link_performance(self.snrs, send_max=send_max, err_min=10 ** 12, return_counters=True,
                                                    stop_early=False)
        if ev is not None:
            ev[1].record()
        counters += tot

    def outputs(self, torch):
        """BER of every point of the sweep"""
        return {"ber_per_point": np.asarray(self.bers, dtype=np.float64)}

    def kernel_units(self):
        return self.units_per_step(1)

    def own_collective(self):
        return True

    def finish(self, counters, steps=1, world=1):
        return {"ber_per_point": [float(b) for b in self.bers], "ebn0_db": self.ebn0, "bit_errors": int(counters[0]),
                "bits": int(counters[2])}

    def e2e_setup(self, torch):
        return None

    def parity(self, torch, frames=4):
        from oracle import oracle
        import helpers
        msg, y, nv = self.link.make_batch(self.snrs[2], 0, torch)
        cnt = torch.zeros(3, dtype=torch.int64, device="cuda")
        dec = self.link.receive_decode_count(msg, y, nv, cnt, torch)[:frames].cpu().numpy()
        yy = y[:frames].cpu().numpy()
        want = []
        for f in range(frames):
            llr = oracle.demodulate(self.link.modem, yy[f].astype(np.complex128), "soft", nv)
            want.append(oracle.viterbi_decode(llr, helpers.k7(), None, "soft"))
        want = np.array(want)
        return {"frames_checked": frames, "bit_mismatches_vs_oracle": int((dec != want).sum()), "bits": int(want.size)}

    def cpu_make(self, frames, seed):
        import helpers
        from commpy_b200.modulation import QAMModem
        rs = np.random.RandomState(seed)
        q = QAMModem(256)
        msgs = rs.randint(0, 2, (frames, self.frame_bits))
        coded = helpers.encode_batch(msgs, helpers.k7(), "cont")
        ns = math.sqrt(2 * q.Es / (0.5 * 10 ** ((12.0 + 10 * math.log10(8)) / 10)))
        y = np.array([q.modulate(c) for c in coded]) + 0.5 * ns * (rs.randn(frames, 1024) + 1j * rs.randn(frames, 1024))
        return (q, y, ns ** 2)

    def cpu_run(self, x, threads):
        import helpers
        from concurrent.futures import ThreadPoolExecutor
        from oracle import oracle
        q, y, nv = x
        tr = helpers.k7()

        def one(f):
            llr = oracle.demodulate(q, y[f], "soft", nv)
            oracle.viterbi_decode(llr, tr, None, "soft")
        with ThreadPoolExecutor(threads) as ex:
            list(ex.map(one, range(len(y))))
        return y.size

    cpu_what = "oracle/commpy_oracle.c (fp64 restatement of modulation.py:100-141 + convcode.py:561-749)"


WORKLOADS = {
    "viterbi_k7_n1024_hard": lambda: ViterbiWorkload("viterbi_k7_n1024_hard", 1024, 65536, 16, "hard"),
    "viterbi_k7_n1024_soft": lambda: ViterbiWorkload("viterbi_k7_n1024_soft", 1024, 65536, 8, "soft",
                                                     metric="codewords/sec (K=7 rate-1/2 soft-decision Viterbi, N=1024)"),
    "viterbi_c2": lambda: ViterbiWorkload("viterbi_c2", 4096, 65536, 2, "soft",
                                          metric="codewords/sec (K=7 rate-1/2 soft-decision Viterbi, N=4096, batch 65536)"),
    "turbo_c3": TurboWorkload,
    "ldpc_c4": LdpcWorkload,
    "link_c5": LinkWorkload,
}
DEFAULT_WORKLOAD = "viterbi_k7_n1024_hard"


def timed_cpu(wl, threads, target_s):
    """oracle on a bounded sample: pilot to size it, then one timed run.  Returns (units/s, units, seconds, frames)."""
    nf = max(2, min(2 * threads, 64))
    pilot = wl.cpu_make(nf, seed=1)
    wl.cpu_run(pilot, threads)                  # (loads the library, warms the caches)
    t0 = time.perf_counter()
    wl.cpu_run(pilot, threads)
    dt = max(time.perf_counter() - t0, 1e-4)
    frames = int(max(nf, min(65536, nf * target_s / dt)))
    x = wl.cpu_make(frames, seed=2)
    t0 = time.perf_counter()
    units = wl.cpu_run(x, threads)
    dt = time.perf_counter() - t0
    return units / dt, units, dt, frames


# ------------------------------------------------------------------------------------------------ reference arm
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    wl = WORKLOADS[args.workload]()
    threads = usable_cores()
    per_step = []
    frames_step = None
    for s in range(args.warmup + args.steps):
        rate, units, dt, frames = timed_cpu(wl, threads, target_s=2.0)
        frames_step = frames
        if s >= args.warmup:
            per_step.append((units, dt))
    tot_u = sum(u for u, _ in per_step)
    tot_t = sum(t for _, t in per_step)
    value = tot_u / tot_t
    line = {
        "impl": "reference", "metric": wl.metric, "value": value, "unit": wl.unit, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / max(1, args.steps),
        "higher_is_better": True, "scaling": wl.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": wl.describe(),
        "cpu_baseline": {"value": value, "unit": wl.unit, "cores": threads, "kind": "port",
                         "sample": "%d frames per step of the same recipe, %s over %d host threads" % (frames_step, wl.cpu_what, threads)},
        "e2e": {"value": value, "unit": wl.unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "the Python reference cannot run on the GPU box; its measured rate in the build container is "
                "~1.5 codewords/s/core for this Viterbi shape (BASELINE.md section 2)",
    }
    emit(line)
    return 0


# ------------------------------------------------------------------------------------------------ B200 arm
def run_b200(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    numa = bind_to_gpu_numa_node(local) if world > 1 else None
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    wl = WORKLOADS[args.workload]()
    wl.make(torch, rank, world)
    K, W = args.steps, args.warmup
    own = getattr(wl, "own_collective", lambda: False)()
    counters = torch.zeros(wl.ncounters, dtype=torch.int64, device="cuda")      # this rank's running totals
    snaps = [torch.zeros(wl.ncounters, dtype=torch.int64, device="cuda") for _ in range(4)]
    pending = []

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step(i, ev=None):
        wl.step(torch, counters, ev)
        if world > 1 and not own:
            # the only collective: the int64 error counters.  Snapshot + asynchronous all-reduce on NCCL's own stream:
            # the decode stream never waits for it (SURVEY 8e: "hidden by running ahead")
            s = snaps[i % len(snaps)]
            s.copy_(counters)
            pending.append(dist.all_reduce(s, op=dist.ReduceOp.SUM, async_op=True))
            if len(pending) >= len(snaps) - 1:
                pending.pop(0).wait()

    for i in range(W):
        step(i)
    for w_ in pending:
        w_.wait()
    pending.clear()
    barrier()
    counters.zero_()
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    e0.record()
    for i in range(K):
        if args.dump_outputs and i == K - 1:
            wl.capture = True
            last_start = counters.clone()
        step(i, kev[i])
    for w_ in pending:
        w_.wait()
    pending.clear()
    e1.record()
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        # before the end-to-end and parity calls below, which reuse the buffers the last step wrote
        outs = wl.outputs(torch)
        outs["error_counters"] = (counters - last_start).cpu().numpy().astype(np.float64)
        dump_outputs(args.dump_outputs, outs)
    ms_total = e0.elapsed_time(e1)
    kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in kev]))
    t = torch.tensor([ms_total, kernel_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, kernel_ms = float(t[0]), float(t[1])
    glob = counters.clone()
    if world > 1 and not own:
        dist.all_reduce(glob, op=dist.ReduceOp.SUM)
    glob = glob.cpu().numpy().astype(np.int64)
    value = wl.units_per_step(world) * K / (ms_total / 1e3)

    # ---- end to end through the public host-buffer API (pinned host memory in, pinned host memory out)
    e2e = None
    info = wl.e2e_setup(torch)
    if info is not None:
        Ke = max(3, min(K, 10))

        def time_calls(fn):
            fn()
            barrier()
            t0 = time.perf_counter()
            for _ in range(Ke):
                fn()
            torch.cuda.synchronize()
            te = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(te, op=dist.ReduceOp.MAX)
            return float(te[0])
        dt = time_calls(wl.e2e_step)
        per_call_units = info["frames_per_call"] * world          # every rank makes the call on its own shard
        e2e = {"value": per_call_units * Ke / dt, "unit": wl.unit, "h2d_bytes_per_step": int(info["h2d"]),
               "d2h_bytes_per_step": int(info["d2h"]), "steps": Ke, "frames_per_step_per_gpu": info["frames_per_call"],
               "api": info["api"]}
        alt = wl.e2e_alt()
        if alt is not None:
            fn, ainfo = alt
            dta = time_calls(fn)
            e2e["byte_per_bit"] = dict(ainfo, value=ainfo["frames_per_call"] * world * Ke / dta, unit=wl.unit)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    peak, peak_src = measured_peak()
    achieved = wl.alg_bytes * wl.kernel_units() / (kernel_ms / 1e3) / 1e9
    line = {
        "metric": wl.metric, "value": value, "unit": wl.unit, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": wl.scaling, "vs_baseline": None,
        "dtype": wl.dtype, "data": "synthetic", "config": wl.describe(),
        "parallelism": "frames sharded over %d GPU(s), no data-path collective; int64 error counters all-reduced "
                       "asynchronously once per step" % world,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": ncu_traffic(wl.kernel), "kernel": wl.kernel, "kernel_ms": kernel_ms,
                     "units_per_timed_launch": wl.kernel_units(), "peak_source": peak_src, "note": wl.bound_note},
        "gpu_launches": int(wl.kernel_launches_per_step * K),
        "clocks": clocks,
        "result": wl.finish(glob, K, world),
    }
    if numa is not None:
        line["numa_node"] = numa
    if e2e is not None:
        line["e2e"] = e2e
    else:
        line["e2e"] = {"value": value, "unit": wl.unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 24,
                       "note": "the link generates its frames on the device (cpb_conv_link_tx): nothing but the three "
                               "counters crosses PCIe, so the device-timed sweep IS the end-to-end call"}
    if world == 1:
        line["parity"] = wl.parity(torch)
        threads = usable_cores()
        rate, units, dt, frames = timed_cpu(wl, threads, target_s=12.0)
        line["cpu_baseline"] = {"value": rate, "unit": wl.unit, "cores": threads, "kind": "port",
                                "sample": "%d frames of the same recipe in %.1f s: %s, %d host threads" % (frames, dt, wl.cpu_what, threads)}
        if not args.no_extras and args.workload == DEFAULT_WORKLOAD:
            line["extras"] = run_extras(torch)
    emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


def run_extras(torch):
    """The other configs, timed briefly on the same GPU (device-resident inputs, CUDA events).  A failure here FAILS the
    bench: an extra that cannot run is a broken hot path."""
    out = {}
    peak, _ = measured_peak()
    for name in ("viterbi_k7_n1024_soft", "viterbi_c2", "turbo_c3", "ldpc_c4", "link_c5"):
        wl = WORKLOADS[name]()
        wl.make(torch, 0, 1)
        counters = torch.zeros(wl.ncounters, dtype=torch.int64, device="cuda")
        wl.step(torch, counters)
        torch.cuda.synchronize()
        counters.zero_()
        reps = 2
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for r in range(reps):
            wl.step(torch, counters, evs[r])
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / reps
        kms = float(np.mean([x.elapsed_time(y) for x, y in evs]))
        rec = {"metric": wl.metric, "value": wl.units_per_step(1) / ms * 1e3, "unit": wl.unit, "ms_per_step": ms,
               "kernel_ms": kms, "roofline_frac": wl.alg_bytes * wl.kernel_units() / kms / 1e6 / peak,
               "result": wl.finish(counters.cpu().numpy(), reps, 1), "parity": wl.parity(torch)}
        out[name] = rec
        del wl
        torch.cuda.empty_cache()
    from commpy_b200.modulation import QAMModem
    q = QAMModem(256)
    n = 1 << 24
    y = torch.view_as_complex((torch.randn(n, 2, device="cuda") * 9).contiguous())
    for _ in range(2):
        q.demodulate_batch(y, "soft", 12.0)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(5):
        q.demodulate_batch(y, "soft", 12.0)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / 5
    out["demap_qam256_soft"] = {"value": n / ms * 1e3, "unit": "symbols/s", "ms": ms, "roofline_frac": 40.0 * n / ms / 1e6 / peak}
    return out


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """--dump-outputs: DIR/<name>.npy per array, float32 / float64 only, at most 64 MB in all"""
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT_BYTES, "outputs to dump take %d bytes" % total
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(path, name + ".npy"), a)


_JSON_FD = None


def emit(line):
    """The one JSON line of the contract, written to the REAL stdout (see main())."""
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    # stdout carries exactly one JSON line.  Libraries may print to fd 1 (NCCL's version banner does when NCCL_DEBUG is
    # set in the environment), so fd 1 is pointed at stderr for the whole run and the line goes to a saved copy.
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (B200 arm, rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 arm")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
