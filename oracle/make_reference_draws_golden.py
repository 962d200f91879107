"""Outputs of the UNMODIFIED reference on the random draws of tests/test_oracle_live_reference.py, for a fixed list of
seeds, so that the test replays them without the reference checkout:

    python oracle/make_reference_draws_golden.py     # writes tests/golden/reference_draws.npz (seconds)

Each seed draws exactly what the test drew from it when it ran the reference directly: Viterbi frames of the K=7 code in
every decoding mode and termination, one map_decode frame of the K=4 RSC, a Gallager (96, 33) min-sum decode, 16-QAM
soft / hard demapping, and the MIMO detectors (kbest, best_first_detector, idd_decoder).  Every array is stacked over
the seeds (first axis).  The design file is not copied: the test rebuilds the parity-check matrix from
tests/golden/ldpc_design.npz.  TEST INFRASTRUCTURE ONLY."""
import importlib
import os
import sys
import warnings
from collections import defaultdict

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path = [p for p in sys.path if os.path.abspath(p or ".") != HERE]
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import numpy as np

import refimport

GOLD = os.path.join(os.path.dirname(HERE), "tests", "golden")
SEEDS = tuple(range(8))
MIMO_SEEDS = (0, 1, 2)
MIMO_SHAPES = ((4, 2), (16, 3), (16, 4))
VITERBI_CASES = tuple((mode, term, tb) for mode in ("hard", "soft", "unquantized") for term, tb in (("cont", None), ("term", 9)))


def viterbi_and_bcjr(rcc, seed, out):
    rs = np.random.RandomState(seed)
    k7 = rcc.Trellis(np.array([6]), np.array([[0o133, 0o171]]))
    rsc = rcc.Trellis(np.array([3]), np.array([[1, 0o15]]), np.array([[0o13]]), "rsc")
    for mode, term, tb in VITERBI_CASES:
        msg = rs.randint(0, 2, 48)
        coded = rcc.conv_encode(msg, k7, term).astype(float)
        if mode == "hard":
            x = np.abs(coded - (rs.rand(len(coded)) < 0.1))
        elif mode == "soft":
            x = (2 * coded - 1) * 2 + rs.randn(len(coded)) * 2.5
        else:
            x = (2 * coded - 1) + rs.randn(len(coded))
        out["vit_%s_%s_x" % (mode, term)].append(x)
        out["vit_%s_%s_ref" % (mode, term)].append(rcc.viterbi_decode(x.copy(), k7, tb, mode))
    N, s2 = 40, 0.9
    sys_, par, la = (-1 + np.sqrt(s2) * rs.randn(N) for _ in range(3))
    with np.errstate(all="ignore"):
        L, bits = rcc.map_decode(sys_, par, rsc, s2, 0.2 * la, "decode")
    for k, v in (("sys", sys_), ("par", par), ("La", 0.2 * la), ("L", L), ("bits", bits)):
        out["map_" + k].append(v)


def ldpc_and_demapper(rcc, rmod, seed, out):
    rs = np.random.RandomState(seed + 1)
    params = rcc.get_ldpc_code_params(os.path.join(refimport.REF_ROOT, "commpy/channelcoding/designs/ldpc/gallager/96.33.964.txt"))
    sigma = 0.9
    llr = 2.0 * (1.0 + sigma * rs.randn(2 * 96)) / sigma ** 2
    out["ldpc_llr"].append(llr.copy())
    dec, llr_out = rcc.ldpc_bp_decode(llr.copy(), params, "MSA", 6)
    out["ldpc_dec"].append(dec)
    out["ldpc_out"].append(llr_out)
    modem = rmod.QAMModem(16)
    y = modem.modulate(rs.randint(0, 2, 4 * 30)) + 0.4 * (rs.randn(30) + 1j * rs.randn(30))
    out["demod_y"].append(y)
    with np.errstate(all="ignore"):
        out["demod_soft"].append(modem.demodulate(y, "soft", 0.7))
    out["demod_hard"].append(modem.demodulate(y, "hard"))


def mimo(rmod, rlinks, seed, out):
    rs = np.random.RandomState(seed)
    for m, n in MIMO_SHAPES:
        rq = rmod.QAMModem(m)
        out["q%d_constellation" % m] = [rq.constellation]
        tag = "mimo_q%d_n%d_" % (m, n)

        def demode(s):
            return rq.demodulate(s, "hard")
        for _ in range(10):
            nb = rq.num_bits_symbol
            h = (rs.randn(n, n) + 1j * rs.randn(n, n)) * np.sqrt(0.5)
            nv = n / 10 ** (rs.uniform(5, 25) / 10)
            y = h.dot(rq.modulate(rs.randint(0, 2, n * nb))) + (rs.randn(n) + 1j * rs.randn(n)) * np.sqrt(nv / 2)
            stack = tuple(rs.randint(1, 6, n - 1))
            out[tag + "y"].append(y)
            out[tag + "h"].append(h)
            out[tag + "nv"].append(nv)
            out[tag + "stack"].append(np.array(stack))
            out[tag + "kbest_hard"].append(rmod.kbest(y, h, rq.constellation, 6))
            out[tag + "kbest_soft"].append(rmod.kbest(y, h, rq.constellation, 6, nv, "soft", demode))
            out[tag + "best_first"].append(rmod.best_first_detector(y, h, rq.constellation, stack, nv, demode, 100))
    rq = rmod.QAMModem(16)

    def detector(y, h, constellation, noise_var, a_priori):
        return rmod.kbest(y, h, constellation, 8, noise_var, "soft", lambda s: rq.demodulate(s, "hard")) + 0.25 * a_priori

    def decoder(llr):
        return np.tanh(llr) * 3 + np.roll(llr, 1)

    def decision(llr):
        return (llr > 0).astype(int)
    nvec, n = 5, 2
    h = (rs.randn(nvec, n, n) + 1j * rs.randn(nvec, n, n)) * np.sqrt(0.5)
    y = np.einsum("ijk,ik->ij", h, rq.modulate(rs.randint(0, 2, nvec * n * 4)).reshape(nvec, n)) + 0.1 * rs.randn(nvec, n)
    ap = rs.randn(nvec * n * 4)
    out["idd_y"].append(y)
    out["idd_h"].append(h)
    out["idd_ap"].append(ap.copy())
    out["idd_ref"].append(rlinks.idd_decoder(detector, decoder, decision, 3)(y, h, rq.constellation, 0.02, ap.copy(), n * 4))


def main():
    warnings.simplefilter("ignore")
    refimport.import_reference()
    rcc = importlib.import_module("commpy.channelcoding")
    rmod = importlib.import_module("commpy.modulation")
    rlinks = importlib.import_module("commpy.links")
    out = defaultdict(list)
    for seed in SEEDS:
        viterbi_and_bcjr(rcc, seed, out)
        ldpc_and_demapper(rcc, rmod, seed, out)
    for seed in MIMO_SEEDS:
        mimo(rmod, rlinks, seed, out)
    arrays = {k: np.array(v[0] if k.endswith("_constellation") else v) for k, v in out.items()}
    path = os.path.join(GOLD, "reference_draws.npz")
    np.savez_compressed(path, **arrays)
    print("wrote", path, {k: v.shape for k, v in arrays.items()})


if __name__ == "__main__":
    main()
