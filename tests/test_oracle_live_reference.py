"""Pin of the oracle and the host-side MIMO mirrors on random draws that the other goldens do not contain: for a fixed list
of seeds, the UNMODIFIED reference's outputs were recorded by oracle/make_reference_draws_golden.py into
tests/golden/reference_draws.npz, and oracle/commpy_oracle.c and commpy_b200's mirrors must reproduce them (bit-exact for
Viterbi and LDPC min-sum incl. out_llrs, 1e-9 for the float outputs)."""
import os

import numpy as np
import pytest
import scipy.sparse as sp

from commpy_b200.channelcoding.convcode import Trellis
from oracle import oracle

pytestmark = pytest.mark.filterwarnings("ignore")

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TB = {"cont": None, "term": 9}


@pytest.fixture(scope="module")
def ref():
    return np.load(os.path.join(GOLD, "reference_draws.npz"))


def test_viterbi_and_bcjr_fresh_cases(ref):
    k7 = Trellis(np.array([6]), np.array([[0o133, 0o171]]))
    rsc = Trellis(np.array([3]), np.array([[1, 0o15]]), np.array([[0o13]]), "rsc")
    for mode in ("hard", "soft", "unquantized"):
        for term, tb in TB.items():
            xs, wants = ref["vit_%s_%s_x" % (mode, term)], ref["vit_%s_%s_ref" % (mode, term)]
            for seed, (x, want) in enumerate(zip(xs, wants)):
                assert np.array_equal(want, oracle.viterbi_decode(x.copy(), k7, tb, mode)), (seed, mode, term, tb)
    for seed in range(len(ref["map_sys"])):
        got = oracle.map_decode(ref["map_sys"][seed], ref["map_par"][seed], rsc, 0.9, ref["map_La"][seed], "decode")
        assert np.allclose(ref["map_L"][seed], got[0], rtol=1e-9, atol=1e-9), seed
        assert np.array_equal(ref["map_bits"][seed], got[1]), seed


def test_ldpc_and_demapper_fresh_cases(ref):
    from commpy_b200.modulation import QAMModem
    design = np.load(os.path.join(GOLD, "ldpc_design.npz"))
    H = sp.coo_matrix((np.ones(len(design["g96_H_rows"]), np.int8), (design["g96_H_rows"], design["g96_H_cols"])),
                      shape=(int(design["g96_n_cnodes"]), int(design["g96_n_vnodes"])))
    params = {"n_vnodes": int(design["g96_n_vnodes"]), "parity_check_matrix": H.tocsc()}
    modem = QAMModem(16)
    np.testing.assert_array_equal(modem.constellation, ref["q16_constellation"])
    for seed in range(len(ref["ldpc_llr"])):
        dec, out = oracle.ldpc_bp_decode(ref["ldpc_llr"][seed].copy(), params, "MSA", 6)
        assert np.array_equal(ref["ldpc_dec"][seed], dec) and np.array_equal(ref["ldpc_out"][seed], out), seed
        y, want = ref["demod_y"][seed], ref["demod_soft"][seed]
        got = oracle.demodulate(modem, y, "soft", 0.7)
        fin = np.isfinite(want)
        assert np.allclose(want[fin], got[fin], rtol=1e-9, atol=1e-9), seed
        assert np.array_equal(ref["demod_hard"][seed], oracle.demodulate(modem, y, "hard")), seed


def test_mimo_mirrors_fresh_cases(ref):
    """host-side MIMO mirrors (kbest, best_first_detector, idd_decoder) against the reference's outputs; the hard demapper
    the detectors call is the oracle's (pinned to the reference by tests/test_oracle_golden.py)"""
    from commpy_b200 import modulation as mod
    from commpy_b200.links import idd_decoder
    for m, n in ((4, 2), (16, 3), (16, 4)):
        mq = mod.QAMModem(m)
        np.testing.assert_array_equal(ref["q%d_constellation" % m], mq.constellation)

        def demode(s):
            return oracle.demodulate(mq, s, "hard")
        tag = "mimo_q%d_n%d_" % (m, n)
        for d in range(len(ref[tag + "y"])):
            y, h, nv, stack = ref[tag + "y"][d], ref[tag + "h"][d], float(ref[tag + "nv"][d]), tuple(ref[tag + "stack"][d])
            msg = "draw %d" % d
            np.testing.assert_allclose(mod.kbest(y, h, mq.constellation, 6), ref[tag + "kbest_hard"][d], atol=1e-12, err_msg=msg)
            np.testing.assert_allclose(mod.kbest(y, h, mq.constellation, 6, nv, "soft", demode), ref[tag + "kbest_soft"][d],
                                       rtol=1e-9, atol=1e-9, err_msg=msg)
            np.testing.assert_allclose(mod.best_first_detector(y, h, mq.constellation, stack, nv, demode, 100),
                                       ref[tag + "best_first"][d], rtol=1e-9, atol=1e-9, err_msg=msg)
    # idd_decoder: the same closures as the reference run, 3 iterations
    mq = mod.QAMModem(16)

    def detector(y, h, constellation, noise_var, a_priori):
        return mod.kbest(y, h, constellation, 8, noise_var, "soft", lambda s: oracle.demodulate(mq, s, "hard")) + 0.25 * a_priori

    def decoder(llr):
        return np.tanh(llr) * 3 + np.roll(llr, 1)

    def decision(llr):
        return (llr > 0).astype(int)
    n = 2
    for seed in range(len(ref["idd_y"])):
        got = idd_decoder(detector, decoder, decision, 3)(ref["idd_y"][seed], ref["idd_h"][seed], mq.constellation, 0.02,
                                                          ref["idd_ap"][seed].copy(), n * 4)
        np.testing.assert_array_equal(got, ref["idd_ref"][seed])
