"""tools/make_golden.py — regenerate tests/golden/*.npz from the UNMODIFIED reference headers.

Runs only in the authoring container (needs /root/reference to build oracle/_ref/libqdsp_ref.so via
oracle/Makefile). The fixtures pin both the C restatement (oracle/port.c) and the CUDA path to outputs
of the reference's own classes on seeded synthetic IQ; the GPU box only ever reads the committed
.npz files. Usage: python tools/make_golden.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import loader  # noqa: E402
from qdsp_b200 import synth  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")

# the case table is shared with tests/cases.py so tests replay exactly these inputs
from tests.cases import CASES, make_input  # noqa: E402

SECOND_FILE_CASES = ("interp", "mm_cf32")


def main():
    loader.build()
    if not loader.have_ref():
        raise SystemExit("oracle/_ref/libqdsp_ref.so missing: /root/reference not available")
    R = loader.ref("generic")
    os.makedirs(OUT, exist_ok=True)
    gold = {}
    # ---- tap designs --------------------------------------------------------------------------
    gold["taps_cfg1"] = R.blackman_taps(300e3, 4 * 2.4e6 / 127, 2.4e6)
    gold["taps_cfg3"] = R.blackman_taps(100e3, 4 * 2.4e6 / 4095, 2.4e6)
    t, i, d = R.vfo_design(2.4e6, 48e3, 48e3)
    gold["taps_cfg2"], gold["id_cfg2"] = t, np.asarray([i, d], np.int32)
    t, i, d = R.vfo_design(61.44e6, 48e3, 48e3)
    gold["taps_cfg4"], gold["id_cfg4"] = t, np.asarray([i, d], np.int32)
    t, i, d = R.vfo_design(250e3, 48e3, 48e3)
    gold["taps_rational"], gold["id_rational"] = t, np.asarray([i, d], np.int32)
    gold["taps_bandpass"] = R.blackman_bandpass_taps(15e3, 4e3, 19e3, 240e3)
    gold["taps_rrc"] = R.rrc_taps(31, 4.0, 1.0, 0.35)
    # the reference's baked MMSE interpolator table (src/dsp/interpolation_taps.h), an input of MMClockRecovery
    gold["interp_taps"] = R.interp_taps()
    # ---- streaming cases ----------------------------------------------------------------------
    for name, c in CASES.items():
        x = make_input(c)
        k = c["kind"]
        if k == "fir":
            y = R.fir_cf32(*c["win"], x, c["block"])
        elif k == "fir_f32":
            y = R.fir_f32(*c["win"], x, c["block"])
        elif k == "resamp":
            y, oc, i, d = R.resamp_cf32(*c["win"], c["in_sr"], c["out_sr"], x, c["block"], vfo_style=c.get("vfo_style", False))
            gold[name + "_oc"] = oc
            gold[name + "_id"] = np.asarray([i, d], np.int32)
        elif k == "resamp_f32":
            y, oc, i, d = R.resamp_f32(*c["win"], c["in_sr"], c["out_sr"], x, c["block"])
            gold[name + "_oc"] = oc
        elif k == "power_decim":
            y, oc = R.power_decim(c["power"], x, c["block"])
            gold[name + "_oc"] = oc
        elif k == "xlator":
            y = R.xlator(c["fs"], c["freq"], x, c["block"])
        elif k == "fm":
            y = R.fm_demod(c["fs"], c["dev"], x, c["block"])
        elif k == "fm_stereo":
            y = R.fm_demod_stereo(c["fs"], c["dev"], x, c["block"])
        elif k == "stereo_fm":
            y = R.stereo_fm(c["fs"], c["dev"], x, c["block"])
        elif k == "vfo":
            y, oc = R.vfo(c["offset"], c["in_sr"], c["out_sr"], c["bw"], x, c["block"])
            gold[name + "_oc"] = oc
        elif k == "vfo_fm":
            y, oc = R.vfo_fm(c["offset"], c["in_sr"], c["out_sr"], c["bw"], c["dev"], x, c["block"])
            gold[name + "_oc"] = oc
        elif k == "channelizer":
            y = R.channelizer_fm(np.asarray(c["offsets"], np.float32), c["in_sr"], c["out_sr"], c["bw"], c["dev"], x, c["block"])
        elif k == "deemp":
            y = R.deemp(c["fs"], c["tau"], x.view(np.float32).reshape(-1, 2), c["block"]).reshape(-1).view(np.complex64)
        elif k == "agc":
            y = R.agc(c["fall"], c["fs"], x, c["block"])
        elif k == "cagc":
            y = R.complex_agc(c["set_point"], c["max_gain"], c["rate"], x, c["block"])
        elif k == "ffagc":
            y, vc = R.ff_agc(x, c["block"])
            gold[name + "_vc"] = vc
        elif k == "costas":
            y = R.costas(c["order"], c["bw"], x, c["block"])
        elif k == "math":
            x2 = make_input(c, "src2")
            y = np.stack([R.math(op, x, x2, c["block"]) for op in range(3)])
        elif k == "layout":
            x2 = make_input(c, "src2") if "src2" in c else None
            y = R.layout(c["op"], x, x2, c["block"])
            if c["op"] == 3:
                y = np.stack(y)
        elif k == "volume":
            y = R.volume(x, c["volume"], c["call_set"], c["muted"], c["block"])
        elif k == "threshold":
            y = R.threshold(x, c["block"])
        elif k == "delay_imag":
            y = R.delay_imag(x, c["block"])
        elif k == "amdemod":
            y = R.amdemod(x, c["block"])
        elif k == "squelch":
            y = R.squelch(c["level"], x, c["block"])
        elif k == "mm":
            y, oc = R.mm(x, c["omega"], c["gain_omega"], c["mu_gain"], c["rel"], c["block"])
            gold[name + "_oc"] = oc
        elif k == "msk":
            y, oc = R.msk_demod(c["fs"], c["dev"], c["baud"], x, c["block"])
            gold[name + "_oc"] = oc
        elif k == "psk":
            y, oc = R.psk_demod(c["order"], c["offset"], c["fs"], c["baud"], x, c["block"])
            gold[name + "_oc"] = oc
        elif k == "ssb":
            y = R.ssbdemod(c["fs"], c["bw"], c["mode"], x, c["block"])
        else:
            raise SystemExit(f"unknown kind {k}")
        gold[name] = np.asarray(y)
        print(f"{name:24s} kind={k:12s} in={len(x):7d} out={np.asarray(y).shape}")
    # the vectors of SECOND_FILE_CASES go to a file of their own, so that neither file exceeds 1 MB
    second = {k: gold.pop(k) for k in list(gold)
              if k in SECOND_FILE_CASES or (k.endswith(("_oc", "_id", "_vc")) and k.rsplit("_", 1)[0] in SECOND_FILE_CASES)}
    for name, arrays in (("reference_vectors.npz", gold), ("reference_vectors_2.npz", second)):
        np.savez_compressed(os.path.join(OUT, name), **arrays)
        print("wrote", os.path.join(OUT, name), os.path.getsize(os.path.join(OUT, name)), "bytes")


if __name__ == "__main__":
    main()
