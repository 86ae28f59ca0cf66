#!/usr/bin/env python
"""Generates tests/golden/*.npz with the UNMODIFIED reference (oracle/_ref/libctcref.so, built by
`make -C oracle ref` from /root/reference).  Run in the build container only; the fixtures are committed so
the GPU box (no /root/reference) can pin both the C oracle and the CUDA path against real reference output.

Each file holds the input (float32 probs, seq_lens) with the decoder parameters and the reference's outputs:
tokens / timesteps (int32, -1 where the reference leaves memory uninitialised), scores (float32), lens,
n_results.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from ctcdecode_b200.synth import ctc_like_probs, flat_probs  # noqa: E402
from oracle.oracle import Reference  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))

# the reference's own fixtures, tests/test_decode.py:13-30 (vocab "'", " ", a, b, c, d, "_"; blank = 6)
PROBS_SEQ1 = [[0.06390443, 0.21124858, 0.27323887, 0.06870235, 0.0361254, 0.18184413, 0.16493624],
              [0.03309247, 0.22866108, 0.24390638, 0.09699597, 0.31895462, 0.0094893, 0.06890021],
              [0.218104, 0.19992557, 0.18245131, 0.08503348, 0.14903535, 0.08424043, 0.08120984],
              [0.12094152, 0.19162472, 0.01473646, 0.28045061, 0.24246305, 0.05206269, 0.09772094],
              [0.1333387, 0.00550838, 0.00301669, 0.21745861, 0.20803985, 0.41317442, 0.01946335],
              [0.16468227, 0.1980699, 0.1906545, 0.18963251, 0.19860937, 0.04377724, 0.01457421]]
PROBS_SEQ2 = [[0.08034842, 0.22671944, 0.05799633, 0.36814645, 0.11307441, 0.04468023, 0.10903471],
              [0.09742457, 0.12959763, 0.09435383, 0.21889204, 0.15113123, 0.10219457, 0.20640612],
              [0.45033529, 0.09091417, 0.15333208, 0.07939558, 0.08649316, 0.12298585, 0.01654384],
              [0.02512238, 0.22079203, 0.19664364, 0.11906379, 0.07816055, 0.22538587, 0.13483174],
              [0.17928453, 0.06065261, 0.41153005, 0.1172041, 0.11880313, 0.07113197, 0.04139363],
              [0.15882358, 0.1235788, 0.23376776, 0.20510435, 0.00279306, 0.05294827, 0.22298418]]


def emit(name, probs, seq_lens=None, **kw):
    probs = np.ascontiguousarray(probs, dtype=np.float32)
    V = probs.shape[2]
    ref = Reference([chr(33 + i) if V < 90 else str(i) for i in range(V)])
    r = ref.decode(probs, seq_lens, num_processes=4, **kw)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), probs=probs,
                        seq_lens=np.zeros(0, np.int32) if seq_lens is None else np.asarray(seq_lens, np.int32),
                        params=np.array([kw.get("beam", 100), kw.get("cutoff_top_n", 40), kw.get("blank_id", 0),
                                         int(kw.get("log_input", False))], np.int64),
                        cutoff_prob=np.array([kw.get("cutoff_prob", 1.0)], np.float64), **r)
    print(name, probs.shape, "n_results", r["n_results"][:4], "top score", r["scores"][:, 0][:4])


L29 = ["_"] + [chr(ord("a") + i) for i in range(26)] + [" ", "'"]
TINY_LM = os.path.join(ROOT, "tests", "data", "tiny_lm.arpa")


def emit_lm(name, probs, alpha, beta, seq_lens=None, **kw):
    """Scorer path of the reference (KenLM + dictionary) on tests/data/tiny_lm.arpa (authored for this repo)."""
    probs = np.ascontiguousarray(probs, dtype=np.float32)
    ref = Reference(L29, model_path=TINY_LM, alpha=alpha, beta=beta)
    r = ref.decode(probs, seq_lens, num_processes=4, **kw)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), probs=probs,
                        seq_lens=np.zeros(0, np.int32) if seq_lens is None else np.asarray(seq_lens, np.int32),
                        params=np.array([kw.get("beam", 100), kw.get("cutoff_top_n", 40), kw.get("blank_id", 0),
                                         int(kw.get("log_input", False))], np.int64),
                        cutoff_prob=np.array([kw.get("cutoff_prob", 1.0)], np.float64),
                        lm=np.array([alpha, beta], np.float64), **r)
    top = ["".join(L29[x] for x in r["tokens"][b, 0, :r["lens"][b, 0]]) for b in range(probs.shape[0])]
    print(name, probs.shape, "n_results", r["n_results"][:4], "top-1", top[:3])


def emit_ref_build_cases():
    """recorded/ref_build_cases.npz: the reference's outputs for tests/test_oracle.py REF_BUILD_CASES (inputs from seeds)"""
    from tests.test_oracle import REF_BUILD_CASES, ref_build_inputs
    arrays = {}
    for i, cfg in enumerate(REF_BUILD_CASES):
        probs, V, kw = ref_build_inputs(cfg)
        r = Reference([str(v) for v in range(V)]).decode(probs, **kw)
        L = max(1, int(r["lens"].max()))
        r["tokens"], r["timesteps"] = r["tokens"][:, :, :L], r["timesteps"][:, :, :L]
        arrays.update({"case%d/%s" % (i, k): v for k, v in r.items()})
    os.makedirs(os.path.join(HERE, "recorded"), exist_ok=True)
    np.savez_compressed(os.path.join(HERE, "recorded", "ref_build_cases.npz"), **arrays)


if __name__ == "__main__":
    from ctcdecode_b200.synth import text_probs
    emit_ref_build_cases()
    texts = ["the cat sat on the mat", "a dog ran fast", "the dog sat on a mat the cat ran"]
    emit_lm("lm_tiny_a15_b08_beam32", text_probs(texts, L29, 160, seed=1).numpy(), 1.5, 0.8, beam=32)
    emit_lm("lm_tiny_a0_b0_beam20", text_probs(texts[:2], L29, 120, seed=2).numpy(), 0.0, 0.0, beam=20)
    emit_lm("lm_tiny_a2_bm1_beam8_ragged", text_probs(texts, L29, 140, seed=3).numpy(), 2.0, -1.0,
            seq_lens=[140, 60, 0], beam=8)
    emit_lm("lm_tiny_noise_beam64", ctc_like_probs(2, 150, 29, seed=4).numpy(), 1.0, 0.5, beam=64)

    kat = np.array([PROBS_SEQ1, PROBS_SEQ2], np.float32)
    emit("ref_kat_beam20", kat, beam=20, blank_id=6)
    emit("ref_kat_beam20_log", np.log(kat), beam=20, blank_id=6, log_input=True)
    emit("ref_kat_beam4_top3", kat, beam=4, blank_id=6, cutoff_top_n=3)
    emit("ref_kat_seqlens", kat, seq_lens=[6, 3], beam=20, blank_id=6)
    emit("c1_T50_V6_beam4", ctc_like_probs(4, 50, 6, seed=1, peak=3.0).numpy(), beam=4)
    emit("c2like_T120_V29_beam32", ctc_like_probs(3, 120, 29, seed=2).numpy(), beam=32)
    emit("c2like_log_T100_V29_beam20", ctc_like_probs(2, 100, 29, seed=3, log=True).numpy(), beam=20, log_input=True)
    emit("topn10_T100_V29_beam16", ctc_like_probs(3, 100, 29, seed=4).numpy(), beam=16, cutoff_top_n=10)
    emit("cp099_T80_V64_beam16", ctc_like_probs(2, 80, 64, seed=5).numpy(), beam=16, cutoff_prob=0.99)
    emit("cp03_T80_V29_beam64", ctc_like_probs(2, 80, 29, seed=6).numpy(), beam=64, cutoff_prob=0.3)
    emit("c4like_T60_V256_beam64", ctc_like_probs(1, 60, 256, seed=7).numpy(), beam=64, cutoff_prob=0.99)
    emit("ragged_T90_V29_beam24", ctc_like_probs(5, 90, 29, seed=8).numpy(), seq_lens=[90, 0, 1, 45, 300], beam=24)
    emit("blank_last_T70_V12_beam8", ctc_like_probs(2, 70, 12, seed=9, blank_id=11).numpy(), beam=8, blank_id=11)
    emit("flat_T60_V29_beam50", flat_probs(2, 60, 29, seed=10).numpy(), beam=50)
