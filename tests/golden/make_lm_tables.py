"""Writes the scorer-path fixtures of tests/test_lm.py from the UNMODIFIED reference build (oracle/_ref/libctcref.so,
`make -C oracle ref`); needs that build, and is run by hand when the cases change:

* tests/golden/<model>.lmtab.gz  every n-gram score the decodes of the tests ask for, as the reference's Scorer gives it
                               (the table of tests/native/lm_replay.cpp).  The n-grams are collected by running each
                               case through the CPU emulation of the CTA program with the reference Scorer behind it.
* tests/golden/recorded/lm_cases_{word,char}.npz   the reference's outputs for the cases that are not fixtures of their own.

    python tests/golden/make_lm_tables.py
"""
import ctypes
import gzip
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from ctcdecode_b200.synth import ctc_like_probs, text_probs  # noqa: E402
from oracle import oracle as orc  # noqa: E402
from tests import emul, golden_util, lm_replay  # noqa: E402
from tests import test_lm as t  # noqa: E402
from tests.parity import compare  # noqa: E402

MODELS = (t.TINY, t.REF_ARPA, t.CHAR_LM)


def start_table(model):
    os.makedirs(os.path.dirname(lm_replay.build()), exist_ok=True)
    ref = orc.Reference(["_", " "], model_path=model)
    vocab = ref.lm_vocabulary()
    with open(lm_replay.table(model), "w") as f:
        f.write("order %d\nchar_based %d\nvocab %d\n" % (ref.max_order(), ref.is_character_based(), len(vocab)))
        f.write("".join(w + "\n" for w in vocab) + "ngrams 0\n")


def record(model, labels, probs, seq_lens, alpha, beta, kw, envs=({},)):
    """Runs one case through the emulation with the reference Scorer behind the table (collecting n-grams) and
    returns the reference's own outputs, checked against what the emulation made of the table."""
    ref = orc.Reference(labels, model_path=model, alpha=alpha, beta=beta)
    ref.lib.ref_scorer_cond_from_words.restype = ctypes.c_double
    rep = lm_replay.Replay(labels, model)
    rep.lib.lm_replay_record.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    rep.lib.lm_replay_record(rep.scorer, ctypes.cast(ref.lib.ref_scorer_cond_from_words, ctypes.c_void_p), ref.scorer)
    want = ref.decode(probs, seq_lens, num_processes=2, **kw)
    char = rep.is_character_based() == 1
    words = [] if char else rep.lm_vocabulary()
    for env in envs:
        old = {k: os.environ.get(k) for k in env}
        os.environ.update(env)
        try:
            got = emul.decode_lm(probs, rep.lib, rep.scorer, labels, words, rep.max_order(), alpha, beta,
                                 seq_lens=seq_lens, char_based=char, **kw)
        finally:
            for k, v in old.items():
                os.environ.pop(k, None) if v is None else os.environ.__setitem__(k, v)
        compare(want, got, None, "recording %s %r" % (os.path.basename(model), env))
    assert rep.lib.lm_replay_save(rep.scorer, rep.path) == 0
    return want, ref


def trimmed(out):
    L = max(1, int(out["lens"].max()))
    return dict(tokens=out["tokens"][:, :, :L], timesteps=out["timesteps"][:, :, :L], scores=out["scores"],
                lens=out["lens"], n_results=out["n_results"])


def main():
    for m in MODELS:
        start_table(m)
    protocols = ({}, {"CTC_EMU_LM_PER_FRAME": "1"}, {"CTC_EMU_LM_CHUNK": "7"})
    word, char = {}, {}
    # fixtures of their own (tests/golden/lm_*.npz)
    for name in golden_util.names(lm=True):
        probs, sl, kw, _, a, b = golden_util.load_lm(name)
        record(t.TINY, t.L29, probs, sl, a, b, kw, protocols)
    for name in golden_util.names_char():
        probs, sl, kw, _, a, b = golden_util.load_lm(name)
        record(t.CHAR_LM, t.LCHAR, probs, sl, a, b, kw, protocols)
    # word-based model
    for i, cfg in enumerate(t.LM_CFGS):
        probs, a, b, kw = t.lm_cfg_inputs(cfg)
        word["cfg%d" % i], _ = record(t.TINY, t.L29, probs, None, a, b, kw)
    kat, _, _, _ = golden_util.load("ref_kat_beam20")
    word["kat"], _ = record(t.REF_ARPA, t.KAT_VOCAB, kat, None, 0.0, 0.0, dict(beam=20, blank_id=6))
    probs = ctc_like_probs(2, 300, 29, seed=5).numpy()
    word["c5_shape"], _ = record(t.REF_ARPA, t.L29, probs, None, 2.0, 1.0, dict(beam=100))
    probs = text_probs(t.TEXTS * 2 + t.TEXTS[:2], t.L29, 400, seed=21).numpy()
    word["live"], _ = record(t.TINY, t.L29, probs, None, 2.0, 1.0, dict(beam=100))
    word["live_reset"], _ = record(t.TINY, t.L29, probs, None, 0.5, -0.25, dict(beam=100))
    probs = text_probs(t.TEXTS, t.L29, 240, seed=41).numpy()
    word["online_offline"], ref = record(t.TINY, t.L29, probs, None, 1.5, 0.7, dict(beam=32))
    states = [ref.state_new(32) for _ in range(3)]
    for a, b in t.ONLINE_CUTS:
        ref.decode_with_states(probs[:, a:b], states, [False] * 3, 32)
    word["online_streaming"] = ref.decode_with_states(probs[:, 200:], states, [True] * 3, 32, max_len=240)
    word["online_streaming"]["n_results"] = word["online_offline"]["n_results"]
    for s in states:
        ref.state_free(s)
    import torch
    probs, _ = t.c5_text_probs(12, 1000, seed=7)
    probs = torch.cat([probs, ctc_like_probs(4, 1000, 29, seed=8)], 0).numpy()
    word["c5"], ref = record(t.REF_ARPA, t.L29, probs, None, 2.0, 1.0, dict(beam=100))
    word["c5"]["dict_size"] = np.array(ref.dict_size())
    # the reference's Scorer::reset_params takes floats: after reset_params(0.3, 0.1) it decodes with float(0.3), float(0.1)
    word["c5_reset"], _ = record(t.REF_ARPA, t.L29, probs[:6], None, float(np.float32(0.3)), float(np.float32(0.1)),
                                 dict(beam=100))
    # character-based model
    for i, cfg in enumerate(t.CHAR_CFGS):
        probs, labels, a, b, kw = t.char_cfg_inputs(cfg)
        char["cfg%d" % i], _ = record(t.CHAR_LM, labels, probs, None, a, b, kw)
    for i, (probs, sl, labels, a, b, kw) in enumerate(t.char_random_configurations()):
        char["trial%d" % i], _ = record(t.CHAR_LM, labels, probs, sl, a, b, kw, protocols)
    probs = ctc_like_probs(16, 300, len(t.LCHAR), seed=51).numpy()
    char["live"], _ = record(t.CHAR_LM, t.LCHAR, probs, None, 1.3, 0.6, dict(beam=100))
    char["live_online"], _ = record(t.CHAR_LM, t.LCHAR, probs[:3], None, 1.3, 0.6, dict(beam=24))
    for group, cases in (("word", word), ("char", char)):
        arrays = {}
        for key, out in cases.items():
            extra = {k: v for k, v in out.items() if k == "dict_size"}
            arrays.update({key + "/" + k: v for k, v in dict(trimmed(out), **extra).items()})
        np.savez_compressed(os.path.join(lm_replay.GOLDEN, "recorded", "lm_cases_%s.npz" % group), **arrays)
    for m in MODELS:
        with open(lm_replay.table(m), "rb") as f, gzip.GzipFile(lm_replay.table(m) + ".gz", "wb", mtime=0) as g:
            g.write(f.read())
        os.replace(lm_replay.table(m) + ".gz", os.path.join(lm_replay.GOLDEN, os.path.basename(lm_replay.table(m)) + ".gz"))


if __name__ == "__main__":
    main()
