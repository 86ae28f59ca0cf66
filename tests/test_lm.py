"""Scorer path (word-based KenLM model + dictionary; BASELINE config 5, reference tests/test_decode.py:55-64).

The language model stays behind the host hook: in these tests the hook answers with the scores the UNMODIFIED
reference Scorer gave for the same n-grams (tests/lm_replay.py, recorded by tests/golden/make_lm_tables.py) so the LM
arithmetic is the reference's own, and everything the product adds -- dictionary automaton, cutoff, LM-term
application, per-node memoisation, final rescoring -- is compared with the reference's recorded results: tokens,
timesteps, lens bit-exact, float32 scores bit-exact.  Where the reference build (oracle/_ref) is present, the fixtures
are also checked against it live."""
import os

import numpy as np
import pytest

from ctcdecode_b200.synth import ctc_like_probs, flat_probs, text_probs
from oracle import oracle as orc
from tests import emul, golden_util, lm_replay
from tests.lm_replay import Replay, recorded
from tests.parity import compare

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TINY = os.path.join(ROOT, "tests", "data", "tiny_lm.arpa")
REF_ARPA = os.path.join(ROOT, "tests", "golden", "test.arpa")  # the reference's own test LM (its tests/test.arpa), a fixture
L29 = ["_"] + [chr(ord("a") + i) for i in range(26)] + [" ", "'"]
TEXTS = ["the cat sat on the mat", "a dog ran fast", "the dog sat on a mat the cat ran"]
# the scorer provider of these tests answers from the scores the original decoder's Scorer gave (tests/lm_replay.py)
PROVIDER = lm_replay.build()


def _emul_lm(ref, probs, labels, alpha, beta, seq_lens=None, **kw):
    return emul.decode_lm(probs, ref.lib, ref.scorer, labels, ref.lm_vocabulary(), ref.max_order(), alpha, beta,
                          seq_lens=seq_lens, **kw)


@pytest.mark.parametrize("per_frame", [False, True, 7], ids=["persistent", "per_frame_launch", "chunks_of_7"])
@pytest.mark.parametrize("name", golden_util.names(lm=True))
def test_emulation_lm_matches_reference_golden(name, per_frame, monkeypatch):
    """the host/kernel protocols: one persistent launch with a per-frame handshake (default), one launch per frame,
    and the streaming shape (launches of 7 frames over saved state)"""
    if per_frame is True:
        monkeypatch.setenv("CTC_EMU_LM_PER_FRAME", "1")
    elif per_frame:
        monkeypatch.setenv("CTC_EMU_LM_CHUNK", str(per_frame))
    probs, seq_lens, kw, gold, alpha, beta = golden_util.load_lm(name)
    got = _emul_lm(Replay(L29, TINY), probs, L29, alpha, beta, seq_lens=seq_lens, **kw)
    compare(gold, got, None, name)
    if orc.reference_available():  # and the fixture still is what the original decoder says
        live = orc.Reference(L29, model_path=TINY, alpha=alpha, beta=beta).decode(probs, seq_lens, num_processes=2, **kw)
        compare(gold, live, None, name + " (live reference)")


LM_CFGS = [
    dict(alpha=1.5, beta=0.8, beam=32, T=160, seed=11),
    dict(alpha=0.0, beta=0.0, beam=20, T=100, seed=12),
    dict(alpha=0.5, beta=-0.5, beam=48, T=200, seed=13),
    dict(alpha=2.0, beta=1.0, beam=16, T=120, seed=14, cutoff_prob=0.99),
    dict(alpha=2.0, beta=1.0, beam=16, T=120, seed=15, log_input=True),
    dict(alpha=1.0, beta=2.0, beam=4, T=150, seed=16),
    dict(alpha=1.0, beta=0.5, beam=64, T=100, seed=17, noise=True),
    dict(alpha=1.0, beta=0.5, beam=30, T=80, seed=18, flat=True),
]


def lm_cfg_inputs(cfg):
    """-> probs, alpha, beta, decoder keywords"""
    cfg = dict(cfg)
    alpha, beta, T, seed = cfg.pop("alpha"), cfg.pop("beta"), cfg.pop("T"), cfg.pop("seed")
    if cfg.pop("noise", False):
        probs = ctc_like_probs(3, T, 29, seed=seed)
    elif cfg.pop("flat", False):
        probs = flat_probs(3, T, 29, seed=seed)
    else:
        probs = text_probs(TEXTS, L29, T, seed=seed)
    if cfg.get("log_input"):
        probs = probs.log()
    return probs.numpy(), alpha, beta, cfg


@pytest.mark.parametrize("cfg", LM_CFGS)
def test_emulation_lm_matches_reference(cfg):
    probs, alpha, beta, kw = lm_cfg_inputs(cfg)
    want = recorded("word", "cfg%d" % LM_CFGS.index(cfg))
    got = _emul_lm(Replay(L29, TINY), probs, L29, alpha, beta, **kw)
    compare(want, got, None, str(cfg))


KAT_VOCAB = ["'", " ", "a", "b", "c", "d", "_"]


@pytest.mark.skipif(not os.path.exists(REF_ARPA), reason="reference test LM not present")
def test_emulation_lm_reference_unit_test_and_config5_shape():
    """reference tests/test_decode.py:55-64 ("a a", 7 results) and a BASELINE config-5 shaped batch (test.arpa,
    alpha 2.0, beta 1.0, beam 100) -- with the reference's own LM file (tests/golden/test.arpa)."""
    kat, _, _, _ = golden_util.load("ref_kat_beam20")
    got = _emul_lm(Replay(KAT_VOCAB, REF_ARPA), kat, KAT_VOCAB, 0.0, 0.0, beam=20, blank_id=6)
    compare(recorded("word", "kat"), got, None, "test_beam_search_decoder_3")
    assert got["n_results"][1] == 7
    assert "".join(KAT_VOCAB[x] for x in got["tokens"][1, 0, :got["lens"][1, 0]]) == "a a"
    probs = ctc_like_probs(2, 300, 29, seed=5).numpy()
    got = _emul_lm(Replay(L29, REF_ARPA), probs, L29, 2.0, 1.0, beam=100)
    compare(recorded("word", "c5_shape"), got, None, "config 5 shape")


def test_scorer_accessors_match_reference():
    ref = Replay(L29, TINY)
    assert ref.max_order() == 3 and ref.is_character_based() == 0
    import ctypes
    from ctcdecode_b200 import _native
    lib = _native.load()
    words = ref.lm_vocabulary()
    cond = ctypes.cast(ref.lib.ref_scorer_cond_from_labels, ctypes.c_void_p).value
    sent = ctypes.cast(ref.lib.ref_scorer_sent_from_labels, ctypes.c_void_p).value
    hooks = _native.ScorerHooks(ref.scorer, cond, sent)
    lab = (ctypes.c_char_p * 29)(*[x.encode() for x in L29])
    wrd = (ctypes.c_char_p * len(words))(*[x.encode() for x in words])
    h = ctypes.c_void_p()
    assert lib.ctcdec_scorer_create(ctypes.byref(hooks), 1.0, 1.0, lab, 29, wrd, len(words), ref.max_order(), 0,
                                    ctypes.byref(h)) == 0
    assert lib.ctcdec_scorer_dict_size(h) == 9   # the original's dictionary: 9 of the 12 LM words are spellable
    lib.ctcdec_scorer_destroy(h)


# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("per_frame", [False, True], ids=["persistent", "per_frame_launch"])
@pytest.mark.parametrize("name", golden_util.names(lm=True))
def test_cuda_lm_matches_reference_golden(name, per_frame, monkeypatch):
    import torch
    import ctcdecode_b200
    if per_frame:
        monkeypatch.setenv("CTCDEC_LM_PER_FRAME", "1")
    probs, seq_lens, kw, gold, alpha, beta = golden_util.load_lm(name)
    dec = ctcdecode_b200.CTCBeamDecoder(L29, model_path=lm_replay.table(TINY), alpha=alpha, beta=beta, beam_width=kw["beam"],
                                        cutoff_top_n=kw["cutoff_top_n"], cutoff_prob=kw["cutoff_prob"],
                                        log_probs_input=kw["log_input"], scorer_provider=PROVIDER)
    assert dec.dict_size() == 9 and dec.max_order() == 3 and dec.character_based() == 0
    sl = None if seq_lens is None else torch.from_numpy(seq_lens)
    out, scores, ts, lens = dec.decode(torch.from_numpy(probs), sl)
    got = dict(tokens=out.numpy(), timesteps=ts.numpy(), scores=scores.numpy(), lens=lens.numpy(),
               n_results=dec.last_n_results.numpy(), ties=dec.last_flags.numpy())
    compare(gold, got, None, name)


@pytest.mark.gpu
def test_cuda_lm_matches_live_reference_and_reset_params():
    """BASELINE config-5 shape on the tiny LM: 8 utterances x T=400, beam 100, alpha 2.0, beta 1.0, against the
    reference Scorer path run on the same box; then reset_params (reference __init__.py:134-136)."""
    import torch
    import ctcdecode_b200
    probs = text_probs(TEXTS * 2 + TEXTS[:2], L29, 400, seed=21)
    want = recorded("word", "live")
    dec = ctcdecode_b200.CTCBeamDecoder(L29, model_path=lm_replay.table(TINY), alpha=2.0, beta=1.0, beam_width=100,
                                        scorer_provider=PROVIDER)
    out, scores, ts, lens = dec.decode(probs)
    got = dict(tokens=out.numpy(), timesteps=ts.numpy(), scores=scores.numpy(), lens=lens.numpy(),
               n_results=dec.last_n_results.numpy(), ties=dec.last_flags.numpy())
    compare(want, got, None, "config-5 shape")
    assert "".join(L29[x] for x in out[0, 0, :lens[0, 0]]) == TEXTS[0]
    dec.reset_params(0.5, -0.25)
    want = recorded("word", "live_reset")
    out, scores, ts, lens = dec.decode(probs.cuda())
    got = dict(tokens=out.numpy(), timesteps=ts.numpy(), scores=scores.numpy(), lens=lens.numpy(),
               n_results=dec.last_n_results.numpy(), ties=dec.last_flags.numpy())
    compare(want, got, None, "after reset_params")


ONLINE_CUTS = [(0, 1), (1, 60), (60, 61), (61, 200)]   # then [200, 240) with end of stream


@pytest.mark.gpu
def test_cuda_online_decoder_with_scorer_matches_reference_online_path():
    """reference tests/test_decode.py:93-115,141-159 shape (OnlineCTCBeamDecoder with a language model, one call and
    several calls), on the tiny LM: chunked decoding through device-resident DecoderStates against the reference's
    own decode-with-states path AND against its offline path -- all beams, scores bit-exact; streams of one call
    end at different times."""
    import torch
    import ctcdecode_b200
    probs = text_probs(TEXTS, L29, 240, seed=41)
    want_off = recorded("word", "online_offline")
    dec = ctcdecode_b200.OnlineCTCBeamDecoder(L29, model_path=lm_replay.table(TINY), alpha=1.5, beta=0.7, beam_width=32,
                                              scorer_provider=PROVIDER)
    assert dec.dict_size() == 9

    def as_dict(res, scores, ts, lens, d):
        return dict(tokens=res.numpy(), timesteps=ts.numpy(), scores=scores.numpy(), lens=lens.numpy(),
                    n_results=d.last_n_results.numpy(), ties=d.last_flags.numpy())
    # one call
    st = [ctcdecode_b200.DecoderState(dec) for _ in range(3)]
    got = as_dict(*dec.decode(probs, st, [True] * 3), dec)
    compare(want_off, got, None, "online+scorer, one call")
    assert "".join(L29[x] for x in got["tokens"][0, 0, :got["lens"][0, 0]]) == TEXTS[0]
    # several calls, against the reference's own streaming path fed the same chunks
    st = [ctcdecode_b200.DecoderState(dec) for _ in range(3)]
    for a, b in ONLINE_CUTS:
        r = dec.decode(probs[:, a:b], st, [False] * 3)
        assert r[0].shape == (3, 0, 0)
    got = as_dict(*dec.decode(probs[:, 200:], st, [True] * 3), dec)
    want = recorded("word", "online_streaming")
    want_c = dict(want, n_results=want_off["n_results"])
    compare(want_c, got, None, "online+scorer, five calls vs reference streaming")
    compare(want_off, got, None, "online+scorer, five calls vs reference offline")
    # a state created without a scorer cannot be mixed with scorer states
    plain = ctcdecode_b200.OnlineCTCBeamDecoder(L29, beam_width=32)
    with pytest.raises(Exception):
        dec.decode(probs[:2, :4], [ctcdecode_b200.DecoderState(dec), ctcdecode_b200.DecoderState(plain)], [False] * 2)


def c5_text_probs(B, T, seed):
    """Posteriors that noisily spell sentences over the words of the reference's test.arpa (BASELINE config 5)."""
    import random
    rng = random.Random(seed)
    words = ["a", "also", "beyond", "call", "concerns", "consider", "for", "higher", "however", "i", "in", "is", "little",
             "loin", "look", "looking", "more", "on", "screening", "small", "the", "to", "watch", "what", "would"]
    texts = []
    for _ in range(B):
        s = ""
        while len(s) < T // 5:
            s += (" " if s else "") + rng.choice(words)
        texts.append(s[: T // 4])
    return text_probs(texts, L29, T, seed=seed), texts


@pytest.mark.gpu
def test_cuda_config5_as_stated_matches_reference():
    """BASELINE config 5 as BASELINE.json states it: the reference's tests/test.arpa, alpha 2.0, beta 1.0, beam 100,
    T = 1000 (12 utterances here; bench.py --config c5 runs the 64), against the reference's own Scorer path on the same
    box: tokens, timesteps, lens identical, float32 scores bit-exact; plus alpha / beta that are NOT exact in float32
    after reset_params (reference Scorer::reset_params takes floats, scorer.cpp:122-125)."""
    import torch
    import ctcdecode_b200
    probs, texts = c5_text_probs(12, 1000, seed=7)
    noise = ctc_like_probs(4, 1000, 29, seed=8)
    probs = torch.cat([probs, noise], 0)
    want = recorded("word", "c5")
    dec = ctcdecode_b200.CTCBeamDecoder(L29, model_path=lm_replay.table(REF_ARPA), alpha=2.0, beta=1.0,
                                        beam_width=100, scorer_provider=PROVIDER)
    assert dec.dict_size() == int(want["dict_size"]) and dec.max_order() == 5
    out, scores, ts, lens = dec.decode(probs)
    got = dict(tokens=out.numpy(), timesteps=ts.numpy(), scores=scores.numpy(), lens=lens.numpy(),
               n_results=dec.last_n_results.numpy(), ties=dec.last_flags.numpy())
    checked, skipped = compare(want, got, None, "config 5 (test.arpa)")
    assert checked >= 12
    hits = sum("".join(L29[x] for x in out[b, 0, :lens[b, 0]]) == texts[b] for b in range(12))
    assert hits >= 9, hits  # the posteriors are noisy; most utterances still decode to their sentence
    dec.reset_params(0.3, 0.1)
    want = recorded("word", "c5_reset")
    out, scores, ts, lens = dec.decode(probs[:6])
    got = dict(tokens=out.numpy(), timesteps=ts.numpy(), scores=scores.numpy(), lens=lens.numpy(),
               n_results=dec.last_n_results.numpy(), ties=dec.last_flags.numpy())
    compare(want, got, None, "after reset_params(0.3, 0.1)")


# ---------------------------------------------------------------------------------------------------------------
#  character-based language models (reference scorer.cpp:63-71 / :172-174, ctc_beam_search_decoder.cpp:46, :120-137,
#  :174): no dictionary, an LM term for EVERY appended character, no last-word term at read-out
# ---------------------------------------------------------------------------------------------------------------
CHAR_LM = os.path.join(ROOT, "tests", "data", "char_lm.arpa")
LCHAR = ["_"] + list("abcdefghijklmnop") + ["|", "'", "é", " ", "z", "qu"]   # the last three are not in the model


@pytest.mark.parametrize("per_frame", [False, True, 5], ids=["persistent", "per_frame_launch", "chunks_of_5"])
@pytest.mark.parametrize("name", golden_util.names_char())
def test_emulation_char_lm_matches_reference_golden(name, per_frame, monkeypatch):
    if per_frame is True:
        monkeypatch.setenv("CTC_EMU_LM_PER_FRAME", "1")
    elif per_frame:
        monkeypatch.setenv("CTC_EMU_LM_CHUNK", str(per_frame))
    probs, seq_lens, kw, gold, alpha, beta = golden_util.load_lm(name)
    ref = Replay(LCHAR, CHAR_LM)
    assert ref.is_character_based() == 1 and ref.max_order() == 3
    got = emul.decode_lm(probs, ref.lib, ref.scorer, LCHAR, [], ref.max_order(), alpha, beta, seq_lens=seq_lens,
                         char_based=True, **kw)
    compare(gold, got, None, name)
    if orc.reference_available():  # and the fixture still is what the original decoder says
        live = orc.Reference(LCHAR, model_path=CHAR_LM, alpha=alpha, beta=beta)
        assert live.dict_size() == 0
        compare(gold, live.decode(probs, seq_lens, num_processes=2, **kw), None, name + " (live reference)")


CHAR_CFGS = [
    dict(alpha=1.0, beta=0.3, beam=32, T=80, seed=31),
    dict(alpha=0.0, beta=0.0, beam=16, T=60, seed=32),
    dict(alpha=2.5, beta=-1.0, beam=8, T=100, seed=33, log_input=True),
    dict(alpha=0.7, beta=2.0, beam=64, T=50, seed=34, cutoff_prob=0.95),
    dict(alpha=1.0, beta=1.0, beam=20, T=70, seed=35, blank_id=5, cutoff_top_n=6),
    dict(alpha=1.0, beta=0.5, beam=30, T=40, seed=36, flat=True),
    dict(alpha=1.5, beta=0.2, beam=3, T=120, seed=37, nolabels=True),
]


def char_cfg_inputs(cfg):
    """-> probs, labels, alpha, beta, decoder keywords"""
    cfg = dict(cfg)
    alpha, beta, T, seed = cfg.pop("alpha"), cfg.pop("beta"), cfg.pop("T"), cfg.pop("seed")
    labels = LCHAR
    if cfg.pop("nolabels", False):
        labels = ["_"] + list("abcdefgh")   # no " " label at all: a character-based scorer does not need one
    V = len(labels)
    probs = flat_probs(3, T, V, seed=seed) if cfg.pop("flat", False) else ctc_like_probs(3, T, V, seed=seed)
    if cfg.get("log_input"):
        probs = probs.log()
    return probs.numpy(), labels, alpha, beta, cfg


@pytest.mark.parametrize("cfg", CHAR_CFGS)
def test_emulation_char_lm_matches_reference(cfg):
    probs, labels, alpha, beta, kw = char_cfg_inputs(cfg)
    ref = Replay(labels, CHAR_LM)
    got = emul.decode_lm(probs, ref.lib, ref.scorer, labels, [], ref.max_order(), alpha, beta, char_based=True, **kw)
    compare(recorded("char", "cfg%d" % CHAR_CFGS.index(cfg)), got, None, str(cfg))


@pytest.mark.gpu
@pytest.mark.parametrize("per_frame", [False, True], ids=["persistent", "per_frame_launch"])
@pytest.mark.parametrize("name", golden_util.names_char())
def test_cuda_char_lm_matches_reference_golden(name, per_frame, monkeypatch):
    import torch
    import ctcdecode_b200
    if per_frame:
        monkeypatch.setenv("CTCDEC_LM_PER_FRAME", "1")
    probs, seq_lens, kw, gold, alpha, beta = golden_util.load_lm(name)
    dec = ctcdecode_b200.CTCBeamDecoder(LCHAR, model_path=lm_replay.table(CHAR_LM), alpha=alpha, beta=beta, beam_width=kw["beam"],
                                        cutoff_top_n=kw["cutoff_top_n"], cutoff_prob=kw["cutoff_prob"],
                                        log_probs_input=kw["log_input"], scorer_provider=PROVIDER)
    assert dec.dict_size() == 0 and dec.max_order() == 3 and dec.character_based() == 1
    sl = None if seq_lens is None else torch.from_numpy(seq_lens)
    out, scores, ts, lens = dec.decode(torch.from_numpy(probs), sl)
    got = dict(tokens=out.numpy(), timesteps=ts.numpy(), scores=scores.numpy(), lens=lens.numpy(),
               n_results=dec.last_n_results.numpy(), ties=dec.last_flags.numpy())
    compare(gold, got, None, name)


@pytest.mark.gpu
def test_cuda_char_lm_matches_live_reference_offline_and_online():
    """a config-5 sized batch (16 x T=300, beam 100) with the character model against the reference run on the same
    box, then the same utterances through OnlineCTCBeamDecoder in four chunks (device-resident rows of LM terms that
    grow with the stream)"""
    import torch
    import ctcdecode_b200
    probs = ctc_like_probs(16, 300, len(LCHAR), seed=51)
    want = recorded("char", "live")
    dec = ctcdecode_b200.CTCBeamDecoder(LCHAR, model_path=lm_replay.table(CHAR_LM), alpha=1.3, beta=0.6, beam_width=100,
                                        scorer_provider=PROVIDER)
    out, scores, ts, lens = dec.decode(probs)
    got = dict(tokens=out.numpy(), timesteps=ts.numpy(), scores=scores.numpy(), lens=lens.numpy(),
               n_results=dec.last_n_results.numpy(), ties=dec.last_flags.numpy())
    compare(want, got, None, "character model, 16 x 300, beam 100")
    want = recorded("char", "live_online")
    odec = ctcdecode_b200.OnlineCTCBeamDecoder(LCHAR, model_path=lm_replay.table(CHAR_LM), alpha=1.3, beta=0.6, beam_width=24,
                                               scorer_provider=PROVIDER)
    st = [ctcdecode_b200.DecoderState(odec) for _ in range(3)]
    for a, b in [(0, 1), (1, 130), (130, 131)]:
        odec.decode(probs[:3, a:b], st, [False] * 3)
    res, scores, ts, lens = odec.decode(probs[:3, 131:], st, [True] * 3)
    got = dict(tokens=res.numpy(), timesteps=ts.numpy(), scores=scores.numpy(), lens=lens.numpy(),
               n_results=odec.last_n_results.numpy(), ties=odec.last_flags.numpy())
    compare(want, got, None, "character model, online in four calls")


def char_random_configurations():
    """seeded random walk over (labels, beam, T, alpha, beta, cutoffs, blank position, log input, ragged lengths)
    -> probs, seq_lens, labels, alpha, beta, decoder keywords"""
    rng = np.random.default_rng(2024)
    for trial in range(10):
        nlab = int(rng.integers(4, 24))
        pool = list("abcdefghijklmnop") + ["|", "'", "é", "z", " ", "qu"]
        labels = [pool[i] for i in rng.permutation(len(pool))[:nlab - 1]]
        blank = int(rng.integers(0, nlab))
        labels.insert(blank, "_")
        T, B = int(rng.integers(1, 70)), int(rng.integers(1, 4))
        kw = dict(beam=int(rng.integers(1, 40)), blank_id=blank, cutoff_top_n=int(rng.integers(2, 41)),
                  cutoff_prob=float(rng.choice([1.0, 1.0, 0.999, 0.9])), log_input=bool(rng.integers(0, 2)))
        alpha, beta = float(np.round(rng.uniform(0, 2.5), 2)), float(np.round(rng.uniform(-1, 2), 2))
        probs = (flat_probs(B, T, nlab, seed=int(rng.integers(1 << 30))) if rng.random() < 0.3
                 else ctc_like_probs(B, T, nlab, seed=int(rng.integers(1 << 30)), blank_id=blank))
        if kw["log_input"]:
            probs = probs.log()
        seq_lens = None if rng.random() < 0.5 else rng.integers(0, T + 1, B).astype(np.int32)
        yield probs.numpy(), seq_lens, labels, alpha, beta, kw


def test_emulation_char_lm_random_configurations():
    """the random walk of char_random_configurations over the host / kernel protocols too, with the character model:
    CPU emulation of the CTA program against the reference"""
    for trial, (probs, seq_lens, labels, alpha, beta, kw) in enumerate(char_random_configurations()):
        ref = Replay(labels, CHAR_LM)
        want = recorded("char", "trial%d" % trial)
        env = [{}, {"CTC_EMU_LM_PER_FRAME": "1"}, {"CTC_EMU_LM_CHUNK": "3"}][trial % 3]
        old = {k: os.environ.get(k) for k in env}
        os.environ.update(env)
        try:
            got = emul.decode_lm(probs, ref.lib, ref.scorer, labels, [], ref.max_order(), alpha, beta,
                                 seq_lens=seq_lens, char_based=True, **kw)
        finally:
            for k, v in old.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
        compare(want, got, None, "trial %d: %r labels %d T %d B %d a %.2f b %.2f %s"
                % (trial, kw, len(labels), probs.shape[1], probs.shape[0], alpha, beta, env))
