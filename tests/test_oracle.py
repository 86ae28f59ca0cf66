"""The oracle is pinned before it is trusted: the plain-C restatement (oracle/ctc_oracle.c) must reproduce
(1) the reference's own known answers (reference tests/test_decode.py:13-32,37-91),
(2) the committed outputs of the unmodified reference build (tests/golden, all beams / timesteps / scores),
(3) the reference build's recorded outputs on seeded inputs, and the build itself whenever oracle/_ref is present."""
import numpy as np
import pytest

from ctcdecode_b200.synth import ctc_like_probs, flat_probs
from oracle import oracle as orc
from tests import golden_util
from tests.parity import compare

VOCAB = ["'", " ", "a", "b", "c", "d", "_"]  # reference tests/test_decode.py:13


def _string(tokens, n):
    return "".join(VOCAB[x] for x in tokens[:n])


def test_reference_known_answers(cport):
    probs, _, kw, _ = golden_util.load("ref_kat_beam20")
    r = cport.decode(probs, **kw)
    assert _string(r["tokens"][0, 0], r["lens"][0, 0]) == "acdc"   # test_beam_search_decoder_1
    assert _string(r["tokens"][1, 0], r["lens"][1, 0]) == "b'a"    # test_beam_search_decoder_2 / _batch
    # SURVEY.md Appendix C.3: full golden values of the reference for these inputs
    assert r["scores"][0, 0] == np.float32(6.480283737182617)
    assert list(r["timesteps"][0, 0, :4]) == [0, 1, 4, 5]
    assert list(r["tokens"][1, 3, :4]) == [3, 0, 2, 0] and list(r["timesteps"][1, 3, :4]) == [0, 2, 4, 4]
    lprobs, _, lkw, _ = golden_util.load("ref_kat_beam20_log")      # test_beam_search_decoder_batch_log
    rl = cport.decode(lprobs, **lkw)
    assert _string(rl["tokens"][0, 0], rl["lens"][0, 0]) == "acdc"
    assert _string(rl["tokens"][1, 0], rl["lens"][1, 0]) == "b'a"
    assert np.allclose(rl["scores"], r["scores"], atol=1e-5)


@pytest.mark.parametrize("name", golden_util.names())
def test_cport_matches_reference_golden(cport, name):
    probs, seq_lens, kw, ref = golden_util.load(name)
    got = cport.decode(probs, seq_lens, **kw)
    checked, skipped = compare(ref, got, got["ties"], name)
    assert checked + skipped == probs.shape[0]
    if not name.startswith(("flat", "cp03")):
        assert skipped == 0


REF_BUILD_CASES = [
    dict(B=3, T=150, V=29, seed=11, beam=48),
    dict(B=2, T=90, V=40, seed=12, beam=24, cutoff_top_n=12),
    dict(B=2, T=60, V=300, seed=13, beam=40, cutoff_prob=0.99),
    dict(B=2, T=80, V=29, seed=14, beam=30, cutoff_prob=0.5),
    dict(B=4, T=100, V=29, seed=15, beam=50, flat=True),
]


def ref_build_inputs(cfg):
    """-> probs, V, decoder keywords"""
    cfg = dict(cfg)
    B, T, V, seed = cfg.pop("B"), cfg.pop("T"), cfg.pop("V"), cfg.pop("seed")
    probs = (flat_probs(B, T, V, seed) if cfg.pop("flat", False) else ctc_like_probs(B, T, V, seed)).numpy()
    return probs, V, cfg


@pytest.mark.parametrize("cfg", REF_BUILD_CASES)
def test_cport_matches_reference_build(cport, cfg):
    """against the reference build's recorded outputs for these inputs (tests/golden/make_golden.py), and against the
    build itself when oracle/_ref is present"""
    probs, V, kw = ref_build_inputs(cfg)
    got = cport.decode(probs, **kw)
    compare(golden_util.recorded_ref_build(REF_BUILD_CASES.index(cfg)), got, got["ties"], str(cfg))
    if orc.reference_available():
        compare(orc.Reference([str(i) for i in range(V)]).decode(probs, **kw), got, got["ties"], str(cfg) + " (live)")


def test_cport_streaming_equals_offline(cport):
    """DecoderState::next in chunks == one call (reference ctc_beam_search_decoder.cpp:230-243)."""
    probs = ctc_like_probs(1, 97, 29, seed=21).numpy()
    off = cport.decode(probs, beam=20)
    st = cport.state_new(29, 20)
    for a, b in [(0, 10), (10, 11), (11, 60), (60, 97)]:
        cport.state_next(st, probs[0, a:b])
    on = cport.state_decode(st, 20, 97)
    cport.state_free(st)
    n = on["n_results"]
    assert n == off["n_results"][0]
    assert np.array_equal(on["scores"][:n].view(np.int32), off["scores"][0, :n].view(np.int32))
    assert np.array_equal(on["lens"][:n], off["lens"][0, :n])
    for p in range(n):
        L = on["lens"][p]
        assert np.array_equal(on["tokens"][p, :L], off["tokens"][0, p, :L])
        assert np.array_equal(on["timesteps"][p, :L], off["timesteps"][0, p, :L])
