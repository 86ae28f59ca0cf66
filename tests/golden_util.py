"""Loads tests/golden/*.npz (outputs of the unmodified reference, see tests/golden/make_golden.py)."""
import glob
import os

import numpy as np

HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def names(lm=False):
    """Fixture names; the scorer-path fixtures (lm_*) are listed separately."""
    allf = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(HERE, "*.npz")))
    return [n for n in allf if n.startswith("lm_") == lm and not n.startswith("lmchar_")]


def names_char():
    """Fixtures of the scorer path with a character-based model (tests/golden/make_golden_char.py)."""
    return sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(HERE, "lmchar_*.npz")))


def load_lm(name):
    z = np.load(os.path.join(HERE, name + ".npz"))
    probs, seq_lens, kw, ref = load(name)
    return probs, seq_lens, kw, ref, float(z["lm"][0]), float(z["lm"][1])


def recorded_ref_build(i):
    """The reference build's outputs for tests/test_oracle.py REF_BUILD_CASES[i] (tests/golden/make_golden.py)."""
    z = np.load(os.path.join(HERE, "recorded", "ref_build_cases.npz"))
    return {f.split("/", 1)[1]: z[f] for f in z.files if f.startswith("case%d/" % i)}


def load(name):
    z = np.load(os.path.join(HERE, name + ".npz"))
    beam, top_n, blank, log_input = [int(x) for x in z["params"]]
    kw = dict(beam=beam, cutoff_top_n=top_n, blank_id=blank, log_input=bool(log_input),
              cutoff_prob=float(z["cutoff_prob"][0]))
    seq_lens = z["seq_lens"] if z["seq_lens"].size else None
    ref = {k: z[k] for k in ("tokens", "timesteps", "scores", "lens", "n_results")}
    return z["probs"], seq_lens, kw, ref
