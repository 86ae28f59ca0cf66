"""TEST INFRASTRUCTURE ONLY: the scorer provider that answers from recorded language-model scores
(tests/native/lm_replay.cpp), its tables (tests/golden/<model>.lmtab.gz) and the recorded outputs of the original
decoder for the scorer-path tests (tests/golden/recorded/lm_cases_*.npz), all written by tests/golden/make_lm_tables.py."""
import ctypes
import gzip
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "native", "lm_replay.cpp")
_OUT = os.path.join(_HERE, "native", "_build", "liblm_replay.so")
GOLDEN = os.path.join(_HERE, "golden")
_i32p = ctypes.POINTER(ctypes.c_int32)


def build():
    """Path of the provider library, compiled on first use."""
    if not os.path.exists(_OUT) or os.path.getmtime(_OUT) < os.path.getmtime(_SRC):
        os.makedirs(os.path.dirname(_OUT), exist_ok=True)
        tmp = _OUT + ".tmp%d" % os.getpid()
        # libstdc++ stays a shared dependency (as in emul.py): a static copy would clash with the one python loaded
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-nostdlib++", "-pthread", _SRC, "-o", tmp,
                        "-l:libstdc++.so.6", "-lm"], check=True)
        os.replace(tmp, _OUT)
    return _OUT


def table(model_path):
    """Path of the table recorded for a language model file (tests/data/tiny_lm.arpa: tests/golden/tiny_lm.lmtab.gz),
    unpacked on first use beside the provider library."""
    name = os.path.splitext(os.path.basename(model_path))[0] + ".lmtab"
    packed, out = os.path.join(GOLDEN, name + ".gz"), os.path.join(os.path.dirname(_OUT), name)
    if os.path.exists(packed) and (not os.path.exists(out) or os.path.getmtime(out) < os.path.getmtime(packed)):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        tmp = out + ".tmp%d" % os.getpid()
        with gzip.open(packed, "rb") as f, open(tmp, "wb") as g:
            g.write(f.read())
        os.replace(tmp, out)
    return out


class Replay:
    """A scorer of the provider: what the tests hand to the emulated CTA program (lib, scorer) and ask about."""

    def __init__(self, labels, model_path):
        self.lib = ctypes.CDLL(build())
        L = self.lib
        L.ref_scorer_new.restype = ctypes.c_void_p
        L.ref_scorer_new.argtypes = [ctypes.c_double, ctypes.c_double, ctypes.c_char_p,
                                     ctypes.POINTER(ctypes.c_char_p), ctypes.c_int]
        L.ref_scorer_free.argtypes = [ctypes.c_void_p]
        L.ref_scorer_is_character_based.argtypes = [ctypes.c_void_p]
        L.ref_scorer_max_order.argtypes = [ctypes.c_void_p]
        L.ref_scorer_max_order.restype = ctypes.c_size_t
        L.ref_scorer_cond_from_labels.restype = ctypes.c_double
        L.ref_scorer_cond_from_labels.argtypes = [ctypes.c_void_p, _i32p, ctypes.c_int]
        L.ref_scorer_sent_from_labels.restype = ctypes.c_double
        L.ref_scorer_sent_from_labels.argtypes = [ctypes.c_void_p, _i32p, ctypes.c_int]
        L.ref_lm_vocabulary.restype = ctypes.c_size_t
        L.ref_lm_vocabulary.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_size_t]
        L.lm_replay_save.argtypes = [ctypes.c_void_p, ctypes.c_char_p]
        self.path = table(model_path).encode()
        labels_c = (ctypes.c_char_p * len(labels))(*[s.encode() for s in labels])
        self.scorer = L.ref_scorer_new(0.0, 0.0, self.path, labels_c, len(labels))
        assert self.scorer, "cannot read " + self.path.decode()

    def lm_vocabulary(self):
        n = self.lib.ref_lm_vocabulary(self.path, None, 0)
        buf = ctypes.create_string_buffer(n)
        self.lib.ref_lm_vocabulary(self.path, buf, n)
        return buf.value.decode().split("\n")[:-1]

    def max_order(self):
        return int(self.lib.ref_scorer_max_order(self.scorer))

    def is_character_based(self):
        return int(self.lib.ref_scorer_is_character_based(self.scorer))

    def __del__(self):
        if getattr(self, "scorer", None):
            self.lib.ref_scorer_free(self.scorer)
            self.scorer = None


def recorded(group, key):
    """The original decoder's outputs for one case (tokens / timesteps padded with -1 to max(lens) steps)."""
    z = np.load(os.path.join(GOLDEN, "recorded", "lm_cases_%s.npz" % group))
    return {f.split("/", 1)[1]: z[f] for f in z.files if f.startswith(key + "/")}
