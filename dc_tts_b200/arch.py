"""Layer tables of the five DC-TTS networks, derived from the reference builders.

Each network in /root/reference/networks.py is a straight-line chain of three block
kinds (modules.py): `C` = conv1d (+LN +act), `HC` = highway conv, `D` = stride-2
transposed conv (+LN).  This module states those chains as data so that the host
wrappers, the parameter store, the oracle tests and the C library's own table
(csrc/dctts_nets.cu) can be cross-checked against one another.

Scope names follow the running counter `i` of the reference (e.g. networks.py:23-68).
"""
from collections import namedtuple

from .hyperparams import Hyperparams as hp

# Most characters (attention keys) per utterance a handle with hp.max_N <= 192 takes, as the shipped LJ hyper-parameters
# have.  The library fixes each handle's capacity at creation, max(192, round_up(max_N, 64)) for max_N <= 512, and
# reports it (Engine.KEY_CAPACITY); this value is the fallback for engines that do not.  A training batch with longer
# text fails in the library and is skipped by the trainer loop.
ATTENTION_KEY_CAPACITY = 192

# kind: "C" | "HC" | "D";  act: None | "relu";  pad: "SAME" | "CAUSAL"
Layer = namedtuple("Layer", "kind scope cin cout size rate pad act")


def _F():
    return 1 + hp.n_fft // 2


def textenc_layers():
    """networks.py:23-68 (embed_1 is handled separately; channels 128 -> 2d)."""
    d2 = 2 * hp.d
    L, i = [], 2
    L.append(Layer("C", "C_%d" % i, hp.e, d2, 1, 1, "SAME", "relu")); i += 1
    L.append(Layer("C", "C_%d" % i, d2, d2, 1, 1, "SAME", None)); i += 1
    for _ in range(2):
        for j in range(4):
            L.append(Layer("HC", "HC_%d" % i, d2, d2, 3, 3 ** j, "SAME", None)); i += 1
    for _ in range(2):
        L.append(Layer("HC", "HC_%d" % i, d2, d2, 3, 1, "SAME", None)); i += 1
    for _ in range(2):
        L.append(Layer("HC", "HC_%d" % i, d2, d2, 1, 1, "SAME", None)); i += 1
    return L


def audioenc_layers():
    """networks.py:81-124, all causal."""
    d = hp.d
    L, i = [], 1
    L.append(Layer("C", "C_%d" % i, hp.n_mels, d, 1, 1, "CAUSAL", "relu")); i += 1
    L.append(Layer("C", "C_%d" % i, d, d, 1, 1, "CAUSAL", "relu")); i += 1
    L.append(Layer("C", "C_%d" % i, d, d, 1, 1, "CAUSAL", None)); i += 1
    for _ in range(2):
        for j in range(4):
            L.append(Layer("HC", "HC_%d" % i, d, d, 3, 3 ** j, "CAUSAL", None)); i += 1
    for _ in range(2):
        L.append(Layer("HC", "HC_%d" % i, d, d, 3, 3, "CAUSAL", None)); i += 1
    return L


def audiodec_layers():
    """networks.py:166-209, all causal; the last C (-> n_mels) yields the logits."""
    d = hp.d
    L, i = [], 1
    L.append(Layer("C", "C_%d" % i, 2 * d, d, 1, 1, "CAUSAL", None)); i += 1
    for j in range(4):
        L.append(Layer("HC", "HC_%d" % i, d, d, 3, 3 ** j, "CAUSAL", None)); i += 1
    for _ in range(2):
        L.append(Layer("HC", "HC_%d" % i, d, d, 3, 1, "CAUSAL", None)); i += 1
    for _ in range(3):
        L.append(Layer("C", "C_%d" % i, d, d, 1, 1, "CAUSAL", "relu")); i += 1
    L.append(Layer("C", "C_%d" % i, d, hp.n_mels, 1, 1, "CAUSAL", None)); i += 1
    return L


def ssrn_layers():
    """networks.py:223-290, all SAME; time axis doubles at each D."""
    c, F = hp.c, _F()
    L, i = [], 1
    L.append(Layer("C", "C_%d" % i, hp.n_mels, c, 1, 1, "SAME", None)); i += 1
    for j in range(2):
        L.append(Layer("HC", "HC_%d" % i, c, c, 3, 3 ** j, "SAME", None)); i += 1
    for _ in range(2):
        L.append(Layer("D", "D_%d" % i, c, c, 3, 1, "SAME", None)); i += 1
        for j in range(2):
            L.append(Layer("HC", "HC_%d" % i, c, c, 3, 3 ** j, "SAME", None)); i += 1
    L.append(Layer("C", "C_%d" % i, c, 2 * c, 1, 1, "SAME", None)); i += 1
    for _ in range(2):
        L.append(Layer("HC", "HC_%d" % i, 2 * c, 2 * c, 3, 1, "SAME", None)); i += 1
    L.append(Layer("C", "C_%d" % i, 2 * c, F, 1, 1, "SAME", None)); i += 1
    for _ in range(2):
        L.append(Layer("C", "C_%d" % i, F, F, 1, 1, "SAME", "relu")); i += 1
    L.append(Layer("C", "C_%d" % i, F, F, 1, 1, "SAME", None))
    return L


NETWORKS = {
    "Text2Mel/TextEnc": textenc_layers,
    "Text2Mel/AudioEnc": audioenc_layers,
    "Text2Mel/AudioDec": audiodec_layers,
    "SSRN": ssrn_layers,
}


def param_shapes():
    """TF variable name -> shape for every trainable variable on the path
    (SURVEY.md App. C; names follow the scope strings at train.py:49-76,
    modules.py:32,46,189-190 and the tf.layers defaults `conv1d`,
    `conv2d_transpose`, `kernel`, `bias`, `gamma`, `beta`)."""
    shapes = {"Text2Mel/TextEnc/embed_1/lookup_table": (len(hp.vocab), hp.e)}
    for net, fn in NETWORKS.items():
        for l in fn():
            base = "%s/%s" % (net, l.scope)
            if l.kind == "C":
                shapes[base + "/conv1d/kernel"] = (l.size, l.cin, l.cout)
                shapes[base + "/conv1d/bias"] = (l.cout,)
                shapes[base + "/normalize/gamma"] = (l.cout,)
                shapes[base + "/normalize/beta"] = (l.cout,)
            elif l.kind == "HC":
                shapes[base + "/conv1d/kernel"] = (l.size, l.cin, 2 * l.cout)
                shapes[base + "/conv1d/bias"] = (2 * l.cout,)
                for h in ("H1", "H2"):
                    shapes[base + "/%s/gamma" % h] = (l.cout,)
                    shapes[base + "/%s/beta" % h] = (l.cout,)
            else:  # D
                shapes[base + "/conv2d_transpose/kernel"] = (1, l.size, l.cout, l.cin)
                shapes[base + "/conv2d_transpose/bias"] = (l.cout,)
                shapes[base + "/normalize/gamma"] = (l.cout,)
                shapes[base + "/normalize/beta"] = (l.cout,)
    return shapes
