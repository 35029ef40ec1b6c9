"""Generates golden fixtures from the REFERENCE'S OWN CODE (modules.py, networks.py, train.py, data_load.py, utils.py
of a checkout of the reference project), executed under the TensorFlow API stand-in of tf_shim.py -- same seeded
inputs as make_golden.py and the tests, so the fixture sets are directly comparable.  Run from the repo root:
    python tests/golden/make_golden_refshim.py REFERENCE_DIR      (~10 min: 210 full-graph passes on the CPU)
"""
import os
import sys
import time
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
import tf_shim                                                   # noqa: E402
from dc_tts_b200.data_load import load_data                      # noqa: E402
from dc_tts_b200.hyperparams import Hyperparams as hp            # noqa: E402
from dc_tts_b200.params import init_params, synthetic_text       # noqa: E402
from oracle import ref_features as rf                            # noqa: E402
from oracle import ref_train as rtr                              # noqa: E402
from oracle import ref_vocoder as rv                             # noqa: E402

REF = os.path.abspath(sys.argv[1])
P = init_params(0, "perturbed")
store = tf_shim.Store(P)
tf_shim.install(store, REF)

# 1. one full-graph pass (train.py:48-68) on seeded inputs
L = synthetic_text(1, 60, seed=3)
mels = np.random.default_rng(11).uniform(0, 1, (1, hp.max_T, hp.n_mels)).astype(np.float32)
pma = np.array([7], np.int32)
o = tf_shim.run_graph(L, mels, pma, fetch=("Y", "max_attentions", "alignments", "Q", "K", "R"))
np.savez_compressed(os.path.join(HERE, "refshim_t2m_forward.npz"), Y=o["Y"], max_attentions=o["max_attentions"],
                    Q_sub=o["Q"][:, ::10, :16], K_sub=o["K"][:, ::10, :16], R_sub=o["R"][:, ::10, ::16],
                    align_win=o["alignments"][:, 7:10, :])

# 2. SSRN on a short mel (12 frames -> 48 x 1025)
Ys = np.random.default_rng(12).uniform(0, 1, (1, 12, hp.n_mels)).astype(np.float32)
zl, z = tf_shim.run_ssrn(Ys)
np.savez_compressed(os.path.join(HERE, "refshim_ssrn_T12.npz"), Z=z, Z_logits_sub=zl[:, :, ::8])
missing = sorted(set(P) - store.requested)
assert not missing, "variables the reference graph never asked for: %s" % missing[:5]

# 3. the synthesize loop (synthesize.py:45-57) on Harvard sentence #1: 210 full-graph passes, then SSRN
Lh = load_data("synthesize", os.path.join(ROOT, "harvard_sentences.txt"))[:1]
t0 = time.time()
r = tf_shim.synthesize(Lh)
np.savez_compressed(os.path.join(HERE, "refshim_synth_harvard1.npz"), L=Lh, Y=r["Y"], p_hist=r["p_hist"],
                    max_attentions=r["max_attentions"], Z_sub=r["Z"][:, ::8, ::8])
print("synthesis loop: %.0f s" % (time.time() - t0))

# 4. three steps of the loop on a batch of two, SSRN of the first 8 frames, and every variable the two graphs ask
#    for with the shape they ask for it with (a fresh store, so nothing else is counted)
store = tf_shim.Store(P)
tf_shim.install(store, REF)
r = tf_shim.synthesize(synthetic_text(2, 40, seed=5), steps=3, with_ssrn=False)
_, z = tf_shim.run_ssrn(r["Y"][:, :8])
names = sorted(store.requested)
np.savez_compressed(os.path.join(HERE, "refshim_few_steps.npz"), Y=r["Y"][:, :8], p_hist=r["p_hist"], Z=z,
                    names=np.array(names),
                    shapes=np.array([",".join(map(str, store.requested_shapes[n] or ())) for n in names]))

# 5. host-side pieces: the text adaptor on the reference's own harvard_sentences.txt (data_load.py:79-86), its
#    vocabulary, utils.guided_attention (utils.py:134-140) and the Noam schedule (utils.py:141-145)
tf_shim.install(tf_shim.Store({}), REF)
import data_load as ref_dl                                       # noqa: E402
import hyperparams as ref_hp                                     # noqa: E402
import utils as ref_utils                                        # noqa: E402
ref_hp.Hyperparams.test_data = os.path.join(REF, "harvard_sentences.txt")
texts = ref_dl.load_data("synthesize")
c2i, i2c = ref_dl.load_vocab()
vocab = "".join(i2c[i] for i in range(len(i2c)))
lr_steps = np.array([0, 1, 3999, 4000, 123456])
np.savez_compressed(os.path.join(HERE, "refshim_host.npz"), harvard_L=texts, vocab=np.array(vocab),
                    vocab_index=np.array([c2i[c] for c in vocab]), guided_attention=ref_utils.guided_attention(),
                    lr_steps=lr_steps, lr=np.array([float(ref_utils.learning_rate_decay(hp.lr, int(s))) for s in lr_steps]))

# 6. utils.spectrogram2wav / load_spectrograms with the absent `librosa` replaced by the restated primitives
#    (oracle/ref_vocoder.py, ref_features.py): how the reference COMPOSES them, 3 Griffin-Lim iterations
wavs = {}
ref_utils.librosa = types.SimpleNamespace(
    stft=lambda y, n_fft=None, hop_length=None, win_length=None: rv.stft(np.asarray(y, np.float32), n_fft, hop_length, win_length),
    istft=lambda S, hop_length=None, win_length=None, window="hann": rv.istft(S, hop_length, win_length),
    effects=types.SimpleNamespace(trim=lambda y: (lambda se: (y[se[0]:se[1]], se))(rv.trim_indices(np.asarray(y)))),
    filters=types.SimpleNamespace(mel=lambda sr, n_fft, n_mels: rf.mel_basis(sr, n_fft, n_mels)),
    load=lambda fpath, sr=None: (wavs[fpath], sr))
n_iter = ref_hp.Hyperparams.n_iter
ref_hp.Hyperparams.n_iter = 3
rng = np.random.default_rng(0)
mag = rng.uniform(0.2, 0.8, (40, 1 + hp.n_fft // 2)).astype(np.float32)
wav = ref_utils.spectrogram2wav(mag)
t = np.arange(int(hp.sr * 0.8)) / hp.sr
y = (0.2 * np.sin(2 * np.pi * 300 * t) + 0.02 * rng.standard_normal(t.size)).astype(np.float32)
y[:2000] *= 1e-5
wavs["LJ001-0001.wav"] = y
fname, mel, mg = ref_utils.load_spectrograms("LJ001-0001.wav")
ref_hp.Hyperparams.n_iter = n_iter
np.savez_compressed(os.path.join(HERE, "refshim_vocoder.npz"), wav=wav, fname=np.array(fname), mel=mel, mag=mg)

# 7. the losses of the reference's TRAINING graphs (train.py Graph(num=1 / num=2, mode="train")) on fixed batches, with
#    the oracle's deterministic dropout mask plugged into every dropout the graph places
tf_shim.install(tf_shim.Store(P), REF)
Lt = synthetic_text(2, 50, seed=7)
melt = np.random.default_rng(3).uniform(0, 1, (2, hp.max_T, hp.n_mels)).astype(np.float32)
t2m = {}
rate0 = ref_hp.Hyperparams.dropout_rate
for seed, rate in ((11, hp.dropout_rate), (0, 0.0)):
    ref_hp.Hyperparams.dropout_rate = rate
    t2m[seed] = tf_shim.run_train_graph(Lt, melt, lambda x, r, i, seed=seed: x * rtr.dropout_keep(x.shape, i, seed, r))
ref_hp.Hyperparams.dropout_rate = rate0
mels2 = np.random.default_rng(3).uniform(0, 1, (2, 12, hp.n_mels)).astype(np.float32)
mags2 = np.random.default_rng(4).uniform(0, 1, (2, 48, 1 + hp.n_fft // 2)).astype(np.float32)
ssrn, ssrn_calls = tf_shim.run_train_graph_ssrn(mels2, mags2, lambda x, r, i: x * rtr.dropout_keep(x.shape, i, 9, r))
T2M_KEYS, SSRN_KEYS = ("loss", "loss_mels", "loss_bd1", "loss_att"), ("loss", "loss_mags", "loss_bd2")
np.savez_compressed(os.path.join(HERE, "refshim_train_losses.npz"),
                    t2m_seeds=np.array([11, 0]), t2m_rates=np.array([hp.dropout_rate, 0.0]),
                    t2m_losses=np.array([[t2m[s][0][k] for k in T2M_KEYS] for s in (11, 0)]),
                    t2m_dropout_calls=np.array([t2m[s][1] for s in (11, 0)]),
                    ssrn_losses=np.array([ssrn[k] for k in SSRN_KEYS]), ssrn_dropout_calls=np.array(ssrn_calls))
print("reference-under-shim fixtures written to %s" % HERE)
