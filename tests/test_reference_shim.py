"""Parity against the REFERENCE'S OWN SOURCE.  tests/golden/refshim_*.npz were produced by importing the
reference project's {modules,networks,train,data_load,utils}.py and executing them under the TensorFlow API
stand-in tests/golden/tf_shim.py (generator: tests/golden/make_golden_refshim.py).  They pin everything the
reference's Python decides (topology, dilations, paddings, scopes/variable names and shapes, the decoder shift,
the window mask, the text adaptor, the training losses, how the vocoder composes its primitives); the TF op
semantics themselves are the shim's restatement (see its header).

  * CPU: the oracle's restatements vs these fixtures.
  * GPU: the CUDA path vs these fixtures."""
import os
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, golden
from dc_tts_b200.hyperparams import Hyperparams as hp
from dc_tts_b200.params import init_params, synthetic_text
from oracle import ref_numpy as rn
from oracle import ref_torch as rt

TOL = 1e-3            # north_star: max-abs on mel / linear magnitudes


@pytest.fixture(scope="module")
def P():
    return init_params(0, "perturbed")


def _inputs_forward():
    L = synthetic_text(1, 60, seed=3)
    mels = np.random.default_rng(11).uniform(0, 1, (1, hp.max_T, hp.n_mels)).astype(np.float32)
    return L, mels, np.array([7], np.int32)


def test_oracle_full_graph_vs_reference_code(P):
    g = golden("refshim_t2m_forward.npz")
    L, mels, pma = _inputs_forward()
    o = rt.text2mel_forward(P, L, mels, pma)
    assert np.abs(o["Y"].numpy() - g["Y"]).max() < 2e-5
    assert np.array_equal(o["max_attentions"].numpy(), g["max_attentions"])
    assert np.abs(o["Q"].numpy()[:, ::10, :16] - g["Q_sub"]).max() < 1e-4
    assert np.abs(o["K"].numpy()[:, ::10, :16] - g["K_sub"]).max() < 1e-4
    assert np.abs(o["R"].numpy()[:, ::10, ::16] - g["R_sub"]).max() < 1e-4
    assert np.abs(o["alignments"].numpy()[:, 7:10, :] - g["align_win"]).max() < 1e-5
    # and the two fixture sets (oracle-made, reference-made) agree
    g0 = golden("t2m_forward.npz")
    assert np.abs(g0["Y"] - g["Y"]).max() < 2e-5 and np.array_equal(g0["max_attentions"], g["max_attentions"])


def test_oracle_ssrn_vs_reference_code(P):
    g = golden("refshim_ssrn_T12.npz")
    Y = np.random.default_rng(12).uniform(0, 1, (1, 12, hp.n_mels)).astype(np.float32)
    zl, z = rt.SSRN(P, torch.from_numpy(Y))
    assert np.abs(z.numpy() - g["Z"]).max() < 2e-5
    assert np.abs(zl.numpy()[:, :, ::8] - g["Z_logits_sub"]).max() < 5e-4
    zl2, z2 = rn.SSRN(P, Y)
    assert np.abs(np.asarray(z2) - g["Z"]).max() < 2e-5


def test_oracle_synthesis_loop_vs_reference_code():
    """210 free-running steps of the reference's loop (synthesize.py:45-57) on Harvard sentence 1: identical window
    trajectory, mel within float32 noise -- against the oracle-made fixture of the same run."""
    g, g0 = golden("refshim_synth_harvard1.npz"), golden("synth_harvard1.npz")
    assert np.array_equal(g["L"], g0["L"])
    assert np.array_equal(g["p_hist"], g0["p_hist"])
    assert np.abs(g["Y"] - g0["Y"]).max() < 1e-4
    assert np.abs(g["Z_sub"] - g0["Z_sub"]).max() < 1e-4


def test_reference_code_live_few_steps(P):
    """Three steps of the reference's loop on a batch of two and its SSRN on the first 8 frames (refshim_few_steps.npz)
    vs the oracle's literal schedule, and the variables the reference's graphs asked for vs the parameter schema."""
    g = golden("refshim_few_steps.npz")
    L = synthetic_text(2, 40, seed=5)
    with torch.no_grad():
        o = rt.synthesize(P, L, steps=3, literal=True, record=True)
    assert np.abs(g["Y"][:, :3] - o["Y"].numpy()[:, :3]).max() < 2e-5
    assert np.array_equal(g["p_hist"], o["p_hist"].numpy()[:, :3])
    _, z2 = rt.SSRN(P, torch.from_numpy(g["Y"]))
    assert np.abs(g["Z"] - z2.numpy()).max() < 2e-5
    # the graph asked for exactly the variables of the schema (SURVEY.md App. C), with the schema's shapes
    requested = {str(n): tuple(int(s) for s in str(sh).split(",")) for n, sh in zip(g["names"], g["shapes"])}
    assert requested == {n: v.shape for n, v in P.items()}
    # an unknown or mis-shaped variable is an error of the shim that recorded them, not a silent default
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import tf_shim
    name = "Text2Mel/TextEnc/C_2/conv1d/kernel"
    bad = dict(P); bad[name] = np.zeros((1, 128, 511), np.float32)
    with pytest.raises(ValueError):
        tf_shim.Store(bad).get(name, requested[name])
    with pytest.raises(KeyError):
        tf_shim.Store(P).get(name + "_1", requested[name])


# ------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_cuda_full_graph_vs_reference_code(engine, path):
    g = golden("refshim_t2m_forward.npz")
    L, mels, pma = _inputs_forward()
    Y, M, A = engine.text2mel_forward(L, mels, pma)
    assert np.abs(Y.cpu().numpy() - g["Y"]).max() < TOL
    assert np.array_equal(M.cpu().numpy(), g["max_attentions"])
    assert np.abs(A.cpu().numpy()[:, 7:10, :] - g["align_win"]).max() < 1e-4


@pytest.mark.gpu
def test_cuda_ssrn_vs_reference_code(engine, path):
    g = golden("refshim_ssrn_T12.npz")
    Y = np.random.default_rng(12).uniform(0, 1, (1, 12, hp.n_mels)).astype(np.float32)
    _, Z = engine.ssrn(Y, want_logits=False)
    assert np.abs(Z.cpu().numpy() - g["Z"]).max() < TOL


@pytest.mark.gpu
def test_cuda_synthesis_vs_reference_code(engine):
    """The CUDA-graph decode loop + SSRN vs the reference's own loop run under the shim (Harvard sentence 1)."""
    g = golden("refshim_synth_harvard1.npz")
    Y, Pm, M, A = engine.text2mel_generate(g["L"], want_final_attention=True)
    assert np.array_equal(Pm.cpu().numpy(), g["p_hist"])
    assert np.abs(Y.cpu().numpy() - g["Y"]).max() < TOL
    assert np.array_equal(M.cpu().numpy(), g["max_attentions"])
    _, Z = engine.ssrn(Y, want_logits=False)
    assert np.abs(Z.cpu().numpy()[:, ::8, ::8] - g["Z_sub"]).max() < TOL


# ------------------------------------------------------------------------------------------- host-side pieces
def test_text_adaptor_vs_reference_code():
    """data_load.load_data("synthesize") of the reference itself (data_load.py:79-86) on its own harvard_sentences.txt,
    and its load_vocab() (refshim_host.npz), vs the mirror in dc_tts_b200/data_load.py: all 20 sentences, every id."""
    g = golden("refshim_host.npz")
    ref = g["harvard_L"]
    from dc_tts_b200.data_load import load_data, load_vocab
    mine = load_data("synthesize", os.path.join(ROOT, "harvard_sentences.txt"))
    assert ref.shape == (20, hp.max_N) and ref.dtype == np.int32
    assert np.array_equal(ref, mine)
    vocab = str(g["vocab"])
    assert load_vocab() == ({c: int(i) for c, i in zip(vocab, g["vocab_index"])}, dict(enumerate(vocab)))
    assert np.array_equal(golden("refshim_synth_harvard1.npz")["L"], ref[:1])


def test_training_constants_vs_reference_code():
    """utils.guided_attention (utils.py:134-140) and the Noam schedule (utils.py:141-145) of the reference itself
    (refshim_host.npz)."""
    from oracle import ref_train as rtr
    g = golden("refshim_host.npz")
    np.testing.assert_allclose(g["guided_attention"], rtr.guided_attention(), rtol=0, atol=1e-7)
    assert list(g["lr_steps"]) == [0, 1, 3999, 4000, 123456]
    for gs, lr in zip(g["lr_steps"], g["lr"]):
        assert float(lr) == pytest.approx(rtr.learning_rate(int(gs)), rel=1e-6)


def test_vocoder_and_feature_composition_vs_reference_code(monkeypatch):
    """utils.spectrogram2wav / get_spectrograms / load_spectrograms of the reference itself (refshim_vocoder.npz), run
    with the absent `librosa` replaced by the restated primitives (oracle/ref_vocoder.py, ref_features.py): pins how
    the reference COMPOSES them (de-normalisation, power, Griffin-Lim loop, lfilter, trim; pre-emphasis, mel, dB,
    normalisation, reduction) -- the primitives themselves stay a restatement."""
    from oracle import ref_features as rf
    from oracle import ref_vocoder as rv
    g = golden("refshim_vocoder.npz")
    monkeypatch.setattr(hp, "n_iter", 3)
    rng = np.random.default_rng(0)
    mag = rng.uniform(0.2, 0.8, (40, 1 + hp.n_fft // 2)).astype(np.float32)
    ref_wav = g["wav"]
    mine, _, _ = rv.spectrogram2wav(mag, n_iter=3)
    assert ref_wav.shape == mine.shape and np.abs(ref_wav - mine).max() <= 1e-6 * max(1.0, np.abs(mine).max())
    t = np.arange(int(hp.sr * 0.8)) / hp.sr
    y = (0.2 * np.sin(2 * np.pi * 300 * t) + 0.02 * rng.standard_normal(t.size)).astype(np.float32)
    y[:2000] *= 1e-5
    fname, mel, mg = str(g["fname"]), g["mel"], g["mag"]
    mel2, mg2 = rf.load_spectrograms(y)
    assert fname == "LJ001-0001.wav" and mel.shape == mel2.shape and mg.shape == mg2.shape
    assert np.abs(mel - mel2).max() < 1e-6 and np.abs(mg - mg2).max() < 1e-6
