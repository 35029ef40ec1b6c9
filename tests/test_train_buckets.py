"""Training on length-bucketed batches at the bucket's own shape (reference data_load.py:122-129, dynamic_pad=True).
CPU: the shaped oracle (tests/oracle_buckets.py) against the losses of the reference's OWN training graphs on bucket-shaped
batches (tests/golden/refshim_train_buckets.npz, written by make_golden_buckets.py), and the trainer loop / Graph(mode="train")
feeding those batches unpadded, skipping the ones beyond the attention key capacity."""
import os

import numpy as np
import pytest
import torch

import oracle_buckets as ob
from conftest import golden
from dc_tts_b200 import trainer
from dc_tts_b200.arch import ATTENTION_KEY_CAPACITY
from dc_tts_b200.hyperparams import Hyperparams as hp
from dc_tts_b200.params import init_params, synthetic_text
from oracle import ref_train as rtr

T2M_KEYS, SSRN_KEYS = ("loss", "loss_mels", "loss_bd1", "loss_att"), ("loss", "loss_mags", "loss_bd2")


def _close(got, ref):
    return abs(got - ref) < 2e-6 * max(1.0, abs(ref))


def test_fixture_covers_the_bucket_shapes():
    g = golden("refshim_train_buckets.npz")
    shapes = [tuple(s) for s in g["t2m_shapes"]]
    assert any(n % 8 and t % 8 and n < 32 and t < 32 for n, t in shapes)            # small, neither a multiple of 8
    assert any(hp.max_N < n <= ATTENTION_KEY_CAPACITY for n, _ in shapes)           # more characters than max_N
    assert any(t > hp.max_T for _, t in shapes)                                     # more frames than max_T
    assert any(100 <= n <= hp.max_N and 100 <= t <= hp.max_T for n, t in shapes)    # a realistic bucket
    assert all(t % 2 for t in g["ssrn_T"]) and len(g["ssrn_T"]) >= 2
    assert list(g["rates"]) == [0.0, hp.dropout_rate]


@pytest.mark.parametrize("i", range(4))
def test_oracle_losses_vs_reference_training_graph_buckets(i):
    g = golden("refshim_train_buckets.npz")
    P = init_params(0, "perturbed")
    T = {n: torch.tensor(np.asarray(P[n], np.float32)) for n in rtr.text2mel_names()}
    N_b, T_b = (int(x) for x in g["t2m_shapes"][i])
    L, mels = ob.bucket_inputs(int(g["B"]), N_b, T_b, int(g["input_seed"]))
    assert L.shape == (int(g["B"]), N_b) and mels.shape == (int(g["B"]), T_b, hp.n_mels)
    for j, (seed, rate) in enumerate(zip(g["seeds"], g["rates"])):
        assert g["t2m_dropout_calls"][i, j] == (38 if rate > 0 else 0)             # one dropout per block
        with torch.no_grad():
            o = ob.forward(T, L, mels, int(seed), float(rate))
        for k, ref in zip(T2M_KEYS, g["t2m_losses"][i, j]):
            assert _close(float(o[k]), ref), (N_b, T_b, rate, k, float(o[k]), ref)


def test_oracle_ssrn_losses_vs_reference_training_graph_buckets():
    g = golden("refshim_train_buckets.npz")
    P = init_params(0, "perturbed")
    W = {n: torch.tensor(np.asarray(P[n], np.float32)) for n in rtr.ssrn_names()}
    for i, T_b in enumerate(g["ssrn_T"]):
        mels, mags = ob.ssrn_inputs(int(g["B"]), int(T_b), int(g["input_seed"]))
        for j, (seed, rate) in enumerate(zip(g["seeds"], g["rates"])):
            assert g["ssrn_dropout_calls"][i, j] == (16 if rate > 0 else 0)
            with torch.no_grad():
                o = ob.forward_ssrn(W, mels, mags, int(seed), float(rate))
            for k, ref in zip(SSRN_KEYS, g["ssrn_losses"][i, j]):
                assert _close(float(o[k]), ref), (int(T_b), rate, k, float(o[k]), ref)


def test_shaped_oracle_is_the_fixed_oracle_at_the_fixed_shape():
    P = init_params(0, "perturbed")
    T = {n: torch.tensor(np.asarray(P[n], np.float32)) for n in rtr.text2mel_names()}
    L = synthetic_text(1, 50, seed=7)
    mels = np.random.default_rng(3).uniform(0, 1, (1, hp.max_T, hp.n_mels)).astype(np.float32)
    with torch.no_grad():
        a, b = ob.forward(T, L, mels, 11, 0.05), rtr.forward(T, L, mels, 11, 0.05)
    for k in T2M_KEYS:
        assert float(a[k]) == float(b[k]), k
    assert ob.attention_window(185, 9) == (hp.max_N, 9) and ob.attention_window(30, 214) == (30, hp.max_T)


def test_bucket_parity_cases_clear_the_relu_noise():
    """The premise of the fp32 parity cases of test_gpu_train_buckets.py (see test_train._tie_free): every ReLU pre-activation clears zero by more than
    the float32 forward noise (~1e-6 Text2Mel, ~4e-6 SSRN)."""
    P = init_params(0, "perturbed")
    from test_gpu_train_buckets import SSRN_CASES, T2M_CASES
    for B, N_b, T_b, rate, seed, tc in T2M_CASES:
        if tc == 0:
            L, mels = ob.bucket_inputs(B, N_b, T_b, seed)
            assert ob.t2m_relu_margin(P, L, mels, seed, rate) > 1e-5, (B, N_b, T_b)
    for B, T_b, rate, seed in SSRN_CASES:
        mels, _ = ob.ssrn_inputs(B, T_b, seed)
        assert ob.ssrn_relu_margin(P, mels, seed, rate) > 4e-6, (B, T_b)



# ------------------------------------------------------------------------------- trainer loop and Graph, fake engine
class ShapeRecorder:
    """Stand-in engine that records the shapes of every step it is given."""

    def __init__(self):
        self.calls, self.init = [], None

    def train_init(self, B):
        self.init = ("t2m", B)

    def train_init_ssrn(self, B, T):
        self.init = ("ssrn", B, T)

    def train_step(self, L, mels, global_step=0, seed=0, apply=True):
        self.calls.append((L.shape, mels.shape))
        return {"loss": 1.0, "loss_mels": 0.3, "loss_bd1": 0.69, "loss_att": 0.01}

    def train_step_ssrn(self, mels, mags, global_step=0, seed=0, apply=True):
        self.calls.append((mels.shape, mags.shape))
        return {"loss": 1.0, "loss_mags": 0.3, "loss_bd2": 0.7}

    def restore_training(self, logdir, scope):
        return None

    def save_checkpoint(self, prefix, gs, scope):
        pass


def _corpus(n=48, long_every=0, seed=1):
    """Synthetic utterances with varied text lengths and frames = ~1.2 x characters; every `long_every`-th one is longer
    than the attention key capacity."""
    rng = np.random.default_rng(seed)
    lens = [int(x) for x in rng.integers(12, 170, n)]
    if long_every:
        lens = [ATTENTION_KEY_CAPACITY + 20 if i % long_every == 0 else l for i, l in enumerate(lens)]
    texts = [rng.integers(2, 30, l).astype(np.int32) for l in lens]
    frames = [int(1.2 * l) + 5 for l in lens]
    fpaths = ["wavs/U%03d.wav" % i for i in range(n)]
    store = {os.path.basename(p): (np.full((t, hp.n_mels), 0.5, np.float32), np.full((4 * t, 1 + hp.n_fft // 2), 0.5, np.float32))
             for p, t in zip(fpaths, frames)}
    loader = lambda p: (os.path.basename(p),) + store[os.path.basename(p)]
    return fpaths, lens, texts, loader


@pytest.mark.parametrize("num", [1, 2])
def test_trainer_takes_bucketed_batches_unpadded(tmp_path, num):
    fpaths, lens, texts, loader = _corpus()
    batches = list(trainer.bucketed_batches(fpaths, lens, texts, B=4, seed=3, loader=loader, epochs=2))
    eng = ShapeRecorder()
    gs = trainer.train(num, eng, iter(batches), num_iterations=10 ** 6, logdir=str(tmp_path / "ld"), global_step=0,
                       log=lambda *_: None)
    assert gs == len(batches) == len(eng.calls)
    if num == 1:
        assert eng.calls == [(b[0].shape, b[1].shape) for b in batches]
    else:
        assert eng.calls == [(b[1].shape, b[2].shape) for b in batches]
        assert eng.init == ("ssrn", 4, batches[0][1].shape[1])
    assert len({c[0] for c in eng.calls}) > 3                                      # several bucket shapes, none padded


def test_trainer_skips_and_counts_batches_beyond_the_key_capacity(tmp_path):
    fpaths, lens, texts, loader = _corpus(n=64, long_every=5)
    batches = list(trainer.bucketed_batches(fpaths, lens, texts, B=4, seed=3, loader=loader, epochs=2))
    over = sum(1 for b in batches if b[0].shape[1] > ATTENTION_KEY_CAPACITY)
    assert over > 0
    eng, logged = ShapeRecorder(), []
    gs = trainer.train(1, eng, iter(batches), num_iterations=10 ** 6, logdir=str(tmp_path / "ld"), global_step=0, log=logged.append)
    assert gs == len(batches) - over == len(eng.calls)
    assert all(c[0][1] <= ATTENTION_KEY_CAPACITY for c in eng.calls)
    assert any(("skipped %d batches" % over) in m for m in logged), logged


def test_graph_train_takes_bucketed_batches(tmp_path):
    from dc_tts_b200.train import Graph, Session
    fpaths, lens, texts, loader = _corpus(n=64, long_every=5)
    batches = list(trainer.bucketed_batches(fpaths, lens, texts, B=4, seed=3, loader=loader, epochs=1))
    fits = [b for b in batches if b[0].shape[1] <= ATTENTION_KEY_CAPACITY]
    for num in (1, 2):
        eng = ShapeRecorder()
        g = Graph(num=num, engine=eng, batches=iter(batches))
        with Session() as sess:
            for _ in fits:
                sess.run([g.global_step, g.train_op])
        want = [(b[0].shape, b[1].shape) if num == 1 else (b[1].shape, b[2].shape) for b in fits]
        assert eng.calls == want
        last = max(i for i, b in enumerate(batches) if b[0].shape[1] <= ATTENTION_KEY_CAPACITY)
        assert g.skipped_batches == sum(1 for b in batches[:last] if b[0].shape[1] > ATTENTION_KEY_CAPACITY) > 0
