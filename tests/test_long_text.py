"""Text longer than 192 characters (hp.max_N up to 512), on the CPU: the oracle against the reference's own graphs run
with max_N / max_T raised to (300, 320) (tests/golden/refshim_long.npz, generator make_golden_long.py), and the trainer
loop following an engine's key capacity instead of the 192 of the LJ hyper-parameters."""
import os
import sys

import numpy as np
import pytest
import torch

import oracle_buckets as ob
from conftest import GOLDEN, golden
from dc_tts_b200 import trainer
from dc_tts_b200.arch import ATTENTION_KEY_CAPACITY
from dc_tts_b200.hyperparams import Hyperparams as hp
from dc_tts_b200.params import init_params
from oracle import ref_torch as rt

sys.path.insert(0, GOLDEN)
from make_golden_long import MAX_N, MAX_T, STEPS, long_inputs  # noqa: E402

T2M_KEYS = ("loss", "loss_mels", "loss_bd1", "loss_att")


@pytest.fixture()
def long_hp(monkeypatch):
    monkeypatch.setattr(hp, "max_N", MAX_N)
    monkeypatch.setattr(hp, "max_T", MAX_T)


@pytest.fixture(scope="module")
def P():
    return init_params(0, "perturbed")


def test_fixture_inputs_are_the_generator_inputs():
    g = golden("refshim_long.npz")
    L, _, pma = long_inputs()
    assert (int(g["max_N"]), int(g["max_T"])) == (MAX_N, MAX_T)
    assert np.array_equal(g["L"], L) and np.array_equal(g["pma"], pma)
    assert g["max_attentions"][0].max() >= MAX_N - 5                     # the window of row 0 near the end of its keys
    assert os.path.getsize(os.path.join(GOLDEN, "refshim_long.npz")) < 250 * 1024


def test_oracle_full_graph_vs_reference_long(long_hp, P):
    g = golden("refshim_long.npz")
    L, mels, pma = long_inputs()
    with torch.no_grad():
        o = rt.text2mel_forward(P, L, mels, pma)
    assert np.abs(o["Y"].numpy() - g["Y"]).max() < 2e-5
    assert np.array_equal(o["max_attentions"].numpy(), g["max_attentions"])


def test_oracle_few_steps_vs_reference_long(long_hp, P):
    g = golden("refshim_long.npz")
    L, _, _ = long_inputs()
    with torch.no_grad():
        o = rt.synthesize(P, L, steps=STEPS, literal=False, record=True)
    assert np.array_equal(o["p_hist"].numpy(), g["loop_p_hist"])
    assert np.abs(o["Y"].numpy()[:, :STEPS] - g["loop_Y"]).max() < 2e-5


def test_oracle_losses_vs_reference_long(long_hp, P):
    g = golden("refshim_long.npz")
    B, seed_in = int(g["B"]), int(g["input_seed"])
    W = {n: torch.tensor(np.asarray(P[n], np.float32)) for n in P}
    for i, (N_b, T_b) in enumerate(g["t2m_shapes"]):
        L, mels = ob.bucket_inputs(B, int(N_b), int(T_b), seed_in)
        for j, (seed, rate) in enumerate(zip(g["seeds"], g["rates"])):
            with torch.no_grad():
                out = ob.forward(W, L, mels, int(seed), float(rate))
            for k, ref in zip(T2M_KEYS, g["t2m_losses"][i, j]):
                assert abs(float(out[k]) - ref) < 2e-6 * max(1.0, abs(ref)), (int(N_b), int(T_b), float(rate), k, float(out[k]), ref)


class CapacityRecorder:
    """Stand-in engine with a key capacity of 320 characters, recording the shape of every step."""
    KEY_CAPACITY = 320

    def __init__(self):
        self.calls = []

    def train_init(self, B):
        pass

    def train_step(self, L, mels, global_step=0, seed=0, apply=True):
        self.calls.append(L.shape)
        return {"loss": 1.0, "loss_mels": 0.3, "loss_bd1": 0.69, "loss_att": 0.01}

    def restore_training(self, logdir, scope):
        return None

    def save_checkpoint(self, prefix, gs, scope):
        pass


def _long_corpus(n=96, seed=4):
    """Text lengths from 150 to 340 characters: many buckets above 192, some above 320."""
    rng = np.random.default_rng(seed)
    lens = [int(x) for x in rng.integers(150, 341, n)]
    texts = [rng.integers(2, 30, l).astype(np.int32) for l in lens]
    fpaths = ["wavs/U%03d.wav" % i for i in range(n)]
    store = {os.path.basename(p): (np.full((l // 2, hp.n_mels), 0.5, np.float32), np.full((2 * l, 1 + hp.n_fft // 2), 0.5, np.float32))
             for p, l in zip(fpaths, lens)}
    loader = lambda p: (os.path.basename(p),) + store[os.path.basename(p)]
    return fpaths, lens, texts, loader


def test_trainer_follows_the_engine_key_capacity(tmp_path):
    fpaths, lens, texts, loader = _long_corpus()
    batches = list(trainer.bucketed_batches(fpaths, lens, texts, B=4, seed=3, loader=loader, epochs=2))
    over = sum(1 for b in batches if b[0].shape[1] > CapacityRecorder.KEY_CAPACITY)
    between = sum(1 for b in batches if ATTENTION_KEY_CAPACITY < b[0].shape[1] <= CapacityRecorder.KEY_CAPACITY)
    assert over > 0 and between > 0
    eng, logged = CapacityRecorder(), []
    gs = trainer.train(1, eng, iter(batches), num_iterations=10 ** 6, logdir=str(tmp_path / "ld"), global_step=0, log=logged.append)
    assert gs == len(batches) - over == len(eng.calls)
    assert eng.calls == [b[0].shape for b in batches if b[0].shape[1] <= CapacityRecorder.KEY_CAPACITY]
    assert any(("skipped %d batches with more than 320 characters" % over) in m for m in logged), logged


def test_graph_train_follows_the_engine_key_capacity():
    from dc_tts_b200.train import Graph, Session
    fpaths, lens, texts, loader = _long_corpus(seed=5)
    batches = list(trainer.bucketed_batches(fpaths, lens, texts, B=4, seed=3, loader=loader, epochs=1))
    fits = [b for b in batches if b[0].shape[1] <= CapacityRecorder.KEY_CAPACITY]
    assert any(b[0].shape[1] > ATTENTION_KEY_CAPACITY for b in fits)
    eng = CapacityRecorder()
    g = Graph(num=1, engine=eng, batches=iter(batches))
    with Session() as sess:
        for _ in fits:
            sess.run([g.global_step, g.train_op])
    assert eng.calls == [b[0].shape for b in fits]
    last = max(i for i, b in enumerate(batches) if b[0].shape[1] <= CapacityRecorder.KEY_CAPACITY)
    assert g.skipped_batches == sum(1 for b in batches[:last] if b[0].shape[1] > CapacityRecorder.KEY_CAPACITY)


def test_fits_key_capacity_takes_the_capacity():
    L = np.zeros((2, 300), np.int32)
    assert not trainer.fits_key_capacity(L)
    assert trainer.fits_key_capacity(L, 320)
    assert trainer.key_capacity(object()) == ATTENTION_KEY_CAPACITY == 192
    assert trainer.key_capacity(CapacityRecorder()) == 320
