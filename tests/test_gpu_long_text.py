"""Text longer than 192 characters on the GPU.  A handle's key capacity is max(192, round_up(max_N, 64)) for max_N <= 512
(include/dctts.h: dctts_get_option "key_capacity"); every test here raises Hyperparams.max_N / max_T as a user with longer
text would, creates its own Engine, and lets the oracle read the same class.

  * creation and limits;
  * dctts_attention at N from 193 to 512 on the tcgen05 and the fp32 kernel, dense and under the monotonic window;
  * synthesis at (max_N, max_T) = (300, 320) against the reference's own graphs (tests/golden/refshim_long.npz) and the
    oracle's free-running schedule, on both decode paths, and SSRN on the 320-frame result;
  * training at (300, 320): losses against the reference's training graph, gradients / Adam / weights against
    tests/oracle_buckets.py, workspace growth, and the trainer loop on text up to 320 characters."""
import sys

import numpy as np
import pytest
import torch

import oracle_buckets as ob
from conftest import GOLDEN, golden
from dc_tts_b200 import trainer
from dc_tts_b200.hyperparams import Hyperparams as hp
from dc_tts_b200.params import init_params
from oracle import ref_torch as rt
from test_gpu_bench_shapes import _compare_prefix
from test_gpu_train_buckets import PROBES, T2M_KEYS, _close_losses, _same_tensors
from test_train import _compare_grads, _tie_free

sys.path.insert(0, GOLDEN)
from make_golden_long import MAX_N, MAX_T, STEPS, long_inputs  # noqa: E402

pytestmark = pytest.mark.gpu
TOL = 1e-3


@pytest.fixture(scope="module", autouse=True)
def long_hp():
    with pytest.MonkeyPatch.context() as m:
        m.setattr(hp, "max_N", MAX_N)
        m.setattr(hp, "max_T", MAX_T)
        yield


def _engine(P=None, tc=None):
    from dc_tts_b200.engine import Engine
    e = Engine(0)
    if P is not None:
        e.load_params(P)
    if tc is not None:
        e.set_option("train_tc", tc)
    return e


@pytest.fixture(scope="module")
def P():
    return init_params(0, "perturbed")


# ---------------------------------------------------------------------------------------------- 1. creation and limits
@pytest.mark.parametrize("max_N,cap", [(180, 192), (192, 192), (193, 256), (300, 320), (512, 512)])
def test_key_capacity(monkeypatch, max_N, cap):
    monkeypatch.setattr(hp, "max_N", max_N)
    e = _engine()
    assert e.get_option("key_capacity") == e.KEY_CAPACITY == cap
    e.close()


def test_create_rejects_more_than_512_characters(monkeypatch):
    from dc_tts_b200.engine import DcttsError
    monkeypatch.setattr(hp, "max_N", 513)
    with pytest.raises(DcttsError, match="512"):
        _engine()


def test_entry_points_reject_text_beyond_the_capacity(P):
    from dc_tts_b200.engine import DcttsError
    e = _engine(P)
    assert e.KEY_CAPACITY == 320
    rng = np.random.default_rng(0)
    Q, K = rng.uniform(-1, 1, (1, 8, hp.d)).astype(np.float32), rng.uniform(-1, 1, (1, 321, hp.d)).astype(np.float32)
    e.attention(Q, K[:, :320], K[:, :320])
    with pytest.raises(DcttsError, match="key capacity"):
        e.attention(Q, K, K)
    e.train_init(2, 0.0)
    e.train_reserve(320, 40)
    with pytest.raises(DcttsError, match="key capacity"):
        e.train_reserve(321, 40)
    L, mels = ob.bucket_inputs(2, 321, 20, 0)
    with pytest.raises(DcttsError, match="key capacity"):
        e.train_step(L, mels)
    L, mels = ob.bucket_inputs(2, 320, 20, 0)
    assert np.isfinite(e.train_step(L, mels)["loss"])
    e.close()


# ---------------------------------------------------------------------------------------------- 2. dctts_attention
@pytest.fixture(scope="module")
def engine512():
    with pytest.MonkeyPatch.context() as m:
        m.setattr(hp, "max_N", 512)
        e = _engine()
    assert e.KEY_CAPACITY == 512
    yield e
    e.close()


def _check_attention(R, A, M, Rr, Ar, Mr):
    assert np.abs(R - Rr).max() < 1e-4
    assert np.abs(A - Ar).max() < 1e-5
    # argmax: rows whose best two probabilities lie within float32 noise may pick either
    top2 = np.sort(Ar, axis=1)[:, -2:, :]                                 # (B, 2, T)
    clear = (top2[:, 1] - top2[:, 0]) > 1e-5
    assert clear.mean() > 0.9
    assert np.array_equal(M[clear], Mr[clear])


@pytest.mark.parametrize("tensor_path", [1, 0], ids=["tcgen05", "fp32"])
@pytest.mark.parametrize("N", [193, 256, 257, 320, 511, 512])
def test_attention_long(engine512, monkeypatch, N, tensor_path):
    e = engine512
    e.set_tensor_path(tensor_path)
    B, T = 3, 300
    rng = np.random.default_rng(N)
    Q = rng.uniform(-1, 1, (B, T, hp.d)).astype(np.float32)
    K = rng.uniform(-1, 1, (B, N, hp.d)).astype(np.float32)
    V = rng.uniform(-1, 1, (B, N, hp.d)).astype(np.float32)
    monkeypatch.setattr(hp, "max_N", N)                                   # the oracle's window mask spans the N keys
    tq, tk, tv = torch.from_numpy(Q), torch.from_numpy(K), torch.from_numpy(V)
    R, A, M = e.attention(Q, K, V)
    Rr, Ar, Mr = rt.Attention(tq, tk, tv, False, None)
    _check_attention(R.cpu().numpy(), A.cpu().numpy(), M.cpu().numpy(), Rr.numpy(), Ar.numpy(), Mr.numpy())
    pma = np.array([0, N // 2, N - 1], np.int32)
    R, A, M = e.attention(Q, K, V, True, pma)
    Rr, Ar, Mr = rt.Attention(tq, tk, tv, True, pma)
    A = A.cpu().numpy()
    _check_attention(R.cpu().numpy(), A, M.cpu().numpy(), Rr.numpy(), Ar.numpy(), Mr.numpy())
    for b, p in enumerate(pma):
        live = np.zeros(N, bool); live[p:p + hp.attention_win_size] = True
        assert (A[b][~live] == 0).all()                                   # exact zeros outside the window
    e.set_tensor_path(1)


# ---------------------------------------------------------------------------------------------- 3. synthesis at (300, 320)
@pytest.fixture(scope="module")
def synth_engine(P):
    e = _engine(P)
    yield e
    e.close()


@pytest.mark.parametrize("tensor_path", [1, 0], ids=["tcgen05", "fp32"])
def test_text2mel_forward_vs_reference_long(synth_engine, tensor_path):
    g = golden("refshim_long.npz")
    L, mels, pma = long_inputs()
    synth_engine.set_tensor_path(tensor_path)
    try:
        Y, M, _ = synth_engine.text2mel_forward(L, mels, pma)
    finally:
        synth_engine.set_tensor_path(1)
    assert np.abs(Y.cpu().numpy() - g["Y"]).max() < TOL
    assert np.array_equal(M.cpu().numpy(), g["max_attentions"])


@pytest.mark.parametrize("decode_mode", [1, 0], ids=["cluster", "graph"])
def test_generate_few_steps_vs_reference_long(synth_engine, decode_mode):
    g = golden("refshim_long.npz")
    L, _, _ = long_inputs()
    synth_engine.set_option("decode_mode", decode_mode)
    try:
        Y, Pw, _, _ = synth_engine.text2mel_generate(L, steps=STEPS)
    finally:
        synth_engine.set_option("decode_mode", 1)
    assert np.array_equal(Pw.cpu().numpy()[:, :STEPS], g["loop_p_hist"])
    assert np.abs(Y.cpu().numpy()[:, :STEPS] - g["loop_Y"]).max() < TOL


@pytest.fixture(scope="module")
def oracle_run(P):
    L, _, _ = long_inputs()
    with torch.no_grad():
        r = rt.synthesize(P, L, steps=MAX_T, literal=False, record=True)
    return L, r["Y"].numpy(), r["p_hist"].numpy(), r["margin_hist"].numpy()


@pytest.mark.parametrize("decode_mode", [1, 0], ids=["cluster", "graph"])
def test_generate_320_frames_vs_oracle(synth_engine, oracle_run, P, decode_mode):
    L, Yo, Po, margin = oracle_run
    synth_engine.set_option("decode_mode", decode_mode)
    try:
        Y, Pw, _, _ = synth_engine.text2mel_generate(L)
    finally:
        synth_engine.set_option("decode_mode", 1)
    Y, Pw = Y.cpu().numpy(), Pw.cpu().numpy()
    assert Y.shape == (2, MAX_T, hp.n_mels)
    assert _compare_prefix(Y, Pw, Yo, Po, margin, MAX_T) >= MAX_T
    _, Z = synth_engine.ssrn(Y, want_logits=False)                        # SSRN on the 320-frame mel
    with torch.no_grad():
        _, Zr = rt.SSRN(P, torch.from_numpy(Y))
    assert Z.shape == (2, 4 * MAX_T, 1 + hp.n_fft // 2)
    assert np.abs(Z.cpu().numpy() - Zr.numpy()).max() < TOL


# ---------------------------------------------------------------------------------------------- 4. training at (300, 320)
@pytest.mark.parametrize("tc", [7, 0])
def test_losses_vs_reference_training_graph_long(tc):
    g = golden("refshim_long.npz")
    B, seed_in = int(g["B"]), int(g["input_seed"])
    e = _engine(init_params(0, "perturbed"), tc)
    for j, (seed, rate) in enumerate(zip(g["seeds"], g["rates"])):
        e.train_init(B, float(rate))
        for i, (N_b, T_b) in enumerate(g["t2m_shapes"]):
            L, mels = ob.bucket_inputs(B, int(N_b), int(T_b), seed_in)
            out = e.train_step(L, mels, global_step=0, seed=int(seed), apply=False)
            for k, ref in zip(T2M_KEYS, g["t2m_losses"][i, j]):
                assert abs(out[k] - ref) < 1e-5 * max(1.0, abs(ref)), (int(N_b), int(T_b), float(rate), k, out[k], ref)
    e.close()


# the tie-free parameter set for both kernel sets: at B = 32 and 300+ characters some ReLU pre-activation of the plain set
# sits within the forward noise of zero, and a flipped mask would test the coin flip instead of the arithmetic
LONG_CASES = [(2, 257, 40, 0.05, 11, 7), (32, 320, 70, 0.05, 5, 7), (2, 320, 330, 0.0, 0, 0), (32, 257, 40, 0.05, 3, 0)]


@pytest.mark.parametrize("B,N_b,T_b,rate,seed,tc", LONG_CASES)
def test_shaped_step_vs_oracle_long(B, N_b, T_b, rate, seed, tc):
    P = _tie_free(init_params(0, "perturbed"))
    L, mels = ob.bucket_inputs(B, N_b, T_b, seed)
    newP, st, info = ob.train_step(P, L, mels, global_step=7, seed=seed, rate=rate)
    e = _engine(P, tc)
    e.train_init(B, rate)
    out = e.train_step(L, mels, global_step=7, seed=seed, apply=False)
    for k in T2M_KEYS:
        assert abs(out[k] - info[k]) < 1e-5 * max(1.0, abs(info[k])), (k, out[k], info[k])
    _compare_grads(e, info["grads"])
    e.train_apply(7)
    for n in PROBES:
        m, v = st[n]
        np.testing.assert_allclose(e.train_tensor(n, "m"), m, rtol=2e-3, atol=max(1e-9, 1e-4 * np.abs(m).max()))
        np.testing.assert_allclose(e.train_tensor(n, "v"), v, rtol=4e-3, atol=max(1e-14, 4e-4 * np.abs(v).max()))
        step = np.abs(newP[n] - P[n]).max()
        assert np.abs(e.train_tensor(n, "param") - newP[n]).max() <= 0.05 * step + 2.4e-7, n
    e.close()


@pytest.mark.parametrize("tc", [7, 0])
def test_growth_to_320_characters_matches_a_reserved_handle(tc):
    """A handle initialised for (300, 320) grows to (320, 400) between steps with live Adam state; it matches a handle
    reserved for (320, 400) before its first step in losses, gradients, weights and Adam moments."""
    P = _tie_free(init_params(0, "perturbed"))
    seq = [(40, 30, 0), (320, 400, 1), (MAX_N, MAX_T, 2), (40, 30, 3)]
    grow, big = _engine(P, tc), _engine(P, tc)
    grow.train_init(3, 0.05); big.train_init(3, 0.05)
    big.train_reserve(320, 400)
    for N_b, T_b, gs in seq:
        L, mels = ob.bucket_inputs(3, N_b, T_b, gs)
        a = grow.train_step(L, mels, global_step=gs, seed=gs)
        b = big.train_step(L, mels, global_step=gs, seed=gs)
        _close_losses(a, b, 1e-4)
    _same_tensors(grow, big, PROBES, ("grad", "param", "m", "v"), 1e-3)
    grow.close(); big.close()


def test_trainer_on_text_up_to_320_characters(tmp_path):
    rng = np.random.default_rng(7)
    n = 48
    lens = [int(x) for x in rng.integers(150, 320, n)]
    lens[0] = 319                                                         # with E: 320 characters
    texts = [np.concatenate([rng.integers(2, 30, l), [1]]).astype(np.int32) for l in lens]
    store = {}
    for i, l in enumerate(lens):
        T = l // 2 + 10
        store["U%03d" % i] = (rng.uniform(0, 1, (T, hp.n_mels)).astype(np.float32), np.zeros((4 * T, 1 + hp.n_fft // 2), np.float32))
    loader = lambda p: (p,) + store[p]
    batches = list(trainer.bucketed_batches(list(store), [len(t) for t in texts], texts, B=4, seed=0, loader=loader, epochs=1))
    assert max(b[0].shape[1] for b in batches) > 256
    e = _engine(init_params(1))
    shapes, losses, logged = [], [], []

    class Recorder:
        def __getattr__(self, name):
            return getattr(e, name)

        def train_step(self, L, mels, **k):
            shapes.append(np.shape(L)[1]); out = e.train_step(L, mels, **k); losses.append(out["loss"]); return out

    gs = trainer.train(1, Recorder(), iter(batches), num_iterations=10 ** 6, logdir=str(tmp_path / "ld"), global_step=0,
                       save_every=10 ** 6, log=logged.append)
    assert gs == len(batches) == len(shapes)
    assert not any("skipped" in m for m in logged), logged
    assert max(shapes) > 256 and np.all(np.isfinite(losses))
    e.close()
