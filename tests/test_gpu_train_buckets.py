"""Training steps at the shape of a length bucket (include/dctts.h: dctts_train_step_shaped, dctts_train_step_ssrn_shaped,
dctts_train_reserve) on the GPU: the fixed shape unchanged, losses against the reference's own training graphs
(tests/golden/refshim_train_buckets.npz), gradients / Adam / weights against the shaped oracle (tests/oracle_buckets.py),
workspace growth without stale state, and the trainer loop fed `bucketed_batches` end to end.

The training step sums gradients with float atomics, so two runs of the same step agree to rounding, not bit for bit
(test_train.py: test_cuda_training_reduces_loss_and_is_deterministic); run-to-run comparisons below use that tolerance."""
import ctypes as C

import numpy as np
import pytest

import oracle_buckets as ob
from conftest import golden
from dc_tts_b200 import trainer
from dc_tts_b200.hyperparams import Hyperparams as hp
from dc_tts_b200.params import init_params
from oracle import ref_train as rtr
from test_gpu_trainer_run import _write_dataset
from test_train import _compare_grads, _tie_free

pytestmark = pytest.mark.gpu

F = 1 + hp.n_fft // 2
T2M_KEYS, SSRN_KEYS = ("loss", "loss_mels", "loss_bd1", "loss_att"), ("loss", "loss_mags", "loss_bd2")


def _engine(P, tc=7):
    from dc_tts_b200.engine import Engine
    e = Engine(0)
    e.load_params(P)
    e.set_option("train_tc", tc)
    return e


def _shaped_step(e, L, mels, gs, seed, apply=False):
    """dctts_train_step_shaped called directly (Engine.train_step sends (max_N, max_T) to dctts_train_step)."""
    from dc_tts_b200.engine import _ptr
    L = e._i32(L); mels = e._f32(mels)
    out = (C.c_float * 4)()
    e._check(e._lib.dctts_train_step_shaped(e._h, _ptr(L), L.shape[1], _ptr(mels), mels.shape[1], L.shape[0], gs, seed,
                                            float(hp.lr), int(apply), out, e._stream()), "dctts_train_step_shaped")
    return dict(zip(T2M_KEYS, out))


def _shaped_step_ssrn(e, mels, mags, gs, seed, apply=False):
    from dc_tts_b200.engine import _ptr
    mels = e._f32(mels); mags = e._f32(mags)
    out = (C.c_float * 4)()
    e._check(e._lib.dctts_train_step_ssrn_shaped(e._h, _ptr(mels), _ptr(mags), mels.shape[0], mels.shape[1], gs, seed,
                                                 float(hp.lr), int(apply), out, e._stream()), "dctts_train_step_ssrn_shaped")
    return dict(zip(SSRN_KEYS, out))


def _same_tensors(a, b, names, whats=("grad",), rel=1e-4):
    """Equal up to the reordering of float atomics: per tensor, max |a - b| <= rel * max |a|."""
    for n in names:
        for w in whats:
            x, y = a.train_tensor(n, w), b.train_tensor(n, w)
            assert np.abs(x - y).max() <= rel * np.abs(x).max() + 1e-30, (n, w, np.abs(x - y).max(), np.abs(x).max())


def _close_losses(a, b, rel=1e-5):
    for k in a:
        assert abs(a[k] - b[k]) <= rel * max(1.0, abs(b[k])), (k, a[k], b[k])


# ---------------------------------------------------------------------------------------------- 1. unchanged default
def test_shaped_step_at_the_fixed_shape_is_the_fixed_step():
    P = _tie_free(init_params(0, "perturbed"))
    L, mels = ob.bucket_inputs(2, hp.max_N, hp.max_T, 3)
    e = _engine(P)
    e.train_init(2, 0.05)
    fixed = e.train_step(L, mels, global_step=7, seed=11, apply=False)
    ref = _engine(P); ref.train_init(2, 0.05)
    ref.train_step(L, mels, global_step=7, seed=11, apply=False)
    shaped = _shaped_step(e, L, mels, 7, 11)
    _close_losses(shaped, fixed)
    _same_tensors(e, ref, rtr.text2mel_names())
    e.close(); ref.close()


def test_shaped_ssrn_step_at_the_init_length_is_the_fixed_step():
    P = init_params(0, "perturbed")
    mels, mags = ob.ssrn_inputs(2, 12, 3)
    e = _engine(P); e.train_init_ssrn(2, 12, 0.05)
    ref = _engine(P); ref.train_init_ssrn(2, 12, 0.05)
    fixed = e.train_step_ssrn(mels, mags, global_step=3, seed=9, apply=False)
    ref.train_step_ssrn(mels, mags, global_step=3, seed=9, apply=False)
    shaped = _shaped_step_ssrn(e, mels, mags, 3, 9)
    _close_losses(shaped, fixed)
    _same_tensors(e, ref, rtr.ssrn_names())
    e.close(); ref.close()


# ---------------------------------------------------------------------------------------------- 2. reference losses
@pytest.mark.parametrize("tc", [7, 0])
def test_losses_vs_reference_training_graph_buckets(tc):
    g = golden("refshim_train_buckets.npz")
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
    e = _engine(init_params(0, "perturbed"), tc)
    for j, (seed, rate) in enumerate(zip(g["seeds"], g["rates"])):
        e.train_init_ssrn(B, int(g["ssrn_T"][0]), float(rate))
        for i, T_b in enumerate(g["ssrn_T"]):
            mels, mags = ob.ssrn_inputs(B, int(T_b), seed_in)
            out = e.train_step_ssrn(mels, mags, global_step=0, seed=int(seed), apply=False)
            for k, ref in zip(SSRN_KEYS, g["ssrn_losses"][i, j]):
                assert abs(out[k] - ref) < 1e-5 * max(1.0, abs(ref)), (int(T_b), float(rate), k, out[k], ref)
    e.close()


# ---------------------------------------------------------------------------------------------- 3. gradients, Adam, weights
# tc = 7 (tcgen05 GEMMs) on the tie-free set; tc = 0 (fp32 CUDA cores) on the plain set at cases whose ReLU margin clears the
# forward noise (test_train_buckets.py: test_bucket_parity_cases_clear_the_relu_noise)
T2M_CASES = [(2, 23, 17, 0.05, 11, 7), (2, 185, 9, 0.0, 0, 7), (3, 30, 214, 0.05, 4, 7), (32, 110, 150, 0.05, 5, 7),
             (2, 23, 17, 0.05, 11, 0), (2, 185, 9, 0.0, 0, 0), (2, 61, 45, 0.0, 7, 0)]
SSRN_CASES = [(2, 9, 0.05, 3), (1, 13, 0.0, 0), (2, 23, 0.0, 0)]


@pytest.mark.parametrize("B,N_b,T_b,rate,seed,tc", T2M_CASES)
def test_shaped_step_vs_oracle(B, N_b, T_b, rate, seed, tc):
    P = init_params(0, "perturbed")
    if tc:
        P = _tie_free(P)
    L, mels = ob.bucket_inputs(B, N_b, T_b, seed)
    newP, st, info = ob.train_step(P, L, mels, global_step=7, seed=seed, rate=rate)
    e = _engine(P, tc)
    e.train_init(B, rate)
    out = e.train_step(L, mels, global_step=7, seed=seed, apply=False)
    for k in T2M_KEYS:
        assert abs(out[k] - info[k]) < 1e-5 * max(1.0, abs(info[k])), (k, out[k], info[k])
    _compare_grads(e, info["grads"])
    e.train_apply(7)
    for n in ("Text2Mel/TextEnc/embed_1/lookup_table", "Text2Mel/TextEnc/HC_7/conv1d/kernel", "Text2Mel/AudioEnc/C_1/conv1d/kernel",
              "Text2Mel/AudioDec/HC_3/H2/gamma", "Text2Mel/AudioDec/C_11/conv1d/bias", "Text2Mel/AudioEnc/HC_9/H1/beta"):
        m, v = st[n]
        np.testing.assert_allclose(e.train_tensor(n, "m"), m, rtol=2e-3, atol=max(1e-9, 1e-4 * np.abs(m).max()))
        np.testing.assert_allclose(e.train_tensor(n, "v"), v, rtol=4e-3, atol=max(1e-14, 4e-4 * np.abs(v).max()))
        step = np.abs(newP[n] - P[n]).max()
        assert np.abs(e.train_tensor(n, "param") - newP[n]).max() <= 0.05 * step + 2.4e-7, n
    e.close()


@pytest.mark.parametrize("B,T_b,rate,seed", SSRN_CASES)
def test_shaped_ssrn_step_vs_oracle(B, T_b, rate, seed):
    P = init_params(0, "perturbed")
    mels, mags = ob.ssrn_inputs(B, T_b, seed)
    newP, st, info = ob.train_step_ssrn(P, mels, mags, global_step=3999, seed=seed, rate=rate)
    e = _engine(P)
    e.train_init_ssrn(B, 12, rate)                         # initialised for another length: the step follows the batch
    out = e.train_step_ssrn(mels, mags, global_step=3999, seed=seed, apply=False)
    for k in SSRN_KEYS:
        assert abs(out[k] - info[k]) < 1e-5 * max(1.0, abs(info[k])), (k, out[k], info[k])
    _compare_grads(e, info["grads"])
    e.train_apply(3999)
    for n in ("SSRN/D_4/conv2d_transpose/kernel", "SSRN/HC_12/conv1d/kernel", "SSRN/C_16/conv1d/bias", "SSRN/C_15/normalize/gamma"):
        m, v = st[n]
        np.testing.assert_allclose(e.train_tensor(n, "m"), m, rtol=2e-3, atol=max(1e-9, 1e-4 * np.abs(m).max()))
        step = np.abs(newP[n] - P[n]).max()
        assert np.abs(e.train_tensor(n, "param") - newP[n]).max() <= 0.05 * step + 2.4e-7, n
    e.close()


def test_shaped_step_rejects_what_it_cannot_read():
    from dc_tts_b200.engine import DcttsError
    e = _engine(init_params(0, "perturbed"))
    e.train_init(2, 0.0)
    L, mels = ob.bucket_inputs(2, 193, 20, 0)
    with pytest.raises(DcttsError):
        e.train_step(L, mels)                                                   # beyond the key capacity
    with pytest.raises(DcttsError):
        e.train_reserve(200, 20)
    e.train_init_ssrn(2, 12, 0.0)
    e.train_reserve(200, 20)                                                    # SSRN has no keys: N is ignored
    mels, mags = ob.ssrn_inputs(2, 12, 0)
    with pytest.raises(DcttsError):
        e.train_step_ssrn(mels, mags[:, :47])                                   # mags must hold 4 T frames
    e.close()


# ---------------------------------------------------------------------------------------------- 4. no stale state
PROBES = ("Text2Mel/TextEnc/embed_1/lookup_table", "Text2Mel/TextEnc/HC_7/conv1d/kernel", "Text2Mel/AudioEnc/C_1/conv1d/kernel",
          "Text2Mel/AudioDec/HC_3/H2/gamma", "Text2Mel/AudioDec/C_11/conv1d/bias")


SSRN_PROBES = ("SSRN/D_4/conv2d_transpose/kernel", "SSRN/HC_12/conv1d/kernel", "SSRN/C_15/normalize/gamma", "SSRN/C_16/conv1d/bias")


def _three_steps_of_moments(grown, fresh, name):
    """Adam's v after three steps differs from v after one step: growth did not reset the moments."""
    v = grown.train_tensor(name, "v")
    assert np.abs(v - fresh.train_tensor(name, "v")).max() > 1e-3 * np.abs(v).max(), name


@pytest.mark.parametrize("tc", [7, 0])
def test_growth_keeps_the_optimiser_state_and_leaves_nothing_behind(tc):
    """dctts_train_init sizes the workspace for (max_N, max_T).  Shape A, then B beyond that capacity in both N and T (the
    workspace grows between steps with live Adam moments), then the fixed shape and A again on the grown workspace, on one
    handle -- against a handle reserved for B before its first step: the same losses, gradients, weights and Adam moments
    (up to float-atomic rounding)."""
    P = _tie_free(init_params(0, "perturbed"))
    seq = [(23, 17, 0), (185, 240, 1), (hp.max_N, hp.max_T, 2), (23, 17, 3)]
    assert seq[1][0] > hp.max_N and seq[1][1] > hp.max_T                   # beyond the init capacity: step 1 grows `grow`
    grow, big = _engine(P, tc), _engine(P, tc)
    grow.train_init(3, 0.05); big.train_init(3, 0.05)
    big.train_reserve(185, 240)
    for N_b, T_b, gs in seq:
        L, mels = ob.bucket_inputs(3, N_b, T_b, gs)
        a = grow.train_step(L, mels, global_step=gs, seed=gs)
        b = big.train_step(L, mels, global_step=gs, seed=gs)
        _close_losses(a, b, 1e-4)
    _same_tensors(grow, big, PROBES, ("grad", "param", "m", "v"), 1e-3)
    fresh = _engine(P, tc); fresh.train_init(3, 0.05)
    L, mels = ob.bucket_inputs(3, 23, 17, 3)
    fresh.train_step(L, mels, global_step=3, seed=3)
    _three_steps_of_moments(grow, fresh, "Text2Mel/AudioDec/C_11/conv1d/bias")
    grow.close(); big.close(); fresh.close()


@pytest.mark.parametrize("tc", [7, 0])
def test_ssrn_growth_keeps_the_optimiser_state_and_leaves_nothing_behind(tc):
    """dctts_train_init_ssrn(T = 12) sizes the workspace for 12 frames; a 30-frame batch grows it between steps, then the
    fixed-shape entry point runs at T = 12 on the grown workspace -- against a handle reserved for 30 frames from the start."""
    P = init_params(0, "perturbed")
    seq = [(12, 0), (30, 1), (12, 2)]
    grow, big = _engine(P, tc), _engine(P, tc)
    grow.train_init_ssrn(2, 12, 0.05); big.train_init_ssrn(2, 12, 0.05)
    big.train_reserve(0, 30)
    for T_b, gs in seq:
        mels, mags = ob.ssrn_inputs(2, T_b, gs)
        a = grow.train_step_ssrn(mels, mags, global_step=gs, seed=gs)
        b = big.train_step_ssrn(mels, mags, global_step=gs, seed=gs)
        _close_losses(a, b, 1e-4)
    _same_tensors(grow, big, SSRN_PROBES, ("grad", "param", "m", "v"), 1e-3)
    fresh = _engine(P, tc); fresh.train_init_ssrn(2, 12, 0.05)
    mels, mags = ob.ssrn_inputs(2, 12, 2)
    fresh.train_step_ssrn(mels, mags, global_step=2, seed=2)
    _three_steps_of_moments(grow, fresh, "SSRN/C_16/conv1d/bias")
    grow.close(); big.close(); fresh.close()


# ---------------------------------------------------------------------------------------------- 5. trainer end to end
def _bucketed_dataset(tmp_path, seed=0):
    d = _write_dataset(tmp_path, n=40, seed=seed)
    fpaths, lens, texts = trainer.load_train_data(d)
    loader = lambda p: trainer._load_spectrograms_npy(p, str(tmp_path / "mels"), str(tmp_path / "mags"))
    return fpaths, lens, texts, loader


@pytest.mark.parametrize("num", [1, 2])
def test_trainer_on_bucketed_batches(tmp_path, num):
    from dc_tts_b200.checkpoint import latest_checkpoint
    fpaths, lens, texts, loader = _bucketed_dataset(tmp_path)
    P = init_params(1)
    e = _engine(P)
    logdir = str(tmp_path / ("logdir/LJ01-%d" % num))
    shapes, losses = [], []

    class Recorder:
        """Passes every call to the engine, keeping the batch shapes and the losses."""
        def __getattr__(self, name):
            return getattr(e, name)

        def train_step(self, L, mels, **k):
            shapes.append(np.shape(L)[1:] + np.shape(mels)[1:2]); out = e.train_step(L, mels, **k); losses.append(out["loss"]); return out

        def train_step_ssrn(self, mels, mags, **k):
            shapes.append(np.shape(mels)[1:2]); out = e.train_step_ssrn(mels, mags, **k); losses.append(out["loss"]); return out

    batches = trainer.bucketed_batches(fpaths, lens, texts, B=4, seed=0, loader=loader)
    gs = trainer.train(num, Recorder(), batches, num_iterations=300, logdir=logdir, save_every=150, log=lambda s: None)
    assert gs == 301 and len(losses) == 301
    assert len(set(shapes)) > 3                                                  # the steps followed the buckets
    assert np.all(np.isfinite(losses)) and np.mean(losses[-50:]) < np.mean(losses[:50]), (losses[:5], losses[-5:])
    ck = latest_checkpoint(logdir)
    assert ck is not None and ck.endswith("model_gs_000k")                        # written at 150 and 300
    more = []
    gs2 = trainer.train(num, e, trainer.bucketed_batches(fpaths, lens, texts, B=4, seed=1, loader=loader), num_iterations=301,
                        logdir=logdir, save_every=150, log=more.append)
    assert gs2 == 302 and any("resumed" in s and "300" in s for s in more)
    e.close()


def test_graph_train_across_buckets(tmp_path):
    from dc_tts_b200.train import Graph, Session
    fpaths, lens, texts, loader = _bucketed_dataset(tmp_path, seed=2)
    e = _engine(init_params(1))
    seen = []

    def tap(it):
        for b in it:
            seen.append(b[1].shape[1])
            yield b

    g = Graph(num=2, mode="train", engine=e, batches=tap(trainer.bucketed_batches(fpaths, lens, texts, B=4, seed=0, loader=loader)))
    with Session() as sess:
        out = [sess.run([g.global_step, g.train_op, g.loss]) for _ in range(12)]
    assert [int(o[0]) for o in out] == list(range(1, 13))
    assert all(np.isfinite(o[2]) for o in out) and len(set(seen)) > 2
    e.close()
