"""One Text2Mel training step (BASELINE config 5; reference train.py mode "train", num=1).
CPU: the autograd oracle against the losses of the reference's OWN training graph executed under the TF API stand-in
with the shared deterministic dropout mask (tests/golden/refshim_train_losses.npz, written by make_golden_refshim.py),
optimiser arithmetic.  GPU: CUDA losses, every gradient, and the Adam update against the oracle."""
import numpy as np
import pytest
import torch

from conftest import golden
from dc_tts_b200.hyperparams import Hyperparams as hp
from dc_tts_b200.params import init_params, synthetic_text
from oracle import ref_train as rtr


def _batch(B, seed=3):
    L = synthetic_text(B, 50, seed=7)
    mels = np.random.default_rng(seed).uniform(0, 1, (B, hp.max_T, hp.n_mels)).astype(np.float32)
    return L, mels


def test_dropout_hash_properties():
    k = rtr.dropout_keep((4, 100, 256), 5, 11, 0.05)
    assert set(np.unique(k)) == {np.float32(0), np.float32(1 / 0.95)}
    assert abs((k == 0).mean() - 0.05) < 0.005
    assert np.array_equal(k, rtr.dropout_keep((4, 100, 256), 5, 11, 0.05))            # stateless
    assert not np.array_equal(k, rtr.dropout_keep((4, 100, 256), 6, 11, 0.05))        # per block
    assert not np.array_equal(k, rtr.dropout_keep((4, 100, 256), 5, 12, 0.05))        # per step
    assert np.all(rtr.dropout_keep((3, 7), 0, 0, 0.0) == 1)


def test_schedule_and_guided_attention():
    assert abs(rtr.learning_rate(0) - 0.001 * 4000 ** 0.5 * 4000 ** -1.5) < 1e-15       # utils.py:141-145
    assert abs(rtr.learning_rate(3999) - 0.001) < 1e-12 and rtr.learning_rate(15999) == pytest.approx(0.0005)
    W = rtr.guided_attention()
    assert W.shape == (hp.max_N, hp.max_T) and W[0, 0] == 0 and W.max() < 1
    assert abs(W[90, 0] - (1 - np.exp(-(0.5 ** 2) / 0.08))) < 1e-6


def test_oracle_losses_vs_reference_training_graph():
    g = golden("refshim_train_losses.npz")
    P = init_params(0, "perturbed")
    L, mels = _batch(2)
    assert list(g["t2m_seeds"]) == [11, 0] and list(g["t2m_rates"]) == [hp.dropout_rate, 0.0]
    for (seed, rate), losses, ncalls in zip(((11, hp.dropout_rate), (0, 0.0)), g["t2m_losses"], g["t2m_dropout_calls"]):
        assert ncalls == (38 if rate > 0 else 0)                                       # one dropout per block
        T = {n: torch.tensor(np.asarray(P[n], np.float32)) for n in rtr.text2mel_names()}
        with torch.no_grad():
            o = rtr.forward(T, L, mels, seed, rate)
        for k, ref in zip(("loss", "loss_mels", "loss_bd1", "loss_att"), losses):
            assert abs(float(o[k]) - ref) < 2e-6 * max(1.0, abs(ref)), (k, float(o[k]), ref)


def test_oracle_ssrn_losses_vs_reference_training_graph():
    g = golden("refshim_train_losses.npz")
    P = init_params(0, "perturbed")
    mels = np.random.default_rng(3).uniform(0, 1, (2, 12, hp.n_mels)).astype(np.float32)
    mags = np.random.default_rng(4).uniform(0, 1, (2, 48, 1 + hp.n_fft // 2)).astype(np.float32)
    assert g["ssrn_dropout_calls"] == 16
    T = {n: torch.tensor(np.asarray(P[n], np.float32)) for n in rtr.ssrn_names()}
    with torch.no_grad():
        o = rtr.forward_ssrn(T, mels, mags, 9)
    for k, ref in zip(("loss", "loss_mags", "loss_bd2"), g["ssrn_losses"]):
        assert abs(float(o[k]) - ref) < 2e-6 * max(1.0, abs(ref)), (k, float(o[k]), ref)


def test_oracle_step_arithmetic():
    P = init_params(0, "perturbed")
    L, mels = _batch(1)
    newP, st, info = rtr.train_step(P, L, mels, global_step=0, seed=5)
    g = info["grads"]
    assert len(g) == len(rtr.text2mel_names()) == 209 and all(np.abs(v).max() <= 1 for v in g.values())
    assert np.abs(g["Text2Mel/TextEnc/embed_1/lookup_table"][0]).max() == 0            # zero-padded row gets no gradient
    n = "Text2Mel/AudioDec/C_11/conv1d/bias"
    # first Adam step: m = 0.1 g, v = 0.001 g^2, update = lr_t m / (sqrt v + eps) ~ lr sign(g)
    lr = rtr.learning_rate(0)
    upd = P[n] - newP[n]
    big = np.abs(g[n]) > 1e-6
    assert np.array_equal(np.sign(upd[big]), np.sign(g[n][big]))
    assert np.all(np.abs(np.abs(upd[big]) / lr - 1) < 0.1)                              # (float32 resolution of the parameter)
    assert "SSRN/C_1/conv1d/kernel" in newP and newP["SSRN/C_1/conv1d/kernel"] is P["SSRN/C_1/conv1d/kernel"]


# ------------------------------------------------------------------------------------------- GPU
def _compare_grads(eng, grads, names=None, rtol=2e-3):
    worst = 0.0
    for n in (names or grads):
        g = eng.train_tensor(n, "grad")
        ref = grads[n]
        assert g.shape == ref.shape, n
        scale = max(np.abs(ref).max(), 1e-8)
        err = np.abs(np.clip(g, -1, 1) - ref).max() / scale
        worst = max(worst, err)
        assert err < rtol, (n, err, scale)
    return worst


def _tie_free(P):
    """The same parameters with every ReLU block pushed away from zero (LayerNorm beta += 8: all pre-activations clear zero by
    more than 1).  ReLU is discontinuous: a pre-activation within the forward noise of zero flips its mask and moves the block's
    gradients by ~1e-2 of their max-norm and everything upstream by ~3e-3 (_RELU_TIE below; with ~600k ReLU units at B = 2 a
    few always sit within 1e-5 of zero).  The float32 CUDA-core forward (noise ~1e-6) passes on hand-picked seeds; the
    split-fp16 tensor-core forward is fp32-grade but ~5x noisier, so its gradient parity is asserted on the tie-free set,
    where the comparison tests the arithmetic and not the coin flips (tools/train_grad_report_t2m.py shows the deviation of
    the plain set entering exactly at one ReLU block)."""
    from dc_tts_b200 import arch
    P = dict(P)
    for net, layers in (("TextEnc", arch.textenc_layers()), ("AudioEnc", arch.audioenc_layers()), ("AudioDec", arch.audiodec_layers())):
        for l in layers:
            if l.kind == "C" and l.act == "relu":
                n = "Text2Mel/%s/%s/normalize/beta" % (net, l.scope)
                P[n] = (np.asarray(P[n], np.float32) + 8.0).astype(np.float32)
    return P


def _t2m_relu_margin(P, B, rate, seed):
    """Smallest |pre-activation| over every ReLU block of the oracle's Text2Mel training forward."""
    L, mels = _batch(B)
    T = {n: torch.tensor(np.asarray(P[n], np.float32)) for n in rtr.text2mel_names()}
    seen, orig = [], torch.relu
    torch.relu = lambda z: (seen.append(float(z.detach().abs().min())), orig(z))[1]
    try:
        with torch.no_grad():
            rtr.forward(T, L, mels, seed, rate)
    finally:
        torch.relu = orig
    assert len(seen) == 6                                   # TextEnc C_2, AudioEnc C_1 C_2, AudioDec C_8 C_9 C_10
    return min(seen)


def test_tie_free_set_has_no_relu_near_zero():
    """The premise of the tensor-core gradient-parity cases: on the plain set some ReLU pre-activation sits within the forward
    noise of zero (so a correct fp32-grade forward may flip its mask), on the tie-free set none comes closer than 1."""
    P = init_params(0, "perturbed")
    assert _t2m_relu_margin(P, 2, 0.05, 11) < 1e-4
    assert _t2m_relu_margin(_tie_free(P), 2, 0.05, 11) > 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("B,rate,seed,tc", [(2, 0.0, 0, 7), (2, 0.05, 11, 7), (3, 0.05, 4, 7), (2, 0.0, 0, 0), (2, 0.05, 11, 0), (3, 0.05, 4, 0),
                                            (32, 0.05, 5, 7)])
def test_cuda_train_step_vs_oracle(B, rate, seed, tc):
    """tc = 7: the three conv-GEMMs of every block (forward, data gradient, weight gradient) on tcgen05 (split-fp16 x3,
    kernels_gemm_tc.cu), compared on the tie-free parameter set; tc = 0: fp32 CUDA-core kernels on the plain set.
    B = 32 is BASELINE config 5's batch."""
    from dc_tts_b200.engine import Engine
    P = init_params(0, "perturbed")
    if tc:
        P = _tie_free(P)
    eng = Engine(0)
    eng.load_params(P)
    eng.set_option("train_tc", tc)
    eng.train_init(B, rate)
    L, mels = _batch(B)
    newP, st, info = rtr.train_step(P, L, mels, global_step=7, seed=seed, rate=rate)
    out = eng.train_step(L, mels, global_step=7, seed=seed, apply=False)
    for k in ("loss", "loss_mels", "loss_bd1", "loss_att"):
        assert abs(out[k] - info[k]) < 1e-5 * max(1.0, abs(info[k])), (k, out[k], info[k])
    _compare_grads(eng, info["grads"])
    assert eng.train_grads().numel() >= 23970288
    # the optimiser: parameters, m and v after the update
    eng.train_apply(7)
    for n in ("Text2Mel/TextEnc/embed_1/lookup_table", "Text2Mel/TextEnc/HC_7/conv1d/kernel", "Text2Mel/AudioEnc/C_1/conv1d/kernel",
              "Text2Mel/AudioDec/HC_3/H2/gamma", "Text2Mel/AudioDec/C_11/conv1d/bias", "Text2Mel/AudioEnc/HC_9/H1/beta"):
        m, v = st[n]
        # element-wise 2e-3, with an absolute floor RELATIVE TO THE TENSOR (1e-4 of its largest moment): the split-fp16 GEMMs
        # round against the per-tensor scale, so elements far below the tensor's maximum carry that absolute error
        np.testing.assert_allclose(eng.train_tensor(n, "m"), m, rtol=2e-3, atol=max(1e-9, 1e-4 * np.abs(m).max()))
        np.testing.assert_allclose(eng.train_tensor(n, "v"), v, rtol=4e-3, atol=max(1e-14, 4e-4 * np.abs(v).max()))
        step = np.abs(newP[n] - P[n]).max()
        assert np.abs(eng.train_tensor(n, "param") - newP[n]).max() <= 0.05 * step + 2.4e-7, n      # + 2 ulp at 1.0


@pytest.mark.gpu
def test_cuda_training_reduces_loss_and_is_deterministic():
    from dc_tts_b200.engine import Engine
    P = init_params(1)
    L, mels = _batch(4, seed=9)
    runs = []
    for _ in range(2):
        eng = Engine(0)
        eng.load_params(P)
        eng.train_init(4)
        runs.append([eng.train_step(L, mels, global_step=4000 + i, seed=i)["loss"] for i in range(8)])
    assert runs[0][-1] < runs[0][0]                                                    # same batch, lr 1e-3: the loss falls
    # float atomics reorder sums only: the first steps agree to 1e-4; Adam (a sign-like update where |g| ~ sqrt(v)) amplifies the
    # last-bit differences from step to step, so the whole 8-step trajectory is held to 5e-3 (observed: 4e-4 at step 5)
    assert np.allclose(runs[0][:3], runs[1][:3], rtol=1e-4)
    assert np.allclose(runs[0], runs[1], rtol=5e-3)


@pytest.mark.gpu
def test_cuda_train_checkpoint_roundtrip(tmp_path):
    """train -> save (TF bundle, train.py:152) -> restore into a fresh handle (synthesize.py:31-41) -> same outputs as
    the trained handle; and the trained handle refuses the stale tcgen05 weight planes."""
    from dc_tts_b200 import checkpoint as ck
    from dc_tts_b200.engine import Engine
    P = init_params(2)
    L, mels = _batch(2, seed=5)
    eng = Engine(0)
    eng.load_params(P)
    eng.train_init(2)
    for i in range(3):
        eng.train_step(L, mels, global_step=4000 + i, seed=i)
    prefix = eng.save_text2mel_checkpoint(str(tmp_path / "LJ01-1" / "model_gs_004k"), 4003)
    ck.save_checkpoint(str(tmp_path / "LJ01-2" / "model_gs_000k"), {k: v for k, v in P.items() if k.startswith("SSRN/")})
    got = ck.load_checkpoint(prefix, names=["gs/global_step", "Text2Mel/AudioDec/C_11/conv1d/bias", "Text2Mel/AudioDec/C_11/conv1d/bias/Adam"])
    assert int(got["gs/global_step"]) == 4003 and np.abs(got["Text2Mel/AudioDec/C_11/conv1d/bias/Adam"]).max() > 0
    assert np.abs(got["Text2Mel/AudioDec/C_11/conv1d/bias"] - P["Text2Mel/AudioDec/C_11/conv1d/bias"]).max() > 1e-4   # it moved
    fresh = Engine(0)
    fresh.restore(str(tmp_path / "LJ01-1"), str(tmp_path / "LJ01-2"))
    fresh.set_tensor_path(0)
    pma = np.zeros(2, np.int32)
    ya = eng.text2mel_forward(L, mels, pma)[0]
    yb = fresh.text2mel_forward(L, mels, pma)[0]
    assert torch.equal(ya, yb)
    with pytest.raises(RuntimeError):
        eng.set_tensor_path(1)


_RELU_TIE = ("not a defect: in this configuration a pre-activation of the ReLU block SSRN/C_14 lies 1.2e-7 from zero (float32 "
             "resolution), so two correct float32 forward passes legitimately disagree on that element's ReLU mask; the flipped element "
             "moves C_14's gradients by up to 4e-2 of their max-norm and everything upstream by ~3e-3 "
             "(test_ssrn_relu_margins_explain_the_tie_case, tools/train_grad_report.py)")


def _ssrn_relu_margins(B, T, rate, seed):
    """Smallest |pre-activation| of the two ReLU blocks of SSRN (C_14, C_15) in the oracle's forward pass."""
    from dc_tts_b200 import arch
    from oracle import ref_torch as rt
    P = init_params(0, "perturbed")
    W = {n: torch.tensor(np.asarray(P[n], np.float32)) for n in rtr.ssrn_names()}
    x = torch.as_tensor(np.random.default_rng(3).uniform(0, 1, (B, T, hp.n_mels)).astype(np.float32))
    out = {}
    for c, l in enumerate(arch.ssrn_layers()):
        scope = "SSRN/%s" % l.scope
        if l.kind == "C":
            y = rt._conv(x, W[scope + "/conv1d/kernel"], W[scope + "/conv1d/bias"], l.rate, l.pad)
            z = rt.normalize(y, W[scope + "/normalize/gamma"], W[scope + "/normalize/beta"])
            if l.act == "relu":
                out[l.scope] = float(z.abs().min())
                z = torch.relu(z)
            x = z
        elif l.kind == "HC":
            x = rt.hc(W, x, scope, l.rate, l.pad)
        else:
            x = rt.conv1d_transpose(W, x, scope)
        if rate > 0:
            x = x * torch.from_numpy(rtr.dropout_keep(tuple(x.shape), c, seed, rate))
    return out


def test_ssrn_relu_margins_explain_the_tie_case():
    """ReLU is discontinuous: gradient parity between two float32 implementations needs every ReLU pre-activation to clear
    zero by more than the forward noise (~4e-6 here).  The configurations used as GPU parity cases do; (2, 16, 0.0, 0) does not."""
    assert min(_ssrn_relu_margins(2, 16, 0.0, 0).values()) < 1e-6
    assert min(_ssrn_relu_margins(2, 12, 0.05, 9).values()) > 4e-6
    assert min(_ssrn_relu_margins(1, 8, 0.0, 0).values()) > 4e-6
    assert min(_ssrn_relu_margins(2, 14, 0.0, 7).values()) > 4e-6


@pytest.mark.gpu
@pytest.mark.parametrize("B,T,rate,seed", [pytest.param(2, 16, 0.0, 0, marks=pytest.mark.xfail(reason=_RELU_TIE, strict=False)),
                                           (2, 12, 0.05, 9), (1, 8, 0.0, 0), (2, 14, 0.0, 7)])
def test_cuda_ssrn_train_step_vs_oracle(B, T, rate, seed):
    """The SSRN trainer (train.py num=2): transposed-conv blocks, C = 1024 highway blocks and the F = 1025 wide blocks.
    The first case is kept as a documented ReLU tie (see _RELU_TIE)."""
    from dc_tts_b200.engine import Engine
    P = init_params(0, "perturbed")
    eng = Engine(0)
    eng.load_params(P)
    eng.train_init_ssrn(B, T, rate)
    mels = np.random.default_rng(3).uniform(0, 1, (B, T, hp.n_mels)).astype(np.float32)
    mags = np.random.default_rng(4).uniform(0, 1, (B, 4 * T, 1 + hp.n_fft // 2)).astype(np.float32)
    newP, st, info = rtr.train_step_ssrn(P, mels, mags, global_step=3999, seed=seed, rate=rate)
    out = eng.train_step_ssrn(mels, mags, global_step=3999, seed=seed, apply=False)
    for k in ("loss", "loss_mags", "loss_bd2"):
        assert abs(out[k] - info[k]) < 1e-5 * max(1.0, abs(info[k])), (k, out[k], info[k])
    assert len(info["grads"]) == 80
    _compare_grads(eng, info["grads"])
    eng.train_apply(3999)
    for n in ("SSRN/D_4/conv2d_transpose/kernel", "SSRN/D_7/conv2d_transpose/bias", "SSRN/HC_12/conv1d/kernel", "SSRN/C_13/conv1d/kernel",
              "SSRN/C_16/conv1d/bias", "SSRN/C_15/normalize/gamma", "SSRN/HC_2/H1/beta"):
        m, v = st[n]
        np.testing.assert_allclose(eng.train_tensor(n, "m"), m, rtol=2e-3, atol=max(1e-9, 1e-4 * np.abs(m).max()))
        step = np.abs(newP[n] - P[n]).max()
        assert np.abs(eng.train_tensor(n, "param") - newP[n]).max() <= 0.05 * step + 2.4e-7, n


@pytest.mark.gpu
@pytest.mark.parametrize("num", [1, 2])
def test_cuda_training_resumes_from_its_own_checkpoint(tmp_path, num):
    """ADVICE r1: a restarted run must continue, not start over.  Train 3 steps, save (variables + Adam slots + gs +
    beta powers), restore into a fresh handle with Engine.restore_training, take one more step on both: identical losses
    and identical updated weights (what tf.train.Supervisor's restore gives train.py:144)."""
    from dc_tts_b200 import checkpoint as ck
    from dc_tts_b200.engine import Engine
    P = init_params(2)
    scope = "Text2Mel" if num == 1 else "SSRN"
    T = hp.max_T if num == 1 else 12
    L, mels = _batch(2, seed=5)
    mels = mels[:, :T]
    mags = np.random.default_rng(4).uniform(0, 1, (2, 4 * T, 1 + hp.n_fft // 2)).astype(np.float32)

    def init(e):
        e.load_params(P)
        e.train_init(2, 0.0) if num == 1 else e.train_init_ssrn(2, T, 0.0)

    def step(e, gs):
        return e.train_step(L, mels, global_step=gs, seed=gs) if num == 1 else e.train_step_ssrn(mels, mags, global_step=gs, seed=gs)

    a = Engine(0); init(a)
    for gs in range(3):
        step(a, gs)
    logdir = str(tmp_path / ("LJ01-%d" % num))
    a.save_checkpoint(logdir + "/model_gs_000k", 3, scope)
    got = ck.load_checkpoint(logdir + "/model_gs_000k", ["beta1_power", "beta2_power", "gs/global_step"])
    assert abs(float(got["beta1_power"]) - 0.9 ** 4) < 1e-7 and int(got["gs/global_step"]) == 3
    b = Engine(0); init(b)
    assert b.restore_training(str(tmp_path / "nothing-here"), scope) is None
    assert b.restore_training(logdir, scope) == 3
    probe = "Text2Mel/AudioDec/HC_4/conv1d/kernel" if num == 1 else "SSRN/D_4/conv2d_transpose/kernel"
    for what in ("param", "m", "v"):                                   # the restored state is the saved state, bit for bit
        assert np.array_equal(a.train_tensor(probe, what), b.train_tensor(probe, what)), what
    la, lb = step(a, 3), step(b, 3)
    for k in la:                                                       # float atomics reorder sums: tolerance, not bits
        assert abs(la[k] - lb[k]) <= 1e-4 * max(1.0, abs(la[k])), k
    for what in ("param", "m", "v"):
        x, y = a.train_tensor(probe, what), b.train_tensor(probe, what)
        assert np.abs(x - y).max() <= 1e-3 * np.abs(x).max() + 1e-12, what
    a.close(); b.close()
