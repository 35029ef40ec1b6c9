"""Test infrastructure: the autograd oracle of oracle/ref_train.py for a length-bucketed batch of ANY shape, as the
reference trains on them (data_load.py:122-129, dynamic_pad=True).  oracle/ref_train.py is kept as it is; it pins the
fixed (max_N, max_T) batches, and this module reuses its blocks, dropout mask and optimiser.

Text2Mel on L (B, N_b), mels (B, T_b, n_mels): TextEnc and the attention keys run over N_b rows, AudioEnc / AudioDec over
T_b frames, the mel losses average over B T_b n_mels.  Guided attention (train.py:91-95): W is always (max_N, max_T); A is
padded with -1 and cut to [:max_N, :max_T], so only the window n < N_w = min(N_b, max_N), t < T_w = min(T_b, max_T)
contributes, loss_att = sum_window |A W| / (B N_w T_w).  At (max_N, max_T) this is exactly ref_train.forward.
SSRN on mels (B, T_b, n_mels) / mags (B, 4 T_b, F): ref_train.forward_ssrn has no fixed extent and is used as it is."""
import numpy as np
import torch

from dc_tts_b200 import arch
from dc_tts_b200.hyperparams import Hyperparams as hp
from oracle import ref_torch as rt
from oracle import ref_train as rtr

forward_ssrn = rtr.forward_ssrn
train_step_ssrn = rtr.train_step_ssrn


def attention_window(N_b, T_b):
    """(N_w, T_w): the part of the alignments the guided-attention term covers."""
    return min(N_b, hp.max_N), min(T_b, hp.max_T)


def forward(P, L, mels, seed=0, rate=None):
    rate = hp.dropout_rate if rate is None else rate
    mels = torch.as_tensor(mels, dtype=torch.float32)
    S = torch.cat((torch.zeros_like(mels[:, :1, :]), mels[:, :-1, :]), 1)
    c = [0]
    x = rt.embed(P, torch.as_tensor(L), "Text2Mel/TextEnc/embed_1").to(torch.float32)
    x = rtr._chain(P, x, "Text2Mel/TextEnc", arch.textenc_layers(), c, seed, rate)
    K, V = torch.chunk(x, 2, dim=-1)
    Q = rtr._chain(P, S, "Text2Mel/AudioEnc", arch.audioenc_layers(), c, seed, rate)
    R, alignments, _ = rt.Attention(Q, K, V, False, None)
    logits = rtr._chain(P, R, "Text2Mel/AudioDec", arch.audiodec_layers(), c, seed, rate)
    Y = torch.sigmoid(logits)
    loss_mels = (Y - mels).abs().mean()
    loss_bd1 = torch.nn.functional.binary_cross_entropy_with_logits(logits, mels)
    B = alignments.shape[0]
    N_w, T_w = attention_window(alignments.shape[1], alignments.shape[2])
    A = alignments[:, :N_w, :T_w]
    gts = torch.from_numpy(rtr.guided_attention()[:N_w, :T_w])
    loss_att = (A * gts).abs().sum() / float(B * N_w * T_w)
    return dict(loss=loss_mels + loss_bd1 + loss_att, loss_mels=loss_mels, loss_bd1=loss_bd1, loss_att=loss_att,
                Y=Y, logits=logits, alignments=alignments, Q=Q, K=K, V=V, R=R)


def train_step(P, L, mels, state=None, global_step=0, seed=0, rate=None, lr=None, beta1=0.9, beta2=0.999, eps=1e-8):
    """One Text2Mel optimiser step on a batch of any shape: (new params, Adam state, info with losses and clipped grads)."""
    names = rtr.text2mel_names()
    T = {n: torch.tensor(np.asarray(P[n], np.float32), requires_grad=True) for n in names}
    out = forward(T, L, mels, seed, rate)
    out["loss"].backward()
    newP, newstate, grads, lr_now = rtr._adam(P, names, T, state, global_step, lr, beta1, beta2, eps)
    info = {k: float(out[k].detach()) for k in ("loss", "loss_mels", "loss_bd1", "loss_att")}
    info["grads"] = grads
    info["lr"] = lr_now
    return newP, newstate, info


def bucket_inputs(B, N_b, T_b, seed):
    """Seeded inputs of one bucket: row 0 holds N_b characters (the longest member), the others are shorter and zero
    padded to N_b like dynamic_pad does; mels uniform in [0, 1)."""
    L = np.zeros((B, N_b), np.int32)
    rng = np.random.default_rng([seed, N_b, T_b])
    for b in range(B):
        n = N_b if b == 0 else max(1, N_b - 1 - int(rng.integers(0, max(1, N_b // 3))))
        L[b, :n - 1] = rng.integers(2, len(hp.vocab), size=n - 1)
        L[b, n - 1] = 1                                                   # E
    mels = rng.uniform(0, 1, (B, T_b, hp.n_mels)).astype(np.float32)
    return L, mels


def ssrn_inputs(B, T_b, seed):
    rng = np.random.default_rng([seed, T_b])
    mels = rng.uniform(0, 1, (B, T_b, hp.n_mels)).astype(np.float32)
    mags = rng.uniform(0, 1, (B, 4 * T_b, 1 + hp.n_fft // 2)).astype(np.float32)
    return mels, mags


def t2m_relu_margin(P, L, mels, seed, rate):
    """Smallest |pre-activation| over the six ReLU blocks of the Text2Mel training forward.  ReLU is discontinuous: two
    correct float32 forward passes agree on every mask only where this clears their noise."""
    W = {n: torch.tensor(np.asarray(P[n], np.float32)) for n in rtr.text2mel_names()}
    seen, orig = [], torch.relu
    torch.relu = lambda z: (seen.append(float(z.detach().abs().min())), orig(z))[1]
    try:
        with torch.no_grad():
            forward(W, L, mels, seed, rate)
    finally:
        torch.relu = orig
    return min(seen)


def ssrn_relu_margin(P, mels, seed, rate):
    """Smallest |pre-activation| of SSRN's two ReLU blocks (C_14, C_15) in the training forward."""
    W = {n: torch.tensor(np.asarray(P[n], np.float32)) for n in rtr.ssrn_names()}
    x = torch.as_tensor(mels)
    out = []
    for c, l in enumerate(arch.ssrn_layers()):
        scope = "SSRN/%s" % l.scope
        if l.kind == "C":
            z = rt.normalize(rt._conv(x, W[scope + "/conv1d/kernel"], W[scope + "/conv1d/bias"], l.rate, l.pad),
                             W[scope + "/normalize/gamma"], W[scope + "/normalize/beta"])
            if l.act == "relu":
                out.append(float(z.abs().min()))
                z = torch.relu(z)
            x = z
        elif l.kind == "HC":
            x = rt.hc(W, x, scope, l.rate, l.pad)
        else:
            x = rt.conv1d_transpose(W, x, scope)
        if rate > 0:
            x = x * torch.from_numpy(rtr.dropout_keep(tuple(x.shape), c, seed, rate))
    return min(out)
