"""Training steps at the shape of a length bucket against the fixed 180 x 210 step (BASELINE config 5), one GPU, CUDA events.
    python tools/bench_train_buckets.py [--batch 32 --reps 3 --steps 5 --batches 60]
Prints one JSON line:
  t2m_grid    ms per Text2Mel step at each (N_b, T_b), timed alternately with the fixed step in the same process
  ssrn        ms per SSRN step at each T_b, alternately with the step at T = 210
  throughput  useful (unpadded) mel frames per second over a seeded synthetic LJ-like corpus pushed through
              trainer.bucketed_batches: every batch at its own shape, against the same batches padded by
              trainer.pad_to_fixed (which drops the ones longer than 180 / 210)
The card's name and power limit are read in the same run and printed with the numbers.  Inputs are uploaded before the
timed windows; each step reads its losses back (one synchronisation per step, as the trainer loop does)."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from dc_tts_b200 import trainer
from dc_tts_b200.engine import Engine
from dc_tts_b200.hyperparams import Hyperparams as hp
from dc_tts_b200.params import init_params

ap = argparse.ArgumentParser()
ap.add_argument("--batch", type=int, default=32)
ap.add_argument("--reps", type=int, default=3, help="alternations of shaped / fixed timing windows per shape")
ap.add_argument("--steps", type=int, default=5, help="steps per timing window")
ap.add_argument("--batches", type=int, default=60, help="bucketed batches in the throughput run")
ap.add_argument("--utterances", type=int, default=13100, help="size of the synthetic corpus (LJ Speech has 13,100 clips)")
a = ap.parse_args()
B, F = a.batch, 1 + hp.n_fft // 2
dev = torch.device("cuda", 0)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:                                     # noqa: BLE001 -- the numbers stay valid without it
        q = "nvidia-smi unavailable: %s" % e
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def timed(fn, n):
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for i in range(n):
        fn(i)
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1)


def alternate(shaped, fixed):
    """Median ms per step of `shaped` and of `fixed`, windows interleaved so that clock drift hits both alike."""
    shaped(0); fixed(0); torch.cuda.synchronize()
    s, f = [], []
    for _ in range(a.reps):
        s.append(timed(shaped, a.steps) / a.steps)
        f.append(timed(fixed, a.steps) / a.steps)
    return float(np.median(s)), float(np.median(f))


def text_batch(N, T, seed):
    rng = np.random.default_rng(seed)
    L = np.zeros((B, N), np.int32)
    for b in range(B):
        n = int(rng.integers(max(1, N // 2), N + 1)) if b else N
        L[b, :n] = rng.integers(2, len(hp.vocab), n)
    return torch.from_numpy(L).to(dev), torch.from_numpy(rng.uniform(0, 1, (B, T, hp.n_mels)).astype(np.float32)).to(dev)


P = init_params(0)
out = {"metric": "bucketed_train_useful_mel_frames_per_sec", "card": card(), "batch": B, "dropout": hp.dropout_rate,
       "config": "Text2Mel / SSRN train step (fwd + bwd + clip + Adam), tcgen05 GEMMs (train_tc 7)"}

# ------------------------------------------------------------------ Text2Mel grid vs the fixed step
eng = Engine(0)
eng.load_params(P)
eng.train_init(B)
eng.train_reserve(hp.max_N + 12, hp.max_T + 30)
Lf, mf = text_batch(hp.max_N, hp.max_T, 0)
fixed = lambda i: eng.train_step(Lf, mf, global_step=4000 + i, seed=i)
grid = []
for N, T in [(40, 50), (60, 80), (80, 100), (100, 130), (120, 150), (140, 180), (160, 200), (180, 210), (185, 240),
             (40, 200), (160, 60)]:
    Ls, ms = text_batch(N, T, N * 1000 + T)
    t_s, t_f = alternate(lambda i: eng.train_step(Ls, ms, global_step=4000 + i, seed=i), fixed)
    grid.append({"N_b": N, "T_b": T, "ms_shaped": round(t_s, 3), "ms_fixed_180x210": round(t_f, 3), "ratio": round(t_s / t_f, 3)})
out["t2m_grid"] = grid

# ------------------------------------------------------------------ throughput over a synthetic LJ-like corpus
# text lengths ~ LJ Speech (mean ~100 normalised characters, a few beyond 180); frames (after the r = 4 reduction) ~ 1.3
# per character with +-15 % speaking-rate spread
rng = np.random.default_rng(2026)
n_utt = a.utterances
lens = np.clip(np.round(rng.normal(100, 38, n_utt)), 8, 200).astype(int)
frames = np.maximum(4, np.round(lens * 1.3 * rng.uniform(0.85, 1.15, n_utt))).astype(int)
texts = [rng.integers(2, len(hp.vocab), n).astype(np.int32) for n in lens]
fpaths = ["wavs/LJ%05d.wav" % i for i in range(n_utt)]
idx = {p: i for i, p in enumerate(fpaths)}
mel_rng = np.random.default_rng(7)
loader = lambda p: (p, mel_rng.uniform(0, 1, (frames[idx[p]], hp.n_mels)).astype(np.float32),
                    np.zeros((4 * frames[idx[p]], 1), np.float32))          # mags are not used by the Text2Mel step
batches = []
for L, mels, _, names, _ in trainer.bucketed_batches(fpaths, list(lens), texts, B=B, seed=0, loader=loader):
    batches.append((L, mels, int(sum(frames[idx[n]] for n in names))))
    if len(batches) == a.batches:
        break
shaped_in = [(torch.from_numpy(L).to(dev), torch.from_numpy(m).to(dev), u) for L, m, u in batches if trainer.fits_key_capacity(L)]
fixed_in = []
for L, m, u in batches:
    pf = trainer.pad_to_fixed(L, m, np.zeros((B, 4 * m.shape[1], 1), np.float32))
    if pf is not None:
        fixed_in.append((torch.from_numpy(pf[0]).to(dev), torch.from_numpy(pf[1]).to(dev), u))
eng.train_step(*shaped_in[0][:2], global_step=4000, seed=0)
eng.train_step(*fixed_in[0][:2], global_step=4000, seed=0)
torch.cuda.synchronize()
ms_b = timed(lambda i: eng.train_step(shaped_in[i][0], shaped_in[i][1], global_step=4000 + i, seed=i), len(shaped_in))
ms_f = timed(lambda i: eng.train_step(fixed_in[i][0], fixed_in[i][1], global_step=4000 + i, seed=i), len(fixed_in))
useful_b, useful_f = sum(u for _, _, u in shaped_in), sum(u for _, _, u in fixed_in)
out["throughput"] = {"batches": len(batches), "mean_N_b": float(np.mean([b[0].shape[1] for b in batches])),
                     "mean_T_b": float(np.mean([b[1].shape[1] for b in batches])),
                     "bucketed": {"steps": len(shaped_in), "ms": round(ms_b, 1), "useful_frames": useful_b,
                                  "useful_mel_frames_per_sec": useful_b * 1e3 / ms_b},
                     "pad_to_fixed": {"steps": len(fixed_in), "dropped_batches": len(batches) - len(fixed_in), "ms": round(ms_f, 1),
                                      "useful_frames": useful_f, "useful_mel_frames_per_sec": useful_f * 1e3 / ms_f}}
out["value"] = useful_b * 1e3 / ms_b
out["unit"] = "mel frames/s"
out["speedup_vs_pad_to_fixed"] = (useful_b / ms_b) / (useful_f / ms_f)
eng.close()

# ------------------------------------------------------------------ SSRN at several T_b vs T = 210
eng = Engine(0)
eng.load_params(P)
eng.train_init_ssrn(B, hp.max_T)
g = np.random.default_rng(1)
up = lambda *s: torch.from_numpy(g.uniform(0, 1, s).astype(np.float32)).to(dev)
mf, gf = up(B, hp.max_T, hp.n_mels), up(B, 4 * hp.max_T, F)
fixed = lambda i: eng.train_step_ssrn(mf, gf, global_step=4000 + i, seed=i)
ssrn = []
for T in (25, 50, 100, 150, 210):
    ms, gs = up(B, T, hp.n_mels), up(B, 4 * T, F)
    t_s, t_f = alternate(lambda i: eng.train_step_ssrn(ms, gs, global_step=4000 + i, seed=i), fixed)
    ssrn.append({"T_b": T, "ms_shaped": round(t_s, 3), "ms_fixed_210": round(t_f, 3), "ratio": round(t_s / t_f, 3)})
out["ssrn"] = ssrn
eng.close()
print(json.dumps(out))
