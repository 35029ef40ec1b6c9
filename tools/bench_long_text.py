"""Text longer than 192 characters on one GPU, CUDA events.
    python tools/bench_long_text.py [--batch 32 --reps 3 --iters 20 --out profiles/r04_bench_long_text.json]
Writes (and prints) one JSON object:
  attention   ms per dctts_attention call (dense, as the training forward runs it; B x max_T queries, max_T = 320) at
              N in {192, 256, 320, 512}, tcgen05 kernel (tensor path 1) and fp32 kernel (tensor path 0) timed alternately;
              each call includes the conversion of Q, K, V to split-fp16 planes on the tcgen05 path and writes the
              (B, N, T) alignments
  t2m_step    ms per Text2Mel training step (fwd + bwd + clip + Adam, train_tc 7) at (N_b, T_b) = (180, 210) on a handle
              with the LJ hyper-parameters (max_N 180, max_T 210) and at (256, 300), (320, 400) on a (300, 320) handle
  generate    ms for text2mel_generate (all 320 frames, persistent decode) + SSRN at max_N 300, max_T 320, B utterances
The card's name and power limit are read in the same run and recorded with the numbers."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from dc_tts_b200.engine import Engine
from dc_tts_b200.hyperparams import Hyperparams as hp
from dc_tts_b200.params import init_params, synthetic_text

ap = argparse.ArgumentParser()
ap.add_argument("--batch", type=int, default=32)
ap.add_argument("--reps", type=int, default=3, help="timing windows per measurement (median taken)")
ap.add_argument("--iters", type=int, default=20, help="calls per attention timing window")
ap.add_argument("--steps", type=int, default=5, help="training steps per timing window")
ap.add_argument("--out", default=None, help="also write the JSON here")
a = ap.parse_args()
B = a.batch
dev = torch.device("cuda", 0)
LJ = (hp.max_N, hp.max_T)


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


def engine(max_N, max_T, P=None):
    hp.max_N, hp.max_T = max_N, max_T
    e = Engine(0)
    if P is not None:
        e.load_params(P)
    return e


def text_batch(N, T, seed):
    rng = np.random.default_rng(seed)
    L = np.zeros((B, N), np.int32)
    for b in range(B):
        n = int(rng.integers(max(1, N // 2), N + 1)) if b else N
        L[b, :n - 1] = rng.integers(2, len(hp.vocab), n - 1)
        L[b, n - 1] = 1
    return torch.from_numpy(L).to(dev), torch.from_numpy(rng.uniform(0, 1, (B, T, hp.n_mels)).astype(np.float32)).to(dev)


P = init_params(0)
out = {"metric": "long_text", "card": card(), "batch": B}

# ------------------------------------------------------------------ attention alone, tcgen05 vs fp32
e = engine(512, 320)
T = hp.max_T
rng = np.random.default_rng(0)
att = []
for N in (192, 256, 320, 512):
    Q, K, V = (torch.from_numpy(rng.uniform(-1, 1, s).astype(np.float32)).to(dev) for s in ((B, T, hp.d), (B, N, hp.d), (B, N, hp.d)))
    run = {}
    for tp in (1, 0, 1, 0):                                    # warm both, then time both
        e.set_tensor_path(tp)
        e.attention(Q, K, V)
        torch.cuda.synchronize()
    ms = {1: [], 0: []}
    for _ in range(a.reps):
        for tp in (1, 0):
            e.set_tensor_path(tp)
            ms[tp].append(timed(lambda i: e.attention(Q, K, V), a.iters) / a.iters)
    att.append({"N": N, "T": T, "ms_tcgen05": round(float(np.median(ms[1])), 4), "ms_fp32": round(float(np.median(ms[0])), 4),
                "fp32_over_tcgen05": round(float(np.median(ms[0]) / np.median(ms[1])), 2)})
    print(att[-1], flush=True)
out["attention"] = att
e.close()

# ------------------------------------------------------------------ Text2Mel training step
steps = []
for (mN, mT), (N, T) in [(LJ, (180, 210)), ((300, 320), (256, 300)), ((300, 320), (320, 400))]:
    e = engine(mN, mT, P)
    e.train_init(B)
    e.train_reserve(N, T)
    L, m = text_batch(N, T, N * 1000 + T)
    e.train_step(L, m, global_step=4000, seed=0)
    torch.cuda.synchronize()
    w = [timed(lambda i: e.train_step(L, m, global_step=4000 + i, seed=i), a.steps) / a.steps for _ in range(a.reps)]
    steps.append({"max_N": mN, "max_T": mT, "N_b": N, "T_b": T, "ms": round(float(np.median(w)), 3)})
    print(steps[-1], flush=True)
    e.close()
out["t2m_step"] = steps

# ------------------------------------------------------------------ generate + SSRN at (300, 320)
e = engine(300, 320, P)
L = torch.from_numpy(synthetic_text(B, 280, seed=0)).to(dev)


def synth(_):
    Y, _, _, _ = e.text2mel_generate(L)
    e.ssrn(Y, want_logits=False)


synth(0)
torch.cuda.synchronize()
w = [timed(synth, 1) for _ in range(a.reps)]
out["generate"] = {"max_N": 300, "max_T": 320, "chars": 280, "B": B, "ms_generate_plus_ssrn": round(float(np.median(w)), 1),
                   "decode_mode": e.get_option("decode_mode")}
print(out["generate"], flush=True)
e.close()
hp.max_N, hp.max_T = LJ

s = json.dumps(out)
print(s)
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(s + "\n")
