"""Generates tests/golden/refshim_long.npz: the REFERENCE'S OWN graphs (train.py Graph, networks.py, synthesize.py's loop),
executed under the TensorFlow API stand-in of tf_shim.py with the reference's Hyperparams.max_N / max_T raised to
(300, 320), as a user with longer text would set them in hyperparams.py.  The parameters are init_params(0, "perturbed");
every dropout the training graph places gets the oracle's deterministic mask, as in make_golden_buckets.py.  Contents:
  * one full-graph pass of Graph(mode="synthesize") at B = 2: row 0 holds 285 characters with prev_max_attentions near
    max_N - 3, row 1 is short with the window at 0 (Y, max_attentions);
  * the first steps of synthesize.py:45-54's loop on the same text (Y rows, window trajectory);
  * Text2Mel training losses at (N_b, T_b) = (257, 40), (300, 330), (320, 70) (N_b below, at and above max_N; T_b above
    max_T), with and without dropout, on the seeded inputs of tests/oracle_buckets.py.
Run from the repo root:
    python tests/golden/make_golden_long.py REFERENCE_DIR
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import tf_shim                                                   # noqa: E402
from dc_tts_b200.hyperparams import Hyperparams as hp            # noqa: E402
from dc_tts_b200.params import init_params                       # noqa: E402
from oracle import ref_train as rtr                              # noqa: E402
from oracle_buckets import bucket_inputs                         # noqa: E402

MAX_N, MAX_T = 300, 320
B = 2
INPUT_SEED = 5
STEPS = 4
T2M_SHAPES = [(257, 40), (300, 330), (320, 70)]
RUNS = [(0, 0.0), (11, hp.dropout_rate)]                         # (dropout seed, rate)
T2M_KEYS = ("loss", "loss_mels", "loss_bd1", "loss_att")


def long_inputs():
    """Text (B, MAX_N): row 0 has 285 characters, row 1 has 40, each ended by E; mels uniform in [0, 1); the window of
    row 0 near the end of its keys, of row 1 at 0."""
    L = np.zeros((B, MAX_N), np.int32)
    for b, n in enumerate((285, 40)):
        rng = np.random.default_rng([INPUT_SEED, b])
        L[b, :n] = rng.integers(2, len(hp.vocab), size=n)
        L[b, n] = 1
    mels = np.random.default_rng([INPUT_SEED, 99]).uniform(0, 1, (B, MAX_T, hp.n_mels)).astype(np.float32)
    return L, mels, np.array([MAX_N - 5, 0], np.int32)


if __name__ == "__main__":
    REF = os.path.abspath(sys.argv[1])
    P = init_params(0, "perturbed")
    tf_shim.install(tf_shim.Store(P), REF)
    import hyperparams as ref_hp                                 # noqa: E402  (the reference's, installed above)
    ref_hp.Hyperparams.max_N, ref_hp.Hyperparams.max_T = MAX_N, MAX_T
    hp.max_N, hp.max_T = MAX_N, MAX_T                            # the oracle's guided-attention table follows

    L, mels, pma = long_inputs()
    o = tf_shim.run_graph(L, mels, pma, fetch=("Y", "max_attentions"))
    print("full pass: max_attentions row 0 %s" % o["max_attentions"][0, :8], flush=True)
    r = tf_shim.synthesize(L, steps=STEPS, with_ssrn=False)
    print("loop: p_hist %s" % r["p_hist"].tolist(), flush=True)

    rate0 = ref_hp.Hyperparams.dropout_rate
    t2m_losses = np.zeros((len(T2M_SHAPES), len(RUNS), 4))
    for i, (N_b, T_b) in enumerate(T2M_SHAPES):
        Lb, mb = bucket_inputs(B, N_b, T_b, INPUT_SEED)
        for j, (seed, rate) in enumerate(RUNS):
            ref_hp.Hyperparams.dropout_rate = rate
            losses, _ = tf_shim.run_train_graph(Lb, mb, lambda x, r, k, seed=seed: x * rtr.dropout_keep(x.shape, k, seed, r))
            t2m_losses[i, j] = [losses[k] for k in T2M_KEYS]
            print("text2mel N_b=%d T_b=%d rate=%.2f: %s" % (N_b, T_b, rate, losses), flush=True)
    ref_hp.Hyperparams.dropout_rate = rate0

    out = os.path.join(HERE, "refshim_long.npz")
    np.savez_compressed(out, max_N=np.array(MAX_N), max_T=np.array(MAX_T), B=np.array(B), input_seed=np.array(INPUT_SEED),
                        L=L, pma=pma, Y=o["Y"], max_attentions=o["max_attentions"],
                        loop_Y=r["Y"][:, :STEPS], loop_p_hist=r["p_hist"],
                        t2m_shapes=np.array(T2M_SHAPES), seeds=np.array([s for s, _ in RUNS]),
                        rates=np.array([r_ for _, r_ in RUNS]), t2m_losses=t2m_losses)
    print("written %s (%d bytes)" % (out, os.path.getsize(out)))
