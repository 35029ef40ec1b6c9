"""Generates tests/golden/refshim_train_buckets.npz: the losses of the REFERENCE'S OWN training graphs (train.py
Graph(num=1 / num=2, mode="train"), executed under the TensorFlow API stand-in of tf_shim.py) on length-bucketed batches
of their own shape -- what data_load.py:122-129 (bucket_by_sequence_length, dynamic_pad=True) feeds them.  The parameters
are init_params(0, "perturbed"); every dropout the graph places gets the oracle's deterministic mask, as in section 7 of
make_golden_refshim.py.  Inputs come from tests/oracle_buckets.py (bucket_inputs / ssrn_inputs) with the seeds recorded
in the file.  Run from the repo root:
    python tests/golden/make_golden_buckets.py REFERENCE_DIR
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
from oracle_buckets import bucket_inputs, ssrn_inputs            # noqa: E402

REF = os.path.abspath(sys.argv[1])
P = init_params(0, "perturbed")
tf_shim.install(tf_shim.Store(P), REF)
import hyperparams as ref_hp                                     # noqa: E402  (the reference's, installed above)

B = 2
INPUT_SEED = 5
# (N_b, T_b): small, neither a multiple of 8; N_b > max_N; T_b > max_T; a realistic LJ bucket
T2M_SHAPES = [(23, 17), (185, 9), (30, 214), (110, 150)]
SSRN_T = [9, 23]
RUNS = [(0, 0.0), (11, hp.dropout_rate)]                         # (dropout seed, rate)
T2M_KEYS, SSRN_KEYS = ("loss", "loss_mels", "loss_bd1", "loss_att"), ("loss", "loss_mags", "loss_bd2")

rate0 = ref_hp.Hyperparams.dropout_rate
t2m_losses, t2m_calls = np.zeros((len(T2M_SHAPES), len(RUNS), 4)), np.zeros((len(T2M_SHAPES), len(RUNS)), np.int64)
for i, (N_b, T_b) in enumerate(T2M_SHAPES):
    L, mels = bucket_inputs(B, N_b, T_b, INPUT_SEED)
    for j, (seed, rate) in enumerate(RUNS):
        ref_hp.Hyperparams.dropout_rate = rate
        losses, calls = tf_shim.run_train_graph(L, mels, lambda x, r, k, seed=seed: x * rtr.dropout_keep(x.shape, k, seed, r))
        t2m_losses[i, j] = [losses[k] for k in T2M_KEYS]
        t2m_calls[i, j] = calls
        print("text2mel N_b=%d T_b=%d rate=%.2f: %s" % (N_b, T_b, rate, losses), flush=True)
ssrn_losses, ssrn_calls = np.zeros((len(SSRN_T), len(RUNS), 3)), np.zeros((len(SSRN_T), len(RUNS)), np.int64)
for i, T_b in enumerate(SSRN_T):
    mels, mags = ssrn_inputs(B, T_b, INPUT_SEED)
    for j, (seed, rate) in enumerate(RUNS):
        ref_hp.Hyperparams.dropout_rate = rate
        losses, calls = tf_shim.run_train_graph_ssrn(mels, mags, lambda x, r, k, seed=seed: x * rtr.dropout_keep(x.shape, k, seed, r))
        ssrn_losses[i, j] = [losses[k] for k in SSRN_KEYS]
        ssrn_calls[i, j] = calls
        print("ssrn T_b=%d rate=%.2f: %s" % (T_b, rate, losses), flush=True)
ref_hp.Hyperparams.dropout_rate = rate0

np.savez_compressed(os.path.join(HERE, "refshim_train_buckets.npz"),
                    B=np.array(B), input_seed=np.array(INPUT_SEED),
                    t2m_shapes=np.array(T2M_SHAPES), ssrn_T=np.array(SSRN_T),
                    seeds=np.array([s for s, _ in RUNS]), rates=np.array([r for _, r in RUNS]),
                    t2m_losses=t2m_losses, t2m_dropout_calls=t2m_calls,
                    ssrn_losses=ssrn_losses, ssrn_dropout_calls=ssrn_calls)
print("written %s" % os.path.join(HERE, "refshim_train_buckets.npz"))
