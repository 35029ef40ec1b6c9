"""The trainer loop around `Engine.train_step` / `train_step_ssrn` -- what `python train.py 1|2` does in the reference
(/root/reference/train.py:137-160: one optimiser step per batch, a checkpoint `model_gs_{NNN}k` every 1000 steps in
`hp.logdir + "-" + num`, stop after hp.num_iterations) on top of the LJ transcript parser of data_load.py:41-56 and the
pre-computed `mels/*.npy`, `mags/*.npy` of prepo.py (data_load.py:104-112).

Batching: `bucketed_batches` restates the reference's length-bucketed, dynamically padded queue (data_load.py:88-131:
shuffled stream, buckets by text length every 20 characters, a full bucket emits a batch padded to its own longest
member).  `train` takes those batches as they are and every step runs at the bucket's own shape, as the reference does:
TextEnc and the attention over the bucket's N_b characters, the audio networks over its T_b frames, the losses averaged
over that extent and the guided-attention term over the window n < min(N_b, max_N), t < min(T_b, max_T) (train.py:85-95);
the SSRN trainer follows each bucket's T_b.  A bucket whose text is longer than the engine's key capacity
(`Engine.KEY_CAPACITY`: 192 characters for hp.max_N <= 192, up to 512 as hp.max_N grows) is skipped and counted.
`fixed_size_batches` (plain shuffled batches) and `pad_to_fixed` (a bucket padded out to hp.max_N / hp.max_T) give the
fixed shapes (B, max_N) / (B, max_T, n_mels) / (B, 4 max_T, F) of BASELINE config 5.
"""
import codecs
import os

import numpy as np

from .arch import ATTENTION_KEY_CAPACITY
from .data_load import load_vocab, text_normalize
from .hyperparams import Hyperparams as hp


def load_train_data(data_dir=None):
    """data_load.py:41-56 (LJ Speech): transcript.csv -> (wav paths, text lengths, int32 id arrays ending in E)."""
    data_dir = data_dir or hp.data
    char2idx, _ = load_vocab()
    fpaths, text_lengths, texts = [], [], []
    for line in codecs.open(os.path.join(data_dir, "transcript.csv"), "r", "utf-8").readlines():
        fname, _, text = line.strip().split("|")
        ids = np.array([char2idx[ch] for ch in text_normalize(text) + "E"], np.int32)
        fpaths.append(os.path.join(data_dir, "wavs", fname + ".wav"))
        text_lengths.append(len(ids))
        texts.append(ids)
    return fpaths, text_lengths, texts


def _load_spectrograms_npy(fpath, mels_dir="mels", mags_dir="mags"):
    """data_load.py:105-109: what prepo.py wrote for this wav."""
    fname = os.path.basename(fpath)
    return fname, np.load(os.path.join(mels_dir, fname.replace("wav", "npy"))), np.load(os.path.join(mags_dir, fname.replace("wav", "npy")))


def fixed_size_batches(fpaths, texts, B=None, seed=0, loader=_load_spectrograms_npy, epochs=None, rank=0, world=1):
    """Shuffled batches of exactly B utterances, zero-padded to (B, max_N), (B, max_T, n_mels), (B, 4 max_T, F).
    Utterances that do not fit are skipped; an incomplete last batch of an epoch is dropped (num_batch = len // B,
    data_load.py:97).  Data-parallel runs: every rank draws the SAME permutation (same seed) and keeps every
    world-th utterance, so the ranks' batches are disjoint."""
    B = B or hp.B
    F = 1 + hp.n_fft // 2
    rng = np.random.default_rng(seed)
    epoch = 0
    while epochs is None or epoch < epochs:
        yielded = 0
        order = rng.permutation(len(fpaths))[rank::world]
        L = np.zeros((B, hp.max_N), np.int32)
        mels = np.zeros((B, hp.max_T, hp.n_mels), np.float32)
        mags = np.zeros((B, hp.max_T * hp.r, F), np.float32)
        names, n = [], 0
        for i in order:
            text = texts[i]
            if len(text) > hp.max_N:
                continue
            fname, mel, mag = loader(fpaths[i])
            if mel.shape[0] > hp.max_T or mag.shape[0] > hp.max_T * hp.r:
                continue
            L[n, :len(text)] = text
            mels[n, :mel.shape[0]] = mel
            mags[n, :mag.shape[0]] = mag
            names.append(fname)
            n += 1
            if n == B:
                yield L, mels, mags, names
                yielded += 1
                L = np.zeros_like(L); mels = np.zeros_like(mels); mags = np.zeros_like(mags)
                names, n = [], 0
        if yielded == 0:                          # ADVICE r1: never spin forever re-reading a data set that cannot fill a batch
            raise ValueError("fixed_size_batches: fewer than B=%d utterances fit max_N=%d / max_T=%d (of %d)"
                             % (B, hp.max_N, hp.max_T, len(fpaths)))
        epoch += 1


def bucket_boundaries(text_lengths):
    """data_load.py:125: `[i for i in range(minlen + 1, maxlen - 1, 20)]`."""
    return list(range(min(text_lengths) + 1, max(text_lengths) - 1, 20))


def bucket_index(length, boundaries):
    """tf.contrib.training.bucket_by_sequence_length: bucket k holds boundaries[k-1] <= length < boundaries[k]
    (bucket 0: length < boundaries[0]; the last bucket: length >= boundaries[-1])."""
    return int(np.searchsorted(np.asarray(boundaries), length, side="right"))


def bucketed_batches(fpaths, text_lengths, texts, B=None, seed=0, loader=_load_spectrograms_npy, epochs=None):
    """The reference's input pipeline (data_load.py:88-131) without TensorFlow queues: a shuffled stream of utterances
    (slice_input_producer :99) is routed by TEXT length into buckets (boundaries :125); a bucket that has collected B
    utterances emits them as one batch, every tensor padded with zeros to the longest member of THAT batch
    (dynamic_pad=True, :128): L (B, N_b) int32, mels (B, T_b, n_mels), mags (B, 4 T_b', F).  Buckets keep their partial
    contents across epochs like the TF queue does; nothing is dropped except what never fills a bucket.
    Yields (L, mels, mags, names, bucket); `train` takes them at that shape.  `pad_to_fixed` turns a batch into the fixed
    (max_N, max_T) shapes of BASELINE config 5."""
    B = B or hp.B
    bounds = bucket_boundaries(text_lengths)
    pending = [[] for _ in range(len(bounds) + 1)]
    rng = np.random.default_rng(seed)
    epoch = 0
    while epochs is None or epoch < epochs:
        emitted = 0
        for i in rng.permutation(len(fpaths)):
            k = bucket_index(text_lengths[i], bounds)
            fname, mel, mag = loader(fpaths[i])
            pending[k].append((texts[i], mel, mag, fname))
            if len(pending[k]) == B:
                items, pending[k] = pending[k], []
                N_b = max(len(t) for t, _, _, _ in items)
                T_b = max(m.shape[0] for _, m, _, _ in items)
                Tm_b = max(g.shape[0] for _, _, g, _ in items)
                L = np.zeros((B, N_b), np.int32)
                mels = np.zeros((B, T_b, hp.n_mels), np.float32)
                mags = np.zeros((B, Tm_b, items[0][2].shape[1]), np.float32)
                for b, (t, m, g, _) in enumerate(items):
                    L[b, :len(t)] = t; mels[b, :m.shape[0]] = m; mags[b, :g.shape[0]] = g
                emitted += 1
                yield L, mels, mags, [it[3] for it in items], k
        if emitted == 0 and epochs is None and epoch >= 64:
            raise ValueError("bucketed_batches: no bucket reaches B=%d utterances" % B)
        epoch += 1


def pad_to_fixed(L, mels, mags):
    """A bucketed batch in the fixed shapes of BASELINE config 5 ((B, max_N), (B, max_T, n_mels), (B, 4 max_T, F)),
    or None when the bucket is longer than those (the reference has no such limit while training; BASELINE config 5 fixes
    N = 180, T = 210).  Zero padding is what dynamic_pad already appended, just further."""
    B, N_b = L.shape
    T_b, Tm_b = mels.shape[1], mags.shape[1]
    if N_b > hp.max_N or T_b > hp.max_T or Tm_b > hp.max_T * hp.r:
        return None
    Lf = np.zeros((B, hp.max_N), np.int32); Lf[:, :N_b] = L
    mf = np.zeros((B, hp.max_T, mels.shape[2]), np.float32); mf[:, :T_b] = mels
    gf = np.zeros((B, hp.max_T * hp.r, mags.shape[2]), np.float32); gf[:, :Tm_b] = mags
    return Lf, mf, gf


def checkpoint_name(logdir, gs):
    """train.py:152."""
    return os.path.join(logdir, "model_gs_{}".format(str(gs // 1000).zfill(3) + "k"))


def fits_key_capacity(L, capacity=ATTENTION_KEY_CAPACITY):
    """Whether a batch's text fits `capacity` characters (an engine's KEY_CAPACITY)."""
    return np.shape(L)[1] <= capacity


def key_capacity(engine):
    """The engine's key capacity; ATTENTION_KEY_CAPACITY for an engine that does not report one."""
    return getattr(engine, "KEY_CAPACITY", ATTENTION_KEY_CAPACITY)


def train(num, engine, batches, num_iterations=None, logdir=None, global_step=None, save_every=1000, log=print, resume=True,
          rank=0, world=1, allreduce=None):
    """train.py:137-160 for num = 1 (Text2Mel) or 2 (SSRN).  `batches` yields (L, mels, mags, names) or the
    (L, mels, mags, names, bucket) of `bucketed_batches`, each step at its batch's own shape; a batch with more than
    the engine's KEY_CAPACITY characters is skipped (the next batch takes its step) and the number skipped is logged.
    `engine` is an `Engine` with parameters loaded.  Like tf.train.Supervisor (train.py:144), a `logdir` that already holds a checkpoint
    is RESUMED: variables, Adam slots and the global step come back from it (`resume=False` or an explicit `global_step`
    starts over).  Data parallel (BASELINE config 5, `world` > 1): every rank feeds its own disjoint `batches`, the step
    runs with apply=False, `allreduce` (default dc_tts_b200.parallel.allreduce_mean_) averages the flat gradient arena,
    every rank applies the identical Adam update, dropout masks differ per rank (seed = gs * world + rank) and only rank 0
    writes checkpoints; ranks may hold buckets of different shapes in the same step.  Returns the final global step."""
    if num not in (1, 2):
        raise ValueError("num: 1 for Text2Mel, 2 for SSRN (train.py:139)")
    num_iterations = hp.num_iterations if num_iterations is None else num_iterations
    logdir = logdir or (hp.logdir + "-" + str(num))
    os.makedirs(logdir, exist_ok=True)
    gs = int(global_step or 0)
    initialised = False
    skipped = 0
    capacity = key_capacity(engine)
    for batch in batches:
        L, mels, mags = batch[:3]
        if not fits_key_capacity(L, capacity):
            skipped += 1
            continue
        if not initialised:
            if num == 1:
                engine.train_init(len(L))
            else:
                engine.train_init_ssrn(len(L), mels.shape[1])
            if resume and global_step is None:
                restored = engine.restore_training(logdir, "Text2Mel" if num == 1 else "SSRN")
                if restored is not None:
                    gs = restored
                    log("resumed from %s at global step %d" % (logdir, gs))
            initialised = True
        if world > 1:
            if allreduce is None:
                from .parallel import allreduce_mean_ as allreduce
            seed = gs * world + rank
            if num == 1:
                losses = engine.train_step(L, mels, global_step=gs, seed=seed, apply=False)
            else:
                losses = engine.train_step_ssrn(mels, mags, global_step=gs, seed=seed, apply=False)
            allreduce(engine.train_grads())
            engine.train_apply(gs)
        elif num == 1:
            losses = engine.train_step(L, mels, global_step=gs, seed=gs)
        else:
            losses = engine.train_step_ssrn(mels, mags, global_step=gs, seed=gs)
        gs += 1                                   # apply_gradients(..., global_step=...) increments (train.py:131)
        if gs % save_every == 0 and rank == 0:    # train.py:151-152
            engine.save_checkpoint(checkpoint_name(logdir, gs), gs, "Text2Mel" if num == 1 else "SSRN")
            log("step %d  %s" % (gs, "  ".join("%s %.4f" % kv for kv in sorted(losses.items()))))
        if gs > num_iterations:                   # train.py:160
            break
    if skipped:
        log("skipped %d batches with more than %d characters (attention key capacity)" % (skipped, capacity))
    return gs
