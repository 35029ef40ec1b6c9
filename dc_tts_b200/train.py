"""`Graph(mode="synthesize")` -- the object synthesize.py talks to
(/root/reference/train.py:21-80, synthesize branch :43-46, :48-68, :74-80).

The reference builds a symbolic TF graph and evaluates it with `sess.run(fetches,
feed_dict)`.  Here the attributes (`L, mels, prev_max_attentions, S, K, V, Q, R,
alignments, max_attentions, Y_logits, Y, Z_logits, Z, global_step`) are lightweight
symbols and `Session.run` evaluates them eagerly on the GPU, so that the reference's
loop (synthesize.py:47-57) runs unmodified in structure.  `Graph.generate` is the fast
path: the whole loop on the device, replayed from a CUDA graph.

`Graph(num, mode="train")` is the reference's training object (train.py:22-135): `num_batch`, `global_step`, `lr`, the
losses and `train_op` are fetchable with `Session.run` exactly as train.py:148 does (`sess.run([g.global_step,
g.train_op])`): fetching `train_op` takes the next batch of the input pipeline (data_load.get_batch -> here an iterator of
(L, mels, mags, ...) batches, dc_tts_b200/trainer.py: `bucketed_batches` as they come, or fixed-size batches) and runs ONE
optimiser step at that batch's own shape -- forward with dropout, the losses of train.py:83-113, backward, clipping, Adam
with the Noam rate (train.py:120-131) -- through `Engine.train_step` / `train_step_ssrn`.  A batch with more characters
than the engine's key capacity (Engine.KEY_CAPACITY) is skipped and counted in `skipped_batches`.  Plots and summaries
(train.py:100-104,116-119,154-157) are out of scope.
"""
import numpy as np
import torch

from .data_load import load_vocab
from .engine import get_engine
from .hyperparams import Hyperparams as hp
from .modules import variable_scope
from .networks import Attention, AudioDec, AudioEnc, SSRN, TextEnc


class Symbol:
    """Placeholder / fetchable node of the synthesize graph."""

    def __init__(self, graph, name):
        self.graph, self.name = graph, name

    def __repr__(self):
        return "<dc_tts_b200 graph tensor %s>" % self.name


_TEXT2MEL = ("S", "K", "V", "Q", "R", "alignments", "max_attentions", "Y_logits", "Y")
_FUSED_OK = {"Y", "max_attentions", "alignments", "global_step"}


_TRAIN = {1: ("loss", "loss_mels", "loss_bd1", "loss_att"), 2: ("loss", "loss_mags", "loss_bd2")}


class Graph:
    def __init__(self, num=1, mode="train", engine=None, fused=True, batches=None, num_batch=None, global_step=0):
        """mode "synthesize": the inference graph.  mode "train" (the reference default): `num` = 1 trains Text2Mel, 2 SSRN;
        `batches` is the input pipeline, an iterator of (L, mels, mags, ...) tuples, e.g. trainer.bucketed_batches(...)."""
        if mode not in ("train", "synthesize"):
            raise ValueError("mode: 'train' or 'synthesize' (train.py:22)")
        self.char2idx, self.idx2char = load_vocab()
        self.engine = engine or get_engine()
        self.fused = fused
        self.mode, self.num = mode, num
        if mode == "train":
            if num not in (1, 2):
                raise ValueError("num: 1 for Text2Mel, 2 for SSRN (train.py:24)")
            if batches is None:
                raise ValueError("Graph(mode='train') needs `batches`: the reference reads them from data_load.get_batch(); "
                                 "here pass trainer.bucketed_batches(...) or trainer.fixed_size_batches(...)")
            self.batches = iter(batches)
            self.num_batch = num_batch                       # train.py:33; only used for the progress bar
            self.global_step_value = int(global_step)
            self.last = {}
            self.skipped_batches = 0
            self._initialised = False
            for name in ("global_step", "train_op", "lr") + _TRAIN[num]:
                setattr(self, name, Symbol(self, name))
            return
        self.global_step_value = 0          # `gs/global_step` (train.py:79-80); no checkpoint offline
        for name in ("L", "mels", "prev_max_attentions") + _TEXT2MEL + ("Z_logits", "Z", "global_step"):
            setattr(self, name, Symbol(self, name))

    # ---------------------------------------------------------------- evaluation
    def _text2mel(self, L, mels, pma, want):
        """train.py:48-68 evaluated block by block through networks.py."""
        e = self.engine
        mels = e._f32(mels)
        vals = {}
        with variable_scope("Text2Mel"):
            vals["S"] = torch.cat((torch.zeros_like(mels[:, :1, :]), mels[:, :-1, :]), 1)     # train.py:51
            with variable_scope("TextEnc"):
                vals["K"], vals["V"] = TextEnc(L, training=False, fused=self.fused)
            with variable_scope("AudioEnc"):
                vals["Q"] = AudioEnc(vals["S"], training=False, fused=self.fused)
            with variable_scope("Attention"):
                vals["R"], vals["alignments"], vals["max_attentions"] = Attention(
                    vals["Q"], vals["K"], vals["V"], mononotic_attention=True, prev_max_attentions=pma)
            with variable_scope("AudioDec"):
                vals["Y_logits"], vals["Y"] = AudioDec(vals["R"], training=False, fused=self.fused)
        return vals

    def _train_run(self, names):
        """One `sess.run` of the training graph: fetching train_op consumes a batch and applies one update."""
        from .utils import learning_rate_decay
        if "train_op" in names:
            from .trainer import fits_key_capacity, key_capacity
            L, mels, mags = next(self.batches)[:3]
            while not fits_key_capacity(L, key_capacity(self.engine)):
                self.skipped_batches += 1
                L, mels, mags = next(self.batches)[:3]
            if not self._initialised:
                if self.num == 1:
                    self.engine.train_init(len(L))
                else:
                    self.engine.train_init_ssrn(len(L), mels.shape[1])
                self._initialised = True
            gs = self.global_step_value
            if self.num == 1:
                self.last = self.engine.train_step(L, mels, global_step=gs, seed=gs)
            else:
                self.last = self.engine.train_step_ssrn(mels, mags, global_step=gs, seed=gs)
            self.global_step_value = gs + 1                   # apply_gradients(global_step=...) increments (train.py:131)
        out = {"train_op": None, "global_step": np.int64(self.global_step_value),
               "lr": np.float32(learning_rate_decay(hp.lr, self.global_step_value))}
        for k in _TRAIN[self.num]:
            if k in names and k not in self.last:
                raise ValueError("%s: no training step has run yet (fetch it together with train_op)" % k)
            out[k] = np.float32(self.last.get(k, np.nan))
        return out

    def run(self, fetches, feed_dict=None, as_numpy=True):
        """`sess.run` equivalent.  Feeding `self.Y` cuts Text2Mel out of the evaluation,
        exactly as feeding g.Y does in the reference (synthesize.py:57)."""
        single = isinstance(fetches, Symbol)
        names = [fetches.name] if single else [f.name for f in fetches]
        if self.mode == "train":
            vals = self._train_run(names)
            out = [vals[n] for n in names]
            return out[0] if single else out
        feed = {k.name: v for k, v in (feed_dict or {}).items()}
        vals = dict(global_step=np.int64(self.global_step_value))
        need_t2m = any(n in _TEXT2MEL for n in names if n not in feed) or \
            (any(n in ("Z", "Z_logits") for n in names) and "Y" not in feed)
        if need_t2m:
            for k in ("L", "mels", "prev_max_attentions"):
                if k not in feed:
                    raise ValueError("placeholder %s must be fed" % k)
            if self.fused and set(names) <= _FUSED_OK:
                Y, M, A = self.engine.text2mel_forward(feed["L"], feed["mels"], feed["prev_max_attentions"],
                                                       want_alignments="alignments" in names)
                vals.update(Y=Y, max_attentions=M, alignments=A)
            else:
                vals.update(self._text2mel(feed["L"], feed["mels"], feed["prev_max_attentions"], names))
        vals.update(feed)
        if any(n in ("Z", "Z_logits") for n in names):
            with variable_scope("SSRN"):                                                      # train.py:74-77
                vals["Z_logits"], vals["Z"] = SSRN(vals["Y"], training=False, fused=self.fused)
        out = []
        for n in names:
            v = vals[n]
            if as_numpy and isinstance(v, torch.Tensor):
                v = v.cpu().numpy()
            out.append(v)
        return out[0] if single else out

    # ---------------------------------------------------------------- fast path
    def generate(self, L, steps=0):
        """synthesize.py:45-54 entirely on the device: returns the mel tensor Y
        (B, max_T, n_mels) as a CUDA tensor plus the prev_max_attentions history."""
        Y, P, _, _ = self.engine.text2mel_generate(L, steps)
        return Y, P


class Session:
    """Minimal stand-in for tf.Session used as `with Session() as sess: sess.run(...)`."""

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False

    def run(self, fetches, feed_dict=None):
        g = (fetches if isinstance(fetches, Symbol) else fetches[0]).graph
        return g.run(fetches, feed_dict)
