"""Engine: one libdctts_b200 handle bound to one GPU, driven with torch device tensors.

torch is used here for device memory and streams only; every computation goes through
the C-ABI (include/dctts.h).  This object plays the role of the reference's
`tf.Session` + restored variables (/root/reference/synthesize.py:28-41).
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from .hyperparams import Hyperparams as hp
from .params import check_params


class DcttsError(RuntimeError):
    pass


def _ptr(t):
    return C.c_void_p(0) if t is None else C.c_void_p(t.data_ptr())


class Engine:
    def __init__(self, device=0, hparams=hp):
        self._lib = _lib.load()
        if not torch.cuda.is_available():
            raise DcttsError("dc_tts_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.device = torch.device("cuda", device)
        self.hp = hparams
        self.F = 1 + hparams.n_fft // 2
        st = _lib.HParams(len(hparams.vocab), hparams.e, hparams.d, hparams.c, hparams.n_mels,
                          hparams.n_fft, hparams.max_N, hparams.max_T, hparams.attention_win_size, hparams.r)
        h = _lib.Handle()
        torch.cuda.init()
        with torch.cuda.device(self.device):
            torch.zeros(1, device=self.device)          # make sure the primary context exists
            rc = self._lib.dctts_create(C.byref(st), device, C.byref(h))
        if rc != 0:
            raise DcttsError("dctts_create: " + self._lib.dctts_last_error(None).decode())
        self._h = h
        self.params_loaded = False
        # characters per utterance every entry point of this handle takes: max(192, round_up(max_N, 64)) (include/dctts.h)
        self.KEY_CAPACITY = self.get_option("key_capacity")

    # ------------------------------------------------------------------ plumbing
    def close(self):
        if getattr(self, "_h", None):
            self._lib.dctts_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise DcttsError("%s: %s" % (what, self._lib.dctts_last_error(self._h).decode()))

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _f32(self, x):
        if isinstance(x, np.ndarray):
            x = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32))
        return x.to(device=self.device, dtype=torch.float32).contiguous()

    def _i32(self, x):
        if isinstance(x, np.ndarray):
            x = torch.from_numpy(np.ascontiguousarray(x, dtype=np.int32))
        return torch.as_tensor(x).to(device=self.device, dtype=torch.int32).contiguous()

    def _empty(self, *shape, dtype=torch.float32):
        return torch.empty(shape, device=self.device, dtype=dtype)

    # ------------------------------------------------------------------ parameters
    def stage_params(self, params):
        """Stage some variables (e.g. one of the two checkpoints of synthesize.py:31-41); commit_params() uploads."""
        for name, arr in params.items():
            a = np.ascontiguousarray(arr, dtype=np.float32)
            shape = (C.c_int64 * a.ndim)(*a.shape)
            self._check(self._lib.dctts_set_param(self._h, name.encode(), a.ctypes.data_as(C.c_void_p),
                                                   shape, a.ndim), "dctts_set_param(%s)" % name)

    def commit_params(self):
        """Fails (library error) when a variable of the path is missing or mis-shaped."""
        self._check(self._lib.dctts_commit_params(self._h), "dctts_commit_params")
        self.params_loaded = True
        return int(self._lib.dctts_num_params(self._h))

    def load_params(self, params):
        """Stage every variable (TF names, SURVEY.md App. C) and commit them to the device."""
        check_params(params)
        self.stage_params(params)
        return self.commit_params()

    def restore(self, text2mel_dir, ssrn_dir=None):
        """synthesize.py:31-41: the latest Text2Mel checkpoint of `<logdir>-1` and SSRN checkpoint of `<logdir>-2`
        (TF tensor bundles, read without TensorFlow by dc_tts_b200/checkpoint.py)."""
        from .checkpoint import Saver, latest_checkpoint
        Saver(var_list=["Text2Mel"]).restore(self, latest_checkpoint(text2mel_dir))
        Saver(var_list=["SSRN", "gs"]).restore(self, latest_checkpoint(ssrn_dir if ssrn_dir is not None else text2mel_dir))
        return self.commit_params()

    def set_tensor_path(self, mode):
        self._check(self._lib.dctts_set_tensor_path(self._h, int(mode)), "dctts_set_tensor_path")

    def set_option(self, name, value):
        """Kernel-variant switch (include/dctts.h: dctts_set_option), e.g. ("decode_mode", 0) for the graph-per-frame loop."""
        self._check(self._lib.dctts_set_option(self._h, name.encode(), int(value)), "dctts_set_option(%s)" % name)

    def get_option(self, name):
        v = C.c_int32(0)
        self._check(self._lib.dctts_get_option(self._h, name.encode(), C.byref(v)), "dctts_get_option(%s)" % name)
        return int(v.value)

    def decode_stats(self):
        """(frames with a receptive-field recompute summed over clusters, utterance-frames recomputed, clusters)."""
        a, b, c = C.c_int32(0), C.c_int32(0), C.c_int32(0)
        self._check(self._lib.dctts_decode_stats(self._h, C.byref(a), C.byref(b), C.byref(c)), "dctts_decode_stats")
        return int(a.value), int(b.value), int(c.value)

    def decode_profile(self):
        """Lap timers (SM cycles) of the last persistent decode run with option decode_prof = 1; see include/dctts.h."""
        v = (C.c_int64 * 14)()
        self._check(self._lib.dctts_decode_profile(self._h, v, 14), "dctts_decode_profile")
        names = ["start", "stream_wait", "gemv", "release", "gather", "cluster_barrier", "layernorm", "mix", "attention",
                 "re_attention", "re_gemm", "re_layernorm", "re_barriers", "frame"]
        return dict(zip(names, [int(x) for x in v]))

    def reserve(self, batch):
        self._check(self._lib.dctts_reserve(self._h, int(batch)), "dctts_reserve")

    def bench_block(self, scope, B, L, iters=5, warmup=2):
        """Mean device milliseconds of each kernel of one block (roofline leg of bench.py)."""
        ms = (C.c_float * 8)()
        n = C.c_int32(0)
        self._check(self._lib.dctts_bench_block(self._h, scope.encode(), B, L, iters, warmup, ms, C.byref(n),
                                                self._stream()), "dctts_bench_block")
        return [float(ms[i]) for i in range(n.value)]

    def launch_count(self):
        return int(self._lib.dctts_launch_count(self._h))

    # ------------------------------------------------------------------ building blocks
    def embed(self, scope, ids):
        ids = self._i32(ids)
        B, N = ids.shape
        out = self._empty(B, N, self.hp.e)
        self._check(self._lib.dctts_embed(self._h, scope.encode(), _ptr(ids), B, N, _ptr(out), self._stream()), "dctts_embed")
        return out

    def normalize(self, scope, x):
        x = self._f32(x)
        Cc = x.shape[-1]
        out = torch.empty_like(x)
        self._check(self._lib.dctts_normalize(self._h, scope.encode(), _ptr(x), x.numel() // Cc, Cc, _ptr(out),
                                              self._stream()), "dctts_normalize")
        return out

    def conv1d(self, scope, x, filters, rate=1, causal=False, act=0):
        x = self._f32(x)
        B, L, _ = x.shape
        out = self._empty(B, L, filters)
        self._check(self._lib.dctts_conv1d(self._h, scope.encode(), _ptr(x), B, L, rate, int(causal), act,
                                           _ptr(out), self._stream()), "dctts_conv1d")
        return out

    def hc(self, scope, x, rate=1, causal=False):
        x = self._f32(x)
        B, L, _ = x.shape
        out = torch.empty_like(x)
        self._check(self._lib.dctts_hc(self._h, scope.encode(), _ptr(x), B, L, rate, int(causal), _ptr(out),
                                       self._stream()), "dctts_hc")
        return out

    def conv1d_transpose(self, scope, x):
        x = self._f32(x)
        B, L, Cc = x.shape
        out = self._empty(B, 2 * L, Cc)
        self._check(self._lib.dctts_conv1d_transpose(self._h, scope.encode(), _ptr(x), B, L, _ptr(out),
                                                     self._stream()), "dctts_conv1d_transpose")
        return out

    # ------------------------------------------------------------------ networks
    def textenc(self, L):
        L = self._i32(L)
        B, N = L.shape
        if N != self.hp.max_N:
            raise DcttsError("TextEnc: text must be padded to max_N=%d (reference networks.py:145)" % self.hp.max_N)
        self._check_keys("textenc", N)
        K, V = self._empty(B, N, self.hp.d), self._empty(B, N, self.hp.d)
        self._check(self._lib.dctts_textenc(self._h, _ptr(L), B, _ptr(K), _ptr(V), self._stream()), "dctts_textenc")
        return K, V

    def audioenc(self, S):
        S = self._f32(S)
        B, T, _ = S.shape
        Q = self._empty(B, T, self.hp.d)
        self._check(self._lib.dctts_audioenc(self._h, _ptr(S), B, T, _ptr(Q), self._stream()), "dctts_audioenc")
        return Q

    def attention(self, Q, K, V, monotonic=False, prev_max_attentions=None):
        Q, K, V = self._f32(Q), self._f32(K), self._f32(V)
        B, T, d = Q.shape
        N = K.shape[1]
        pma = self._i32(prev_max_attentions) if monotonic else None
        R = self._empty(B, T, 2 * d)
        A = self._empty(B, N, T)
        M = self._empty(B, T, dtype=torch.int64)
        self._check(self._lib.dctts_attention(self._h, _ptr(Q), _ptr(K), _ptr(V), B, T, N, int(bool(monotonic)),
                                              _ptr(pma), _ptr(R), _ptr(A), _ptr(M), self._stream()), "dctts_attention")
        return R, A, M

    def audiodec(self, R):
        R = self._f32(R)
        B, T, _ = R.shape
        logits, Y = self._empty(B, T, self.hp.n_mels), self._empty(B, T, self.hp.n_mels)
        self._check(self._lib.dctts_audiodec(self._h, _ptr(R), B, T, _ptr(logits), _ptr(Y), self._stream()), "dctts_audiodec")
        return logits, Y

    def ssrn(self, Y, want_logits=True, out=None):
        """`out`: optional preallocated contiguous (B, 4T, F) float32 CUDA tensor (e.g. a slice of a gather buffer)."""
        Y = self._f32(Y)
        B, T, _ = Y.shape
        if out is not None:
            if tuple(out.shape) != (B, T * self.hp.r, self.F) or out.dtype != torch.float32 or not out.is_contiguous() \
                    or out.device != self.device:
                raise DcttsError("ssrn: `out` must be a contiguous float32 (B, 4T, F) tensor on this engine's device")
        Z = out if out is not None else self._empty(B, T * self.hp.r, self.F)
        logits = self._empty(B, T * self.hp.r, self.F) if want_logits else None
        self._check(self._lib.dctts_ssrn(self._h, _ptr(Y), B, T, _ptr(logits), _ptr(Z), self._stream()), "dctts_ssrn")
        return logits, Z

    # ------------------------------------------------------------------ graph level
    def text2mel_forward(self, L, mels, prev_max_attentions, want_alignments=True):
        L, mels, pma = self._i32(L), self._f32(mels), self._i32(prev_max_attentions)
        B = L.shape[0]
        if L.shape[1] != self.hp.max_N or mels.shape[1] != self.hp.max_T:
            raise DcttsError("synthesize graph needs N == max_N and T == max_T (reference networks.py:145)")
        self._check_keys("text2mel_forward", L.shape[1])
        Y = self._empty(B, self.hp.max_T, self.hp.n_mels)
        M = self._empty(B, self.hp.max_T, dtype=torch.int64)
        A = self._empty(B, self.hp.max_N, self.hp.max_T) if want_alignments else None
        self._check(self._lib.dctts_text2mel_forward(self._h, _ptr(L), _ptr(mels), _ptr(pma), B, _ptr(Y), _ptr(M),
                                                     _ptr(A), self._stream()), "dctts_text2mel_forward")
        return Y, M, A

    def text2mel_generate(self, L, steps=0, want_final_attention=False):
        L = self._i32(L)
        B = L.shape[0]
        Y = self._empty(B, self.hp.max_T, self.hp.n_mels)
        P = self._empty(B, self.hp.max_T, dtype=torch.int32)
        M = self._empty(B, self.hp.max_T, dtype=torch.int64) if want_final_attention else None
        A = self._empty(B, self.hp.max_N, self.hp.max_T) if want_final_attention else None
        self._check(self._lib.dctts_text2mel_generate(self._h, _ptr(L), B, int(steps), _ptr(Y), _ptr(P), _ptr(M),
                                                      _ptr(A), self._stream()), "dctts_text2mel_generate")
        return Y, P, M, A

    def spectrogram2wav(self, mag, n_iter=-1):
        """utils.py:67-94 for a batch: mag (B, T, F) in [0,1] -> (untrimmed wav (B, hop*(T-1)) CUDA tensor,
        trim (B, 2) int32 numpy [start, end) as librosa.effects.trim would keep)."""
        mag = self._f32(mag)
        if mag.dim() == 2:
            mag = mag[None]
        B, T, F = mag.shape
        h = self.hp
        self._check(self._lib.dctts_set_vocoder_params(self._h, h.hop_length, h.win_length, float(h.power), float(h.max_db),
                                                       float(h.ref_db), float(h.preemphasis), int(h.n_iter)),
                    "dctts_set_vocoder_params")
        wav = self._empty(B, h.hop_length * (T - 1))
        trim = np.zeros((B, 2), np.int32)
        self._check(self._lib.dctts_spectrogram2wav(self._h, _ptr(mag), B, T, int(n_iter), _ptr(wav),
                                                    trim.ctypes.data_as(C.c_void_p), self._stream()), "dctts_spectrogram2wav")
        return wav, trim

    def get_spectrograms(self, wav, sr=None):
        """utils.py:20-65 from a loaded waveform (1-D float32, hp.sr): -> (mel (T, n_mels), mag (T, F)) CUDA tensors and
        the [start, end) sample range librosa.effects.trim keeps."""
        h = self.hp
        wav = self._f32(wav).reshape(-1)
        n = wav.numel()
        self._check(self._lib.dctts_set_vocoder_params(self._h, h.hop_length, h.win_length, float(h.power), float(h.max_db),
                                                       float(h.ref_db), float(h.preemphasis), int(h.n_iter)),
                    "dctts_set_vocoder_params")
        cap = 1 + n // h.hop_length
        mel = self._empty(cap, h.n_mels)
        mag = self._empty(cap, self.F)
        t = C.c_int32(0)
        trim = (C.c_int32 * 2)()
        self._check(self._lib.dctts_get_spectrograms(self._h, _ptr(wav), n, int(sr or h.sr), _ptr(mel), _ptr(mag), cap,
                                                     C.byref(t), trim, self._stream()), "dctts_get_spectrograms")
        return mel[:t.value], mag[:t.value], (int(trim[0]), int(trim[1]))

    # ------------------------------------------------------------------ training step (BASELINE config 5)
    def train_init(self, B, dropout_rate=None):
        """Allocates the training workspace for batches of B utterances (train.py mode "train", num=1)."""
        rate = self.hp.dropout_rate if dropout_rate is None else dropout_rate
        self._check(self._lib.dctts_train_init(self._h, int(B), float(rate)), "dctts_train_init")

    def _check_keys(self, what, N):
        if N > self.KEY_CAPACITY:
            raise DcttsError("%s: N = %d characters exceeds the attention kernels' key capacity (%d)" % (what, N, self.KEY_CAPACITY))

    def train_step(self, L, mels, global_step=0, seed=0, lr=None, apply=True):
        """One Text2Mel optimiser step on L (B, N) int32 / mels (B, T, n_mels): forward with dropout, losses
        (train.py:83-99), backward, clip, Adam (train.py:122-132).  Returns {loss, loss_mels, loss_bd1, loss_att}.
        (max_N, max_T) batches run the fixed-shape step; any other shape -- a length bucket of `bucketed_batches`, as the
        reference trains on them -- runs at its own extent (N <= KEY_CAPACITY; the workspace grows as needed)."""
        L = self._i32(L); mels = self._f32(mels)
        if L.dim() != 2 or mels.dim() != 3 or mels.shape[0] != L.shape[0] or mels.shape[2] != self.hp.n_mels:
            raise DcttsError("train_step: L must be (B, N) and mels (B, T, n_mels); got %s, %s" % (tuple(L.shape), tuple(mels.shape)))
        B, N = L.shape
        T = mels.shape[1]
        self._check_keys("train_step", N)
        out = (C.c_float * 4)()
        args = (int(global_step), int(seed) & 0xffffffff, float(self.hp.lr if lr is None else lr), 1 if apply else 0, out, self._stream())
        if (N, T) == (self.hp.max_N, self.hp.max_T):
            self._check(self._lib.dctts_train_step(self._h, _ptr(L), _ptr(mels), B, *args), "dctts_train_step")
        else:
            self._check(self._lib.dctts_train_step_shaped(self._h, _ptr(L), N, _ptr(mels), T, B, *args), "dctts_train_step_shaped")
        return {"loss": out[0], "loss_mels": out[1], "loss_bd1": out[2], "loss_att": out[3]}

    def train_init_ssrn(self, B, T=None, dropout_rate=None):
        """Training workspace for the SSRN trainer (train.py num=2): mels (B, T, n_mels) -> mags (B, 4T, F).
        Measured parity: all 80 gradient tensors within 6e-6 of the autograd checker's (DESIGN.md 8e)."""
        rate = self.hp.dropout_rate if dropout_rate is None else dropout_rate
        self._check(self._lib.dctts_train_init_ssrn(self._h, int(B), int(self.hp.max_T if T is None else T), float(rate)),
                    "dctts_train_init_ssrn")
        self._ssrn_T = int(self.hp.max_T if T is None else T)

    def train_step_ssrn(self, mels, mags, global_step=0, seed=0, lr=None, apply=True):
        """One SSRN optimiser step on ground-truth mels (B, T, n_mels) / mags (B, 4T, F) (train.py:69-72,100-108,122-132).
        The T given to train_init_ssrn runs the fixed-shape step; any other T runs at its own extent."""
        mels = self._f32(mels); mags = self._f32(mags)
        if mels.dim() != 3 or mags.dim() != 3 or mags.shape[0] != mels.shape[0] or mels.shape[2] != self.hp.n_mels \
                or mags.shape[2] != self.F or mags.shape[1] != self.hp.r * mels.shape[1]:
            raise DcttsError("train_step_ssrn: mels must be (B, T, n_mels) and mags (B, %d T, %d); got %s, %s"
                             % (self.hp.r, self.F, tuple(mels.shape), tuple(mags.shape)))
        B, T = mels.shape[0], mels.shape[1]
        out = (C.c_float * 4)()
        args = (int(global_step), int(seed) & 0xffffffff, float(self.hp.lr if lr is None else lr), 1 if apply else 0, out, self._stream())
        if T == getattr(self, "_ssrn_T", None):
            self._check(self._lib.dctts_train_step_ssrn(self._h, _ptr(mels), _ptr(mags), B, *args), "dctts_train_step_ssrn")
        else:
            self._check(self._lib.dctts_train_step_ssrn_shaped(self._h, _ptr(mels), _ptr(mags), B, T, *args), "dctts_train_step_ssrn_shaped")
        return {"loss": out[0], "loss_mags": out[1], "loss_bd2": out[2]}

    def train_reserve(self, N, T):
        """Pre-size the training workspace for steps up to N characters and T mel frames (SSRN: N is ignored), so that
        no later bucket has to grow it.  Growing never loses the variables, gradients or Adam moments.  On a Text2Mel
        handle an N above KEY_CAPACITY raises DcttsError (library check)."""
        self._check(self._lib.dctts_train_reserve(self._h, int(N), int(T)), "dctts_train_reserve")

    def train_apply(self, global_step, lr=None):
        self._check(self._lib.dctts_train_apply(self._h, int(global_step), float(self.hp.lr if lr is None else lr), self._stream()),
                    "dctts_train_apply")

    def train_grads(self):
        """The flat float32 gradient arena as a CUDA tensor sharing the library's memory (all-reduce it in a
        data-parallel job between train_step(apply=False) and train_apply)."""
        ptr, n = C.c_void_p(), C.c_int64(0)
        self._check(self._lib.dctts_train_grads(self._h, C.byref(ptr), C.byref(n)), "dctts_train_grads")

        class _View:
            __cuda_array_interface__ = {"shape": (n.value,), "typestr": "<f4", "data": (ptr.value, False), "version": 2}
        return torch.as_tensor(_View(), device=self.device)

    def train_tensor(self, name, what="param"):
        """Copy of a Text2Mel variable / its gradient / Adam m / v, in the TF variable's shape."""
        from .arch import param_shapes
        shape = param_shapes()[name]
        out = np.empty(shape, np.float32)
        self._check(self._lib.dctts_train_tensor(self._h, name.encode(), {"param": 0, "grad": 1, "m": 2, "v": 3}[what],
                                                 out.ctypes.data_as(C.c_void_p), out.size), "dctts_train_tensor(%s)" % name)
        return out

    def train_set_tensor(self, name, array, what="param"):
        """Upload a variable / Adam m / Adam v of the network being trained from the TF layout (resume)."""
        from .arch import param_shapes
        a = np.ascontiguousarray(array, dtype=np.float32)
        if tuple(a.shape) != tuple(param_shapes()[name]):
            raise DcttsError("train_set_tensor(%s): shape %s, expected %s" % (name, a.shape, param_shapes()[name]))
        self._check(self._lib.dctts_train_set_tensor(self._h, name.encode(), {"param": 0, "m": 2, "v": 3}[what],
                                                     a.ctypes.data_as(C.c_void_p), a.size), "dctts_train_set_tensor(%s)" % name)

    def restore_training(self, logdir, scope="Text2Mel"):
        """What tf.train.Supervisor does when `logdir` already holds a checkpoint (train.py:144): every variable of the
        network being trained, its Adam slots (`<name>/Adam`, `<name>/Adam_1`) and `gs/global_step` come back from the
        latest bundle, so a restarted run continues the Noam schedule and the Adam state instead of overwriting
        model_gs_001k from scratch.  Call after train_init / train_init_ssrn.  Returns the restored global step, or None
        when the directory holds no checkpoint."""
        from .arch import param_shapes
        from .checkpoint import latest_checkpoint, list_variables, load_checkpoint
        path = latest_checkpoint(logdir)
        if path is None:
            return None
        avail = {n for n, _, _ in list_variables(path)}
        names = [n for n in param_shapes() if n.startswith(scope + "/")]
        missing = [n for n in names if n not in avail]
        if missing:
            raise DcttsError("restore_training: %s lacks %s" % (path, ", ".join(missing[:3])))
        for n in names:
            want = [n] + [n + sfx for sfx in ("/Adam", "/Adam_1") if n + sfx in avail]
            t = load_checkpoint(path, want)
            self.train_set_tensor(n, t[n], "param")
            if n + "/Adam" in t:
                self.train_set_tensor(n, t[n + "/Adam"], "m")
            if n + "/Adam_1" in t:
                self.train_set_tensor(n, t[n + "/Adam_1"], "v")
        gs = 0
        if "gs/global_step" in avail:
            gs = int(load_checkpoint(path, ["gs/global_step"])["gs/global_step"])
        return gs

    def save_checkpoint(self, prefix, global_step, scope="Text2Mel"):
        """What `sv.saver.save(sess, logdir + '/model_gs_...')` writes at train.py:152 for the network being trained
        (`scope` "Text2Mel" or "SSRN"): every variable of the scope, its Adam slots (`<name>/Adam`, `<name>/Adam_1`),
        the optimiser's `beta1_power` / `beta2_power` (TF's Adam keeps beta^t as variables; a TF train-graph
        Saver.restore expects them) and `gs/global_step`, as a TF tensor bundle."""
        from .arch import param_shapes
        from .checkpoint import save_checkpoint
        out = {"gs/global_step": np.array(global_step, np.int32),
               "beta1_power": np.array(0.9 ** (global_step + 1), np.float32),      # after t applies TF holds beta^(t+1)
               "beta2_power": np.array(0.999 ** (global_step + 1), np.float32)}
        for name in param_shapes():
            if name.startswith(scope + "/"):
                out[name] = self.train_tensor(name, "param")
                out[name + "/Adam"] = self.train_tensor(name, "m")
                out[name + "/Adam_1"] = self.train_tensor(name, "v")
        return save_checkpoint(prefix, out)

    def save_text2mel_checkpoint(self, prefix, global_step):
        return self.save_checkpoint(prefix, global_step, "Text2Mel")

    def synthesize_host(self, L_host, Y_host=None, Z_host=None):
        """synthesize.py:45-57 with host (ideally pinned) tensors in and out."""
        L_host = torch.as_tensor(L_host, dtype=torch.int32).contiguous()
        B = L_host.shape[0]
        if Z_host is None:
            Z_host = torch.empty((B, self.hp.max_T * self.hp.r, self.F), dtype=torch.float32).pin_memory()
        if Y_host is None:
            Y_host = torch.empty((B, self.hp.max_T, self.hp.n_mels), dtype=torch.float32).pin_memory()
        self._check(self._lib.dctts_synthesize_host(self._h, _ptr(L_host), B, _ptr(Y_host), _ptr(Z_host)),
                    "dctts_synthesize_host")
        return Y_host, Z_host


_default = None


def get_engine():
    """The process-wide default engine (used by modules.py / networks.py wrappers)."""
    global _default
    if _default is None:
        import os
        _default = Engine(int(os.environ.get("LOCAL_RANK", "0")))
    return _default


def set_engine(e):
    global _default
    _default = e
    return e
