"""TEST INFRASTRUCTURE -- a minimal eager stand-in for the slice of the TensorFlow 1.x API that the
reference's synthesis graph touches, so that the reference's OWN source files (modules.py, networks.py,
train.py: Graph(mode="synthesize") of a checkout of the reference project) can be imported and executed
without TensorFlow.  make_golden_refshim.py uses it to record the refshim_*.npz fixtures.

What this pins and what it does not:
  * pinned: everything the reference's Python decides -- layer order and counts, kernel sizes, dilation
    schedules, paddings, activations, the highway mix, the one-frame shift of the decoder input, the attention
    window mask, scope nesting and therefore every variable NAME and SHAPE (the store below rejects any name
    the graph asks for that SURVEY.md App. C / dc_tts_b200.arch.param_shapes() does not list, and reports
    names that were never asked for).
  * not pinned: the numerical semantics of the TF ops themselves (conv1d SAME/dilated padding,
    conv2d_transpose SAME stride 2, contrib layer_norm eps = 1e-12, softmax, ...), which are restated here from
    TF's documentation a third time (independently of oracle/ref_numpy.py and oracle/ref_torch.py: this file
    uses tap-wise numpy matmuls).  Parity therefore stays "unpinned" at the op level.

Execution model: eager.  `tf.placeholder` returns the next value of a feed queue, so a graph is evaluated by
constructing the reference's Graph object once per `run` (the constructor IS the graph definition);
variables live in a name -> array store that persists across constructions.
"""
import contextlib
import sys
import types

import numpy as np


class T(np.ndarray):
    """ndarray with the two static-shape calls the reference makes."""

    class _Shape(tuple):
        def as_list(self):
            return list(self)

    def get_shape(self):
        return T._Shape(self.shape)


def _t(x, dtype=None):
    return np.asarray(x, dtype=dtype).view(T)


class Store:
    """Variables by full TF name.  Strict: unknown names and shape mismatches raise."""

    def __init__(self, values):
        self.values = {k: np.asarray(v) for k, v in values.items()}
        self.requested = set()
        self.requested_shapes = {}          # name -> the shape the graph asked for (None: it named no shape)

    def get(self, name, shape=None):
        if name not in self.values:
            raise KeyError("the reference graph asked for variable %r, which the parameter schema does not list" % name)
        v = self.values[name]
        if shape is not None and tuple(int(s) for s in shape) != v.shape:
            raise ValueError("variable %s: graph wants shape %s, store has %s" % (name, tuple(shape), v.shape))
        self.requested.add(name)
        self.requested_shapes[name] = None if shape is None else tuple(int(s) for s in shape)
        return _t(v)


class _State:
    store = None
    scope = []
    feeds = []
    layer_counts = {}
    dropout_hook = None
    dropout_calls = 0


def _full(name):
    return "/".join(_State.scope + [name])


@contextlib.contextmanager
def variable_scope(name_or_scope, default_name=None, reuse=None):
    name = name_or_scope if name_or_scope is not None else default_name
    _State.scope.append(name)
    try:
        yield name
    finally:
        _State.scope.pop()


def get_variable(name, dtype=None, shape=None, initializer=None, trainable=True):
    return _State.store.get(_full(name), shape)


def placeholder(dtype, shape=None, name=None):
    if not _State.feeds:
        raise RuntimeError("tf.placeholder: no feed value queued")
    return _t(_State.feeds.pop(0), dtype)


def Variable(initial_value, name=None, trainable=True, dtype=None):
    return _t(initial_value)


# ---- tf.layers ----------------------------------------------------------------------------
def _layer_scope(base):
    """tf.layers names a layer `base`, `base_1`, ... per enclosing scope; the reference wraps every layer in its
    own variable_scope, so a second layer of the same kind in one scope would be a bug worth hearing about."""
    key = ("/".join(_State.scope), base)
    n = _State.layer_counts.get(key, 0)
    _State.layer_counts[key] = n + 1
    return base if n == 0 else "%s_%d" % (base, n)


def layers_conv1d(inputs, filters, kernel_size, dilation_rate=1, padding="valid", use_bias=True,
                  kernel_initializer=None, reuse=None, strides=1, activation=None, name=None):
    x = np.asarray(inputs, np.float32)
    B, L, cin = x.shape
    k, r = int(kernel_size), int(dilation_rate)
    with variable_scope(name or _layer_scope("conv1d")):
        W = np.asarray(get_variable("kernel", shape=(k, cin, filters)))
        b = np.asarray(get_variable("bias", shape=(filters,))) if use_bias else None
    if padding.lower() == "same":
        total = (k - 1) * r
        left = total // 2                      # TF SAME, stride 1: the extra cell goes to the right
        x = np.pad(x, [(0, 0), (left, total - left), (0, 0)])
    elif padding.lower() != "valid":
        raise ValueError(padding)
    Lout = x.shape[1] - (k - 1) * r
    y = np.zeros((B, Lout, filters), np.float32)
    for j in range(k):
        y += x[:, j * r:j * r + Lout, :] @ W[j]
    if b is not None:
        y += b
    return _t(y)


def layers_conv2d_transpose(inputs, filters, kernel_size, strides=(1, 1), padding="valid", activation=None,
                            kernel_initializer=None, use_bias=True, name=None):
    x = np.asarray(inputs, np.float32)
    B, H, Wd, cin = x.shape
    assert H == 1 and tuple(kernel_size) == (1, 3) and tuple(strides) == (1, 2) and padding.lower() == "same", \
        "the shim implements the one transposed convolution the reference uses"
    with variable_scope(name or _layer_scope("conv2d_transpose")):
        K = np.asarray(get_variable("kernel", shape=(1, 3, filters, cin)))          # (h, w, out, in)
        b = np.asarray(get_variable("bias", shape=(filters,))) if use_bias else None
    # gradient of a SAME, stride-2, width-3 convolution whose input had width 2*Wd: that forward pass pads one
    # cell on the RIGHT only, so its transpose scatters y[2t + j] += x[t] . K[j]^T and keeps columns [0, 2*Wd)
    full = np.zeros((B, 2 * Wd + 1, filters), np.float32)
    for j in range(3):
        full[:, j:j + 2 * Wd:2, :] += x[:, 0] @ K[0, j].T
    y = full[:, :2 * Wd, :]
    if b is not None:
        y = y + b
    return _t(y[:, None])


def layers_dropout(inputs, rate=0.5, training=False, name=None):
    """Identity at inference.  In training TF draws from its own random stream, which cannot be reproduced: the
    caller plugs a deterministic mask in (`_State.dropout_hook(x, rate, call_index)`), so that the PLACEMENT and
    scaling of every dropout in the reference's graph is what gets exercised."""
    if not training or rate == 0:
        return inputs
    assert _State.dropout_hook is not None, "training-mode dropout needs a mask hook"
    out = _State.dropout_hook(np.asarray(inputs), rate, _State.dropout_calls)
    _State.dropout_calls += 1
    return _t(out)


def contrib_layer_norm(inputs, begin_norm_axis=1, begin_params_axis=-1, scope=None, reuse=None, center=True, scale=True):
    x = np.asarray(inputs, np.float32)
    assert begin_norm_axis in (-1, x.ndim - 1)
    with variable_scope(scope, "LayerNorm"):
        beta = np.asarray(get_variable("beta", shape=x.shape[-1:]))
        gamma = np.asarray(get_variable("gamma", shape=x.shape[-1:]))
    mean = x.mean(-1, keepdims=True, dtype=np.float32)
    var = ((x - mean) ** 2).mean(-1, keepdims=True, dtype=np.float32)           # tf.nn.moments
    inv = gamma / np.sqrt(var + np.float32(1e-12))                               # tf.nn.batch_normalization
    return _t(x * inv + (beta - mean * inv))


# ---- tf.* / tf.nn -------------------------------------------------------------------------
def sequence_mask(lengths, maxlen):
    return _t(np.arange(int(maxlen))[None, :] < np.asarray(lengths)[:, None])


def softmax(x, axis=-1, name=None):
    x = np.asarray(x, np.float32)
    e = np.exp(x - x.max(axis, keepdims=True))
    return _t(e / e.sum(axis, keepdims=True))


def sigmoid(x, name=None):
    x = np.asarray(x, np.float32)
    return _t(np.float32(1) / (np.float32(1) + np.exp(-x)))


def matmul(a, b, transpose_a=False, transpose_b=False):
    a, b = np.asarray(a), np.asarray(b)
    if transpose_a: a = np.swapaxes(a, -1, -2)
    if transpose_b: b = np.swapaxes(b, -1, -2)
    return _t(a @ b)


def install(store, reference_dir):
    """Registers the stand-in modules and puts the reference checkout `reference_dir` on sys.path.  Returns the
    `tensorflow` module."""
    _State.store = store
    tf = types.ModuleType("tensorflow")
    tf.float32, tf.int32, tf.int64, tf.string = np.float32, np.int32, np.int64, object
    tf.variable_scope = variable_scope
    tf.get_variable = get_variable
    tf.placeholder = placeholder
    tf.Variable = Variable
    tf.concat = lambda values, axis, name=None: _t(np.concatenate([np.asarray(v) for v in values], axis))
    tf.zeros = lambda shape, dtype=np.float32, name=None: _t(np.zeros(shape, dtype))
    tf.ones = lambda shape, dtype=np.float32, name=None: _t(np.ones(shape, dtype))
    tf.zeros_like = lambda x, **k: _t(np.zeros_like(np.asarray(x)))
    tf.ones_like = lambda x, **k: _t(np.ones_like(np.asarray(x)))
    tf.split = lambda x, n, axis=0, **k: [_t(p) for p in np.split(np.asarray(x), n, axis)]
    tf.expand_dims = lambda x, axis, **k: _t(np.expand_dims(np.asarray(x), axis))
    tf.squeeze = lambda x, axis=None, **k: _t(np.squeeze(np.asarray(x), axis))
    tf.transpose = lambda x, perm=None, **k: _t(np.transpose(np.asarray(x), perm))
    tf.tile = lambda x, multiples, **k: _t(np.tile(np.asarray(x), multiples))
    tf.where = lambda c, a, b, **k: _t(np.where(np.asarray(c), np.asarray(a), np.asarray(b)))
    tf.equal = lambda a, b, **k: _t(np.asarray(a) == b)
    tf.not_equal = lambda a, b, **k: _t(np.asarray(a) != b)
    tf.logical_or = lambda a, b, **k: _t(np.logical_or(np.asarray(a), np.asarray(b)))
    tf.to_float = lambda x, **k: np.float32(x) if np.isscalar(x) else _t(np.asarray(x, np.float32))
    tf.rsqrt = lambda x, **k: np.float32(1) / np.sqrt(np.float32(x)) if np.isscalar(x) else _t(1 / np.sqrt(np.asarray(x, np.float32)))
    tf.argmax = lambda x, axis=None, **k: _t(np.argmax(np.asarray(x), axis).astype(np.int64))
    tf.matmul = matmul
    tf.sequence_mask = sequence_mask
    tf.convert_to_tensor = lambda x, **k: _t(x)
    tf.abs = lambda x, **k: _t(np.abs(np.asarray(x)))
    tf.reduce_mean = lambda x, axis=None, **k: np.asarray(x).mean(axis, dtype=np.float64).astype(np.float32)
    tf.reduce_sum = lambda x, axis=None, **k: np.asarray(x).sum(axis, dtype=np.float64).astype(np.float32)
    tf.minimum = lambda a, b, **k: np.minimum(a, b)
    tf.clip_by_value = lambda x, lo, hi, **k: _t(np.clip(np.asarray(x), lo, hi))

    def _pad(x, paddings, mode="CONSTANT", constant_values=0, **k):
        return _t(np.pad(np.asarray(x), paddings, mode="constant", constant_values=constant_values))
    tf.pad = _pad

    class _Adam:                                     # the optimiser itself is not exercised under the shim
        def __init__(self, learning_rate=None, **k): self.learning_rate = learning_rate
        def compute_gradients(self, loss): return []
        def apply_gradients(self, gvs, global_step=None): return None
    tf.train = types.SimpleNamespace(AdamOptimizer=_Adam)
    def _bce(logits=None, labels=None, **k):
        x, z = np.asarray(logits, np.float32), np.asarray(labels, np.float32)
        return _t(np.maximum(x, 0) - x * z + np.log1p(np.exp(-np.abs(x))))          # TF's documented stable form
    tf.nn = types.SimpleNamespace(sigmoid_cross_entropy_with_logits=_bce, relu=lambda x, name=None: _t(np.maximum(np.asarray(x), 0)), sigmoid=sigmoid, softmax=softmax,
                                  embedding_lookup=lambda table, ids, **k: _t(np.asarray(table)[np.asarray(ids)]))
    tf.layers = types.SimpleNamespace(conv1d=layers_conv1d, conv2d_transpose=layers_conv2d_transpose, dropout=layers_dropout)
    tf.contrib = types.SimpleNamespace(layers=types.SimpleNamespace(layer_norm=contrib_layer_norm,
                                                                    variance_scaling_initializer=lambda *a, **k: None))
    tf.truncated_normal_initializer = lambda *a, **k: None
    tf.constant_initializer = lambda *a, **k: None
    tf.summary = types.SimpleNamespace(scalar=lambda *a, **k: None, image=lambda *a, **k: None, merge_all=lambda *a, **k: None)
    sys.modules["tensorflow"] = tf
    # the reference's utils.py imports these at module level; nothing on the synthesis graph calls into them
    for name in ("librosa", "matplotlib", "matplotlib.pyplot"):
        if name not in sys.modules:
            m = types.ModuleType(name)
            m.use = lambda *a, **k: None
            sys.modules[name] = m
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    if reference_dir not in sys.path:
        sys.path.insert(0, reference_dir)
    return tf


def run_graph(L, mels, prev_max_attentions, fetch=("Y", "max_attentions", "alignments")):
    """One `sess.run` of the reference's synthesis graph (synthesize.py:48-52): builds train.Graph with the three
    placeholders bound to these values and returns the requested attributes as plain arrays.  Unless Z is
    fetched, the SSRN call at train.py:77 is skipped (it does not feed back into Text2Mel and costs 20 GMAC)."""
    import train as ref_train                      # the reference's train.py
    _State.scope = []
    _State.layer_counts = {}
    _State.feeds = [np.asarray(L, np.int32), np.asarray(mels, np.float32), np.asarray(prev_max_attentions, np.int32)]
    real_ssrn = ref_train.SSRN
    if not any(k.startswith("Z") for k in fetch):
        ref_train.SSRN = lambda Y, training=True: (None, None)
    try:
        g = ref_train.Graph(mode="synthesize")
    finally:
        ref_train.SSRN = real_ssrn
    assert not _State.feeds
    return {k: np.asarray(getattr(g, k)) for k in fetch}


def run_ssrn(Y):
    """`sess.run(g.Z, {g.Y: Y})` (synthesize.py:57): feeding g.Y replaces AudioDec's output, so the fetched value is
    the reference's SSRN(Y) under the "SSRN" scope (train.py:76-77)."""
    import networks as ref_networks
    _State.scope = []
    _State.layer_counts = {}
    with variable_scope("SSRN"):
        Z_logits, Z = ref_networks.SSRN(_t(np.asarray(Y, np.float32)), training=False)
    return np.asarray(Z_logits), np.asarray(Z)


def synthesize(L, steps=None, with_ssrn=True):
    """The loop of the reference's synthesize.py:45-57 around the reference's graph."""
    import hyperparams as ref_hp
    hp = ref_hp.Hyperparams
    L = np.asarray(L, np.int32)
    steps = hp.max_T if steps is None else steps
    Y = np.zeros((len(L), hp.max_T, hp.n_mels), np.float32)
    prev = np.zeros((len(L),), np.int32)
    hist = np.zeros((len(L), steps), np.int32)
    out = None
    for j in range(steps):
        hist[:, j] = prev
        out = run_graph(L, Y, prev)
        Y[:, j, :] = out["Y"][:, j, :]
        prev = out["max_attentions"][:, j].astype(np.int32)
    Z = run_ssrn(Y)[1] if with_ssrn else None
    return {"Y": Y, "Z": Z, "p_hist": hist, "max_attentions": out["max_attentions"], "alignments": out["alignments"]}


def run_train_graph_ssrn(mels, mags, dropout_hook):
    """The reference's TRAINING graph for SSRN (train.py Graph(num=2, mode="train")): losses on a fixed batch."""
    import train as ref_train
    _State.scope = []
    _State.layer_counts = {}
    _State.dropout_hook = dropout_hook
    _State.dropout_calls = 0
    mels = _t(np.asarray(mels, np.float32)); mags = _t(np.asarray(mags, np.float32))
    real = ref_train.get_batch
    ref_train.get_batch = lambda: (_t(np.zeros((len(mels), 4), np.int32)), mels, mags, None, 1)
    try:
        g = ref_train.Graph(num=2, mode="train")
    finally:
        ref_train.get_batch = real
        _State.dropout_hook = None
    return {k: float(np.asarray(getattr(g, k))) for k in ("loss", "loss_mags", "loss_bd2")}, _State.dropout_calls


def run_train_graph(L, mels, dropout_hook):
    """The reference's TRAINING graph for Text2Mel (train.py Graph(num=1, mode="train")): get_batch() is replaced
    by the given fixed-size batch, the optimiser by a stub; returns the three losses and the total."""
    import train as ref_train
    _State.scope = []
    _State.layer_counts = {}
    _State.dropout_hook = dropout_hook
    _State.dropout_calls = 0
    L = _t(np.asarray(L, np.int32)); mels = _t(np.asarray(mels, np.float32))
    real = ref_train.get_batch
    ref_train.get_batch = lambda: (L, mels, None, None, 1)
    try:
        g = ref_train.Graph(num=1, mode="train")
    finally:
        ref_train.get_batch = real
        _State.dropout_hook = None
    return {k: float(np.asarray(getattr(g, k))) for k in ("loss", "loss_mels", "loss_bd1", "loss_att")}, _State.dropout_calls
