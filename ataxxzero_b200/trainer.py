"""The training side of the reference's ``model.Network`` (model.py:81-142) on the device: ``Trainer.train(minibatch, lr)``,
``Trainer.run_on_samples`` losses, ``Trainer.network()`` for ``save_model``.  Every FLOP runs in libataxxzero.so
(csrc/az_train.cu: tcgen05 forward conv / data gradient / weight gradient kernels, batch-norm and head kernels, momentum
update); this module only binds the C ABI."""
import ctypes as C

import numpy as np

from . import _native, model
from ._native import AZ_FEATURES, AZ_LOGITS, check, lib, register

_vp = C.c_void_p
register("az_trainer_create", C.c_int, [_vp, C.c_int, C.c_int, C.POINTER(_vp)])
register("az_trainer_destroy", None, [_vp])
register("az_trainer_load", C.c_int, [_vp, _vp, C.c_size_t])
register("az_trainer_step", C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_float, _vp])
register("az_trainer_set_games", C.c_int, [_vp, _vp, C.c_size_t])
register("az_trainer_step_picks", C.c_int, [_vp, _vp, _vp, C.c_int, C.c_float, _vp])
register("az_trainer_eval", C.c_int, [_vp, _vp, _vp, _vp, C.c_int, _vp, _vp, _vp])
register("az_trainer_export", C.c_int, [_vp, _vp, C.c_size_t])
register("az_trainer_launches", C.c_ulonglong, [_vp])
register("az_trainer_last_step_ms", C.c_float, [_vp])
register("az_trainer_debug_read", C.c_int, [_vp, C.c_char_p, C.c_int, C.c_int, _vp, C.c_size_t])


def _batch_arrays(features, policies, values):
    f = np.ascontiguousarray(features, dtype=np.int8)
    p = np.ascontiguousarray(policies, dtype=np.float32)
    v = np.ascontiguousarray(values, dtype=np.float32).reshape(-1)
    n = len(v)
    if f.size != n * AZ_FEATURES or p.size != n * AZ_LOGITS:
        raise ValueError("minibatch shapes disagree: features %r, policies %r, values %r" % (f.shape, p.shape, v.shape))
    return f, p, v, n


class Trainer:
    """``model.Network(scope, build_training=True)`` + its session (model.py:24-34,81-101)."""

    def __init__(self, ctx, network, max_batch=512):
        if network.filters != model.Network.FILTERS:
            raise ValueError("libataxxzero.so trains %d-filter networks, got %d" % (model.Network.FILTERS, network.filters))
        self.ctx = ctx
        self.blocks = network.blocks
        self.max_batch = int(max_batch)
        self._packed_size = network.packed().size
        self._h = _vp()
        check(lib().az_trainer_create(ctx.handle, self.max_batch, self.blocks, C.byref(self._h)))
        ctx.adopt(self)
        self.load(network)

    def load(self, network):
        """model.load_model into a fresh training graph: gamma = 1, beta = 0, momentum = 0 (train.py:112-120)."""
        packed = network.packed()
        check(lib().az_trainer_load(self._h, _vp(packed.ctypes.data), packed.size))

    def train(self, features, policies, values, learning_rate):
        """One ``network.train(minibatch, learning_rate)`` (model.py:116-127).  Returns (policy, value, regularisation) loss of
        the minibatch before the update."""
        f, p, v, n = _batch_arrays(features, policies, values)
        losses = np.zeros(3, dtype=np.float32)
        check(lib().az_trainer_step(self._h, _vp(f.ctypes.data), _vp(p.ctypes.data), _vp(v.ctypes.data), n, float(learning_rate), _vp(losses.ctypes.data)))
        return float(losses[0]), float(losses[1]), float(losses[2])

    def set_games(self, packed):
        """The games this run samples from (``train_data.pack_entries``): uploaded once, kept on the device."""
        words = np.ascontiguousarray(packed.words, dtype=np.uint32)
        check(lib().az_trainer_set_games(self._h, _vp(words.ctypes.data), words.size))

    def train_picks(self, offsets, meta, learning_rate):
        """One step on samples of the resident games (``train_data.draw_arrays``): sample extraction and the step run
        back to back on the device, nothing but the 12 bytes per sample of its description crosses the bus."""
        o = np.ascontiguousarray(offsets, dtype=np.uint64)
        m = np.ascontiguousarray(meta, dtype=np.uint32)
        if o.shape != m.shape or o.ndim != 1:
            raise ValueError("offsets %r and meta %r must be equally long vectors" % (o.shape, m.shape))
        losses = np.zeros(3, dtype=np.float32)
        check(lib().az_trainer_step_picks(self._h, _vp(o.ctypes.data), _vp(m.ctypes.data), len(o), float(learning_rate), _vp(losses.ctypes.data)))
        return float(losses[0]), float(losses[1]), float(losses[2])

    def losses(self, features, policies, values, outputs=False):
        """``run_on_samples(policy_loss.eval)`` / ``value_loss.eval`` (model.py:129-142): inference-mode batch-norm."""
        f, p, v, n = _batch_arrays(features, policies, values)
        losses = np.zeros(2, dtype=np.float32)
        logits = np.zeros((n, 7, 7, 17), dtype=np.float32) if outputs else None
        vals = np.zeros((n, 1), dtype=np.float32) if outputs else None
        check(lib().az_trainer_eval(self._h, _vp(f.ctypes.data), _vp(p.ctypes.data), _vp(v.ctypes.data), n, _vp(losses.ctypes.data),
                                    _vp(logits.ctypes.data) if outputs else None, _vp(vals.ctypes.data) if outputs else None))
        if outputs:
            return float(losses[0]), float(losses[1]), logits, vals
        return float(losses[0]), float(losses[1])

    def network(self):
        """The current weights + moving statistics as a ``model.Network`` (what ``save_model`` writes, model.py:173-183)."""
        packed = np.zeros(self._packed_size, dtype=np.float32)
        check(lib().az_trainer_export(self._h, _vp(packed.ctypes.data), packed.size))
        f, b = model.Network.FILTERS, self.blocks
        shapes = [(3, 3, 4, f)] + [(3, 3, f, f)] * (2 * b) + [(1, 1, f, model.MOVE_TYPES), (1, 1, f, 1), (49, 1), (1,)]
        conv, off = [], 0
        for shape in shapes:
            size = int(np.prod(shape))
            conv.append(packed[off:off + size].reshape(shape).copy())
            off += size
        bn = []
        for _ in range(2 * (1 + 2 * b)):
            bn.append(packed[off:off + f].copy())
            off += f
        assert off == packed.size
        return model.Network(conv, bn)

    @property
    def launches(self):
        return int(lib().az_trainer_launches(self._h))

    @property
    def last_step_ms(self):
        """Device time of the last step's kernels (CUDA events; minibatch already in HBM)."""
        return float(lib().az_trainer_last_step_ms(self._h))

    def debug_read(self, what, layer=0, n=0):
        """An internal tensor of the last step (test hook; az_train.cu, az_trainer_debug_read).  "z" / "act" / "d_h" take the
        first n boards as [n, 7, 7, F]: "z" is layer ``layer``'s conv output, "act" its input activation (``layer`` 0 the
        input features, ``layer`` = layers the tower output), "d_h" the gradient of the loss with respect to layer 0's
        output after a training step."""
        f = model.Network.FILTERS
        shape = {"z": (n, 7, 7, f), "act": (n, 7, 7, f), "d_h": (n, 7, 7, f), "grad_conv": (3, 3, f, f), "conv": (3, 3, f, f),
                 "grad_gamma": (f,), "grad_beta": (f,), "gamma": (f,), "beta": (f,), "moving": (2, f),
                 "grad_heads": (f * 17 + f + 49 + 1,)}[what]
        out = np.zeros(shape, dtype=np.float32)
        check(lib().az_trainer_debug_read(self._h, what.encode(), int(layer), int(n), _vp(out.ctypes.data), out.size))
        return out

    def close(self):
        if self._h:
            lib().az_trainer_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
