"""Handle of the CUDA policy/value network (rz_net_* in include/rz_engine.h)."""
import ctypes as C

import numpy as np

from . import _cabi
from .agent import model as M

IMPL_AUTO, IMPL_GENERIC, IMPL_TCGEN05 = 0, 1, 2


class Net:
    def __init__(self, model_config, device=0):
        self.mc = model_config
        self.device = device
        self._h = C.c_void_p()
        cfg = _cabi.NetCfg(model_config.cnn_filter_num, model_config.res_layer_num, model_config.value_fc_size,
                           model_config.cnn_filter_size)
        _cabi.check(_cabi.lib().rz_net_create(C.byref(cfg), device, C.byref(self._h)), "rz_net_create")
        n = C.c_size_t()
        _cabi.check(_cabi.lib().rz_net_blob_size(self._h, C.byref(n)), "rz_net_blob_size")
        self.blob_floats = n.value
        assert self.blob_floats == M.blob_size(model_config)
        self.digest = None

    @property
    def handle(self):
        return self._h

    def load_blob(self, blob):
        blob = np.ascontiguousarray(blob, dtype=np.float32)
        _cabi.check(_cabi.lib().rz_net_load_weights(self._h, blob.ctypes.data_as(_cabi.f32p), blob.size), "rz_net_load_weights")
        self.digest = M.blob_digest(blob)

    def load_weights(self, weights):
        self.load_blob(M.weights_to_blob(self.mc, weights))

    def load_blob_dev(self, tensor, stream_ptr=None):
        """tensor: float32 CUDA tensor holding the blob (e.g. after torch.distributed.broadcast)."""
        _cabi.check(_cabi.lib().rz_net_load_weights_dev(self._h, C.c_void_p(tensor.data_ptr()), tensor.numel(), stream_ptr),
                    "rz_net_load_weights_dev")

    def predict_planes(self, planes, impl=IMPL_AUTO):
        """planes uint8 (N,2,8,8) host array -> policy (N,64) float32, value (N,) float32 (host)."""
        planes = np.ascontiguousarray(planes, dtype=np.uint8)
        n = planes.shape[0]
        policy = np.empty((n, 64), np.float32)
        value = np.empty((n,), np.float32)
        _cabi.check(_cabi.lib().rz_net_predict(self._h, planes.ctypes.data_as(_cabi.u8p), policy.ctypes.data_as(_cabi.f32p),
                                                value.ctypes.data_as(_cabi.f32p), n, impl), "rz_net_predict")
        return policy, value

    def predict_dev(self, own_t, enemy_t, policy_t, value_t, n, impl=IMPL_AUTO, stream_ptr=None):
        _cabi.check(_cabi.lib().rz_net_predict_dev(self._h, C.c_void_p(own_t.data_ptr()), C.c_void_p(enemy_t.data_ptr()),
                                                    C.c_void_p(policy_t.data_ptr()), C.c_void_p(value_t.data_ptr()), n, impl,
                                                    stream_ptr), "rz_net_predict_dev")

    def debug_tower_dev(self, own_t, enemy_t, policy_t, value_t, tower_t, n, stream_ptr=None):
        _cabi.check(_cabi.lib().rz_net_debug_tower_dev(self._h, C.c_void_p(own_t.data_ptr()), C.c_void_p(enemy_t.data_ptr()),
                                                        C.c_void_p(policy_t.data_ptr()), C.c_void_p(value_t.data_ptr()),
                                                        C.c_void_p(tower_t.data_ptr()), n, stream_ptr), "rz_net_debug_tower_dev")

    def debug_heads_dev(self, own_t, enemy_t, policy_t, value_t, logits_t, vlogit_t, n, tower_t=None, stream_ptr=None):
        """tcgen05 path with the head outputs before softmax / tanh (and optionally the fp32 tower output)"""
        _cabi.check(_cabi.lib().rz_net_debug_heads_dev(self._h, C.c_void_p(own_t.data_ptr()), C.c_void_p(enemy_t.data_ptr()),
                                                        C.c_void_p(policy_t.data_ptr()), C.c_void_p(value_t.data_ptr()),
                                                        C.c_void_p(tower_t.data_ptr()) if tower_t is not None else None,
                                                        C.c_void_p(logits_t.data_ptr()), C.c_void_p(vlogit_t.data_ptr()), n, stream_ptr),
                    "rz_net_debug_heads_dev")

    def close(self):
        if self._h:
            _cabi.lib().rz_net_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
