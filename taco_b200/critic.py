"""Host-side mirror of the critic branch of ``PPO_ActorCritic`` for rollout inference.

Mirrors (IsaacGymEnvs/algorithms/nets_asymmetry.py), in the configuration the reference trains with
(README.md:60-66: ``--use_critic_encoder=True --critic_encoder_type=LSTM --lenStates=5``):
  * ``LSTMEncoder.forward``                  :128-136  (``nn.LSTM(26, H, num_layers, batch_first=True)``, output ``x[:, -1, :]``)
  * ``MLP.forward`` with Identity output     :23-39, :318
  * ``PPO_ActorCritic.act`` (critic branch)  :350-352  ``value = critic_mlp(critic_encoder(critic_input))``

The math runs in libtaco_b200.so (FP32 CUDA-core kernel, or the tcgen05 bf16 kernel with ``tensor_cores=True``); torch only
provides device memory and the stream.  No CPU fallback.  The tcgen05 kernel takes 1 to 4 stacked LSTM layers (one launch per
layer over chunks of the batch); ``tensor_cores_available`` says whether it takes this critic's shape.  A stacked critic's
workspace belongs to the handle, so one handle runs one ``forward`` at a time.
"""
import ctypes as C

import numpy as np
import torch

from . import _capi
from .actor import _as_f32, _ptr


def _np(t):
    return np.ascontiguousarray(t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else t, dtype=np.float32)


class CriticLSTM:
    def __init__(self, input_size, seq_len, lstm_hidden, mlp_hidden, lstm_layers=1, device="cuda:0"):
        if not torch.cuda.is_available():
            raise RuntimeError("CUDA is not available: the critic kernels have no CPU fallback")
        dev = torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError(f"CriticLSTM runs on CUDA only (got {device!r})")
        self.device_id = dev.index if dev.index is not None else 0
        self.device = f"cuda:{self.device_id}"
        self.input_size, self.seq_len = int(input_size), int(seq_len)
        self.lstm_hidden, self.lstm_layers = int(lstm_hidden), int(lstm_layers)
        self.mlp_sizes = [self.lstm_hidden] + [int(h) for h in mlp_hidden] + [1]
        self._lib = _capi.lib()
        arr = (C.c_int32 * len(self.mlp_sizes))(*self.mlp_sizes)
        h = C.c_void_p()
        _capi.check(self._lib.taco_critic_create(self.device_id, self.input_size, self.seq_len, self.lstm_hidden, self.lstm_layers,
                                                 arr, len(self.mlp_sizes), C.byref(h)), "taco_critic_create")
        self._h = h

    @property
    def n_mlp_layers(self):
        return len(self.mlp_sizes) - 1

    @property
    def tensor_cores_available(self):
        return bool(self._lib.taco_critic_tc_available(self._h))

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device_id).cuda_stream)

    def load(self, lstm_params, mlp_weights, mlp_biases):
        """lstm_params: per LSTM layer (weight_ih (4H, in), weight_hh (4H, H), bias_ih (4H), bias_hh (4H)) in torch's nn.LSTM
        layout (gate blocks i, f, g, o), bottom layer first; mlp_weights[l] (out, in), mlp_biases[l] (out,) like nn.Linear."""
        if len(lstm_params) != self.lstm_layers or len(mlp_weights) != self.n_mlp_layers or len(mlp_biases) != self.n_mlp_layers:
            raise ValueError(f"expected {self.lstm_layers} LSTM layers and {self.n_mlp_layers} MLP layers")
        H = self.lstm_hidden
        flat = []
        for l, prm in enumerate(lstm_params):
            in_l = self.input_size if l == 0 else H
            w_ih, w_hh, b_ih, b_hh = (_as_f32(x, self.device_id) for x in prm)
            if tuple(w_ih.shape) != (4 * H, in_l) or tuple(w_hh.shape) != (4 * H, H) or tuple(b_ih.shape) != (4 * H,) or tuple(b_hh.shape) != (4 * H,):
                raise ValueError(f"LSTM layer {l}: expected weight_ih {(4 * H, in_l)}, weight_hh {(4 * H, H)}, biases {(4 * H,)}")
            flat += [w_ih, w_hh, b_ih, b_hh]
        ws, bs = [], []
        for l in range(self.n_mlp_layers):
            w, b = _as_f32(mlp_weights[l], self.device_id), _as_f32(mlp_biases[l], self.device_id)
            if tuple(w.shape) != (self.mlp_sizes[l + 1], self.mlp_sizes[l]) or tuple(b.shape) != (self.mlp_sizes[l + 1],):
                raise ValueError(f"MLP layer {l}: expected weight {(self.mlp_sizes[l + 1], self.mlp_sizes[l])}, bias {(self.mlp_sizes[l + 1],)}")
            ws.append(w); bs.append(b)
        lp = (C.c_void_p * len(flat))(*[_ptr(a) for a in flat])
        wp = (C.c_void_p * len(ws))(*[_ptr(a) for a in ws])
        bp = (C.c_void_p * len(bs))(*[_ptr(a) for a in bs])
        _capi.check(self._lib.taco_critic_load(self._h, lp, wp, bp, self._stream()), "taco_critic_load")

    def load_modules(self, critic_encoder, critic_mlp):
        """Load from reference-style modules: ``LSTMEncoder`` (its ``.layers`` nn.LSTM) and ``MLP`` (its ``.layers`` Sequential)."""
        lstm = critic_encoder.layers
        if lstm.bidirectional or not lstm.batch_first:
            raise ValueError("the critic kernels implement the unidirectional batch_first LSTM encoder")
        prm = [tuple(getattr(lstm, f"{nm}_l{l}") for nm in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")) for l in range(lstm.num_layers)]
        lin = [m for m in critic_mlp.layers if isinstance(m, torch.nn.Linear)]
        self.load(prm, [m.weight for m in lin], [m.bias for m in lin])

    def forward(self, states, tensor_cores=False, out=None):
        """value (N, 1) = critic_mlp(critic_encoder(states)); states (N, len_states, 26) float32 on the critic's device."""
        if states.device.type != "cuda" or (states.device.index or 0) != self.device_id:
            states = states.to(self.device)
        states = states.float().contiguous()
        if states.dim() != 3 or states.size(1) != self.seq_len or states.size(2) != self.input_size:
            raise ValueError(f"critic input must be (N, {self.seq_len}, {self.input_size}), got {tuple(states.shape)}")
        n = states.size(0)
        if out is None:
            out = torch.empty(n, 1, dtype=torch.float32, device=self.device)
        elif out.dtype != torch.float32 or not out.is_contiguous() or out.numel() != n or out.device.type != "cuda":
            raise ValueError("forward(out=...): contiguous float32 CUDA tensor of N values")
        _capi.check(self._lib.taco_critic_forward(self._h, C.c_void_p(states.data_ptr()), C.c_void_p(out.data_ptr()), n,
                                                  1 if tensor_cores else 0, self._stream()), "taco_critic_forward")
        return out

    __call__ = forward

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.taco_critic_destroy(self._h)
            self._h = C.c_void_p(0)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
