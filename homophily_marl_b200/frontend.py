"""Fused observation front end (SURVEY 8f row f2): u8 obs planes -> conv3x3(3->6)+LeakyReLU -> Linear(->32)+LeakyReLU.

Forward-only replacement, for rollouts, of ``HomophilyAgent.rgb_preprocess`` (src/modules/agents/homophily_agent.py:19-27,
213-214) consuming the env's u8 observation buffer directly (``ssd_frontend_forward``: conv on the CUDA cores, the Linear on
tcgen05 tensor cores with a tf32 hi/lo split and fp32 accumulation in TMEM).  The learner keeps the reference's autograd
module; ``attach_to_mac`` only reroutes the no-grad rollout calls.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _capi


class ObsFrontEnd:
    def __init__(self, conv_w, conv_b, fc_w, fc_b, view, negative_slope=0.01, device="cuda:0"):
        if not torch.cuda.is_available():
            raise RuntimeError("ObsFrontEnd needs a CUDA device (sm_100a); there is no CPU fallback")
        device = torch.device(device)
        self.device = torch.device("cuda", device.index if device.index is not None else torch.cuda.current_device())
        self.view, self.N, self.P = int(view), 2 * int(view) + 1, 2 * int(view) - 1
        arrs = [np.ascontiguousarray(torch.as_tensor(t).detach().cpu().numpy(), dtype=np.float32) for t in (conv_w, conv_b, fc_w, fc_b)]
        if arrs[0].shape != (6, 3, 3, 3) or arrs[1].shape != (6,) or arrs[2].shape != (32, 6 * self.P * self.P) or arrs[3].shape != (32,):
            raise ValueError("expected Conv2d(3,6,3) and Linear(6*(N-2)^2, 32) parameters (config/default.yaml defaults)")
        self.lib = _capi.load()
        self._h = C.c_void_p()
        _capi.check(self.lib.ssd_frontend_create(self.view, arrs[0].ctypes.data, arrs[1].ctypes.data, arrs[2].ctypes.data,
                                                 arrs[3].ctypes.data, float(negative_slope), self.device.index, C.byref(self._h)))

    @classmethod
    def from_module(cls, conv_to_fc, view, device=None):
        """conv_to_fc: the reference's nn.Sequential(Conv2d, LeakyReLU, Flatten, Linear, LeakyReLU)."""
        conv, act, fc = conv_to_fc[0], conv_to_fc[1], conv_to_fc[3]
        device = device or conv.weight.device
        return cls(conv.weight, conv.bias, fc.weight, fc.bias, view, negative_slope=getattr(act, "negative_slope", 0.01), device=device)

    def _buffers(self, obs_buf, rows, agent_stride, out):
        """Validates the obs buffer and ``out`` of one forward; returns ``out`` (allocated when None)."""
        if obs_buf.dtype != torch.uint8 or not obs_buf.is_cuda or not obs_buf.is_contiguous():
            raise ValueError("obs_buf must be a contiguous uint8 CUDA tensor")
        if obs_buf.device != self.device:
            raise ValueError(f"obs_buf is on {obs_buf.device}, the front end on {self.device}")
        if obs_buf.numel() < rows * agent_stride:
            raise ValueError("obs_buf is smaller than rows * agent_stride")
        if out is None:
            return torch.empty((rows, 32), dtype=torch.float32, device=self.device)
        if (not isinstance(out, torch.Tensor) or out.dtype != torch.float32 or out.device != self.device
                or tuple(out.shape) != (rows, 32) or not out.is_contiguous()):
            raise ValueError(f"out must be a contiguous float32 tensor of shape ({rows}, 32) on {self.device}")
        return out

    def forward(self, obs_buf: torch.Tensor, rows: int, agent_stride: int, plane_stride: int, row_stride: int, out=None):
        """obs_buf: u8 CUDA buffer holding `rows` agent views `agent_stride` bytes apart.  Returns f32 [rows, 32].

        One launch on the current stream of the handle's device.  The handle owns the scratch of tiles shared between CTAs, so
        it must not run on two streams at once: concurrent callers (env ranges) each hold their own handle."""
        rows = int(rows)
        out = self._buffers(obs_buf, rows, agent_stride, out)
        if rows == 0:                                         # nothing to launch (an empty tensor may have no storage)
            return out
        with torch.cuda.device(self.device):
            _capi.check(self.lib.ssd_frontend_forward(self._h, obs_buf.data_ptr(), rows, int(agent_stride), int(plane_stride),
                                                      int(row_stride), out.data_ptr(),
                                                      C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))
        return out

    def forward_index4(self, obs_buf: torch.Tensor, rows: int, agent_stride: int, row_stride: int, color_lut, out=None):
        """``forward`` on index4 agent views (pixel x of a row is nibble x: byte x >> 1, low nibble when x is even), each index
        standing for the RGB pixel ``color_lut[index]`` (u8 [16, 3] or [16, 4]).  Bit-identical to ``forward`` on those RGB
        planes; same device, stream and handle rules."""
        rows = int(rows)
        lut = np.asarray(color_lut.cpu() if isinstance(color_lut, torch.Tensor) else color_lut)
        if lut.dtype != np.uint8 or lut.shape not in ((16, 3), (16, 4)):
            raise ValueError(f"color_lut must be a uint8 [16, 3] or [16, 4] array, got {lut.dtype} {lut.shape}")
        rgb0 = np.zeros((16, 4), dtype=np.uint8)
        rgb0[:, :3] = lut[:, :3]
        out = self._buffers(obs_buf, rows, agent_stride, out)
        if rows == 0:
            return out
        with torch.cuda.device(self.device):
            _capi.check(self.lib.ssd_frontend_forward_index4(self._h, obs_buf.data_ptr(), rows, int(agent_stride), int(row_stride),
                                                             rgb0.ctypes.data, out.data_ptr(),
                                                             C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))
        return out

    def forward_env(self, env, obs_buf=None, out=None):
        """All B*n agent views of an ``SSDBatchEnv`` (row order [B][n], as ``batch['obs'].reshape(bs * n, ...)``)."""
        if env.obs_format != "rgb":
            raise ValueError("the fused front end reads RGB planes; this env writes index4 observations")
        lay = env.layout
        return self.forward(env.obs_buf if obs_buf is None else obs_buf, env.B * env.n, lay.obs_agent_stride,
                            lay.obs_plane_stride, lay.obs_row_stride, out=out)

    def forward_env_index4(self, env, obs_buf=None, out=None):
        """``forward_env`` for an ``SSDBatchEnv`` in obs_format "index4": its ``obs_layout`` strides and ``spec.lut`` palette."""
        if env.obs_format != "index4":
            raise ValueError(f"forward_env_index4 reads index4 observations; this env writes {env.obs_format!r}")
        lay = env.obs_layout
        return self.forward_index4(env.obs_buf if obs_buf is None else obs_buf, env.B * env.n, lay.agent_stride, lay.row_stride,
                                   env.spec.lut, out=out)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.ssd_frontend_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MacFrontEnd:
    """Reroutes ``mac.agent.rgb_preprocess`` (homophily_controller.py:132-136) to the fused kernel while a rollout is in
    progress.  The packed weights follow the module's parameters (re-packed when an optimiser step bumped their versions).

    One ``ObsFrontEnd`` per env range, keyed by the range's first agent view: the batched runner rolls ranges out on their own
    streams without host syncs, and a handle's scratch and tile counters serve one forward at a time.

    ``obs_format`` is the format of the env's observation buffer the kernel reads: "rgb" (u8 planes) or "index4" (packed
    colour indices, expanded through ``env.spec.lut`` inside the kernel).  A call raises if the env has switched formats since."""

    def __init__(self, mac, env, obs_format="rgb"):
        if obs_format not in ("rgb", "index4"):
            raise ValueError(f"obs_format must be 'rgb' or 'index4', got {obs_format!r}")
        self.mac, self.env, self.obs_format = mac, env, obs_format
        self.module = mac.agent.conv_to_fc
        self.original = mac.agent.rgb_preprocess
        self.active = False
        self.rows = None                                      # (first agent view, count) of the env range being rolled out
        self._fes, self._stamp = {}, None
        mac.agent.rgb_preprocess = self

    def _front_end(self, first=0):
        stamp = tuple((p.data_ptr(), p._version) for p in self.module.parameters())
        if stamp != self._stamp:                              # new weights: every range's handle is re-packed on its next use
            self._close_all()
            self._stamp = stamp
        fe = self._fes.get(first)
        if fe is None:
            fe = self._fes[first] = ObsFrontEnd.from_module(self.module, self.env.spec.view, device=self.env.device)
        return fe

    def _close_all(self):
        for fe in self._fes.values():
            fe.close()
        self._fes.clear()

    def __call__(self, x):
        first, count = self.rows if self.rows is not None else (0, self.env.B * self.env.n)
        if not self.active or x.shape[0] != count:            # learner path (autograd) / foreign batch: the module
            return self.original(x)
        if self.env.obs_format != self.obs_format:
            raise ValueError(f"the front end reads {self.obs_format!r} observations; the env now writes {self.env.obs_format!r}")
        if self.obs_format == "index4":
            lay = self.env.obs_layout
            return self._front_end(first).forward_index4(self.env.obs_buf.view(-1)[first * lay.agent_stride:], count, lay.agent_stride,
                                                         lay.row_stride, self.env.spec.lut)
        lay = self.env.layout
        return self._front_end(first).forward(self.env.obs_buf.view(-1)[first * lay.obs_agent_stride:], count, lay.obs_agent_stride,
                                              lay.obs_plane_stride, lay.obs_row_stride)

    def __deepcopy__(self, memo):
        """``copy.deepcopy(mac)`` (the learner's target network, homophily_learner.py:47) must not copy the kernel handle: the
        copy of the agent gets its own, unpatched ``rgb_preprocess`` back."""
        import types
        agent_copy = memo.get(id(self.mac.agent))
        if agent_copy is None:
            return self.original
        return types.MethodType(type(self.mac.agent).rgb_preprocess, agent_copy)

    def detach(self):
        self.mac.agent.rgb_preprocess = self.original
        self._close_all()
