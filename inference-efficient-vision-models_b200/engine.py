"""``nn.Module`` drop-ins for the reference's hot path, backed by the sm_100a engine (C ABI).

``B200QuantizedResNet`` stands where the reference holds the FX-converted INT8 ``GraphModule``
(quantization/engines.py:118) and ``B200HalfResNet`` where it holds ``model.half()``
(quantization/engines.py:91-92): the call ``outputs = model(images)`` (engines.py:27,31,60;
quantization/main.py:287) keeps its dtypes and shapes -- f32 NCHW in / f32 logits out for INT8, f16 in /
f16 out for FP16 -- and ``.eval()``, ``.parameters()`` (dtype sniffing at engines.py:20,47),
``.state_dict()`` and ``.to()/.cpu()`` keep working for the callers that touch them.
There is no fallback path: if the CUDA library is missing or no B200 is present, construction raises.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from .netdesc import DTYPE_F16, DTYPE_I8, OP_CONV, OP_HEAD, NetSpec, from_converted, from_half_module, \
    from_quantized_state_dict


def _marshal(net: NetSpec):
    """NetSpec -> (NetDesc, keepalive list)."""
    keep = []
    arr = (_lib.LayerDesc * len(net.layers))()
    for i, L in enumerate(net.layers):
        d = arr[i]
        d.op, d.in_tensor, d.res_tensor, d.out_tensor = L.op, L.in_tensor, L.res_tensor, L.out_tensor
        d.cin, d.cout, d.ksize, d.stride, d.pad, d.relu = L.cin, L.cout, L.ksize, L.stride, L.pad, int(L.relu)
        for field_name, a, dt in (("weight", L.weight, None), ("bias", L.bias, np.float32),
                                  ("w_scale", L.w_scale, np.float32)):
            if a is None:
                setattr(d, field_name, None)
                continue
            a = np.ascontiguousarray(a if dt is None else a.astype(dt))
            keep.append(a)
            setattr(d, field_name, a.ctypes.data)
        d.in_scale, d.in_zp = L.in_scale, L.in_zp
        d.out_scale, d.out_zp = L.out_scale, L.out_zp
        d.res_scale, d.res_zp = L.res_scale, L.res_zp
        d.add_scale, d.add_zp = L.add_scale, L.add_zp
    nd = _lib.NetDesc()
    nd.dtype, nd.num_layers = net.dtype, len(net.layers)
    nd.in_c, nd.in_h, nd.in_w, nd.num_classes = net.in_c, net.in_h, net.in_w, net.num_classes
    nd.in_scale, nd.in_zp = net.in_scale, net.in_zp
    nd.layers = arr
    keep.append(arr)
    return nd, keep


IMAGENET_MEAN = (0.485, 0.456, 0.406)      # quantization/dataset.py:17-18
IMAGENET_STD = (0.229, 0.224, 0.225)


def pil_bilinear_coeffs(in_size: int, out_size: int):
    """Per-output-pixel tables of Pillow's 8-bit bilinear resample (``Resample.c``: ``precompute_coeffs`` followed by
    ``normalize_coeffs_8bpc``) for resizing ``in_size`` to ``out_size`` along one axis: ``bounds[o] = (first source
    index, taps)`` and ``kk[o, :taps]`` = 22-bit fixed-point weights.  Python floats are C doubles and ``int()``
    truncates like the C casts, so the tables equal Pillow's own (tests/test_host.py)."""
    import math
    precision_bits = 32 - 8 - 2
    scale = filterscale = in_size / out_size
    if filterscale < 1.0:
        filterscale = 1.0
    support = filterscale                      # bilinear filter: support 1.0
    ksize = int(math.ceil(support)) * 2 + 1
    bounds = np.zeros((out_size, 2), np.int32)
    kk = np.zeros((out_size, ksize), np.int32)
    inv = 1.0 / filterscale
    for o in range(out_size):
        center = (o + 0.5) * scale
        lo = max(int(center - support + 0.5), 0)
        hi = min(int(center + support + 0.5), in_size)
        weights = []
        for x in range(lo, hi):
            d = abs((x - center + 0.5) * inv)
            weights.append(1.0 - d if d < 1.0 else 0.0)
        total = 0.0
        for w in weights:
            total += w
        for t, w in enumerate(weights):
            if total != 0.0:
                w = w / total
            kk[o, t] = int(w * (1 << precision_bits) - 0.5) if w < 0 else int(w * (1 << precision_bits) + 0.5)
        bounds[o] = (lo, hi - lo)
    return bounds, kk


def input_lut(in_scale: float, in_zp: int, mean=IMAGENET_MEAN, std=IMAGENET_STD) -> np.ndarray:
    """[3, 256] uint8: lut[c, v] = quantize_per_tensor(Normalize(ToTensor(v)))[c], computed with the very torch /
    torchvision ops the reference's transform and converted graph run, one 8-bit level at a time -- the fused
    kernel is therefore bit-identical to the unfused f32 pipeline by construction."""
    from torchvision.transforms import functional as TF
    levels = torch.arange(256, dtype=torch.uint8).view(1, 256, 1).expand(1, 256, 3).contiguous()   # H=1, W=256, C=3
    x = TF.to_tensor(levels.numpy())                         # [3, 1, 256] float32 in [0, 1]: v / 255
    x = TF.normalize(x, list(mean), list(std))
    q = torch.quantize_per_tensor(x, float(in_scale), int(in_zp), torch.quint8).int_repr()
    return np.ascontiguousarray(q.view(3, 256).numpy())


class _B200Engine(nn.Module):
    _torch_dtype = torch.float32

    def __init__(self, net: NetSpec, source=None, device: Optional[int] = None, max_batch: int = 256):
        super().__init__()
        self._lib = _lib.load()          # raises when the CUDA extension has not been built
        if not torch.cuda.is_available():
            raise RuntimeError("B200 engine: no CUDA device visible and there is no CPU fallback")
        self.net = net
        self.device_index = torch.cuda.current_device() if device is None else int(device)
        self.max_batch = int(max_batch)
        self._source = source            # the reference-side module, kept for state_dict()/parameters()
        # One zero-size parameter of the right dtype keeps `next(model.parameters()).dtype`
        # (quantization/engines.py:20,47) meaningful.
        self._dtype_probe = nn.Parameter(torch.empty(0, dtype=self._torch_dtype), requires_grad=False)
        self._handle = C.c_void_p()
        nd, keep = _marshal(net)
        _lib.check(self._lib.ievm_create(C.byref(nd), self.device_index, self.max_batch, C.byref(self._handle)),
                   "ievm_create")
        del keep

    # ---- reference-facing protocol ---------------------------------------------------------
    def forward(self, images: torch.Tensor) -> torch.Tensor:
        if images.dim() != 4 or tuple(images.shape[1:]) != (self.net.in_c, self.net.in_h, self.net.in_w):
            raise ValueError(f"expected [N,{self.net.in_c},{self.net.in_h},{self.net.in_w}], got {tuple(images.shape)}")
        if images.dtype != self._torch_dtype:
            raise TypeError(f"expected {self._torch_dtype} input, got {images.dtype}")
        n = images.shape[0]
        if n == 0:
            return torch.empty((0, self.net.num_classes), dtype=self._torch_dtype, device=images.device)
        if n > self.max_batch:
            return torch.cat([self.forward(images[i:i + self.max_batch]) for i in range(0, n, self.max_batch)])
        if not images.is_cuda:
            return self._forward_host(images)
        self._check_device(images)
        x = images.contiguous()
        out = torch.empty((n, self.net.num_classes), dtype=self._torch_dtype, device=x.device)
        stream = torch.cuda.current_stream(x.device).cuda_stream
        _lib.check(self._forward_fn(self._handle, x.data_ptr(), n, out.data_ptr(), stream), "ievm_forward")
        return out

    def _forward_host(self, images: torch.Tensor) -> torch.Tensor:
        """CPU tensor in, CPU tensor out (the reference's loops hand over CPU batches:
        quantization/engines.py:52-60): H2D copy, forward and D2H copy inside the C call."""
        x = images.contiguous()
        n = x.shape[0]
        out = torch.empty((n, self.net.num_classes), dtype=self._torch_dtype)
        _lib.check(self._forward_host_fn(self._handle, x.data_ptr(), n, out.data_ptr()), "ievm_forward_host")
        return out

    def _check_device(self, t: torch.Tensor) -> None:
        if t.device.index != self.device_index:
            raise ValueError(f"tensor is on cuda:{t.device.index} but this engine is bound to cuda:{self.device_index}")

    # ---- pipelined host path: the reference's evaluation loops hand over one CPU batch per iteration --------------
    def submit(self, images: torch.Tensor) -> "PendingLogits":
        """Enqueue ``model(images)`` for a CPU batch and return at once (``ievm_submit_*_host``): the H2D copy of this
        batch overlaps the forward of the previous one.  ``images`` is what ``forward`` accepts on the CPU (pinned
        memory makes the copy asynchronous) or, for INT8 engines, decoded uint8 ``[N, h, w, 3]`` images.  At most two
        batches are in flight: a third call first settles the oldest one, whose ``.result()`` then returns at once.
        ``.result()`` of the returned object waits for this one's logits (a CPU tensor)."""
        if images.is_cuda:
            raise ValueError("submit() is the host-buffer path; call the engine directly with CUDA tensors")
        n = int(images.shape[0])
        if n == 0 or n > self.max_batch:
            raise ValueError(f"submit() takes 1..{self.max_batch} images per call, got {n}")
        x = images.contiguous()
        if x.dtype == torch.uint8:
            fn = self._submit_u8(x)
        else:
            if x.dim() != 4 or tuple(x.shape[1:]) != (self.net.in_c, self.net.in_h, self.net.in_w):
                raise ValueError(f"expected [N,{self.net.in_c},{self.net.in_h},{self.net.in_w}], got {tuple(x.shape)}")
            if x.dtype != self._torch_dtype:
                raise TypeError(f"expected {self._torch_dtype} input, got {x.dtype}")
            fn = self._submit_fn
        if not hasattr(self, "_out_ring"):       # two pinned logits buffers, one per pipeline slot
            self._out_ring = [torch.empty((self.max_batch, self.net.num_classes), dtype=self._torch_dtype).pin_memory()
                              for _ in range(2)]
            self._out_owner = [None, None]
            self._out_next = 0
        k = self._out_next
        # The call that last used this buffer may not have been read yet: settle it (copy its logits out) before this
        # call's D2H overwrites them.  The C submit waits for that call's slot anyway, so this adds no synchronisation.
        if self._out_owner[k] is not None:
            self._out_owner[k].result()
            self._out_owner[k] = None
        out = self._out_ring[k]
        self._out_next ^= 1
        ticket = C.c_int64(-1)
        _lib.check(fn(self._handle, x.data_ptr(), n, out.data_ptr(), C.byref(ticket)), "ievm_submit_host")
        pending = PendingLogits(self, int(ticket.value), out, n, x)
        self._out_owner[k] = pending
        return pending

    def _submit_u8(self, x: torch.Tensor):
        raise TypeError("uint8 image input belongs to the INT8 engine")

    def state_dict(self, *args, **kwargs):
        if self._source is not None and hasattr(self._source, "state_dict"):
            return self._source.state_dict(*args, **kwargs)
        return super().state_dict(*args, **kwargs)

    def to(self, *args, **kwargs):       # the engine is bound to its B200; .to()/.cpu() are no-ops
        return self

    def cpu(self):
        return self

    def cuda(self, device=None):
        return self

    def half(self):
        if self._torch_dtype != torch.float16:
            raise TypeError("an INT8 engine cannot be cast to half")
        return self

    # ---- engine controls / parity hooks --------------------------------------------------
    def set_option(self, name: str, value: int) -> None:
        _lib.check(self._lib.ievm_set_option(self._handle, name.encode(), int(value)), f"set_option({name})")

    @property
    def launches_per_forward(self) -> int:
        return int(self._lib.ievm_launches_per_forward(self._handle))

    def layer_launch(self, index: int) -> int:
        """Index of the layer whose kernel launch computes layer `index` (a fused 1x1 downsample reports its block's
        first conv, the max-pool of the fused front end reports the stem)."""
        return int(self._lib.ievm_layer_launch(self._handle, index))

    def profile_read(self):
        """[(name, total_ms, calls)] per launch slot accumulated since set_option('profile', 1)."""
        slots = len(self.net.layers) + 1
        ms = (C.c_float * slots)()
        calls = (C.c_int32 * slots)()
        self._lib.ievm_profile_read(self._handle, slots, ms, calls)
        names = ["quantize_input"] + [L.name for L in self.net.layers]
        return [(names[i], float(ms[i]), int(calls[i])) for i in range(slots)]

    def tensor_shape(self, tid: int):
        out = (C.c_int32 * 6)()
        _lib.check(self._lib.ievm_tensor_shape(self._handle, tid, C.byref(out)), "ievm_tensor_shape")
        return tuple(out)

    def read_tensor(self, tid: int) -> np.ndarray:
        """Tensor ``tid`` of the last forward as NCHW over the real channels (needs keep_tensors=1)."""
        n, h, w, c, pitch, elem = self.tensor_shape(tid)
        dt = np.uint8 if elem == 1 else np.float16
        buf = np.empty((n, h, w, pitch), dtype=dt)
        _lib.check(self._lib.ievm_debug_read_tensor(self._handle, tid, buf.ctypes.data, buf.nbytes), "read_tensor")
        return np.ascontiguousarray(buf[..., :c].transpose(0, 3, 1, 2))

    def read_tensor_by_name(self, name: str) -> np.ndarray:
        for tid, nm in self.net.tensor_names.items():
            if nm == name:
                return self.read_tensor(tid)
        raise KeyError(name)

    def conv_accumulators(self, layer_name: str, n: int) -> np.ndarray:
        """Raw tensor-core accumulators of conv ``layer_name`` as NCHW over real channels."""
        for li, L in enumerate(self.net.layers):
            if L.name == layer_name and L.op == OP_CONV:
                _, h, w, c, pitch, _ = self.tensor_shape(L.out_tensor)
                buf = np.empty((n, h, w, pitch), dtype=np.int32)
                _lib.check(self._lib.ievm_debug_conv_acc(self._handle, li, n, buf.ctypes.data, buf.nbytes),
                           "conv_accumulators")
                acc = np.ascontiguousarray(buf[..., :c].transpose(0, 3, 1, 2))
                return acc if self.net.dtype == DTYPE_I8 else acc.view(np.float32)
        raise KeyError(layer_name)

    def debug_frontend(self, images: torch.Tensor, want_acc: bool = True):
        """Run only the fused front end (quantize + stem + ReLU + max-pool) on a CUDA batch: the engine's native input,
        or decoded uint8 ``[N, in_h, in_w, 3]`` images through the lookup table of ``set_input_transform`` (INT8).
        Returns (pooled NCHW over real channels, stem accumulators NCHW or None)."""
        stem, pool = self.net.layers[0], self.net.layers[1]
        n = int(images.shape[0])
        u8 = images.dtype == torch.uint8
        if u8 and (images.dim() != 4 or tuple(images.shape[1:]) != (self.net.in_h, self.net.in_w, 3)):
            raise ValueError(f"expected uint8 [N,{self.net.in_h},{self.net.in_w},3], got {tuple(images.shape)}")
        if u8 and getattr(self, "_lut", None) is None:
            raise ValueError("debug_frontend on uint8 images needs set_input_transform() first")
        _, ho, wo, c, pitch, elem = self.tensor_shape(stem.out_tensor)
        _, ph, pw, _, _, _ = self.tensor_shape(pool.out_tensor)
        dt = np.uint8 if elem == 1 else np.float16
        pooled = np.empty((n, ph, pw, pitch), dtype=dt)
        acc = np.empty((n, ho, wo, pitch), dtype=np.int32) if want_acc else None
        x = images.contiguous()
        _lib.check(self._lib.ievm_debug_frontend(self._handle, x.data_ptr(), int(u8), n, pooled.ctypes.data, pooled.nbytes,
                                                 acc.ctypes.data if want_acc else None, acc.nbytes if want_acc else 0),
                   "debug_frontend")
        pooled = np.ascontiguousarray(pooled[..., :c].transpose(0, 3, 1, 2))
        if want_acc:
            acc = np.ascontiguousarray(acc[..., :c].transpose(0, 3, 1, 2))
            acc = acc if self.net.dtype == DTYPE_I8 else acc.view(np.float32)
        return pooled, acc

    def close(self) -> None:
        if getattr(self, "_handle", None) is not None and self._handle.value:
            self._lib.ievm_destroy(self._handle)
            self._handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class PendingLogits:
    """Logits of a batch handed to ``submit()``; ``result()`` waits (``ievm_wait``) and returns them as a CPU tensor."""

    def __init__(self, engine, ticket, out, n, keepalive):
        self._engine, self._ticket, self._out, self._n, self._keepalive = engine, ticket, out, n, keepalive
        self._value = None

    def result(self) -> torch.Tensor:
        if self._value is None:
            eng = self._engine
            _lib.check(eng._lib.ievm_wait(eng._handle, self._ticket), "ievm_wait")
            self._value = self._out[:self._n].clone()       # the pinned slot is reused two submits later
            self._keepalive = None
        return self._value


class B200QuantizedResNet(_B200Engine):
    """Drop-in for the converted static-INT8 module (fbgemm semantics, bit-exact target)."""
    _torch_dtype = torch.float32

    def __init__(self, net: NetSpec, **kw):
        if net.dtype != DTYPE_I8:
            raise ValueError("expected an INT8 NetSpec")
        super().__init__(net, **kw)
        self._forward_fn = self._lib.ievm_forward_i8
        self._forward_host_fn = self._lib.ievm_forward_i8_host
        self._submit_fn = self._lib.ievm_submit_i8_host

    @classmethod
    def from_converted(cls, gm, **kw) -> "B200QuantizedResNet":
        return cls(from_converted(gm), source=gm, **kw)

    # ---- SURVEY 8(f)-1: the input pipeline in front of the hot path -------------------------
    def set_input_transform(self, mean=IMAGENET_MEAN, std=IMAGENET_STD) -> np.ndarray:
        """Fuse ``T.ToTensor() -> T.Normalize(mean, std)`` (quantization/dataset.py:16-18) and the graph's
        ``quantize_per_tensor`` into the front-end kernel.  Returns the [3, 256] lookup table it uploaded."""
        lut = input_lut(self.net.in_scale, self.net.in_zp, mean, std)
        _lib.check(self._lib.ievm_set_input_lut(self._handle, lut.ctypes.data), "ievm_set_input_lut")
        self._lut = lut
        return lut

    def _submit_u8(self, x: torch.Tensor):
        if getattr(self, "_lut", None) is None:
            self.set_input_transform()
        if x.dim() != 4 or x.shape[3] != 3:
            raise ValueError(f"expected uint8 [N,h,w,3], got {tuple(x.shape)}")
        if tuple(x.shape[1:3]) == (self.net.in_h, self.net.in_w):
            return self._lib.ievm_submit_u8_host
        if getattr(self, "_resize_src", None) != tuple(x.shape[1:3]):
            self.set_resize(x.shape[1], x.shape[2])
        return self._lib.ievm_submit_u8_resize_host

    def set_resize(self, src_h: int, src_w: int) -> None:
        """Install ``T.Resize((in_h, in_w))`` (quantization/dataset.py:15: Pillow's bilinear resample) for decoded
        source images of ``src_h x src_w``."""
        bw, kw = pil_bilinear_coeffs(int(src_w), self.net.in_w)
        bh, kh = pil_bilinear_coeffs(int(src_h), self.net.in_h)
        _lib.check(self._lib.ievm_set_resize(self._handle, int(src_h), int(src_w), bw.ctypes.data, kw.ctypes.data, kw.shape[1],
                                             bh.ctypes.data, kh.ctypes.data, kh.shape[1]), "ievm_set_resize")
        self._resize_src = (int(src_h), int(src_w))

    def debug_resize(self, images: torch.Tensor) -> np.ndarray:
        """Only the resize stage: uint8 CUDA ``[N, h, w, 3]`` -> uint8 ``[N, in_h, in_w, 3]`` (parity hook)."""
        if getattr(self, "_resize_src", None) != tuple(images.shape[1:3]):
            self.set_resize(images.shape[1], images.shape[2])
        x = images.contiguous()
        out = np.empty((x.shape[0], self.net.in_h, self.net.in_w, 3), np.uint8)
        _lib.check(self._lib.ievm_debug_resize(self._handle, x.data_ptr(), x.shape[0], out.ctypes.data, out.nbytes), "debug_resize")
        return out

    def forward_u8(self, images: torch.Tensor) -> torch.Tensor:
        """Decoded 8-bit images ``[N, h, w, 3]`` (HWC, RGB, uint8; CPU or CUDA) -> f32 logits, bit-identical to the
        reference's ``Resize -> ToTensor -> Normalize`` transform followed by the converted module.  Images that are
        already ``in_h x in_w`` skip the resize.  A quarter (or less) of the input bytes over PCIe and HBM."""
        if getattr(self, "_lut", None) is None:
            self.set_input_transform()
        if images.dtype != torch.uint8 or images.dim() != 4 or images.shape[3] != 3:
            raise ValueError(f"expected uint8 [N,h,w,3], got {images.dtype} {tuple(images.shape)}")
        if images.shape[0] == 0:
            return torch.empty((0, self.net.num_classes), dtype=torch.float32, device=images.device)
        if tuple(images.shape[1:3]) != (self.net.in_h, self.net.in_w):
            return self._forward_u8_resize(images)
        n = images.shape[0]
        if n > self.max_batch:
            return torch.cat([self.forward_u8(images[i:i + self.max_batch]) for i in range(0, n, self.max_batch)])
        x = images.contiguous()
        if not x.is_cuda:
            out = torch.empty((n, self.net.num_classes), dtype=torch.float32)
            _lib.check(self._lib.ievm_forward_u8_host(self._handle, x.data_ptr(), n, out.data_ptr()), "ievm_forward_u8_host")
            return out
        self._check_device(x)
        out = torch.empty((n, self.net.num_classes), dtype=torch.float32, device=x.device)
        stream = torch.cuda.current_stream(x.device).cuda_stream
        _lib.check(self._lib.ievm_forward_u8(self._handle, x.data_ptr(), n, out.data_ptr(), stream), "ievm_forward_u8")
        return out

    def _forward_u8_resize(self, images: torch.Tensor) -> torch.Tensor:
        if getattr(self, "_resize_src", None) != tuple(images.shape[1:3]):
            self.set_resize(images.shape[1], images.shape[2])
        n = images.shape[0]
        if n > self.max_batch:
            return torch.cat([self._forward_u8_resize(images[i:i + self.max_batch]) for i in range(0, n, self.max_batch)])
        x = images.contiguous()
        if not x.is_cuda:
            out = torch.empty((n, self.net.num_classes), dtype=torch.float32)
            _lib.check(self._lib.ievm_forward_u8_resize_host(self._handle, x.data_ptr(), n, out.data_ptr()),
                       "ievm_forward_u8_resize_host")
            return out
        self._check_device(x)
        out = torch.empty((n, self.net.num_classes), dtype=torch.float32, device=x.device)
        stream = torch.cuda.current_stream(x.device).cuda_stream
        _lib.check(self._lib.ievm_forward_u8_resize(self._handle, x.data_ptr(), n, out.data_ptr(), stream), "ievm_forward_u8_resize")
        return out

    @classmethod
    def from_quantized_state_dict(cls, sd, **kw) -> "B200QuantizedResNet":
        return cls(from_quantized_state_dict(sd), **kw)


class B200HalfResNet(_B200Engine):
    """Drop-in for ``model.half()`` (student ResNet-18 or ResNet-50 teacher)."""
    _torch_dtype = torch.float16

    def __init__(self, net: NetSpec, **kw):
        if net.dtype != DTYPE_F16:
            raise ValueError("expected an FP16 NetSpec")
        super().__init__(net, **kw)
        self._forward_fn = self._lib.ievm_forward_f16
        self._forward_host_fn = self._lib.ievm_forward_f16_host
        self._submit_fn = self._lib.ievm_submit_f16_host

    @classmethod
    def from_half_module(cls, model, **kw) -> "B200HalfResNet":
        return cls(from_half_module(model), source=model, **kw)


def kd_eval_loss(student_logits: torch.Tensor, teacher_logits: torch.Tensor, labels: torch.Tensor,
                 alpha: float = 0.5, temperature: float = 4.0):
    """Soft-target KD loss of knowledge_distillation/train.py:47-57 on device logits.
    Returns (loss, ce, kd, n_correct) as a 4-element CUDA tensor without synchronising."""
    lib = _lib.load()
    if student_logits.dim() != 2 or student_logits.shape != teacher_logits.shape:
        raise ValueError(f"student / teacher logits must both be [N, classes]: {tuple(student_logits.shape)} vs "
                         f"{tuple(teacher_logits.shape)}")
    if labels.dim() != 1 or labels.shape[0] != student_logits.shape[0]:
        raise ValueError(f"labels must be [N] = [{student_logits.shape[0]}], got {tuple(labels.shape)}")
    if not student_logits.is_cuda or teacher_logits.device != student_logits.device or labels.device != student_logits.device:
        raise ValueError("student logits, teacher logits and labels must live on the same CUDA device")
    s = student_logits.float().contiguous()
    t = teacher_logits.float().contiguous()
    y = labels.to(torch.int64).contiguous()       # a label outside [0, classes) makes the CE term NaN (no out-of-bounds read)
    out3 = torch.empty(3, dtype=torch.float32, device=s.device)
    with torch.cuda.device(s.device):
        _lib.check(lib.ievm_kd_loss(s.data_ptr(), t.data_ptr(), y.data_ptr(), s.shape[0], s.shape[1],
                                    float(temperature), out3.data_ptr(),
                                    torch.cuda.current_stream(s.device).cuda_stream), "ievm_kd_loss")
    loss = (1.0 - alpha) * out3[0] + alpha * out3[1]
    return torch.stack([loss, out3[0], out3[1], out3[2]])


def measure_mma_peak(dtype: str = "i8", device: int = 0, iters: int = 4000) -> float:
    """Tera-ops/s this device's tensor cores sustain on a pure ``tcgen05.mma`` stream (``ievm_probe_mma_peak``):
    the roofline denominator bench.py uses for the tensor-core kernels (no library INT8 GEMM exists to measure against)."""
    lib = _lib.load()
    out = C.c_double(0.0)
    _lib.check(lib.ievm_probe_mma_peak(int(device), 0 if dtype == "i8" else 1, int(iters), C.byref(out)), "ievm_probe_mma_peak")
    return float(out.value)
