"""CPU emulation of the *launch plan* the C library builds (test infrastructure, not a product path).

Executes, with torch on the CPU, exactly what the CUDA kernels are told to do: the layer list, tap
tables (parity views for stride 2, output phases for the folded upsample, concat as K ranges), the
packed K-major weights and the folded scale/shift, all read back through the C ABI's introspection
calls of a host-only handle.  Comparing its output with the oracle validates the host logic (network
structure, key mapping, weight packing, BatchNorm folding, tap geometry) without a GPU; what remains
for the GPU tests is the PTX machinery itself.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from livespeechportraits_b200 import _lib

KIND_HEAD, KIND_S1, KIND_S2, KIND_UP, KIND_TAIL = range(5)


def bf16_bits_to_f32(a: np.ndarray) -> torch.Tensor:
    return torch.from_numpy((a.astype(np.uint32) << 16).view(np.float32).copy())


class HostPlan:
    def __init__(self, variant: str, state_dict: Dict[str, torch.Tensor], ngf: int = 64, num_downs: int = 8,
                 device: int = -1):
        """``device`` -1: a host-only handle; a CUDA ordinal: a handle that can also run lspg_forward."""
        self.lib = _lib.load()
        self.h = C.c_void_p()
        _lib.check(self.lib.lspg_create(C.byref(self.h), _lib.LSPG_VARIANT[variant], ngf, num_downs, 13, 3, device))
        keep, names = [], []
        for k, v in state_dict.items():
            if k.endswith("num_batches_tracked"):
                continue
            names.append(k.encode())
            keep.append(v.detach().float().contiguous())
        arr = (_lib.LspgTensor * len(keep))()
        for i, (nm, t) in enumerate(zip(names, keep)):
            arr[i].name, arr[i].numel = nm, t.numel()
            arr[i].data = C.cast(t.data_ptr(), C.POINTER(C.c_float))
        _lib.check(self.lib.lspg_load_weights(self.h, arr, len(keep)))
        n = C.c_int()
        _lib.check(self.lib.lspg_num_layers(self.h, C.byref(n)))
        self.layers: List[_lib.LspgLayerInfo] = []
        for i in range(n.value):
            info = _lib.LspgLayerInfo()
            _lib.check(self.lib.lspg_layer_info_get(self.h, i, C.byref(info)))
            self.layers.append(info)

    def close(self):
        if self.h:
            self.lib.lspg_destroy(self.h)
            self.h = C.c_void_p()

    PARITY_WEIGHT_SCALE = 256.0          # include/lspg.h: LSPG_PARITY_WEIGHT_SCALE

    def weight_limb(self, i: int, limb: int) -> torch.Tensor:
        """One packed weight limb as an fp32 value, exactly: limb 0 / 1 = PARITY fp16 hi / lo of w * 256, scaled back by the
        power of two; limb 2 = FAST bf16."""
        L = self.layers[i]
        count = L.n_phases * L.cout_pad * L.k_total
        buf = np.zeros(count, np.uint16)
        _lib.check(self.lib.lspg_layer_packed(self.h, i, limb, buf.ctypes.data, count))
        if limb == 2:
            out = bf16_bits_to_f32(buf)
        else:
            out = torch.from_numpy(buf.view(np.float16).astype(np.float32)) / self.PARITY_WEIGHT_SCALE
        return out.view(L.n_phases, L.cout_pad, L.k_total)

    def packed(self, i: int, limbs: int, dtype: torch.dtype = torch.float32) -> torch.Tensor:
        """Weights as the kernels multiply them: ``limbs == 2`` = PARITY (fp16 hi + lo limbs of w * 256, scaled back here,
        summed in ``dtype``: exact in float64), ``limbs == 1`` = FAST (bf16)."""
        if limbs == 1:
            return self.weight_limb(i, 2).to(dtype)
        return self.weight_limb(i, 0).to(dtype) + self.weight_limb(i, 1).to(dtype)

    def affine(self, i: int):
        L = self.layers[i]
        s = np.zeros(L.cout_pad, np.float32)
        b = np.zeros(L.cout_pad, np.float32)
        _lib.check(self.lib.lspg_layer_affine(self.h, i, s.ctypes.data, b.ctypes.data, L.cout_pad))
        return torch.from_numpy(s), torch.from_numpy(b)


def _shift(a: torch.Tensor, dy: int, dx: int) -> torch.Tensor:
    """b[n, y, x] = a[n, y+dy, x+dx], zero outside (what TMA's out-of-bounds fill gives the kernel)."""
    n, h, w, c = a.shape
    out = torch.zeros_like(a)
    ys0, ys1 = max(0, dy), min(h, h + dy)
    xs0, xs1 = max(0, dx), min(w, w + dx)
    if ys1 > ys0 and xs1 > xs0:
        out[:, ys0 - dy:ys1 - dy, xs0 - dx:xs1 - dx] = a[:, ys0:ys1, xs0:xs1]
    return out


def pack_input_s2d(x: torch.Tensor) -> torch.Tensor:
    """aux_kernels.cuh:pack_input_s2d_kernel in torch: [B,13,H,W] -> [B,H/2,W/2,64]."""
    b, c, h, w = x.shape
    s = torch.zeros(b, h // 2, w // 2, 64)
    for py in range(2):
        for px in range(2):
            s[..., (py * 2 + px) * 16:(py * 2 + px) * 16 + c] = x[:, :, py::2, px::2].permute(0, 2, 3, 1)
    return s


# The MMAs a PARITY K step issues, as (activation limb, weight limb): A_hi*B_hi, A_hi*B_lo, A_lo*B_hi (A_lo*B_lo is below
# the fp32 accumulator's resolution and never issued; include/lspg.h).
PARITY_PRODUCTS = ((0, 0), (0, 1), (1, 0))


def layer_linear(plan: HostPlan, i: int, srcs: Sequence, limbs: int = 2, dtype: torch.dtype = torch.float32,
                 device="cpu", products: Optional[Sequence[Tuple[int, int]]] = None) -> torch.Tensor:
    """``scale * conv`` of layer ``i`` (folded BatchNorm scale, no shift / residual / ReLU) as [B, Ho, Wo, cout_pad]: the
    phases of an upsample conv interleaved; for the tail the source grid with column ``(py*2+px)*3 + c``.

    ``srcs``: per concat source, the activation [B,h,w,C] as one tensor or as the tuple of its stored limbs (hi, lo).
    ``products`` None: exact operands - each source's limbs summed and the weight limbs summed, in ``dtype``.  Otherwise a
    list of (activation limb, weight limb) pairs (weight limbs 0 / 1 = PARITY hi / lo), each product accumulated on its own
    into one ``dtype`` accumulator, tap by tap, as the kernels do."""
    L = plan.layers[i]
    limb_srcs = [tuple(t.to(device, dtype) for t in (s if isinstance(s, (tuple, list)) else (s,))) for s in srcs]
    if products is None:
        limb_srcs = [(sum(s[1:], s[0]),) for s in limb_srcs]
        ws = [plan.packed(i, limbs, dtype).to(device)]
        products = ((0, 0),)
    else:
        ws = [plan.weight_limb(i, l).to(device, dtype) for l in range(2)]
    scale = plan.affine(i)[0].to(device, dtype)
    kb_per_tap = sum(int(L.cin[s]) for s in range(L.n_src))
    b, hs, ws_ = limb_srcs[0][0].shape[:3]
    if L.kind == KIND_S2:
        hs, ws_ = hs // 2, ws_ // 2
    phase_out = []
    for z in range(L.n_phases):
        acc = torch.zeros(b, hs, ws_, L.cout_pad, dtype=dtype, device=device)
        for t in range(L.n_taps):
            dx, dy, amap = int(L.tap_dx[z][t]), int(L.tap_dy[z][t]), int(L.tap_map[z][t])
            koff = t * kb_per_tap
            for s in range(L.n_src):
                cin = int(L.cin[s])
                for al, wl in products:
                    a = limb_srcs[s][al]
                    if L.kind == KIND_S2:
                        a = a[:, (amap >> 1)::2, (amap & 1)::2]    # parity view
                    acc += torch.einsum("nyxc,oc->nyxo", _shift(a, dy, dx), ws[wl][z, :, koff:koff + cin])
                koff += cin
        phase_out.append(acc * scale)
    if L.kind != KIND_UP:
        return phase_out[0]
    y = torch.zeros(b, 2 * hs, 2 * ws_, L.cout_pad, dtype=dtype, device=device)
    for z in range(4):
        y[:, (z >> 1)::2, (z & 1)::2] = phase_out[z]
    return y


def run_layer(plan: HostPlan, i: int, srcs: Sequence, res: Optional[torch.Tensor] = None, limbs: int = 2,
              dtype: torch.dtype = torch.float32, device="cpu",
              products: Optional[Sequence[Tuple[int, int]]] = None) -> torch.Tensor:
    """Layer ``i`` of the plan on its concat sources ``srcs`` (see :func:`layer_linear`) and its residual ``res``: the
    stored output [B,h,w,cout_pad], or for the tail the fp32 frame's values as [B,3,H,W].  Runs in ``dtype`` on ``device``
    with torch ops only."""
    L = plan.layers[i]
    y = layer_linear(plan, i, srcs, limbs, dtype, device, products) + plan.affine(i)[1].to(device, dtype)
    if L.kind == KIND_TAIL:
        y = torch.tanh(y)                                          # [B,hs,ws,16]; col = (py*2+px)*3 + c
        b, hs, ws_ = y.shape[:3]
        out = torch.zeros(b, 3, 2 * hs, 2 * ws_, dtype=dtype, device=device)
        for py in range(2):
            for px in range(2):
                for c in range(3):
                    out[:, c, py::2, px::2] = y[..., (py * 2 + px) * 3 + c]
        return out
    if L.res >= 0:
        y = y + res.to(device, dtype)
    if L.relu:
        y = torch.relu(y)
    return y


def run_plan(plan: HostPlan, x: torch.Tensor, limbs: int = 2, round_act=None,
             taps_out: Optional[Dict[int, torch.Tensor]] = None) -> torch.Tensor:
    """Execute the plan on [B,13,H,W] fp32 input.  ``limbs``: 1 = FAST (bf16 weights), 2 = PARITY (fp16 hi+lo weights).
    ``round_act``: optional function applied to every stored activation (e.g. bf16 rounding)."""
    q = round_act or (lambda t: t)
    tensors: Dict[int, torch.Tensor] = {0: q(pack_input_s2d(x))}
    result = None
    for i, L in enumerate(plan.layers):
        srcs = [tensors[L.src[s]] for s in range(L.n_src)]
        y = run_layer(plan, i, srcs, tensors[L.res] if L.res >= 0 else None, limbs)
        if L.kind == KIND_TAIL:
            result = y
            continue
        tensors[L.out] = q(y)
        if taps_out is not None:
            taps_out[L.out] = tensors[L.out]
    return result
