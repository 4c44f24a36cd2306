"""Layer-by-layer check of one or more launch plans on the GPU against float64 references (run by tests/test_gpu_layers.py).

    python tests/layer_parity_worker.py [--geo] [--modes parity,fast] variant,recipe,B,H,W [...]

A script, not a test module: the LSPG_* launch switches are read once per process, so every switch set runs in a process of
its own, under whatever environment the caller set.  Prints one JSON object per line: per config and mode, one record per
layer and one for the input packer and the buffer boundaries.  ``--geo`` needs no GPU: it prints the kernel instantiation
every layer of every config would launch.

For every conv layer the reference is tests/plan_emulator.py:run_layer in float64 on the GPU (torch ops only), fed with the
sources and residual the GPU itself stored, so errors do not compound from layer to layer:

* PARITY: ``max|got - ref| <= D/8 + 2^-21 max|ref|`` where ``D = min(max|scale*conv(a_lo, w_hi)|, max|scale*conv(a_hi,
  w_lo)|)`` on the same operands is the error of a kernel that drops one of its two cross products; the second term is the
  fp16 hi + lo storage of the output.  Every stored element also keeps the limb rule of the epilogues: ``hi`` is an fp16
  nearest to ``hi + lo`` (either neighbour on an exact tie), unless ``|hi|`` saturated at 65504.
* FAST: ``|got - ref| <= ulp_bf16(ref) + 2^-16 max|ref|`` everywhere (the second term covers values that cancel to almost
  zero or sit at a ReLU's edge), and at most 3e-3 of the elements differ from ``bf16_rn(ref)``.
* The tail's fp32 frame against float64 ``tanh``: the D/8 rule in PARITY, ``2^-17`` in FAST.
* No element of any stored tensor is NaN (the workspace starts as 0xFF bytes, a NaN in fp16 and bf16), and ReLU outputs are
  not negative.

Why D/8 and 3e-3 (measured on one B200 at 1000 W, profiles/layer_parity_b200.log): the tensor core's fp32 accumulator is
coarser than round-to-nearest fp32, and its error grows with the K range one accumulator sums.  Over all 15 instantiations
err/D spreads from 0.0015 to 0.126; the top of that range is on layers that sum their whole K (up to 9 x 512) in one tile:
the pair<128> / pair<256> layers of the 16- and 32-frame 512^2 plans (worst: large B, 32 x 512^2, layer 52, pair<128,NL2>,
0.1257, inside D/8 + 2^-21 max|y|) and umma<64> with LSPG_NO_SPLITK=1 (0.105, normal B, 1 x 256^2).  The same umma<64,NL2>
layers of the same config split four or eight ways inside a cluster (LSPG_CLUSTER_SPLIT=1) measure at most 0.027: the
accumulation length, not a missing product - that would measure about 1.  For the same reason the share of FAST elements that
round to the other bf16 neighbour than float64 reaches 1.95e-3 (umma<64,NL1,CSP> x8) while every element stays within half
an ulp plus the floor; a kernel that truncated instead of rounding would show about half.
"""
from __future__ import annotations

import ctypes as C
import json
import math
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import plan_emulator as E  # noqa: E402
from livespeechportraits_b200 import _lib  # noqa: E402
from oracle import f2f_oracle as O  # noqa: E402

MODES = {"fast": 0, "parity": 1}
GUARD = 1 << 16                     # workspace guard band, bytes on each side (a multiple of 1024)
OUT_GUARD = 1024                    # output guard, elements on each side
F32_NAN_BITS = 0x7FC00000
PARITY_D_FRACTION = 1 / 8           # PARITY bound: D * this + 2^-21 max|ref| (see the module docstring)
FAST_MISMATCH = 3e-3                # FAST: largest share of elements that may differ from bf16_rn(float64)


def instantiation(g, kind: int) -> dict:
    """The kernel template lspg.cu:launch_layer picks for this geometry (NL is the mode's)."""
    tail = kind == E.KIND_TAIL
    csp = g.cluster_split > 0
    if g.kernel == 2:
        fam = "pair"
    elif g.kernel == 1:
        fam = "patch"
    else:
        fam = "umma"
    cl = g.cta_cluster if fam == "patch" and not csp else 1      # the CL template argument (a cluster split runs CL = 1 code)
    return {"family": fam, "bn": g.bn, "tail": tail, "csp": csp, "cl": cl, "cta_cluster": g.cta_cluster,
            "splitk_reduce": g.n_split > 1 and not csp}


def inst_name(r: dict, nl) -> str:
    args = [str(r["bn"]), f"NL{nl}"]
    if r["tail"]:
        args.append("TAIL")
    if r["family"] == "patch" and not r["csp"]:
        args.append(f"CL{r['cl']}")
    if r["csp"]:
        args.append("CSP")
    s = f"{r['family']}<{','.join(args)}>"
    if r["cta_cluster"] > 1:
        s += f" x{r['cta_cluster']}"
    if r["splitk_reduce"]:
        s += " +splitk_reduce"
    return s


def geo_records(lib, h, nlayers, B, H, W):
    out = []
    for i in range(nlayers):
        g = _lib.LspgLayerGeo()
        _lib.check(lib.lspg_debug_layer_geo(h, i, B, H, W, C.byref(g)))
        info = _lib.LspgLayerInfo()
        _lib.check(lib.lspg_layer_info_get(h, i, C.byref(info)))
        out.append((info, g, instantiation(g, info.kind)))
    return out


def emit(rec: dict) -> None:
    print(json.dumps(rec), flush=True)


def parse_config(s: str):
    v, r, b, hh, ww = s.split(",")
    return v, r, int(b), int(hh), int(ww)


def run_geo(configs) -> None:
    lib = _lib.load()
    for variant, recipe, B, H, W in configs:
        h = C.c_void_p()
        _lib.check(lib.lspg_create(C.byref(h), _lib.LSPG_VARIANT[variant], 64, 8, 13, 3, -1))
        n = C.c_int()
        lib.lspg_num_layers(h, C.byref(n))
        for i, (info, g, inst) in enumerate(geo_records(lib, h, n.value, B, H, W)):
            emit(dict(type="geo", config=[variant, recipe, B, H, W], layer=i, kind=info.kind, **inst))
        lib.lspg_destroy(h)


# ---------------------------------------------------------------------------------------------------------- inputs
def realistic_input(B, H, W):
    fm, cand = O.make_inputs(B, H, W, seed=21)
    for i in range(1, B):                        # distinct frames (make_inputs repeats one candidate set)
        fm[i] = torch.roll(fm[i], shifts=(3 * i, 5 * i), dims=(1, 2))
        cand[i] = torch.roll(cand[i], shifts=(7 * i, 2 * i), dims=(1, 2))
    return torch.cat([fm, cand], 1).contiguous()


def adversarial_input(B, H, W):
    """Feature maps for every frame and ONE candidate set (passed with batch stride 0), sprinkled with values on fp16 and bf16
    rounding ties, values whose fp16 residual is subnormal or underflows, fp16-subnormal values, +-1 and -0.0."""
    rng = np.random.Generator(np.random.PCG64(77))
    specials = np.array([
        1.0, -1.0, 0.0, -0.0, 0.99999994, -0.99999994,
        1 + 2 ** -11, 1 + 3 * 2 ** -11, -(0.5 + 2 ** -12), 0.25 + 3 * 2 ** -13,        # fp16 ties (to even: down / up)
        1 + 2 ** -8, 1 + 3 * 2 ** -8, -(0.5 + 2 ** -9), 0.75 + 2 ** -9,                 # bf16 ties
        0.125 + 2 ** -20, 0.125 + 3 * 2 ** -26, -(0.5 + 2 ** -25), 1 - 2 ** -20,        # subnormal / underflowing fp16 residuals
        1e-5, -3e-8, 2 ** -25, 2 ** -24, 6.1e-5,                                        # fp16-subnormal values and below
        (1 + 2 ** -11) + 2 ** -23, 1 + 2 ** -8 + 2 ** -11,                               # just past the ties
    ], dtype=np.float32)
    fm = (2 * rng.random((B, 1, H, W), dtype=np.float32) - 1).astype(np.float32)
    cand = (2 * rng.random((1, 12, H, W), dtype=np.float32) - 1).astype(np.float32)
    for a in (fm, cand):
        mask = rng.random(a.shape) < 0.3
        a[mask] = rng.choice(specials, size=int(mask.sum()))
    return torch.from_numpy(fm), torch.from_numpy(cand)


def packed_input_bits(fm: torch.Tensor, cand: torch.Tensor, mode: str):
    """aux_kernels.cuh:pack_input_s2d_kernel with numpy rounding: 16-bit patterns [B,H/2,W/2,64] per limb."""
    B = fm.shape[0]
    x = torch.cat([fm, cand.expand(B, -1, -1, -1)], 1)
    s = E.pack_input_s2d(x).numpy()                         # fp32, channels 13..15 of each group zero
    if mode == "parity":
        hi = s.astype(np.float16)
        lo = (s - hi.astype(np.float32)).astype(np.float16)
        return [hi.view(np.uint16), lo.view(np.uint16)]
    return [torch.from_numpy(s).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)]


# ---------------------------------------------------------------------------------------------------------- the run
class Run:
    def __init__(self, plan: E.HostPlan, B, H, W, mode):
        self.plan, self.lib, self.h = plan, plan.lib, plan.h
        self.B, self.H, self.W, self.mode, self.m = B, H, W, mode, MODES[mode]
        self.nl = 2 if mode == "parity" else 1
        need = C.c_size_t()
        _lib.check(self.lib.lspg_workspace_bytes(self.h, B, H, W, self.m, C.byref(need)))
        self.need = need.value
        self.buf = torch.full((self.need + 2 * GUARD,), 0xFF, dtype=torch.uint8, device="cuda")
        self.ws = self.buf.data_ptr() + GUARD
        self.base = (self.ws + 1023) // 1024 * 1024 - self.buf.data_ptr()      # index of the plan's aligned base in buf
        n_out = B * 3 * H * W
        self.out_buf = torch.full((n_out + 2 * OUT_GUARD,), float("nan"), device="cuda")
        self.out = self.out_buf[OUT_GUARD:OUT_GUARD + n_out].view(B, 3, H, W)
        self.u8_buf = torch.full((n_out + 2 * 256,), 0xAB, dtype=torch.uint8, device="cuda")
        self.u8 = self.u8_buf[256:256 + n_out].view(B, H, W, 3)

    def forward(self, fm, fs, cand, cs, image=False):
        fn = self.lib.lspg_forward_image if image else self.lib.lspg_forward
        out = self.u8 if image else self.out
        _lib.check(fn(self.h, fm, fs, cand, cs, out.data_ptr(), self.B, self.H, self.W, self.ws, self.need, self.m,
                      torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()

    def forward_x(self, x, image=False):
        hw = self.H * self.W
        self.forward(x.data_ptr(), 13 * hw, x.data_ptr() + 4 * hw, 13 * hw, image)

    def stored(self, tid: int):
        """The limbs of activation tensor `tid` as views into the workspace, [B,h,w,C] fp16 (PARITY) / bf16 (FAST)."""
        c, th, tw = C.c_int(), C.c_int(), C.c_int()
        _lib.check(self.lib.lspg_tensor_shape(self.h, tid, self.H, self.W, C.byref(c), C.byref(th), C.byref(tw)))
        n = self.B * th.value * tw.value * c.value
        views = []
        for limb in range(self.nl):
            off = C.c_size_t()
            _lib.check(self.lib.lspg_debug_tensor_offset(self.h, tid, limb, self.B, self.H, self.W, self.m, C.byref(off)))
            s = self.base + off.value
            t = self.buf[s:s + 2 * n].view(torch.float16 if self.nl == 2 else torch.bfloat16)
            views.append(t.view(self.B, th.value, tw.value, c.value))
        return tuple(views)

    def release(self):
        _lib.check(self.lib.lspg_release_workspace(self.h, C.c_void_p(self.ws)))


def ulp_bf16(v: torch.Tensor) -> torch.Tensor:
    _, e = torch.frexp(v)
    return torch.where(v == 0, torch.zeros_like(v), torch.ldexp(torch.ones_like(v), e - 8))


def limb_rule_violations(hi: torch.Tensor, lo: torch.Tensor) -> int:
    """Elements where hi is not an fp16 nearest to hi + lo (exact ties may go either way), saturated |hi| = 65504 exempt."""
    h, s = hi.double(), hi.double() + lo.double()
    r = s.to(torch.float16).double()
    ok = (r == h) | ((s - h).abs() == (s - r).abs()) | (h.abs() == 65504)
    return int((~ok).sum())


def check_layers(run: Run, config, mode):
    plan, dev = run.plan, torch.device("cuda")
    nl = run.nl
    geos = geo_records(run.lib, run.h, len(plan.layers), run.B, run.H, run.W)
    for i, L in enumerate(plan.layers):
        info, g, inst = geos[i]
        srcs = [run.stored(L.src[s]) for s in range(L.n_src)]
        res = sum(t.double() for t in run.stored(L.res)) if L.res >= 0 else None
        with torch.no_grad():
            ref = E.run_layer(plan, i, srcs, res, nl, torch.float64, dev)
            if L.kind == E.KIND_TAIL:
                got, limbs = run.out.double(), None
            else:
                limbs = run.stored(L.out)
                got = sum(t.double() for t in limbs)[..., :ref.shape[-1]]
            rec = dict(type="layer", config=list(config), mode=mode, layer=i, kind=L.kind, key=L.conv_key.decode(),
                       inst=inst_name(inst, nl), nl=nl, **inst)
            max_ref = float(ref.abs().max())
            diff = (got - ref).abs()
            err = float(diff.max())
            rec.update(max_ref=max_ref, err=err, nan=int(torch.isnan(got).sum()))
            rec["negative"] = int((got < 0).sum()) if L.relu else 0
            if nl == 2:
                d_a = float(E.layer_linear(plan, i, srcs, 2, torch.float64, dev, products=[(1, 0)]).abs().max())
                d_w = float(E.layer_linear(plan, i, srcs, 2, torch.float64, dev, products=[(0, 1)]).abs().max())
                D = min(d_a, d_w)
                bound = D * PARITY_D_FRACTION + 2 ** -21 * max_ref
                rec.update(D=D, err_over_D=err / D if D > 0 else (0.0 if err == 0 else math.inf), bound=bound,
                           limb_violations=limb_rule_violations(*limbs) if limbs else 0)
                rec["ok"] = err <= bound and rec["limb_violations"] == 0
            elif L.kind == E.KIND_TAIL:
                bound = 2 ** -17
                rec.update(bound=bound, ok=err <= bound)
            else:
                allowed = ulp_bf16(ref) + 2 ** -16 * max_ref
                rec["err_over_ulp"] = float((diff / allowed).max()) if max_ref > 0 else 0.0
                rec["mismatch"] = float((got != ref.to(torch.bfloat16).double()).double().mean())
                rec["ok"] = rec["err_over_ulp"] <= 1.0 and rec["mismatch"] <= FAST_MISMATCH
            rec["ok"] = bool(rec["ok"] and rec["nan"] == 0 and rec["negative"] == 0)
        emit(rec)
        del srcs, res, ref, got, diff, limbs
    torch.cuda.empty_cache()


def run_config(config, modes):
    variant, recipe, B, H, W = config
    sd = O.make_state_dict(variant, recipe)
    plan = E.HostPlan(variant, sd, device=0)
    try:
        x1 = realistic_input(B, H, W).cuda()
        fm_adv, cand_adv = adversarial_input(B, H, W)
        fm_adv_d, cand_adv_d = fm_adv.cuda(), cand_adv.cuda()
        for mode in modes:
            run = Run(plan, B, H, W, mode)
            run.forward_x(x1)
            nt = C.c_int()
            _lib.check(run.lib.lspg_num_tensors(run.h, C.byref(nt)))
            nan_tensors = [t for t in range(nt.value) if any(bool(torch.isnan(v).any()) for v in run.stored(t))]
            check_layers(run, config, mode)
            out1 = run.out.clone()
            bnd = dict(type="boundary", config=list(config), mode=mode, nan_tensors=nan_tensors,
                       workspace_guards=bool((run.buf[:GUARD] == 0xFF).all() and (run.buf[GUARD + run.need:] == 0xFF).all()))
            ob = run.out_buf.view(torch.int32)
            bnd["out_guards"] = bool((ob[:OUT_GUARD] == F32_NAN_BITS).all() and (ob[-OUT_GUARD:] == F32_NAN_BITS).all())
            bnd["out_nan"] = int(torch.isnan(out1).sum())
            run.forward_x(x1, image=True)
            bnd["u8_guards"] = bool((run.u8_buf[:256] == 0xAB).all() and (run.u8_buf[-256:] == 0xAB).all())
            bnd["u8_equals_tensor2im"] = bool(np.array_equal(run.u8.cpu().numpy(), O.tensor2im(out1.cpu())))
            # the adversarial input, one candidate set broadcast with batch stride 0: the packed input tensor is bit-exact
            run.forward(fm_adv_d.data_ptr(), H * W, cand_adv_d.data_ptr(), 0)
            want = packed_input_bits(fm_adv, cand_adv, mode)
            got = [v.view(torch.int16).cpu().numpy().view(np.uint16) for v in run.stored(0)]
            emit(dict(type="packer", config=list(config), mode=mode,
                      mismatches=[int((a != b).sum()) for a, b in zip(got, want)], elements=int(want[0].size)))
            # the first input again: bit-identical output, nothing depends on what the workspace held before
            run.forward_x(x1)
            bnd["rerun_bit_identical"] = bool(torch.equal(run.out, out1))
            bnd["ok"] = (not nan_tensors and bnd["workspace_guards"] and bnd["out_guards"] and bnd["out_nan"] == 0
                         and bnd["u8_guards"] and bnd["u8_equals_tensor2im"] and bnd["rerun_bit_identical"])
            emit(bnd)
            run.release()
            del run, out1
            torch.cuda.empty_cache()
    finally:
        plan.close()


def main(argv):
    modes = ["parity", "fast"]
    geo = False
    configs = []
    it = iter(argv)
    for a in it:
        if a == "--modes":
            modes = next(it).split(",")
        elif a == "--geo":
            geo = True
        else:
            configs.append(parse_config(a))
    if geo:
        run_geo(configs)
        return 0
    emit(dict(type="device", name=torch.cuda.get_device_name(0),
              env={k: v for k, v in os.environ.items() if k.startswith("LSPG_")}))
    for cfg in configs:
        run_config(cfg, modes)
    return 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
