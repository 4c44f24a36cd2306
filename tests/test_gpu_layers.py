"""Per-layer parity of every conv kernel variant the launch planner can select, against float64 references.

The end-to-end gates (1e-3 on the frame) cannot tell a correct PARITY kernel from one that never issues one of its two cross
products (A_hi*B_lo or A_lo*B_hi): oracle/precision_study.py puts that error at a few 1e-4 end to end.  Here every layer is
checked on its own, fed the activations the GPU stored, against tests/plan_emulator.py:run_layer in float64, with a bound
of 1/8 of the error a dropped product would cause (tests/layer_parity_worker.py lists the rules and the measurements that
set them).

The GPU tests run tests/layer_parity_worker.py once per set of LSPG_* launch switches (the library reads them once per
process); MATRIX lists the switch sets and the configs that reach every kernel instantiation.  The CPU tests prove that the
matrix reaches every instantiation lspg.cu:launch_layer can select, and that the bound rejects a kernel with a missing
limb product while it admits fp32 accumulation.
"""
import json
import os
import subprocess
import sys
from collections import defaultdict

import pytest
import torch

import layer_parity_worker as W
import plan_emulator as E
from oracle import f2f_oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
WORKER = os.path.join(HERE, "layer_parity_worker.py")
MODES = ("parity", "fast")

# (switches, configs (variant, recipe, batch, height, width), what the set reaches)
MATRIX = {
    "default": ({}, [("normal", "A", 1, 256, 256), ("normal", "B", 3, 256, 256), ("normal", "B", 8, 512, 256),
                     ("large", "A", 1, 512, 512), ("large", "B", 32, 512, 512)],
                "finisher split-K, tail CL1, ragged image groups, patch<64,CSP>, the single-frame and the benchmark plans"),
    "cluster_split": ({"LSPG_CLUSTER_SPLIT": "1"}, [("normal", "B", 1, 256, 256), ("large", "B", 2, 512, 512)],
                      "cluster split-K at batch 1-2"),
    "finisher_split": ({"LSPG_CLUSTER_SPLIT": "0"}, [("large", "B", 16, 512, 512)], "splitk_reduce at large batch"),
    "no_splitk": ({"LSPG_NO_SPLITK": "1"}, [("normal", "B", 1, 256, 256)], "unsplit small layers"),
    "no_pair": ({"LSPG_NO_PAIR": "1"}, [("large", "B", 16, 256, 256)], "patch<128> CL2, multicast weights"),
    "no_pair_no_cluster": ({"LSPG_NO_PAIR": "1", "LSPG_NO_CLUSTER": "1"}, [("large", "B", 16, 256, 256)],
                           "patch<128> / patch<64> / tail CL1"),
    "no_patch": ({"LSPG_NO_PATCH": "1"}, [("normal", "B", 2, 256, 256)], "umma<16,TAIL>, umma on every layer"),
}

# Every conv template lspg.cu:launch_layer can launch, as (family, BN, TAIL, CSP, CL), each in both NL = 1 (FAST) and 2.
ALL_INSTANTIATIONS = {
    ("pair", 256, False, False, 1), ("pair", 128, False, False, 1), ("pair", 64, False, False, 1),
    ("patch", 64, False, True, 1), ("umma", 128, False, True, 1), ("umma", 64, False, True, 1),
    ("patch", 16, True, False, 1), ("patch", 16, True, False, 2),
    ("patch", 128, False, False, 1), ("patch", 128, False, False, 2),
    ("patch", 64, False, False, 1), ("patch", 64, False, False, 2),
    ("umma", 16, True, False, 1), ("umma", 128, False, False, 1), ("umma", 64, False, False, 1),
}


def _key(r):
    return (r["family"], r["bn"], r["tail"], r["csp"], r["cl"])


def start_worker(switches, configs, extra=()):
    env = {k: v for k, v in os.environ.items() if not k.startswith("LSPG_")}
    env.update(switches)
    args = [sys.executable, WORKER, *extra] + [",".join(map(str, c)) for c in configs]
    return subprocess.Popen(args, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)


def finish_worker(proc, timeout):
    try:
        out, err = proc.communicate(timeout=timeout)
    except subprocess.TimeoutExpired:
        proc.kill()
        proc.communicate()
        raise
    assert proc.returncode == 0, f"worker failed ({proc.returncode}):\n{out[-4000:]}\n{err[-4000:]}"
    return [json.loads(line) for line in out.splitlines() if line.startswith("{")]


# ------------------------------------------------------------------------------------------------------------ CPU tests
def test_matrix_reaches_every_kernel_instantiation():
    """Coverage of the GPU matrix, from the host planner alone: under each switch set the matrix's configs must together launch
    every conv instantiation of launch_layer (and nothing this table does not know), the split-K finisher, and - since
    every config runs in both modes - each of them and both input packers in FAST and PARITY."""
    assert set(MODES) == {"parity", "fast"}
    seen = defaultdict(set)
    finisher = []
    procs = {name: start_worker(switches, configs, extra=["--geo"]) for name, (switches, configs, _) in MATRIX.items()}
    for name, proc in procs.items():
        for r in finish_worker(proc, timeout=300):
            seen[_key(r)].add(name)
            if r["splitk_reduce"]:
                finisher.append((name, r["config"]))
    assert set(seen) <= ALL_INSTANTIATIONS, f"instantiations this test does not know: {set(seen) - ALL_INSTANTIATIONS}"
    assert set(seen) == ALL_INSTANTIATIONS, f"never launched by the matrix: {ALL_INSTANTIATIONS - set(seen)}"
    assert any(n == "finisher_split" and c[2] >= 8 for n, c in finisher), "splitk_reduce at large batch is not reached"
    for k in sorted(seen, key=str):
        print(f"{k}: {sorted(seen[k])}")


def _limbs(t):
    hi = t.half()
    return hi, (t - hi.float()).half()


@pytest.mark.parametrize("variant", ["normal", "large"])
def test_parity_bound_rejects_a_dropped_product_and_admits_fp32_accumulation(variant):
    """The PARITY bound of the GPU check, on host plans at 256x256 (recipe B), every layer fed the emulator's activations split
    into fp16 limbs: an fp32-accumulating emulation of the three-product scheme (plan_emulator.PARITY_PRODUCTS) stays within
    D/64 of float64, and a kernel that drops A_lo*B_hi or A_hi*B_lo exceeds the GPU check's bound D/8 + 2^-21 max|ref| on
    every layer (measured here: at least 5x above it)."""
    sd = O.make_state_dict(variant, "B")
    plan = E.HostPlan(variant, sd)
    torch.manual_seed(0)
    try:
        fm, cand = O.make_inputs(1, 256, 256)
        taps = {}
        E.run_plan(plan, torch.cat([fm, cand], 1), limbs=2, taps_out=taps)
        taps[0] = E.pack_input_s2d(torch.cat([fm, cand], 1))
        stored = {k: _limbs(v) for k, v in taps.items()}
        worst_ok, worst_drop = 0.0, float("inf")
        for i, L in enumerate(plan.layers):
            srcs = [stored[L.src[s]] for s in range(L.n_src)]
            res = sum(t.double() for t in stored[L.res]) if L.res >= 0 else None
            ref = E.run_layer(plan, i, srcs, res, 2, torch.float64)
            D = min(float(E.layer_linear(plan, i, srcs, 2, torch.float64, products=[p]).abs().max())
                    for p in [(1, 0), (0, 1)])
            bound = D * W.PARITY_D_FRACTION + 2 ** -21 * float(ref.abs().max())
            res32 = res.float() if res is not None else None
            kernel = E.run_layer(plan, i, srcs, res32, 2, torch.float32, products=E.PARITY_PRODUCTS)
            err = float((kernel.double() - ref).abs().max())
            assert err <= D / 64, f"layer {i} ({L.conv_key.decode()}): fp32 emulation err {err:.3g} > D/64 = {D / 64:.3g}"
            worst_ok = max(worst_ok, err / D)
            for drop in [(1, 0), (0, 1)]:
                prods = [p for p in E.PARITY_PRODUCTS if p != drop]
                bad = E.run_layer(plan, i, srcs, res32, 2, torch.float32, products=prods)
                e = float((bad.double() - ref).abs().max())
                assert e > bound, f"layer {i} ({L.conv_key.decode()}): dropping {drop} gives {e:.3g} <= bound {bound:.3g}"
                worst_drop = min(worst_drop, e / bound)
        print(f"{variant}: worst fp32 err/D {worst_ok:.3g}; smallest dropped-product err/bound {worst_drop:.3g}")
    finally:
        plan.close()


# ------------------------------------------------------------------------------------------------------------ GPU tests
def _print_table(name, recs):
    dev = next((r for r in recs if r["type"] == "device"), {})
    print(f"\n=== {name}: {dev.get('name')} env {dev.get('env')}")
    worst = {}
    for r in recs:
        if r["type"] == "layer":
            if r["nl"] == 2:
                print(f"{'x'.join(map(str, r['config'][2:]))} {r['config'][0]:6s} {r['config'][1]} parity L{r['layer']:02d} "
                      f"{r['inst']:34s} err {r['err']:.3g} D {r['D']:.3g} err/D {r['err_over_D']:.4f} max|y| {r['max_ref']:.4g}"
                      f"{'' if r['ok'] else '  FAIL'}")
                k = (r["inst"], "err/D")
                worst[k] = max(worst.get(k, 0.0), r["err_over_D"])
            else:
                stat = (f"err/ulp {r['err_over_ulp']:.3f} mismatch {r['mismatch']:.2e}" if "mismatch" in r
                        else f"err {r['err']:.3g} (tail, bound {r['bound']:.3g})")
                print(f"{'x'.join(map(str, r['config'][2:]))} {r['config'][0]:6s} {r['config'][1]} fast   L{r['layer']:02d} "
                      f"{r['inst']:34s} {stat} max|y| {r['max_ref']:.4g}{'' if r['ok'] else '  FAIL'}")
                if "mismatch" in r:
                    k = (r["inst"], "err/ulp, mismatch")
                    a, b = worst.get(k, (0.0, 0.0))
                    worst[k] = (max(a, r["err_over_ulp"]), max(b, r["mismatch"]))
                else:
                    k = (r["inst"], "err/bound")
                    worst[k] = max(worst.get(k, 0.0), r["err"] / r["bound"])
        elif r["type"] in ("packer", "boundary"):
            print(json.dumps(r))
    print(f"--- {name}: worst per instantiation")
    for (inst, what), v in sorted(worst.items()):
        print(f"  {inst:34s} {what:18s} {v if isinstance(v, float) else v}")


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MATRIX))
def test_every_layer_matches_float64(name):
    switches, configs, _ = MATRIX[name]
    recs = finish_worker(start_worker(switches, configs), timeout=1800)
    _print_table(name, recs)
    layers = [r for r in recs if r["type"] == "layer"]
    assert len({(tuple(r["config"]), r["mode"]) for r in layers}) == len(configs) * len(MODES)
    for r in layers:
        where = f"{r['config']} {r['mode']} layer {r['layer']} {r['key']} [{r['inst']}]"
        assert r["nan"] == 0 and r["negative"] == 0, f"{where}: {r['nan']} NaN, {r['negative']} negative after ReLU"
        if r["nl"] == 2:
            assert r["limb_violations"] == 0, f"{where}: {r['limb_violations']} stored elements break hi = fp16_rn(hi + lo)"
            assert r["err"] <= r["bound"], f"{where}: err {r['err']:.3g} > D/8 + 2^-21 max|y| = {r['bound']:.3g} (D {r['D']:.3g})"
        elif "mismatch" in r:
            assert r["err_over_ulp"] <= 1.0, f"{where}: error {r['err_over_ulp']:.3g} bf16 ulp"
            assert r["mismatch"] <= W.FAST_MISMATCH, f"{where}: {r['mismatch']:.3g} of the elements differ from bf16_rn(float64)"
        else:
            assert r["err"] <= r["bound"], f"{where}: tail err {r['err']:.3g} > {r['bound']:.3g}"
    packers = [r for r in recs if r["type"] == "packer"]
    assert len(packers) == len(configs) * len(MODES)
    for r in packers:
        assert sum(r["mismatches"]) == 0, f"{r['config']} {r['mode']}: packed input differs in {r['mismatches']} elements"
    bounds = [r for r in recs if r["type"] == "boundary"]
    assert len(bounds) == len(configs) * len(MODES)
    for r in bounds:
        assert r["ok"], r
