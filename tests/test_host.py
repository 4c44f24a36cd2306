"""Host-side logic, CPU only: the C ABI loads and exports what include/lspg.h declares, error behaviour,
the drop-in module's state-dict contract, and the launch plan (structure, packing, BatchNorm folding, tap
geometry) executed by the CPU plan emulator against the oracle.  No GPU compute here."""
import ctypes as C
import os
import re
import types

import numpy as np
import pytest
import torch

from livespeechportraits_b200 import _lib
from livespeechportraits_b200.generator import Feature2Face_G
from oracle import f2f_oracle as O
import plan_emulator as E

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def opt(size="normal", **kw):
    d = dict(isTrain=False, size=size, n_downsample_G=8, ngf=64, fp16=0)
    d.update(kw)
    return types.SimpleNamespace(**d)


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "lspg.h")).read()
    declared = set(re.findall(r"^(?:int|const char\*)\s+(lspg_\w+)\s*\(", header, flags=re.M))
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    for name in declared:
        assert getattr(lib, name) is not None


def test_create_argument_errors_and_no_cpu_path():
    lib = _lib.load()
    h = C.c_void_p()
    assert lib.lspg_create(C.byref(h), 7, 64, 8, 13, 3, -1) == -1          # LSPG_EINVAL
    assert b"variant" in lib.lspg_last_error()
    assert lib.lspg_create(C.byref(h), 0, 48, 8, 13, 3, -1) == -1
    assert lib.lspg_create(C.byref(h), 0, 64, 8, 13, 4, -1) == -1
    if not torch.cuda.is_available():
        assert lib.lspg_create(C.byref(h), 0, 64, 8, 13, 3, 0) == -2        # LSPG_ENODEV: no device, no fallback
    assert lib.lspg_create(C.byref(h), 0, 64, 8, 13, 3, -1) == 0
    buf = (C.c_float * 4)()
    rc = lib.lspg_forward(h, buf, 0, buf, 0, buf, 1, 256, 256, buf, 16, 0, None)
    assert rc == -2 and b"no CPU path" in lib.lspg_last_error()
    # the rasteriser entry point has no CPU path either, and validates its arguments first
    assert lib.lspg_draw_feature_maps(h, buf, None, 0, buf, 1, 256, 256, None) == -2 and b"no CPU path" in lib.lspg_last_error()
    assert lib.lspg_draw_feature_maps(h, None, None, 0, buf, 1, 256, 256, None) == -1
    assert lib.lspg_draw_feature_maps(h, buf, buf, 7, buf, 1, 256, 256, None) == -1     # odd shoulder count
    assert lib.lspg_draw_feature_maps(h, buf, None, 0, buf, 0, 256, 256, None) == -1
    need = C.c_size_t()
    assert lib.lspg_workspace_bytes(h, 1, 300, 256, 0, C.byref(need)) == -1  # H must be a multiple of 256
    assert lib.lspg_workspace_bytes(h, 1, 256, 256, 5, C.byref(need)) == -1  # unknown mode
    assert lib.lspg_workspace_bytes(h, 2, 512, 512, 1, C.byref(need)) == 0 and need.value > 0
    lib.lspg_destroy(h)


def test_load_weights_validation_and_module_prefix():
    lib = _lib.load()
    h = C.c_void_p()
    assert lib.lspg_create(C.byref(h), 0, 64, 8, 13, 3, -1) == 0
    w = torch.randn(64, 13, 3, 3)
    arr = (_lib.LspgTensor * 1)()
    arr[0].name = b"module.netG.model.model.0.weight"               # DataParallel prefix is accepted
    arr[0].data = C.cast(w.data_ptr(), C.POINTER(C.c_float))
    arr[0].numel = w.numel()
    assert lib.lspg_load_weights(h, arr, 1) == 0
    arr[0].numel = w.numel() - 1
    assert lib.lspg_load_weights(h, arr, 1) == -1
    assert b"elements" in lib.lspg_last_error()
    lib.lspg_destroy(h)


@pytest.mark.parametrize("variant", ["normal", "large"])
def test_module_state_dict_contract(variant):
    net = Feature2Face_G(opt(variant))
    spec = O.state_dict_spec(variant)
    sd = net.state_dict()
    assert list(sd.keys()) == list(spec.keys())
    assert all(tuple(sd[k].shape) == tuple(s) for k, (r, s) in spec.items())
    res = net.load_state_dict(O.make_state_dict(variant, "B"), strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    # the reference's init_weights (networks.py:347-378) dispatches on class names: the leaves are real modules
    names = {m.__class__.__name__ for m in net.modules()}
    assert "Conv2d" in names and "BatchNorm2d" in names
    n_conv = sum(1 for m in net.modules() if isinstance(m, torch.nn.Conv2d))
    assert n_conv == (76 if variant == "large" else 46)


def test_module_refuses_cpu_and_train_mode():
    net = Feature2Face_G(opt("normal")).eval()
    with pytest.raises(RuntimeError, match="no CPU path"):
        net(torch.zeros(1, 13, 256, 256))
    net.train()
    with pytest.raises(NotImplementedError):
        net(torch.zeros(1, 13, 256, 256))
    with pytest.raises(NotImplementedError):
        Feature2Face_G(opt("small"))


@pytest.mark.parametrize("variant,recipe", [("normal", "B"), ("large", "A")])
def test_launch_plan_reproduces_the_oracle(variant, recipe):
    sd = O.make_state_dict(variant, recipe)
    plan = E.HostPlan(variant, sd)
    try:
        kinds = [L.kind for L in plan.layers]
        assert kinds[0] == E.KIND_HEAD and kinds[-1] == E.KIND_TAIL
        assert len(kinds) == (76 if variant == "large" else 46)
        fm, cand = O.make_inputs(1, 256, 256)
        x = torch.cat([fm, cand], 1)
        ref = O.generator_forward(sd, x, variant)
        out = E.run_plan(plan, x, limbs=2)
        # hi+lo fp16 weights carry 22 mantissa bits: the plan (fp32 activations here) must reproduce the oracle to ~1e-4
        assert (out - ref).abs().max().item() <= 2e-4
        out_bf16 = E.run_plan(plan, x, limbs=1, round_act=lambda t: t.bfloat16().float())
        assert (out_bf16 - ref).abs().max().item() <= 5e-2
    finally:
        plan.close()


def test_bn_fold_matches_batchnorm_formula():
    sd = O.make_state_dict("normal", "B")
    plan = E.HostPlan("normal", sd)
    try:
        for i, L in enumerate(plan.layers):
            s, b = plan.affine(i)
            if L.has_bn:
                key = L.bn_key.decode()
                inv = 1.0 / torch.sqrt(sd[key + ".running_var"] + 1e-5)
                assert torch.allclose(s[: L.cout], sd[key + ".weight"] * inv, rtol=1e-6, atol=1e-7)
                assert torch.allclose(b[: L.cout], sd[key + ".bias"] - sd[key + ".running_mean"] * sd[key + ".weight"] * inv,
                                      rtol=1e-5, atol=1e-6)
            else:
                assert float((s - 1).abs().max()) == 0 and float(b.abs().max()) == 0
    finally:
        plan.close()


def test_flops_accounting_matches_oracle():
    lib = _lib.load()
    for variant in ("normal", "large"):
        h = C.c_void_p()
        assert lib.lspg_create(C.byref(h), _lib.LSPG_VARIANT[variant], 64, 8, 13, 3, -1) == 0
        v = C.c_double()
        assert lib.lspg_flops_per_frame(h, 512, 512, C.byref(v)) == 0
        assert int(v.value) == O.conv_flops_per_frame(variant, 512, 512)
        lib.lspg_destroy(h)


@pytest.mark.skipif(not O.reference_available(), reason="reference checkout not present on this machine")
def test_drop_in_through_the_reference_model_class(tmp_path):
    """create_model -> Feature2FaceModel -> our generator; load_networks round-trips a 'module.'-prefixed pkl."""
    import contextlib
    import io
    import sys
    O.reference_generator("normal")            # puts the reference on sys.path
    from livespeechportraits_b200 import generator as G
    import models.feature2face_G as ref_mod  # type: ignore
    original = ref_mod.Feature2Face_G
    try:
        G.install()
        sd = O.make_state_dict("normal", "B")
        ckpt = tmp_path / "Feature2Face.pkl"
        torch.save({"module." + k: v for k, v in sd.items()}, ckpt)
        o = O.reference_opt("normal", load_epoch=str(ckpt), checkpoints_dir=str(tmp_path))
        with contextlib.redirect_stdout(io.StringIO()):
            from models import create_model  # type: ignore
            model = create_model(o)
            model.setup(o)
            model.eval()
        g = model.Feature2Face_G
        assert isinstance(g, G.Feature2Face_G) and not g.training
        got = g.state_dict()
        assert all(torch.equal(got[k], v) for k, v in sd.items())
        with pytest.raises(RuntimeError, match="no CPU path"):
            model.inference(torch.zeros(1, 1, 256, 256), torch.zeros(1, 12, 256, 256))
    finally:
        ref_mod.Feature2Face_G = original


def test_tile_decode_division_by_multiply_high_is_exact():
    """decode_tile divides tile indices by launch-time constants with multiply-high + shift (csrc/conv_umma.cuh fast_div)."""
    import random
    lib = _lib.load()
    rng = random.Random(0)
    q = C.c_uint32()
    divisors = list(range(1, 300)) + [2 ** k for k in range(1, 31)] + [2 ** k - 1 for k in range(2, 31)] + \
        [2 ** k + 1 for k in range(1, 30)] + [37, 74, 148, 8192, 9472, 65535, 65537, 2 ** 31 - 1] + [rng.randrange(1, 2 ** 31) for _ in range(300)]
    for d in divisors:
        ns = [0, 1, d - 1, d, d + 1, 2 * d - 1, 2 * d, 2 ** 31 - 1, 2 ** 31 - d] + [rng.randrange(0, 2 ** 31) for _ in range(40)]
        for n in ns:
            if 0 <= n < 2 ** 31:
                assert lib.lspg_debug_fast_div(n, d, C.byref(q)) == 0
                assert q.value == n // d, (n, d, q.value)
    assert lib.lspg_debug_fast_div(5, 0, C.byref(q)) == -1
    assert lib.lspg_debug_fast_div(2 ** 31, 3, C.byref(q)) == -1


def _geo_table(variant, batch, height=512, width=512):
    lib = _lib.load()
    h = C.c_void_p()
    assert lib.lspg_create(C.byref(h), _lib.LSPG_VARIANT[variant], 64, 8, 13, 3, -1) == 0
    n = C.c_int()
    assert lib.lspg_num_layers(h, C.byref(n)) == 0
    out = []
    for i in range(n.value):
        g = _lib.LspgLayerGeo()
        assert lib.lspg_debug_layer_geo(h, i, batch, height, width, C.byref(g)) == 0
        info = _lib.LspgLayerInfo()
        assert lib.lspg_layer_info_get(h, i, C.byref(info)) == 0
        out.append((info, g))
    need = C.c_size_t()
    assert lib.lspg_workspace_bytes(h, batch, height, width, 1, C.byref(need)) == 0
    lib.lspg_destroy(h)
    return out, need.value


@pytest.mark.parametrize("variant,batch", [("large", 1), ("large", 16), ("large", 32), ("large", 37), ("normal", 5), ("normal", 32)])
def test_planner_invariants(variant, batch):
    """The launch planner (layer_geo in csrc/lspg.cu) on the host: tile shapes, kernel choice, split-K and wave rules."""
    table, ws = _geo_table(variant, batch)
    sms = 148
    for info, g in table:
        assert g.tile_w * g.tile_h * g.tile_n == 128                       # one UMMA M tile
        assert g.bn in (16, 64, 128, 256) and info.cout_pad % g.bn == 0 and g.n_tiles == info.cout_pad // g.bn
        tiles = g.m_tiles * g.n_tiles * g.n_phases
        if g.kernel == 2:                                                    # cta_group::2: pairs of neighbouring M tiles
            assert g.m_tiles % 2 == 0 and g.n_split == 1 and g.ctas % 2 == 0 and (g.tile_w, g.tile_h) == (8, 16)
        if g.kernel in (1, 2):
            assert info.kind != 2                                            # stride-2 convs use the per-tap kernel
        if g.n_split > 1:
            assert g.kernel != 2
            assert tiles * g.n_split <= sms                                  # split-K never spills into a second wave
            assert (g.n_split - 1) * g.split_len < g.k_items <= g.n_split * g.split_len   # every split has work
            if g.cluster_split:
                # the splits of a tile are one thread-block cluster (DSMEM reduction): portable cluster size, one CTA per
                # (tile, split), nothing in the global scratch, no finisher launch
                assert g.cluster_split == g.n_split and g.n_split in (2, 4, 8)
                assert g.ctas == tiles * g.n_split and g.partial_bytes == 0
                assert g.bn in (64, 128) and info.kind != 4
            else:
                assert g.partial_bytes == g.n_split * tiles * 128 * g.bn * 4
        else:
            assert g.partial_bytes == 0 and g.cluster_split == 0
        # the launch's cluster: CTA pairs, the CTAs of a cluster split, or pairs of patch CTAs that multicast their weight
        # stages when the layer fills a wave without split-K
        if g.kernel == 2:
            assert g.cta_cluster == 2
        elif g.cluster_split:
            assert g.cta_cluster == g.cluster_split
        elif g.kernel == 1:
            assert g.cta_cluster == (2 if g.n_split == 1 and g.m_tiles % 2 == 0 and tiles >= sms else 1)
        else:
            assert g.cta_cluster == 1
        assert 1 <= g.ctas <= sms
    assert ws > max(g.partial_bytes for _, g in table)
    n_split_layers = sum(1 for _, g in table if g.n_split > 1)
    n_cluster = sum(1 for _, g in table if g.cluster_split)
    if batch >= 8:
        assert n_split_layers >= 10 and n_cluster == n_split_layers       # from 8 frames up every split layer reduces inside its cluster
    else:
        assert n_cluster == 0 and (batch != 1 or n_split_layers >= 40)     # below that (measured slower) the finisher kernel stays


@pytest.mark.parametrize("variant,batch,height,width,mode", [("normal", 1, 256, 256, 1), ("normal", 3, 512, 256, 0),
                                                             ("large", 32, 512, 512, 1), ("large", 5, 256, 1024, 0)])
def test_tensor_offsets_are_aligned_disjoint_and_inside_the_workspace(variant, batch, height, width, mode):
    """lspg_debug_tensor_offset: every limb of every activation tensor starts on a 1 KB boundary of the aligned workspace,
    no two overlap, and all of them - and the split-K scratch after them - fit in lspg_workspace_bytes minus the slack that
    aligning the caller's pointer may use."""
    lib = _lib.load()
    h = C.c_void_p()
    assert lib.lspg_create(C.byref(h), _lib.LSPG_VARIANT[variant], 64, 8, 13, 3, -1) == 0
    try:
        need = C.c_size_t()
        assert lib.lspg_workspace_bytes(h, batch, height, width, mode, C.byref(need)) == 0
        nt = C.c_int()
        lib.lspg_num_tensors(h, C.byref(nt))
        spans = []
        for t in range(nt.value):
            c, th, tw = C.c_int(), C.c_int(), C.c_int()
            assert lib.lspg_tensor_shape(h, t, height, width, C.byref(c), C.byref(th), C.byref(tw)) == 0
            nbytes = batch * th.value * tw.value * c.value * 2
            for limb in range(2 if mode == 1 else 1):
                off = C.c_size_t()
                assert lib.lspg_debug_tensor_offset(h, t, limb, batch, height, width, mode, C.byref(off)) == 0
                assert off.value % 1024 == 0
                spans.append((off.value, off.value + nbytes))
        spans.sort()
        assert spans[0][0] == 0
        assert all(a[1] <= b[0] for a, b in zip(spans, spans[1:])), "activation tensors overlap"
        n = C.c_int()
        lib.lspg_num_layers(h, C.byref(n))
        partial = 0
        for i in range(n.value):
            g = _lib.LspgLayerGeo()
            assert lib.lspg_debug_layer_geo(h, i, batch, height, width, C.byref(g)) == 0
            partial = max(partial, g.partial_bytes)
        assert -(-spans[-1][1] // 1024) * 1024 + partial <= need.value - 1024
        off = C.c_size_t()
        assert lib.lspg_debug_tensor_offset(h, nt.value, 0, batch, height, width, mode, C.byref(off)) == -1
        assert lib.lspg_debug_tensor_offset(h, 0, 2 if mode == 1 else 1, batch, height, width, mode, C.byref(off)) == -1
        assert lib.lspg_debug_tensor_offset(h, 0, 0, batch, 300, width, mode, C.byref(off)) == -1
    finally:
        lib.lspg_destroy(h)


def test_planner_picks_the_n_tile_with_fewer_waves():
    def bn_of(batch, cout, hw):
        table, _ = _geo_table("large", batch)
        return {g.bn for info, g in table if info.kind == 1 and info.cout == cout and g.kernel == 2
                and g.m_tiles == batch * (hw // 8) * (hw // 16)}
    # 256 -> 256 @64^2, 16 frames: 256 pairs of N=256 tiles = 4 waves of 74 clusters; 512 pairs of N=128 = 7 half-size waves
    assert bn_of(16, 256, 64) == {128}
    assert bn_of(32, 256, 64) == {256}        # 7 waves vs 14 half-size waves: tie -> the wider tile
    assert bn_of(16, 512, 32) == {256}        # 2 vs 4 half-size: tie
    assert bn_of(32, 512, 32) == {128}        # 4 vs 7 half-size
    # the 64-channel layers always take the resident-weights N=64 pair kernel
    assert bn_of(16, 64, 256) == {64}


@pytest.mark.parametrize("variant", ["normal", "large"])
def test_accepted_shapes_tile_every_level_and_768_is_rejected(variant):
    """check_shape (csrc/lspg.cu): a shape is accepted only if the tiles of every layer cover its grid exactly.  768x768 is a
    multiple of 256 (the reference renders it) but its 24/12/6/3-pixel levels do not tile into the power-of-two boxes: it must
    be refused with LSPG_EINVAL, not rendered wrong."""
    lib = _lib.load()
    h = C.c_void_p()
    assert lib.lspg_create(C.byref(h), _lib.LSPG_VARIANT[variant], 64, 8, 13, 3, -1) == 0
    need = C.c_size_t()
    for (hh, ww) in [(768, 768), (512, 768), (768, 256), (1280, 1024)]:
        assert lib.lspg_workspace_bytes(h, 1, hh, ww, 1, C.byref(need)) == -1, (hh, ww)
        assert b"not supported" in lib.lspg_last_error()
        g = _lib.LspgLayerGeo()
        assert lib.lspg_debug_layer_geo(h, 0, 1, hh, ww, C.byref(g)) == -1
    n = C.c_int()
    lib.lspg_num_layers(h, C.byref(n))
    for (hh, ww) in [(256, 256), (512, 512), (512, 256), (256, 1024), (1024, 1024), (2048, 512)]:
        for batch in (1, 3, 32):
            assert lib.lspg_workspace_bytes(h, batch, hh, ww, 1, C.byref(need)) == 0, (hh, ww, lib.lspg_last_error())
            for i in range(n.value):
                g = _lib.LspgLayerGeo()
                info = _lib.LspgLayerInfo()
                assert lib.lspg_debug_layer_geo(h, i, batch, hh, ww, C.byref(g)) == 0
                assert lib.lspg_layer_info_get(h, i, C.byref(info)) == 0
                c, th, tw = C.c_int(), C.c_int(), C.c_int()
                # sampling grid of the layer = its first source for upsample/tail convs, its output otherwise
                tid = info.src[0] if info.kind in (3, 4) else info.out
                assert lib.lspg_tensor_shape(h, tid, hh, ww, C.byref(c), C.byref(th), C.byref(tw)) == 0
                grid = th.value * tw.value * batch
                assert th.value % g.tile_h == 0 and tw.value % g.tile_w == 0
                assert g.m_tiles * 128 >= grid                                 # tiles cover the grid (image padding only)
                assert g.m_tiles == (tw.value // g.tile_w) * (th.value // g.tile_h) * -(-batch // g.tile_n)
    lib.lspg_destroy(h)


def test_module_copies_do_not_share_the_native_handle():
    """copy.deepcopy / pickling reset the native state (a shared handle would be destroyed twice); DataParallel replication
    over several devices is refused with a pointer to the process-per-GPU path."""
    import copy
    import pickle
    net = Feature2Face_G(opt("normal")).eval()
    net.load_state_dict(O.make_state_dict("normal", "B"))
    net._info_handle()                                   # creates a host-only native handle
    assert net._host_handle
    for clone in (copy.deepcopy(net), pickle.loads(pickle.dumps(net))):
        assert not clone._handle and not clone._host_handle and clone._workspaces == {} and clone._weights_dirty
        assert not clone.training
        a, b = net.state_dict(), clone.state_dict()
        assert list(a) == list(b) and all(torch.equal(a[k], b[k]) for k in a)
        assert all(p is not q for p, q in zip(net.parameters(), clone.parameters()))
        assert clone.launches_per_forward() == net.launches_per_forward()       # the copy builds its own handle on demand
        assert clone._host_handle and clone._host_handle.value != net._host_handle.value
    with pytest.raises(NotImplementedError, match="ShardedRenderer"):
        net._replicate_for_data_parallel()
    with pytest.raises(NotImplementedError, match="ShardedRenderer"):
        torch.nn.parallel.replicate(net, [0, 1]) if torch.cuda.device_count() > 1 else net._replicate_for_data_parallel()


def test_package_exports_public_names():
    import livespeechportraits_b200 as pkg
    for name in ("Feature2Face_G", "install", "ClipRenderer", "ShardedRenderer", "partition"):
        assert hasattr(pkg, name)


def test_planner_invariants_over_random_problem_sizes():
    """Property test of layer_geo / workspace sizing through the C ABI (host only): any accepted (batch, H, W) gives tiles
    that cover every level, split-K that stays inside one wave with non-empty K ranges, cluster splits of portable size, and a
    workspace at least as large as the activations + the largest partial buffer."""
    from hypothesis import given, settings, strategies as st
    lib = _lib.load()
    handles = {}
    for variant in ("normal", "large"):
        h = C.c_void_p()
        assert lib.lspg_create(C.byref(h), _lib.LSPG_VARIANT[variant], 64, 8, 13, 3, -1) == 0
        n = C.c_int()
        lib.lspg_num_layers(h, C.byref(n))
        handles[variant] = (h, n.value)

    @settings(max_examples=60, deadline=None)
    @given(st.sampled_from(["normal", "large"]), st.integers(1, 96), st.sampled_from([256, 512, 1024]), st.sampled_from([256, 512, 1024]),
           st.sampled_from([0, 1]))
    def check(variant, batch, hh, ww, mode):
        h, nl = handles[variant]
        need = C.c_size_t()
        assert lib.lspg_workspace_bytes(h, batch, hh, ww, mode, C.byref(need)) == 0, lib.lspg_last_error()
        act = 0
        nt = C.c_int()
        lib.lspg_num_tensors(h, C.byref(nt))
        for t in range(nt.value):
            c, th, tw = C.c_int(), C.c_int(), C.c_int()
            lib.lspg_tensor_shape(h, t, hh, ww, C.byref(c), C.byref(th), C.byref(tw))
            act += batch * th.value * tw.value * c.value * 2 * (2 if mode == 1 else 1)
        worst_partial = 0
        for i in range(nl):
            g = _lib.LspgLayerGeo()
            assert lib.lspg_debug_layer_geo(h, i, batch, hh, ww, C.byref(g)) == 0
            assert g.tile_w * g.tile_h * g.tile_n == 128 and g.m_tiles >= 1 and g.n_tiles >= 1
            tiles = g.m_tiles * g.n_tiles * g.n_phases
            assert 1 <= g.ctas <= 148
            if g.n_split > 1:
                assert tiles * g.n_split <= 148 and (g.n_split - 1) * g.split_len < g.k_items <= g.n_split * g.split_len
                assert g.cluster_split in (0, 2, 4, 8) and (g.cluster_split == 0 or g.cluster_split == g.n_split)
                assert (g.cluster_split != 0) == (batch >= 8) or g.partial_bytes > 0
            if g.kernel == 2:
                assert g.m_tiles % 2 == 0 and g.ctas % 2 == 0 and g.n_split == 1
            worst_partial = max(worst_partial, g.partial_bytes)
        assert need.value >= act + worst_partial

    try:
        check()
    finally:
        for h, _ in handles.values():
            lib.lspg_destroy(h)
