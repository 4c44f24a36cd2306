"""The oracle against its pins: golden fixtures generated from the reference module (the outputs of its own init and
its tensor2im included, oracle/make_golden_reference_checks.py) and known-answer facts."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import f2f_oracle as O

GOLDEN = sorted(p for p in glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.npz"))
                if not os.path.basename(p).startswith(("raster_", "a2h_", "f2f_")))  # raster_*: tests/test_raster_oracle.py
REF_CHECKS = os.path.join(os.path.dirname(__file__), "golden", "f2f_reference_checks.npz")


def test_key_grammar_and_parameter_counts():
    # SURVEY.md section 4 known-answer facts (probed on the reference module)
    for variant, n_keys, n_params, n_buf in (("large", 441, 121_789_760, 53_961), ("normal", 261, 76_203_840, 31_915)):
        spec = O.state_dict_spec(variant)
        assert len(spec) == n_keys
        params = sum(int(np.prod(s)) for r, s in spec.values() if r in ("conv", "bn_weight", "bn_bias"))
        bufs = sum(int(np.prod(s)) if s else 1 for r, s in spec.values() if r in ("bn_mean", "bn_var", "bn_count"))
        assert params == n_params and bufs == n_buf


def test_algorithmic_flops():
    assert O.conv_flops_per_frame("large", 512, 512) == 249_764_511_744
    assert O.conv_flops_per_frame("normal", 512, 512) == 166_075_564_032
    assert O.conv_flops_per_frame("normal", 1024, 1024) == 4 * 166_075_564_032


def test_zero_in_zero_out():
    sd = O.make_state_dict("normal", "A")
    out = O.generator_forward(sd, torch.zeros(1, 13, 256, 256), "normal")
    assert float(out.abs().max()) == 0.0


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_oracle_matches_reference_golden(path):
    g = np.load(path)
    variant, recipe = str(g["variant"]), str(g["recipe"])
    b, h, w, st = int(g["batch"]), int(g["height"]), int(g["width"]), int(g["stride"])
    sd = O.make_state_dict(variant, recipe)
    fm, cand = O.make_inputs(b, h, w)
    taps = {}
    out = O.inference(sd, fm, cand, variant) if False else O.generator_forward(sd, torch.cat([fm, cand], 1), variant, taps=taps)
    # the restatement and the reference run the same ATen kernels on the same host type: agree to fp32 noise
    assert np.abs(out[:, :, ::st, ::st].numpy() - g["out_sub"]).max() <= 2e-6
    d = out.double()
    assert abs(d.sum().item() - g["out_stats"][0]) <= 1e-3 * max(1.0, abs(g["out_stats"][0]))
    assert np.abs(taps["e1"][:, ::8, ::st * 2, ::st * 2].numpy() - g["e1_sub"]).max() <= 1e-5
    assert np.abs(taps["d1"][:, ::8, ::st * 2, ::st * 2].numpy() - g["d1_sub"]).max() <= 1e-4
    assert out.shape == (b, 3, h, w) and out.dtype == torch.float32
    assert float(out.abs().max()) < 1.0


def test_inference_concat_order():
    sd = O.make_state_dict("normal", "B")
    fm, cand = O.make_inputs(1, 256, 256)
    a = O.inference(sd, fm, cand, "normal")
    b = O.generator_forward(sd, torch.cat([fm, cand], 1), "normal")
    assert torch.equal(a, b)


@pytest.mark.parametrize("variant", ["normal", "large"])
def test_restatement_equals_live_reference_under_its_own_init(variant):
    """The reference module after networks.init_weights('normal', 0.02) under torch.manual_seed(0) (models/networks.py:347-378),
    as tests/golden/f2f_reference_checks.npz stores it: its key list, its weights (per-tensor sums) and its output."""
    g = np.load(REF_CHECKS)
    assert list(g[f"{variant}_keys"]) == list(O.state_dict_spec(variant).keys())
    sd = O.init_weights_state_dict(variant, int(g["init_seed"]))
    sums = np.array([sd[k].double().sum().item() for k in sd])
    assert np.allclose(sums, g[f"{variant}_weight_sums"], rtol=1e-9, atol=1e-9)      # the same weights as the reference's
    fm, cand = O.make_inputs(1, 256, 256, seed=int(g["input_seed"]))
    mine = O.generator_forward(sd, torch.cat([fm, cand], 1), variant)
    st = int(g["stride"])
    assert np.abs(mine[:, :, ::st, ::st].numpy() - g[f"{variant}_out_sub"]).max() <= 1e-6
    d, ref_stats = mine.double(), g[f"{variant}_out_stats"]
    assert abs(d.sum().item() - ref_stats[0]) <= 1e-6 * d.numel()
    assert abs(d.min().item() - ref_stats[2]) <= 1e-6 and abs(d.max().item() - ref_stats[3]) <= 1e-6


def test_tensor2im_restatement():
    g = torch.Generator().manual_seed(9)
    x = torch.tanh(torch.randn(2, 3, 16, 16, generator=g) * 2)
    x[0, 0, 0, 0], x[0, 1, 0, 0], x[0, 2, 0, 0] = -1.0, 1.0, 0.0        # boundary values: 0, 255, 127
    u = O.tensor2im(x)
    assert u.shape == (2, 16, 16, 3) and u.dtype == np.uint8
    assert tuple(u[0, 0, 0]) == (0, 255, 127)
    assert np.array_equal(np.load(REF_CHECKS)["tensor2im"], u)            # the reference's util/util.py:19-42 on x
