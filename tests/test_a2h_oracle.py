"""Row N4 (SURVEY.md 8f), CPU part: the oracle of the Audio2Headpose loop pinned against golden vectors generated from the
reference; the incremental recurrence the CUDA kernel runs checked against the oracle - in its
float64 host emulator (algorithmic equivalence) and with the arrays lsph_load_weights actually packed (host logic of the
C ABI, no GPU); the C ABI's argument checking."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from livespeechportraits_b200 import _lib, headpose
from oracle import a2h_oracle as A
import a2h_incremental as INC

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(os.path.dirname(__file__), "golden", "a2h_B_60.npz")
GOLD_LOOP = os.path.join(os.path.dirname(__file__), "golden", "a2h_live_loop.npz")
# Intra-op CPU threads the reference ran with when tests/golden/a2h_*.npz were written.  ATen's CPU matmuls split their
# sums by thread count (1 or 12+ threads round differently from 2-8), and the loop feeds those last bits back into its
# history, so the restatement reproduces the stored vectors only with the same count.
GOLDEN_THREADS = 8


@pytest.fixture
def golden_threads():
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


def test_known_answers():
    opt = A.default_opt()
    assert A.dilations(opt) == (1, 2, 4, 8, 16, 32, 64) * 2
    assert A.receptive_field(opt) == 255 and opt.A2H_receptive_field == 255          # demo.py:163-166
    assert A.output_size(opt) == 25
    spec = A.state_dict_spec(opt)
    assert len(spec) == 185
    assert sum(int(np.prod(s)) for k, s in spec.items() if not k.endswith("num_batches_tracked")) == 4267939


@pytest.mark.usefixtures("golden_threads")
def test_oracle_matches_golden_from_the_reference():
    """tests/golden/a2h_B_60.npz was written by oracle/make_golden_a2h.py from the UNMODIFIED Audio2HeadposeModel."""
    g = np.load(GOLD)
    opt = A.default_opt()
    sd = A.make_state_dict(opt, str(g["recipe"]), int(g["weight_seed"]))
    audio = A.make_audio_feats(int(g["n_audio"]), opt, int(g["audio_seed"]))
    noise = A.reference_noise(int(g["n_audio"]) - opt.frame_future, opt.A2H_GMM_ndim, 1, int(g["torch_seed"]))
    assert np.array_equal(noise, g["noise"])
    pred, params = A.generate_sequences(sd, audio, g["pre_headpose"], noise, opt, float(g["sigma_scale"]), return_params=True)
    assert np.abs(pred - g["pred"]).max() <= 2e-6
    assert np.abs(params - g["params"]).max() <= 2e-6


@pytest.mark.usefixtures("golden_threads")
def test_oracle_matches_the_live_reference_loop():
    """tests/golden/a2h_live_loop.npz holds what the UNMODIFIED Audio2HeadposeModel computed (oracle/make_golden_reference_checks.py):
    its key list, its generate_sequences loop under torch.manual_seed(11) and one full-window forward of its module."""
    g = np.load(GOLD_LOOP)
    opt = A.default_opt()
    assert list(g["keys"]) == list(A.state_dict_spec(opt).keys())
    for recipe, seed in (("A", 1), ("B", 2)):
        sd = A.make_state_dict(opt, recipe, seed)
        audio = A.make_audio_feats(36, opt, seed)
        pre = np.linspace(-0.2, 0.3, 12).astype(np.float32)
        noise = A.reference_noise(36 - 15, 12, 1, seed=11)
        mine = A.generate_sequences(sd, audio, pre, noise, opt, 0.3)
        ref = g[f"{recipe}_pred"]
        assert ref.shape == (21, 12) and ref.dtype == np.float64
        assert np.abs(ref - mine).max() <= 1e-6, recipe
        # one full-window forward against the module's own forward
        hist = torch.from_numpy(np.random.Generator(np.random.PCG64(11)).standard_normal((1, 255, 12)).astype(np.float32))
        aud = torch.from_numpy(A.make_audio_feats(255, opt, 5)).unsqueeze(0)
        assert torch.allclose(torch.from_numpy(g[f"{recipe}_forward"]), A.audio2headpose_forward(sd, hist, aud, opt), atol=1e-6)


@pytest.mark.parametrize("recipe", ["A", "B"])
def test_incremental_recurrence_equals_the_full_window_loop(recipe):
    opt = A.default_opt()
    sd = A.make_state_dict(opt, recipe)
    audio = A.make_audio_feats(50, opt)
    pre = np.linspace(-0.3, 0.4, 12).astype(np.float32)
    noise = A.reference_noise(35, 12, 1, seed=3)
    ref, rp = A.generate_sequences(sd, audio, pre, noise, opt, 0.3, return_params=True)
    inc, ip = INC.generate_incremental(sd, audio, pre, noise, opt, 0.3, return_params=True)
    assert np.abs(ref - inc).max() <= 2e-5 and np.abs(rp - ip).max() <= 2e-5


def _handle(opt, sd, device=-1):
    lib = _lib.load()
    cfg = headpose.config_from_opt(opt)
    h = C.c_void_p()
    assert lib.lsph_create(C.byref(h), C.byref(cfg), device) == 0, lib.lsph_last_error()
    names, keep = [], []
    for k, v in sd.items():
        if not k.endswith("num_batches_tracked"):
            names.append(("module." + k).encode())                   # the DataParallel prefix is accepted
            keep.append(v.float().contiguous())
    arr = (_lib.LspgTensor * len(keep))()
    for i, (n, t) in enumerate(zip(names, keep)):
        arr[i].name, arr[i].data, arr[i].numel = n, C.cast(t.data_ptr(), C.POINTER(C.c_float)), t.numel()
    assert lib.lsph_load_weights(h, arr, len(keep)) == 0, lib.lsph_last_error()
    return lib, h, (arr, keep)


def test_packed_weights_drive_the_recurrence_to_the_oracle():
    """The arrays the kernel reads (w_fg tap order, residual/skip row order, folded BatchNorm, cond + conv biases), taken
    back through the C ABI of a host-only handle and run through the kernel's recurrence in numpy."""
    opt = A.default_opt()
    sd = A.make_state_dict(opt, "B", 4)
    lib, h, _keep = _handle(opt, sd)
    L, R, S, H = 14, 128, 256, 512

    def packed(which, n):
        buf = np.empty(n, np.float32)
        assert lib.lsph_debug_packed(h, which, buf.ctypes.data_as(C.c_void_p), n) == 0, lib.lsph_last_error()
        return buf.astype(np.float64)
    w_fg = packed(0, L * 2 * R * 2 * R).reshape(L, 2 * R, 2 * R)
    w_rs = packed(1, L * (R + S) * R).reshape(L, R + S, R)
    b_rs = packed(2, L * (R + S)).reshape(L, R + S)
    w_cond = packed(3, L * 2 * R * H).reshape(L * 2 * R, H)
    b_cond = packed(4, L * 2 * R)
    scale0, shift0 = packed(5, H), packed(6, H)
    assert lib.lsph_debug_packed(h, 9, None, 0) == -1
    lib.lsph_destroy(h)
    f64 = lambda k: sd[k].double().numpy()      # noqa: E731
    audio = A.make_audio_feats(44, opt, 2).astype(np.float64)
    pre = np.linspace(0.2, -0.1, 12)
    noise = A.reference_noise(29, 12, 1, seed=8)
    ref, rp = A.generate_sequences(sd, audio.astype(np.float32), pre.astype(np.float32), noise, opt, 0.3, return_params=True)
    lre = INC.lrelu
    # hoisted audio path exactly as the three GEMMs compute it
    ds1 = lre((audio @ f64("audio_downsample.0.weight").T) * scale0 + shift0)
    ds2 = ds1 @ f64("audio_downsample.3.weight").T + f64("audio_downsample.3.bias")
    cond = (ds2 @ w_cond.T + b_cond).reshape(-1, L, 2 * R)
    W1, b1 = f64("WaveNet.start_conv1.weight")[:, :, 0], f64("WaveNet.start_conv1.bias")
    W2, b2 = f64("WaveNet.start_conv2.weight")[:, :, 0], f64("WaveNet.start_conv2.bias")
    E1, e1 = f64("WaveNet.end_conv_1.weight")[:, :, 0], f64("WaveNet.end_conv_1.bias")
    E2, e2 = f64("WaveNet.end_conv_2.weight")[:, :, 0], f64("WaveNet.end_conv_2.bias")
    dil, rf, ff, n_audio = A.dilations(opt), 255, 15, 44
    T = rf - 1 + 29
    X = np.zeros((L, T, R))
    hcur = pre.copy()
    pred, params = np.zeros((29, 12)), np.zeros((29, 25))
    for t in range(T):
        arow = min(max(t + ff - (rf - 1), 0), n_audio - 1)
        x = lre(W2 @ lre(W1 @ hcur + b1) + b2)
        skip = np.zeros(S)
        for l in range(L):
            X[l, t] = x
            xd = X[l, t - dil[l]] if t - dil[l] >= 0 else np.zeros(R)
            fg = w_fg[l] @ np.concatenate([xd, x]) + cond[arow, l]
            z = np.tanh(fg[:R]) / (1.0 + np.exp(-fg[R:]))
            rs = w_rs[l] @ z + b_rs[l]
            skip += rs[R:]
            x = rs[:R] + x
        if t >= rf - 1:
            i = t - (rf - 1)
            out = E2 @ lre(E1 @ lre(skip) + e1) + e2
            params[i] = out
            hcur = noise[i] * (np.exp(-out[13:25]) * 0.3) + out[1:13]
            pred[i] = hcur
    assert np.abs(pred - ref).max() <= 2e-5 and np.abs(params - rp).max() <= 2e-5


def test_c_abi_exports_and_argument_checks():
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "lsph.h")).read()
    declared = set(re.findall(r"^(?:int|const char\*)\s+(lsph_\w+)\s*\(", header, flags=re.M))
    assert declared == set(_lib.SYMBOLS_H), declared ^ set(_lib.SYMBOLS_H)
    opt = A.default_opt()
    h = C.c_void_p()
    for field, bad in (("skip_ch", 128), ("residual_ch", 64), ("kernel_size", 3), ("input_ch", 40), ("ncenter", 0), ("layers", 9)):
        cfg = headpose.config_from_opt(opt)
        setattr(cfg, field, bad)
        assert lib.lsph_create(C.byref(h), C.byref(cfg), -1) == -1, field
    cfg = headpose.config_from_opt(opt)
    if not torch.cuda.is_available():
        assert lib.lsph_create(C.byref(h), C.byref(cfg), 0) == -2                      # no device, no fallback
    assert lib.lsph_create(C.byref(h), C.byref(cfg), -1) == 0
    buf = (C.c_float * 4)()
    assert lib.lsph_generate(h, buf, 40, buf, buf, None, 0.3, buf, None, 0, None) == -2 and b"no CPU path" in lib.lsph_last_error()
    arr = (_lib.LspgTensor * 1)()
    w = torch.zeros(512, 1024)
    arr[0].name, arr[0].data, arr[0].numel = b"audio_downsample.0.weight", C.cast(w.data_ptr(), C.POINTER(C.c_float)), w.numel()
    assert lib.lsph_load_weights(h, arr, 1) == -4 and b"missing parameter" in lib.lsph_last_error()   # every parameter is required
    arr[0].numel = 5
    assert lib.lsph_load_weights(h, arr, 1) == -1
    lib.lsph_destroy(h)
    with pytest.raises(RuntimeError, match="no CPU path"):
        headpose.HeadposeGenerator(opt, A.make_state_dict(opt, "A"), device=torch.device("cpu"))
    with pytest.raises(NotImplementedError):
        headpose.config_from_opt(A.default_opt(feature_decoder="LSTM"))


@pytest.mark.skipif(not A.reference_available(), reason="reference checkout not present on this machine")
def test_install_swaps_the_loop_on_the_reference_model_class():
    """headpose.install() replaces Audio2HeadposeModel.generate_sequences (what demo.py:212 calls); the model object, its
    module and weights stay the reference's own.  Without a GPU the swapped loop refuses to run (no CPU path)."""
    opt = A.default_opt()
    m = A.reference_model(opt, A.make_state_dict(opt, "A"))
    import models.audio2headpose_model as ref_mod  # type: ignore
    original = ref_mod.Audio2HeadposeModel.generate_sequences
    try:
        headpose.install()
        assert ref_mod.Audio2HeadposeModel.generate_sequences is headpose.generate_sequences
        audio = A.make_audio_feats(30, opt)
        assert m.generate_sequences(audio, np.zeros(12, np.float32), fill_zero=False, sigma_scale=0.3, opt=opt) is None   # :161-162
        if not torch.cuda.is_available():
            with pytest.raises(RuntimeError, match="no CPU path"):
                m.generate_sequences(audio, np.zeros(12, np.float32), fill_zero=True, sigma_scale=0.3, opt=opt)
    finally:
        ref_mod.Audio2HeadposeModel.generate_sequences = original
