"""Generate the fixtures of the checks that used to need the reference checkout at test time, by running the UNMODIFIED
reference once.  TEST INFRASTRUCTURE.

    LSP_REFERENCE_ROOT=<LiveSpeechPortraits checkout> PYTHONDONTWRITEBYTECODE=1 python oracle/make_golden_reference_checks.py

Writes
* ``tests/golden/f2f_reference_checks.npz``: per variant, the reference generator's state-dict keys, per-tensor sums of
  the weights ``networks.init_weights('normal', 0.02)`` gives it under ``torch.manual_seed(0)``, and a strided sub-sample
  plus full-tensor statistics of its output on ``make_inputs(1, 256, 256, seed=5)``; and ``util.tensor2im`` of two small
  images (tests/test_oracle.py).
* ``tests/golden/a2h_live_loop.npz``: per recipe, ``Audio2HeadposeModel.generate_sequences`` on seeded weights, audio
  features and torch seed, and one full-window ``Audio2Headpose.forward`` on a seeded history (tests/test_a2h_oracle.py).

Each case is also checked against the restatement here, so a fixture is only written when the oracle agrees with the
reference.
"""
from __future__ import annotations

import contextlib
import io
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
from oracle import a2h_oracle as A  # noqa: E402
from oracle import f2f_oracle as O  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
F2F_STRIDE = 8


def stats(t: torch.Tensor) -> np.ndarray:
    d = t.double()
    return np.array([d.sum().item(), (d * d).sum().item(), d.min().item(), d.max().item()], np.float64)


def tensor2im_inputs() -> torch.Tensor:
    g = torch.Generator().manual_seed(9)
    x = torch.tanh(torch.randn(2, 3, 16, 16, generator=g) * 2)
    x[0, 0, 0, 0], x[0, 1, 0, 0], x[0, 2, 0, 0] = -1.0, 1.0, 0.0        # boundary values: 0, 255, 127
    return x


def history_input() -> torch.Tensor:
    return torch.from_numpy(np.random.Generator(np.random.PCG64(11)).standard_normal((1, 255, 12)).astype(np.float32))


def f2f() -> None:
    out = {}
    for variant in ("normal", "large"):
        net = O.reference_generator(variant)
        torch.manual_seed(0)
        with contextlib.redirect_stdout(io.StringIO()):
            from models import networks  # type: ignore  (reference package)
            networks.init_weights(net, "normal", 0.02)
        net.eval()
        sd = net.state_dict()
        assert list(sd.keys()) == list(O.state_dict_spec(variant).keys())
        mine_sd = O.init_weights_state_dict(variant, 0)
        assert all(torch.equal(sd[k], mine_sd[k]) for k in sd), "init restatement differs from networks.init_weights"
        fm, cand = O.make_inputs(1, 256, 256, seed=5)
        x = torch.cat([fm, cand], 1)
        with torch.no_grad():
            ref = net(x)
        err = (ref - O.generator_forward(sd, x, variant)).abs().max().item()
        assert err <= 1e-6, f"{variant}: restatement differs from the reference by {err}"
        out[f"{variant}_keys"] = np.array(list(sd.keys()))
        out[f"{variant}_weight_sums"] = np.array([sd[k].double().sum().item() for k in sd], np.float64)
        out[f"{variant}_out_sub"] = ref[:, :, ::F2F_STRIDE, ::F2F_STRIDE].numpy()
        out[f"{variant}_out_stats"] = stats(ref)
        print(f"f2f {variant}: {len(sd)} keys, max|ref - restatement| {err:.2e}")
    from util import util as ref_util  # type: ignore  (reference package, on sys.path since reference_generator)
    x = tensor2im_inputs()
    out["tensor2im"] = np.stack([ref_util.tensor2im(x[i]) for i in range(x.shape[0])])
    assert np.array_equal(out["tensor2im"], O.tensor2im(x))
    path = os.path.join(GOLDEN, "f2f_reference_checks.npz")
    np.savez_compressed(path, stride=F2F_STRIDE, input_seed=5, init_seed=0, torch_version=torch.__version__, **out)
    print("wrote", path)


def a2h() -> None:
    opt = A.default_opt()
    out = {}
    for recipe, seed in (("A", 1), ("B", 2)):
        sd = A.make_state_dict(opt, recipe, seed)
        m = A.reference_model(opt, sd)
        net = m.Audio2Headpose
        assert list(net.state_dict().keys()) == list(A.state_dict_spec(opt).keys())
        audio = A.make_audio_feats(36, opt, seed)
        pre = np.linspace(-0.2, 0.3, 12).astype(np.float32)
        noise = A.reference_noise(36 - opt.frame_future, 12, 1, seed=11)
        torch.manual_seed(11)
        with contextlib.redirect_stderr(io.StringIO()):
            ref = m.generate_sequences(audio.copy(), pre, fill_zero=True, sigma_scale=0.3, opt=opt)
        err = np.abs(ref - A.generate_sequences(sd, audio, pre, noise, opt, 0.3)).max()
        assert err <= 1e-6, f"{recipe}: restatement differs from the reference loop by {err}"
        hist = history_input()
        aud = torch.from_numpy(A.make_audio_feats(255, opt, 5)).unsqueeze(0)
        with torch.no_grad():
            fwd = net(hist, aud)
        assert torch.allclose(fwd, A.audio2headpose_forward(sd, hist, aud, opt), atol=1e-6)
        out[f"{recipe}_pred"] = ref
        out[f"{recipe}_forward"] = fwd.numpy()
        print(f"a2h {recipe}: loop {ref.shape} max|ref - restatement| {err:.2e}, forward {tuple(fwd.shape)}")
    out["keys"] = np.array(list(net.state_dict().keys()))
    path = os.path.join(GOLDEN, "a2h_live_loop.npz")
    np.savez_compressed(path, torch_version=torch.__version__, **out)
    print("wrote", path)


if __name__ == "__main__":
    if not O.reference_available():
        raise SystemExit(f"reference checkout not found at {O.REFERENCE_ROOT} (set LSP_REFERENCE_ROOT)")
    torch.set_num_threads(8)          # tests/test_a2h_oracle.py GOLDEN_THREADS: the loop's last bits depend on it
    f2f()
    a2h()
