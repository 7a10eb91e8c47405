"""Pins oracle/svg_oracle.py against fixtures produced by executing the reference (tests/golden/make_golden.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import svg_oracle as O
from tests.golden_cases import CASES, load_case, read_fixture

HERE = os.path.dirname(os.path.abspath(__file__))


def _strided(t, n):
    f = t.reshape(-1)
    if f.numel() <= n:
        return f
    return f[torch.linspace(0, f.numel() - 1, n).long()]


@pytest.mark.parametrize("name", list(CASES))
def test_oracle_matches_reference(name):
    """fp64 oracle == fp64 reference (same seeded weights / inputs): logits, every loss term, every gradient."""
    cfg, fx, full = load_case(name)
    params = O.make_params(cfg, seed=int(fx["seed_params"]), dtype=torch.float64)
    cmd, arg = torch.from_numpy(fx["commands"]).double(), torch.from_numpy(fx["args"]).double()
    label = torch.from_numpy(fx["label"]) if "label" in fx else None
    eps = torch.from_numpy(fx["eps"]) if "eps" in fx else None
    arg_dec = torch.from_numpy(fx["args_dec"]).double() if "args_dec" in fx else None
    out, losses, grads = O.train_step(params, cfg, cmd, arg, label=label, eps=eps, args_dec=arg_dec)
    for k in ("command_logits", "args_logits", "visibility_logits", "mu", "logsigma"):
        if "O_" + k not in fx:
            assert k not in out
            continue
        assert tuple(out[k].shape) == tuple(fx["O_shape_" + k]), k
        got = out[k] if full else _strided(out[k], 4096)
        np.testing.assert_allclose(got.numpy().reshape(-1), fx["O_" + k].reshape(-1), rtol=1e-9, atol=1e-10, err_msg=k)
    for k in ("loss", "loss_cmd", "loss_args", "loss_visibility", "loss_kl"):
        if "L_" + k in fx:
            assert abs(losses[k].item() - float(fx["L_" + k])) <= 1e-10 * max(1.0, abs(float(fx["L_" + k]))), k
        else:
            assert k not in losses
    if "assignment" in fx:      # HierarchicalSelfMatching: the Hungarian assignment itself (model.py:339-350)
        assert out["assignment"].tolist() == fx["assignment"].tolist()
        assert any(row != sorted(row) for row in fx["assignment"].tolist()), "fixture must contain a non-identity assignment"
    assert sorted(grads) == list(fx["param_names"])
    for k, g in grads.items():
        got = g if full else _strided(g, 512)
        scale = float(np.abs(fx["G_" + k]).max()) + 1e-30
        np.testing.assert_allclose(got.numpy().reshape(-1), fx["G_" + k].reshape(-1), rtol=1e-7, atol=1e-9 * scale,
                                   err_msg=k)
        assert abs(g.norm().item() - float(fx["Gnorm_" + k])) <= 1e-9 * float(fx["Gnorm_" + k]) + 1e-30, k


def test_oracle_fp32_close_to_fp64_golden():
    """The fp32 oracle (what the GPU tests and the CPU baseline use) stays within fp32 noise of the fp64 golden."""
    cfg, fx, full = load_case("hier_cfg1")
    params = O.make_params(cfg, seed=int(fx["seed_params"]))
    cmd, arg = torch.from_numpy(fx["commands"]), torch.from_numpy(fx["args"])
    out = O.forward(params, cfg, cmd, arg)
    ls = O.loss(out, cfg)
    got = _strided(out["args_logits"], 4096).numpy()
    np.testing.assert_allclose(got, fx["O_args_logits"].reshape(-1), rtol=1e-3, atol=1e-4)
    assert abs(ls["loss"].item() - float(fx["L_loss"])) < 1e-4 * float(fx["L_loss"])


def test_extended_padding_semantics():
    # clean OR-shift-by-3 (SURVEY.md 8c): prefix of ones grows by 3, independent of prefix length
    for ln in (1, 2, 5, 14, 20, 29):
        cmd = torch.full((1, 1, 32), float(O.CMD_EOS))
        cmd[0, 0, 0] = O.CMD_SOS
        cmd[0, 0, 1:1 + ln] = O.CMD_L
        ext = O.extended_padding(cmd.long())[0, 0]
        k = 1 + ln
        expect = torch.zeros(32)
        expect[:min(32, k)] = 1
        expect[3:min(32, k + 3)] = 1
        assert torch.equal(ext, expect), ln


def test_matmul_modes_are_close():
    cfg, fx, _ = load_case("tiny_hier")
    params = O.make_params(cfg, seed=7)
    cmd, arg = torch.from_numpy(fx["commands"]), torch.from_numpy(fx["args"])
    ref = O.forward(params, cfg, cmd, arg)["args_logits"]
    x3 = O.forward(params, cfg, cmd, arg, matmul="bf16x3")["args_logits"]
    b1 = O.forward(params, cfg, cmd, arg, matmul="bf16")["args_logits"]
    e3, e1 = (x3 - ref).abs().max().item(), (b1 - ref).abs().max().item()
    assert e3 < 2e-4 and e3 < e1 / 20, (e3, e1)


def test_fixtures_regenerate_from_the_reference(tmp_path):
    """Re-runs the fixture generator (tests/golden/make_golden.py) with the fp64 oracle standing in for the reference's
    model and loss, and requires the committed fixtures -- the reference's own results -- to come out again: inputs,
    weights and key set bit for bit, fp64 results to 1e-10 relative (a different BLAS thread split cannot make it flaky).
    Run the generator without --oracle on a checkout of the reference to regenerate the fixtures themselves."""
    import subprocess
    import sys
    names = ["tiny_hier", "edge_hier", "tiny_hier_vae_label", "tiny_one_stage", "tiny_selfmatch", "tiny_sketchformer"]
    r = subprocess.run([sys.executable, os.path.join(HERE, "golden", "make_golden.py"), "--oracle", "--out", str(tmp_path)]
                       + names, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    for n in names:
        new = read_fixture(str(tmp_path), n)
        old = read_fixture(os.path.join(HERE, "golden"), n)
        assert sorted(new) == sorted(old), n
        for k in old:
            if old[k].dtype.kind == "f" and not k.startswith(("commands", "args")):
                np.testing.assert_allclose(new[k], old[k], rtol=1e-10, atol=1e-13, err_msg="%s/%s" % (n, k))
            else:
                assert np.array_equal(new[k], old[k]), (n, k)
