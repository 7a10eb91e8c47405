"""Generates tests/golden/*.npz by EXECUTING THE REFERENCE (alexandre01/deepsvg, a checkout named by $DEEPSVG_REFERENCE).

Run once:  DEEPSVG_REFERENCE=<deepsvg checkout> python tests/golden/make_golden.py [--out DIR] [case ...]
A case whose file would pass 1 MB is split by key into <case>.npz + <case>.part<k>.npz (tests/golden_cases.read_fixture).
With --oracle the fp64 oracle stands in for the reference's model and loss (no checkout needed): the same inputs, weights
and file layout, so tests/test_oracle_golden.py regenerates fixtures with it and compares them with the committed ones.
The reference cannot travel to the GPU box, so its outputs are committed as fixtures; tests/test_oracle_golden.py
pins oracle/svg_oracle.py against them.  Nothing from the reference is copied: it is imported, run, and only
numbers are stored.

Protocol (SURVEY.md 8c): the reference module is run in float64 (`.double()`), eval mode (dropout off), VAE noise injected, and the loss's aliased in-place
`_get_padding_mask(extended=True)` replaced by its clean clone()-based equivalent ("de-aliased oracle").
"""
import glob
import os
import sys
from unittest.mock import MagicMock

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import svg_oracle as O                      # noqa: E402


def load_reference():
    """Imports the reference from $DEEPSVG_REFERENCE (its optional plotting / IO dependencies mocked) and de-aliases its
    padding mask.  Returns its modules."""
    if not os.path.isdir(os.path.join(os.environ.get("DEEPSVG_REFERENCE", ""), "deepsvg")):
        sys.exit("set DEEPSVG_REFERENCE to a checkout of alexandre01/deepsvg (or pass --oracle)")
    sys.path.insert(0, os.environ["DEEPSVG_REFERENCE"])
    for m in ["tensorboardX", "cairosvg", "IPython", "IPython.display", "moviepy", "moviepy.editor", "shapely",
              "shapely.ops", "shapely.geometry", "matplotlib", "matplotlib.pyplot", "svgwrite"]:
        sys.modules.setdefault(m, MagicMock())
    from deepsvg.model import config, loss, model
    loss._get_padding_mask = dealiased_padding_mask
    model._get_padding_mask = dealiased_padding_mask      # perfect_matching (model.py:315) uses the same aliased add
    return config, loss, model


def dealiased_padding_mask(commands, seq_dim=0, extended=False):
    """Same arithmetic as the reference's _get_padding_mask, but the shifted add reads a copy (no aliasing)."""
    with torch.no_grad():
        pm = ((commands == 4).cumsum(dim=seq_dim) == 0).float()
        if extended:
            S = commands.size(seq_dim)
            src = torch.narrow(pm, seq_dim, 0, S - 3).clone()
            torch.narrow(pm, seq_dim, 3, S - 3).add_(src).clamp_(max=1)
        if seq_dim == 0:
            return pm.unsqueeze(-1)
        return pm


CASES = {
    # name: (kind, overrides, batch, store_full)
    "tiny_hier": ("hierarchical", dict(d_model=32, n_heads=4, dim_feedforward=64, dim_z=24, n_layers=2,
                                       n_layers_decode=2, max_num_groups=3, max_seq_len=6, args_dim=15,
                                       use_vae=False), 3, True),
    "tiny_hier_vae_label": ("hierarchical", dict(d_model=32, n_heads=2, dim_feedforward=48, dim_z=16, n_layers=1,
                                                 n_layers_decode=2, max_num_groups=4, max_seq_len=5, args_dim=15,
                                                 use_vae=True, label_condition=True, n_labels=7, dim_label=8),
                            4, True),
    "tiny_one_stage": ("one_stage", dict(d_model=32, n_heads=4, dim_feedforward=64, dim_z=32, n_layers=2,
                                         n_layers_decode=1, max_num_groups=4, max_total_len=12, args_dim=15,
                                         use_vae=True, label_condition=True, n_labels=5, dim_label=8), 3, True),
    "hier_cfg1": ("hierarchical", dict(use_vae=False), 2, False),   # BASELINE.json configs[0]
    # hand-built edge cases (see edge_batch): one-command path, empty paths, paths filled to max_seq_len (no EOS inside
    # the window), the 'a' and 'z' commands, argument values 0 and args_dim - 1
    "edge_hier": ("hierarchical", dict(d_model=32, n_heads=4, dim_feedforward=64, dim_z=24, n_layers=2,
                                       n_layers_decode=2, max_num_groups=3, max_seq_len=6, args_dim=15,
                                       use_vae=False), 4, True),
    # the same edge batch at a configuration the CUDA path supports (head_dim 32), for the GPU parity test
    "edge_d128": ("hierarchical", dict(use_vae=False, d_model=128, n_heads=4, dim_feedforward=256, dim_z=64, n_layers=2,
                                       n_layers_decode=2, max_num_groups=4, max_seq_len=10), 4, False),
    # BASELINE.json configs[4] ("scaled hierarchical, tensor-core stress", SURVEY.md 8d row 5): d_model 512, 8 layers per
    # stack, 16 paths of 64 commands, head_dim 64; 55.8 M parameters are regenerated from the seed, only outputs are stored
    "scaled_cfg5": ("hierarchical", dict(use_vae=False, d_model=512, n_layers=8, n_layers_decode=8, max_num_groups=16,
                                         max_seq_len=64), 2, False),
    # BASELINE.json configs[3] (one-stage fonts, SURVEY.md 8d row 4): G = 1 grouped tensors of 50 commands, 52 labels, VAE
    "fonts_cfg4": ("one_stage", dict(use_vae=True, label_condition=True, n_labels=52, max_total_len=50), 3, False),
    # HierarchicalSelfMatching (model/config.py:101-108): Hungarian assignment of predicted slots to target paths
    "tiny_selfmatch": ("hierarchical", dict(d_model=32, n_heads=4, dim_feedforward=64, dim_z=24, n_layers=2,
                                            n_layers_decode=2, max_num_groups=4, max_seq_len=6, args_dim=15,
                                            use_vae=False, self_match=True), 5, True),
    "selfmatch_d128": ("hierarchical", dict(use_vae=False, d_model=128, n_heads=4, dim_feedforward=256, dim_z=64, n_layers=2,
                                            n_layers_decode=2, max_num_groups=4, max_seq_len=10, self_match=True), 6, False),
    # Sketchformer (model/config.py:74-80): one-stage, autoregressive decoder (causal mask, embedded shifted targets),
    # relative argument targets (2 * args_dim classes)
    "tiny_sketchformer": ("one_stage", dict(d_model=32, n_heads=4, dim_feedforward=64, dim_z=32, n_layers=2,
                                            n_layers_decode=2, max_num_groups=4, max_total_len=12, args_dim=15,
                                            use_vae=True, pred_mode="autoregressive", rel_targets=True), 3, True),
    "sketchformer_d128": ("one_stage", dict(d_model=128, n_heads=4, dim_feedforward=256, dim_z=64, n_layers=2,
                                            n_layers_decode=2, max_num_groups=4, max_total_len=30, use_vae=False,
                                            pred_mode="autoregressive", rel_targets=True), 4, False),
}


def edge_batch(cfg):
    """4 icons x G paths x (S + 2) positions.  Commands: m=0 l=1 c=2 a=3 EOS=4 SOS=5 z=6 (difflib/tensor.py:10-21)."""
    M_, L_, C_, A_, Z_ = O.CMD_M, O.CMD_L, O.CMD_C, 3, 6
    G, S = cfg.max_num_groups, cfg.max_seq_len
    cyc = [L_, C_, A_, Z_, L_, M_, C_, A_]
    full = lambda k: [M_] + [cyc[(j + k) % len(cyc)] for j in range(S - 1)]      # a path filled to max_seq_len
    pad = lambda icon: icon + [[] for _ in range(G - len(icon))]
    paths = [
        pad([[M_]]),                                               # a one-command path, the others empty (invisible)
        [full(p) for p in range(G)],                               # every path at max_seq_len (no EOS inside the window)
        pad([[M_, Z_], [M_, A_, A_, C_]]),
        pad([[M_] + [C_] * (S - 1), [M_, L_], [M_, L_, L_]]),
    ]
    cmd = torch.full((len(paths), G, S + 2), float(O.CMD_EOS))
    arg = torch.full((len(paths), G, S + 2, cfg.n_args), -1.0)
    g = torch.Generator().manual_seed(31)
    for i, icon in enumerate(paths):
        for p, body in enumerate(icon):
            cmd[i, p, 0] = O.CMD_SOS
            if not body:
                continue
            b = torch.tensor(body)
            cmd[i, p, 1:1 + len(body)] = b.float()
            vals = torch.randint(0, cfg.args_dim, (len(body), cfg.n_args), generator=g).float()
            vals[0, :] = 0.0                       # smallest argument value
            vals[-1, :] = float(cfg.args_dim - 1)   # largest
            m = O.CMD_ARGS_MASK[b].float()
            arg[i, p, 1:1 + len(body)] = vals * m - (1 - m)
    return cmd, arg
WEIGHTS = dict(O.DEFAULT_WEIGHTS)


def ref_cfg(config, kind, over):
    c = (config.HierarchicalSelfMatching() if over.get("self_match") else config.Hierarchical()) if kind == "hierarchical" \
        else config.OneStageOneShot()
    for k, v in over.items():
        setattr(c, k, v)
    if "max_total_len" not in over:
        c.max_total_len = c.max_num_groups * c.max_seq_len
    c.num_groups_proposal = c.max_num_groups
    return c


def sample(t, n=4096):
    f = t.reshape(-1)
    if f.numel() <= n:
        return f.clone()
    idx = torch.linspace(0, f.numel() - 1, n).long()
    return f[idx]


def run_reference(kind, over, cfg_o, params, cmd, arg, arg_dec, label, eps):
    """The reference's SVGTransformer + SVGLoss + backward in fp64.  Returns (out, losses, grads, assignment or None)."""
    config, loss, model_mod = load_reference()
    cfg_r = ref_cfg(config, kind, over)
    model = model_mod.SVGTransformer(cfg_r).double()   # fp64: no ReLU-boundary chaos between two implementations
    sd = model.state_dict()
    # the oracle's parameter inventory must be exactly the reference's parameters
    ref_param_names = {k for k, _ in model.named_parameters()}
    assert ref_param_names == set(params), (ref_param_names ^ set(params))
    for k, v in params.items():
        assert tuple(sd[k].shape) == tuple(v.shape), (k, sd[k].shape, v.shape)
    model.load_state_dict(params, strict=False)
    model.eval()
    loss_fn = loss.SVGLoss(cfg_r)
    kw = {"label": label} if label is not None else {}
    if eps is not None:
        real = torch.randn_like
        torch.randn_like = lambda s, *a, **k: eps.reshape(s.shape).to(s.dtype)
    captured = {}
    if getattr(cfg_r, "self_match", False):
        orig_pm = model.perfect_matching

        def spy(*a):
            captured["asg"] = orig_pm(*a)
            return captured["asg"]
        model.perfect_matching = spy
    try:
        out = model(cmd, arg, cmd, arg_dec, params={}, **kw)
    finally:
        if eps is not None:
            torch.randn_like = real
    losses = loss_fn(out, None, weights=WEIGHTS)
    model.zero_grad()
    losses["loss"].backward()
    grads = {k: (p.grad if p.grad is not None else torch.zeros_like(p)) for k, p in model.named_parameters()}
    return out, losses, grads, captured.get("asg")


def run_oracle(kind, over, cfg_o, params, cmd, arg, arg_dec, label, eps):
    """oracle/svg_oracle.py in fp64 on the same inputs and weights, in place of the reference (--oracle)."""
    out, losses, grads = O.train_step(params, cfg_o, cmd, arg, label=label, eps=eps, weights=WEIGHTS,
                                      args_dec=arg_dec if arg_dec is not arg else None)
    return out, losses, grads, out.get("assignment")


def run_case(name, run_model=run_reference):
    kind, over, batch, full = CASES[name]
    cfg_o = O.make_cfg(kind, **over)
    params = O.make_params(cfg_o, seed=7, dtype=torch.float64)
    cmd, arg = edge_batch(cfg_o) if name.startswith("edge") else O.synth_batch(cfg_o, batch, seed=99)
    assert cmd.shape[0] == batch
    cmd, arg = cmd.double(), arg.double()
    arg_dec = arg
    if over.get("rel_targets"):
        # relative-argument targets (SVGTensor.get_relative_args, difflib/tensor.py:150-168): ids in [0, 2*args_dim-2] on
        # the slots the command uses, -1 elsewhere; drawn at random here (the model only sees them as class ids)
        m = O.CMD_ARGS_MASK[cmd.long()].double()
        vals = torch.randint(0, 2 * cfg_o.args_dim - 1, arg.shape, generator=torch.Generator().manual_seed(41)).double()
        arg_dec = vals * m - (1 - m)
    label = None
    if cfg_o.label_condition:
        label = torch.randint(0, cfg_o.n_labels, (batch,), generator=torch.Generator().manual_seed(5))
    eps = None
    if cfg_o.use_vae:
        eps = torch.randn(batch, cfg_o.dim_z, generator=torch.Generator().manual_seed(6)).double()
    out, losses, grads, asg = run_model(kind, over, cfg_o, params, cmd, arg, arg_dec, label, eps)

    fx = {"commands": cmd.float().numpy(), "args": arg.float().numpy(), "seed_params": np.int64(7)}
    if arg_dec is not arg:
        fx["args_dec"] = arg_dec.float().numpy()
    if asg is not None:
        fx["assignment"] = asg.reshape(batch, -1).numpy()     # what the reference's perfect_matching picked
    if label is not None:
        fx["label"] = label.numpy()
    if eps is not None:
        fx["eps"] = eps.numpy()
    for k in ("loss", "loss_cmd", "loss_args", "loss_visibility", "loss_kl"):
        if k in losses:
            fx["L_" + k] = np.float64(losses[k].item())
    keys = ["command_logits", "args_logits"] + (["visibility_logits"] if "visibility_logits" in out else []) + \
           (["mu", "logsigma"] if "mu" in out else [])
    for k in keys:
        t = out[k].detach().contiguous()
        fx["O_shape_" + k] = np.array(t.shape)
        fx["O_" + k] = (t if full else sample(t)).numpy()
    fx["param_names"] = np.array(sorted(grads))
    for k, g in grads.items():
        fx["Gnorm_" + k] = np.float64(g.double().norm().item())
        fx["G_" + k] = (g if full else sample(g, 512)).detach().numpy()
    kb = save_fixture(OUT_DIR, name, fx) // 1024
    print(name, {k: float(v) for k, v in fx.items() if k.startswith("L_")}, kb, "KB")


MAX_FILE_BYTES = 1 << 20


def save_fixture(out_dir, name, fx):
    """Writes `fx` as out_dir/name.npz, split by key into name.npz, name.part1.npz, ... when one file would pass
    MAX_FILE_BYTES (compressed).  Returns the total size in bytes."""
    for p in glob.glob(os.path.join(out_dir, name + ".part*.npz")):
        os.remove(p)
    keys = list(fx)
    for n in range(1, len(keys) + 1):
        paths = [os.path.join(out_dir, name + (".npz" if i == 0 else ".part%d.npz" % i)) for i in range(n)]
        for path, chunk in zip(paths, np.array_split(np.array(keys, dtype=object), n)):
            np.savez_compressed(path, **{k: fx[k] for k in chunk})
        sizes = [os.path.getsize(p) for p in paths]
        if max(sizes) <= MAX_FILE_BYTES:
            return sum(sizes)
        for p in paths[1:]:
            os.remove(p)
    raise RuntimeError("%s: a single array passes %d bytes" % (name, MAX_FILE_BYTES))


OUT_DIR = HERE

if __name__ == "__main__":
    torch.manual_seed(0)
    argv = sys.argv[1:]
    if "--out" in argv:                      # tests/test_oracle_golden.py regenerates into a scratch directory
        OUT_DIR = argv[argv.index("--out") + 1]
        del argv[argv.index("--out"):argv.index("--out") + 2]
        os.makedirs(OUT_DIR, exist_ok=True)
    runner = run_reference
    if "--oracle" in argv:
        argv.remove("--oracle")
        runner = run_oracle
    for n in (argv or CASES):
        run_case(n, runner)
