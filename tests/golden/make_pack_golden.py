"""Generates tests/golden/pack_batch.npz by EXECUTING the reference's batch assembly
(SVGTensorDataset.get_data, svgtensor_dataset.py:164-205, with SVGTensor.add_eos/add_sos/pad, difflib/tensor.py:108-143)
on random raw path tensors.  Run once: DEEPSVG_REFERENCE=<deepsvg checkout> python tests/golden/make_pack_golden.py
Only numbers are stored; tests/test_pack.py checks deepsvg_b200.pack_icons (native packer) against them.
"""
import os
import sys
from types import SimpleNamespace
from unittest.mock import MagicMock

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
if not os.path.isdir(os.path.join(os.environ.get("DEEPSVG_REFERENCE", ""), "deepsvg")):
    sys.exit("set DEEPSVG_REFERENCE to a checkout of alexandre01/deepsvg")
sys.path.insert(0, os.environ["DEEPSVG_REFERENCE"])
for m in ["tensorboardX", "cairosvg", "IPython", "IPython.display", "moviepy", "moviepy.editor", "shapely",
          "shapely.ops", "shapely.geometry", "matplotlib", "matplotlib.pyplot", "svgwrite", "pandas", "PIL", "PIL.Image",
          "networkx", "sklearn", "sklearn.cluster", "bs4", "numpy.core.multiarray"]:
    if m not in ("pandas", "numpy.core.multiarray"):
        sys.modules.setdefault(m, MagicMock())

from deepsvg.svgtensor_dataset import SVGTensorDataset  # noqa: E402

MASK = np.array([[0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1], [0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1], [0, 0, 0, 0, 0, 1, 1, 1, 1, 1, 1],
                 [1, 1, 1, 1, 1, 0, 0, 0, 0, 1, 1], [0] * 11, [0] * 11, [0] * 11])
ARG_COLS = [1, 2, 3, 4, 5, 8, 9, 10, 11, 12, 13]


def random_icon(rng, G, S, total):
    """Raw per-path (len, 14) tensors as SVG.to_tensor(concat_groups=False) produces them: col 0 command, unused args -1."""
    n_paths = int(rng.integers(1, G + 1))
    paths, budget = [], total
    for _ in range(n_paths):
        ln = int(rng.integers(1, min(S, budget - 1) + 1)) if budget > 2 else 0
        if ln == 0:
            break
        budget -= ln
        cmds = rng.integers(1, 4, size=ln)            # l, c, a
        cmds[0] = 0                                    # m
        if ln > 2 and rng.random() < 0.3:
            cmds[-1] = 6                               # z
        t = np.full((ln, 14), -1.0, dtype=np.float32)
        t[:, 0] = cmds
        vals = rng.integers(0, 256, size=(ln, 11))
        m = MASK[cmds]
        t[:, ARG_COLS] = np.where(m == 1, vals, -1)
        t[:, 6:8] = rng.integers(0, 256, size=(ln, 2))   # start_pos: present in the raw data, dropped by args()
        paths.append(torch.from_numpy(t))
    return paths


def main():
    rng = np.random.default_rng(17)
    G, S, TOTAL = 8, 30, 100
    fake = SimpleNamespace(MAX_NUM_GROUPS=G, MAX_SEQ_LEN=S, MAX_TOTAL_LEN=TOTAL, PAD_VAL=-1, model_args=None)
    icons = [random_icon(rng, G, S, TOTAL) for _ in range(24)]
    icons[3] = [icons[3][0][:1]]                                  # a one-command path, the others missing
    icons[5] = [torch.from_numpy(np.concatenate([p.numpy()[:1], np.repeat(p.numpy()[:1], S - 1, 0)])) for p in icons[5][:2]]  # paths filled to MAX_SEQ_LEN
    rows, offsets = [], [0]
    want = {k: [] for k in ("commands", "args", "commands_grouped", "args_grouped")}
    for paths in icons:
        res = SVGTensorDataset.get_data(fake, [p.clone() for p in paths], [0] * len(paths),
                                        model_args=["commands", "args", "commands_grouped", "args_grouped"])
        for k in want:
            want[k].append(res[k].numpy())
        for g in range(G):
            if g < len(paths):
                rows.append(paths[g].numpy())
                offsets.append(offsets[-1] + paths[g].shape[0])
            else:
                offsets.append(offsets[-1])
    fx = {"rows": np.concatenate(rows, 0), "offsets": np.array(offsets, dtype=np.int64), "G": np.int64(G), "S": np.int64(S),
          "TOTAL": np.int64(TOTAL)}
    for k, v in want.items():
        fx["want_" + k] = np.stack(v, 0)
    np.savez_compressed(os.path.join(HERE, "pack_batch.npz"), **fx)
    print({k: v.shape for k, v in fx.items() if hasattr(v, "shape")})


if __name__ == "__main__":
    main()
