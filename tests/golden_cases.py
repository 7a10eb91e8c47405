"""The fixture cases of tests/golden/make_golden.py, restated so the tests do not import the generator
(which needs a checkout of the original deepsvg)."""
import glob
import os

import numpy as np

from oracle import svg_oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))

CASES = {
    "tiny_hier": ("hierarchical", dict(d_model=32, n_heads=4, dim_feedforward=64, dim_z=24, n_layers=2,
                                       n_layers_decode=2, max_num_groups=3, max_seq_len=6, args_dim=15,
                                       use_vae=False), True),
    "tiny_hier_vae_label": ("hierarchical", dict(d_model=32, n_heads=2, dim_feedforward=48, dim_z=16, n_layers=1,
                                                 n_layers_decode=2, max_num_groups=4, max_seq_len=5, args_dim=15,
                                                 use_vae=True, label_condition=True, n_labels=7, dim_label=8), True),
    "tiny_one_stage": ("one_stage", dict(d_model=32, n_heads=4, dim_feedforward=64, dim_z=32, n_layers=2,
                                         n_layers_decode=1, max_num_groups=4, max_total_len=12, args_dim=15,
                                         use_vae=True, label_condition=True, n_labels=5, dim_label=8), True),
    "hier_cfg1": ("hierarchical", dict(use_vae=False), False),
    # hand-built edge cases: one-command path, empty paths, paths filled to max_seq_len, 'a' / 'z' commands, extreme arg values
    "edge_hier": ("hierarchical", dict(d_model=32, n_heads=4, dim_feedforward=64, dim_z=24, n_layers=2,
                                       n_layers_decode=2, max_num_groups=3, max_seq_len=6, args_dim=15,
                                       use_vae=False), True),
    "edge_d128": ("hierarchical", dict(use_vae=False, d_model=128, n_heads=4, dim_feedforward=256, dim_z=64, n_layers=2,
                                       n_layers_decode=2, max_num_groups=4, max_seq_len=10), False),
    # BASELINE.json configs[4] and configs[3] (SURVEY.md 8d rows 5 and 4)
    "scaled_cfg5": ("hierarchical", dict(use_vae=False, d_model=512, n_layers=8, n_layers_decode=8, max_num_groups=16,
                                         max_seq_len=64), False),
    "fonts_cfg4": ("one_stage", dict(use_vae=True, label_condition=True, n_labels=52, max_total_len=50), False),
    # HierarchicalSelfMatching (model/config.py:101-108)
    "tiny_selfmatch": ("hierarchical", dict(d_model=32, n_heads=4, dim_feedforward=64, dim_z=24, n_layers=2,
                                            n_layers_decode=2, max_num_groups=4, max_seq_len=6, args_dim=15,
                                            use_vae=False, self_match=True), True),
    "selfmatch_d128": ("hierarchical", dict(use_vae=False, d_model=128, n_heads=4, dim_feedforward=256, dim_z=64, n_layers=2,
                                            n_layers_decode=2, max_num_groups=4, max_seq_len=10, self_match=True), False),
    # Sketchformer (model/config.py:74-80): autoregressive decoder, relative argument targets
    "tiny_sketchformer": ("one_stage", dict(d_model=32, n_heads=4, dim_feedforward=64, dim_z=32, n_layers=2,
                                            n_layers_decode=2, max_num_groups=4, max_total_len=12, args_dim=15,
                                            use_vae=True, pred_mode="autoregressive", rel_targets=True), True),
    "sketchformer_d128": ("one_stage", dict(d_model=128, n_heads=4, dim_feedforward=256, dim_z=64, n_layers=2,
                                            n_layers_decode=2, max_num_groups=4, max_total_len=30, use_vae=False,
                                            pred_mode="autoregressive", rel_targets=True), False),
}


def read_fixture(directory, name):
    """The arrays of fixture `name`: directory/name.npz plus the name.part<k>.npz files of a case that
    make_golden.py split to keep every file under 1 MB."""
    fx = {}
    for p in [os.path.join(directory, name + ".npz")] + sorted(glob.glob(os.path.join(directory, name + ".part*.npz"))):
        fx.update(np.load(p, allow_pickle=False))
    return fx


def load_case(name):
    kind, over, full = CASES[name]
    cfg = O.make_cfg(kind, **over)
    fx = read_fixture(os.path.join(HERE, "golden"), name)
    return cfg, fx, full
