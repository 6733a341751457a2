"""Shared helpers for the parity tests: golden loading and synthetic tensors."""
import json
import os

import numpy as np
import torch

from oracle import raft_oracle as O
from oracle import synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    recipe = json.loads(bytes(z["recipe"]).decode())
    return recipe, {k: z[k] for k in z.files if k != "recipe"}


def check_sample(mine, g, key, tol):
    """``mine`` (a whole tensor) against a reference output stored as a sample (oracle/make_golden.py ``_sampled``): same
    shape, every sampled element within ``tol``, and the sum and absolute sum over all elements within what an
    element-wise bound of ``tol`` allows."""
    assert tuple(mine.shape) == tuple(g[key + "_shape"]), (tuple(mine.shape), g[key + "_shape"])
    flat = mine.detach().double().cpu().reshape(-1).numpy()
    err = np.abs(flat[synth.sample_index(flat.size, g[key].size)] - g[key]).max()
    assert err < tol, (key, err)
    total, abs_total, _ = g[key + "_sums"]
    assert abs(flat.sum() - total) < tol * flat.size, key
    assert abs(np.abs(flat).sum() - abs_total) < tol * flat.size, key


def e2e_inputs(recipe):
    """(state_dict, images, kwargs) rebuilt from a golden recipe (see oracle/make_golden.py)."""
    kw = dict(recipe["kwargs"])
    shapes = O.state_dict_shapes(recipe["variant"], kw.get("corr_levels", 4), kw.get("corr_radius"))
    sd = synth.synth_state_dict(shapes, recipe["wseed"])
    img = torch.from_numpy(synth.synth_images(recipe["batch"], recipe["height"], recipe["width"], recipe["iseed"], recipe["kind"]))
    return sd, img, kw


E2E = ["e2e_raft_small_cfg1", "e2e_raft_small_b2", "e2e_raft_noise", "e2e_raft_smooth_b2", "e2e_raft_altcorr", "e2e_raft_r3_l3", "e2e_gma"]
