"""Shared test helpers: golden fixtures, seeded weights (cached)."""
import functools
import os

import numpy as np
import torch

import cir_b200 as cir

syn = cir.synthetic
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name))
    return {k: z[k] for k in z.files}


@functools.lru_cache(maxsize=4)
def weights(seed, style, head_gain, cross_gain=1.0):
    return (syn.make_stage1_state_dict(seed, 384, style),
            syn.make_stage2_state_dict(seed, 384, style, head_gain=head_gain, cross_gain=cross_gain))


def golden_weights(g):
    return weights(int(g["seed"]), str(g["style"]), float(g["head_gain"]), float(g["cross_gain"]) if "cross_gain" in g else 1.0)


def golden_images(g):
    """The gallery images a fixture was generated from (its ``images`` key names the generator)."""
    fn = syn.make_diverse_images if ("images" in g and str(g["images"]) == "diverse") else syn.make_images
    return fn(int(g["G"]), 384, seed=1)
