"""Inputs and sampling of the golden fixtures that are regenerated rather than stored.

TEST INFRASTRUCTURE.  ``oracle/make_golden.py`` records the reference's outputs on these
inputs, and the tests regenerate the same inputs and check them against the sha256 stored
beside the outputs, so a fixture needs no copy of its inputs.  Long filtered outputs are stored
at the columns ``sample_columns`` picks, which keeps every fixture file under 1 MB.
"""

from __future__ import annotations

import hashlib

import numpy as np

from pyparrm_b200.synthetic import make_recording

# filter_edges.npz: (filter_half_width, omit_n_samples, filter_direction, period_half_width)
# for every shape in EDGE_SHAPES, case = filter index * len(EDGE_SHAPES) + shape index
EDGE_FILTERS = ((2000, 0, "both", None), (2000, 0, "past", None), (2000, 0, "future", None),
                (300, 2, "both", 0.5), (2499, 10, "both", None))
EDGE_SHAPES = ((2, 5000), (1, 50), (3, 1), (1, 4001), (2, 2000), (1, 777))


def sha(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def filter_edges_inputs() -> list:
    """The input of every filter_edges case: the seeded recording for the (2, 5000) shape,
    seeded foreign data (N(10, 1)) for the others."""
    rng = np.random.default_rng(11)
    base = make_recording(2, 5000, 2000, 130, seed=9)
    return [base if shape == (2, 5000) else rng.standard_normal(shape) + 10.0
            for _ in EDGE_FILTERS for shape in EDGE_SHAPES]


def checked_filter_edges_inputs(g) -> list:
    """``filter_edges_inputs()``, each checked against the sha256 recorded in fixture ``g``."""
    xs = filter_edges_inputs()
    assert len(xs) == int(g["n_cases"])
    for case, x in enumerate(xs):
        assert sha(x) == str(g[f"case{case}_x_sha256"]), f"filter_edges case {case}: input differs"
    return xs


def sample_columns(n_times: int, taps, n_interior: int = 2000, seed: int = 0) -> np.ndarray:
    """Columns of a [channels, n_times] filtered output worth storing: every column within the
    taps' reach of either edge (where taps run off the recording) and a seeded sample of
    ``n_interior`` columns between them."""
    reach = int(np.abs(np.asarray(taps)).max()) + 1
    edges = np.union1d(np.arange(min(reach, n_times)), np.arange(max(n_times - reach, 0), n_times))
    interior = np.setdiff1d(np.arange(n_times), edges)
    pick = np.random.default_rng(seed).choice(interior, min(n_interior, interior.size), replace=False)
    return np.union1d(edges, pick).astype(np.int32)
