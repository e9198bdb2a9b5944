"""Shared test helpers (checkpoint stand-ins, module trees).  Test infrastructure only."""
import os

import torch

from oracle.checkpoint_standins import state_dict as checkpoint  # noqa: F401  (seeded stand-ins of the vendored weights)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def pillow_resize_cases():
    """The cases of tests/golden/pillow_resize.npz as (input, Pillow's output, filter).  The inputs are consecutive draws
    of np.random.default_rng(0) (scripts/make_golden.py); one that is not stored (keeps the file under 1 MB) is replayed
    from that generator, and every stored one is checked against the same replay."""
    import numpy as np
    g = np.load(os.path.join(ROOT, "tests", "golden", "pillow_resize.npz"))
    rng = np.random.default_rng(0)
    cases, n = [], 0
    while f"out{n}" in g:
        if f"in{n}" in g:
            im = g[f"in{n}"]
            assert np.array_equal(rng.integers(0, 256, im.shape, dtype=np.uint8), im), f"case {n}: replay"
        else:
            im = rng.integers(0, 256, tuple(g[f"shape{n}"]), dtype=np.uint8)
        cases.append((im, g[f"out{n}"], int(g[f"filter{n}"])))
        n += 1
    return cases


class _Node(torch.nn.Module):
    def forward(self, x):
        return x


def module_tree(state_dict) -> torch.nn.Module:
    """A module whose parameters carry exactly the dotted names of `state_dict` (for TorchScript archives shaped like
    the ones `clip.load` downloads)."""
    root = _Node()
    for key, value in state_dict.items():
        parts = key.split('.')
        m = root
        for p in parts[:-1]:
            if not hasattr(m, p):
                m.add_module(p, _Node())
            m = getattr(m, p)
        m.register_parameter(parts[-1], torch.nn.Parameter(value.clone(), requires_grad=False))
    return root
