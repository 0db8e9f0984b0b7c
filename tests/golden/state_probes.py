"""Compact fingerprint of a state dict, shared by make_golden_reference_state.py and the tests that compare same-seed
construction with the original project's modules."""
import numpy as np


def probe(t, n=64):
    """(flat positions, values there, float64 sum) of tensor t; the positions are seeded by the tensor's size."""
    a = t.detach().cpu().numpy().reshape(-1)
    idx = np.random.default_rng(a.size).choice(a.size, size=min(n, a.size), replace=False) if a.size else np.zeros(0, np.int64)
    return idx.astype(np.int64), a[idx], np.float64(a.astype(np.float64).sum())


def assert_state_matches(sd, g, prefix):
    """State dict sd has the golden's names in order, its shapes, its values at the probed positions (exactly) and its sums."""
    assert list(sd) == [str(k) for k in g[prefix + ".names"]]
    for k, v in sd.items():
        assert tuple(v.shape) == tuple(g[f"{prefix}.{k}.shape"]), k
        a = v.detach().cpu().numpy().reshape(-1)
        assert np.array_equal(a[g[f"{prefix}.{k}.idx"]], g[f"{prefix}.{k}.val"]), k
        s = float(g[f"{prefix}.{k}.sum"])
        assert abs(float(a.astype(np.float64).sum()) - s) <= 1e-9 * max(1.0, abs(s)), k
