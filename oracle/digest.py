"""TEST INFRASTRUCTURE - compact digests shared by oracle/make_golden.py (which writes them from the reference) and the tests (which
recompute them from the oracle / the CUDA path): fixed random cotangents for the train-mode probe loss, a per-tensor gradient digest and
the row sample that keeps large outputs in a fixture under 1 MB."""
import numpy as np
import torch


def keep_rows(arrs, key, step):
    """replaces arrs[key] by every `step`-th row of it (last axis kept whole) and records the step and the full shape.  A step coprime
    with the map sizes makes the kept rows visit every channel, anchor and upsampling phase."""
    a = np.asarray(arrs[key])
    arrs[f"{key}_shape"] = np.array(a.shape)
    arrs[f"{key}_step"] = np.int64(step)
    arrs[key] = np.ascontiguousarray(a.reshape(-1, a.shape[-1])[::step])


def fixture_shape(g, key):
    """the full shape of what the reference computed for `key`, also when fixture `g` keeps only rows of it"""
    return tuple(int(v) for v in g[f"{key}_shape"]) if f"{key}_step" in g else g[key].shape


def fixture_pair(g, key, mine):
    """(mine, reference) over what fixture `g` stores of `key`: the whole array, or the rows keep_rows() kept (full shapes checked)"""
    mine = np.asarray(mine)
    if f"{key}_step" not in g:
        return mine, g[key]
    assert mine.shape == fixture_shape(g, key), (key, mine.shape)
    return mine.reshape(-1, mine.shape[-1])[::int(g[f"{key}_step"])], g[key]


def train_probe_tensors(shapes_raw, shapes_seg, seed=11):
    """the fixed random cotangents R_i, S_k of the scalar L = sum_i <x_i, R_i> + sum_k <seg_k, S_k> (same generator in the tests)"""
    rs = np.random.RandomState(seed)
    return ([torch.from_numpy(rs.normal(0, 1, s).astype(np.float32)) for s in shapes_raw],
            [torch.from_numpy(rs.normal(0, 1, s).astype(np.float32) * 0.05) for s in shapes_seg])


def grad_digest(g: torch.Tensor):
    """[L2 norm, sum, 32 leading values, 32 strided values] of one gradient tensor"""
    f = g.detach().reshape(-1).double()
    idx = torch.linspace(0, f.numel() - 1, 32).long()
    lead = torch.zeros(32, dtype=torch.float64)
    lead[:min(32, f.numel())] = f[:32]
    return torch.cat([f.norm().view(1), f.sum().view(1), lead, f[idx]]).numpy()
