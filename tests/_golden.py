"""Stored outputs of the reference's own CUDA extensions and RenderCNN module (tests/golden/ref_cuda_ops.npz, written on a
B200 by tests/golden/make_golden_cuda.py), so the tests that compare with them run where the reference is absent.

Every array keeps a seeded sample of its elements (`<key>.idx`, `<key>.val`) and its largest magnitude (`<key>.absmax`,
which check_close compares over the whole array);
an array the tests compare exactly also keeps the SHA-256 of all its bytes (`<key>.sha256`), taken after -0.0 is made +0.0
where the tests compare values rather than bits."""
import hashlib
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'ref_cuda_ops.npz')
SAMPLE = 2048


def _flat(t):
    return t.detach().contiguous().cpu().numpy().reshape(-1)


def _sha(a, values=False):
    if values:
        a = np.where(a == 0, np.zeros_like(a), a)
    return hashlib.sha256(a.tobytes()).hexdigest()


def record(out, key, t, seed, exact=False, values=False, n=SAMPLE, idx=None):
    a = _flat(t)
    if idx is None:
        idx = np.random.default_rng(seed).choice(a.size, size=min(n, a.size), replace=False)
    idx = np.sort(np.asarray(idx, dtype=np.int32))
    out[key + '.idx'] = idx
    out[key + '.val'] = a[idx]
    out[key + '.absmax'] = np.float64(np.abs(a.astype(np.float64)).max()) if a.size else np.float64(0.0)
    if exact:
        out[key + '.sha256'] = np.array(_sha(a, values))


def load():
    return np.load(PATH)


def absmax(g, key):
    return float(g[key + '.absmax'])


def check_exact(g, key, t, values=False):
    """Bit for bit; with values=True, equal as numbers (-0.0 == +0.0)."""
    a = _flat(t)
    ref = g[key + '.val']
    assert a.dtype == ref.dtype, (key, a.dtype, ref.dtype)
    got = a[g[key + '.idx']]
    if values:
        np.testing.assert_array_equal(got, ref, err_msg=key)
    else:
        assert got.tobytes() == ref.tobytes(), '%s: %d of %d sampled elements differ' % (
            key, int((got.view(np.uint8).reshape(got.size, -1) != ref.view(np.uint8).reshape(ref.size, -1)).any(-1).sum()),
            ref.size)
    assert _sha(a, values) == str(g[key + '.sha256']), '%s: the sample matches, the whole array does not' % key


def check_close(g, key, t, rtol, atol):
    """Elementwise on the stored sample; over the whole array, its largest magnitude within the same tolerance."""
    a = _flat(t)
    np.testing.assert_allclose(a[g[key + '.idx']], g[key + '.val'], rtol=rtol, atol=atol, err_msg=key)
    ref_max = absmax(g, key)
    got_max = float(np.abs(a.astype(np.float64)).max()) if a.size else 0.0
    assert abs(got_max - ref_max) <= atol + rtol * ref_max, '%s: max |x| %.6e, stored %.6e' % (key, got_max, ref_max)
