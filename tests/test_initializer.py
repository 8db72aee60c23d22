"""pb_bss_b200.initializer against outputs of the unmodified reference (tests/golden/initializer.npz,
oracle/make_golden.py: make_initializer).  The random and the flag initialisers run on the host (they must consume
NumPy's global stream like the reference, pb_bss/initializer/iid.py); deflationSeed composes device kernels."""
import os

import numpy as np
import pytest

GOLD = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'initializer.npz'))


def test_iid_initialisers_consume_the_global_stream_like_the_reference():
    from pb_bss_b200.initializer import iid
    Y = np.ones([4, 5, 3])
    for name in ('uniform_normalized', 'dirichlet_uniform', 'one_hot'):
        for pf in (False, True):
            np.random.seed(0)
            got = getattr(iid, name)(Y, 2, permutation_free=pf)
            np.testing.assert_array_equal(got, GOLD[f'{name}_{int(pf)}'], err_msg=f'{name} permutation_free={pf}')
            assert got.shape == (4, 2, 5)
    np.random.seed(0)
    np.testing.assert_array_equal(iid.dirichlet(np.ones([2, 7, 3]), 3, alpha=3), GOLD['dirichlet_a3'])
    # doctest values of the reference (iid.py:30-35)
    np.random.seed(0)
    np.testing.assert_allclose(iid.uniform_normalized(Y, 2)[0, 0], [0.45937056, 0.62040588, 0.40331128, 0.36119761, 0.52491232],
                               atol=1e-8)


def test_flag_initialiser():
    from pb_bss_b200.initializer import deterministic
    np.testing.assert_array_equal(deterministic.flag(np.ones([4, 5, 3]), 2, permutation_free=True), GOLD['flag_2'])
    np.testing.assert_allclose(deterministic.flag(np.ones([1, 5, 3]), 4, minimum=0.1, permutation_free=True),
                               GOLD['flag_4_min'], rtol=1e-15)
    with pytest.raises(NotImplementedError):
        deterministic.flag(np.ones([1, 5, 3]), 2)
    with pytest.raises(AssertionError):
        deterministic.flag(np.ones([1, 5, 3]), 2, permutation_free=True, minimum=0.6)


@pytest.mark.gpu
def test_deflation_seed_matches_reference():
    from oracle import synth
    from pb_bss_b200.initializer import deflation
    # the inputs of oracle/make_golden.py: make_initializer, regenerated from the same seeds
    y = synth.structured_stft(257, 60, 4, 3, seed=17)[0]
    sal = np.random.RandomState(2).uniform(0.1, 1, size=(257, 60))
    got = deflation.deflationSeed(y, 3, permutation_free=True)
    assert got.shape == (3, 257, 60)
    np.testing.assert_allclose(got, GOLD['deflation_pf'], rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(deflation.deflationSeed(y, 3, permutation_free=False, neighbors=3),
                               GOLD['deflation_nopf'], rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(deflation.deflationSeed(y, 2, saliencies=sal, eps=1e-3),
                               GOLD['deflation_with_sal'], rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(got.sum(0), 1, atol=1e-12)
    import torch
    t = deflation.deflationSeed(torch.from_numpy(y).cuda(), 3)
    assert t.is_cuda and tuple(t.shape) == (3, 257, 60)
    with pytest.raises(AssertionError):
        deflation.deflationSeed(y[:100], 3)   # F must be 257 or 513 (deflation.py:34)
