"""CPU-side checks of sample_batch / rand_batch / resample_batch: list lengths and ksType are validated in Python before
any handle is made or any library call is issued, so these pass without a device."""
import numpy as np
import pytest

import kde_b200 as K
from tests.util import mixture


@pytest.fixture(scope="module")
def dens():
    rng = np.random.default_rng(0)
    return [K.kde(mixture(rng, d, 20), [0.3] * d) for d in (1, 2, 3)]


def test_length_mismatches_are_refused_before_the_call(dens):
    for kw in ({"Np": [5, 5]}, {"Np": [5] * 3, "seeds": [1, 2]}, {"Np": [5] * 3, "randU": [None]},
               {"Np": [5] * 3, "randN": [None, None, None, None]}):
        with pytest.raises(K.KDEError):
            K.sample_batch(dens, **kw)
    with pytest.raises(K.KDEError):  # randN[i] must be d_i x Np[i]
        K.sample_batch(dens, [5] * 3, randN=[None, np.zeros((3, 5)), None])
    with pytest.raises(K.KDEError):
        K.rand_batch(dens, [1, 2])
    with pytest.raises(K.KDEError):
        K.resample_batch(dens, [5, 5])
    with pytest.raises(K.KDEError):
        K.resample_batch(dens, seeds=[1])


def test_discrete_is_refused_as_resample_refuses_it(dens):
    with pytest.raises(K.KDEError, match="discrete"):
        K.resample_batch(dens, ksType=":discrete")
    with pytest.raises(K.KDEError, match="discrete"):
        K.resample(dens[0], ksType=":discrete")


def test_exported():
    for name in ("sample_batch", "rand_batch", "resample_batch"):
        assert name in K.__all__ and callable(getattr(K, name))
