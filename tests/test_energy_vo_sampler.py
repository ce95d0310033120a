"""Batched draws of the weighting matrices (BaseSampler.sample_V_batch), which the batched energy-type VO update uses in place
of one sample_V() call per data point and Newton iteration: same matrices, same order, no GPU needed."""
import numpy as np

import gpde_b200  # noqa: F401
from gpde_b200 import VirtualObservables as VO
from gpde_b200.physics import BoundaryConditionEnsemble, setup_physics


def _host_query_point():
    ph = setup_physics(2, 2, 3, "NDP")
    bce = BoundaryConditionEnsemble(ph, 1, "NDP", rng=np.random.RandomState(0))
    x = np.random.RandomState(1).normal(size=ph['fom'].dim_in)
    return VO.QuerryPoint(ph['fom'], x, bce[0])


def test_rbf_sample_V_batch_equals_sequential_draws_on_the_host():
    qp = _host_query_point()
    s = VO.RadialBasisFunctionSampler(qp, 0.2, 6)
    np.random.seed(7)
    seq = [s.sample_V() for _ in range(5)]
    after_seq = np.random.uniform()
    np.random.seed(7)
    batch = s.sample_V_batch(5)
    assert isinstance(batch, np.ndarray) and batch.shape == (5, qp.dim_out, 6)
    assert np.array_equal(batch, np.stack(seq))
    assert np.random.uniform() == after_seq            # the global stream advanced by exactly the same draws


def test_default_sample_V_batch_stacks_sample_V_calls_in_order():
    qp = _host_query_point()

    class Counting(VO.BaseSampler):
        calls = 0

        def _sample(self):
            Counting.calls += 1
            return np.full((qp.dim_out, 2), float(Counting.calls))

    batch = Counting(qp).sample_V_batch(4)
    assert batch.shape == (4, qp.dim_out, 2) and Counting.calls == 4
    assert [float(v[0, 0]) for v in batch] == [1.0, 2.0, 3.0, 4.0]
