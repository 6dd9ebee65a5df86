"""Call ordering: a device-pointer query followed at once by another call on the same index.

A device-pointer ``sknnr_kneighbors`` call returns before its kernels are through: they run on the
caller's stream, in the buffers of the index's first slots, until the caller synchronises.  A call
that reuses one of those slots must wait for them first.  ``transform`` runs in slot 0, whose
projected queries the refine and exhaustive kernels of the device-pointer call still read.

Whether a missing wait shows up here depends on timing (the query is sized to run for tens of
milliseconds, so the ``transform`` lands inside it), so this test is not certain to fail without
the wait.  It pins down the ordering, which no other test covers.
"""

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def test_transform_right_after_device_pointer_query_leaves_both_results_intact():
    import torch

    from sknnr_b200._engine import KNNIndex

    rng = np.random.default_rng(11)
    n_ref, d, n_q, k = 50_000, 32, 1_000_000, 5
    center = rng.standard_normal(d) * 10.0
    scale = rng.uniform(0.5, 2.0, d)
    R = rng.standard_normal((n_ref, d)) * scale + center
    ix = KNNIndex((R - center) / scale, center, scale, None, rng.standard_normal((n_ref, 3)))
    X = rng.standard_normal((n_q, d)) * scale + center
    T = rng.standard_normal((20_000, d)) * scale + center   # other rows; few, so transform lands early

    ref = ix.query(X, k, weights="distance", with_pred=True)
    z_ref = ix.transform(T)

    x_d = torch.from_numpy(X).cuda()
    outs = [torch.full((n_q, k), -1.0, dtype=torch.float64, device="cuda"),
            torch.full((n_q, k), -1, dtype=torch.int64, device="cuda"),
            torch.full((n_q, 3), -1.0, dtype=torch.float64, device="cuda")]
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    ix.query_device(x_d.data_ptr(), False, n_q, d, k, dist_ptr=outs[0].data_ptr(), idx_ptr=outs[1].data_ptr(),
                    pred_ptr=outs[2].data_ptr(), weights="distance", stream=stream.cuda_stream)
    z = ix.transform(T)          # no synchronisation in between
    torch.cuda.synchronize()

    assert np.array_equal(z, z_ref)
    for got, want in zip(outs, ref):
        got = got.cpu().numpy()
        assert got.dtype == want.dtype and got.shape == want.shape
        assert np.array_equal(got, want)
