"""Host-side weight repacking (packing.py) checked on CPU against the oracle's literal restatement of the
reference layers: the algebraic rewrites the CUDA path relies on must be exact up to fp32 rounding."""
import numpy as np
import torch

from mocha_sigasia2023_b200 import packing, weights


def _spatial_conv_ref(x, w, b, A):
    """SpatialConv of the reference (net/blocks.py:55-66): 1x1 conv to K*Cout channels, then
    einsum('nkctv,kvw->nctw'). x [N, Cin, T, V], w [K*Cout, Cin], b [K*Cout], A [K, V, V]."""
    K = A.shape[0]
    y = np.einsum("oc,nctv->notv", w, x) + b[None, :, None, None]
    n, kc, t, v = y.shape
    y = y.reshape(n, K, kc // K, t, v)
    return np.einsum("nkctv,kvw->nctw", y, A)


def test_augmented_weight_layout():
    """The augmented gcn weight is [_gcn_first's weight | the K per-partition biases | zeros], its width padded to the
    next multiple of 16 (one tcgen05 K step; the GEMM's TMA boxes zero-fill the rest of the last 64-column k-block)."""
    sd = {k: v.detach().to(torch.float32) for k, v in weights.generator_state_dict(1777).items()}
    w4, b, A = sd["mot_embedding.2.blk.gcn.conv.weight"], sd["mot_embedding.2.blk.gcn.conv.bias"], sd["mot_embedding.2.A_j"]
    K = A.shape[0]
    wp, _ = packing._gcn_first(w4, b, A)
    co, kp = wp.shape
    w16 = packing._gcn_first_aug(w4, b, A)
    assert w16.shape == (co, (kp + K + 15) // 16 * 16) and w16.shape[1] % 16 == 0
    assert torch.equal(w16[:, :kp], wp)
    assert torch.equal(w16[:, kp:kp + K], b.reshape(K, co).t())
    assert not w16[:, kp + K:].any()


def test_gcn_first_and_augmented_weights_reproduce_spatial_conv():
    """_gcn_first (aggregate first, bias table) and _gcn_first_aug (biases as extra K columns multiplying
    the adjacency column sums, K padded to one tcgen05 K step of 16) are both the reference SpatialConv."""
    sd = {k: v.detach().to(torch.float32) for k, v in weights.generator_state_dict(1777).items()}
    w4 = sd["mot_embedding.2.blk.gcn.conv.weight"]
    b = sd["mot_embedding.2.blk.gcn.conv.bias"]
    A = sd["mot_embedding.2.A_j"]
    K, V = A.shape[0], A.shape[1]
    cin = w4.shape[1]
    rng = np.random.default_rng(0)
    x = rng.standard_normal((2, cin, 3, V)).astype(np.float64)
    want = _spatial_conv_ref(x, w4[:, :, 0, 0].numpy().astype(np.float64), b.numpy().astype(np.float64),
                             A.numpy().astype(np.float64))                      # [N, Cout, T, V]
    # aggregate first: agg[n,t,w, k*Cin+ci] = sum_u x[n,ci,t,u] A[k,u,w]
    agg = np.einsum("nctu,kuw->ntwkc", x, A.numpy().astype(np.float64)).reshape(2, 3, V, K * cin)
    wp, bias2d = packing._gcn_first(w4, b, A)
    got = agg @ wp.numpy().astype(np.float64).T + bias2d.numpy().astype(np.float64)[None, None]
    np.testing.assert_allclose(got.transpose(0, 3, 1, 2), want, rtol=1e-6, atol=1e-6)
    # augmented: rows get the K column sums appended, then zero padding up to the padded K
    wa = packing._gcn_first_aug(w4, b, A).numpy().astype(np.float64)
    assert wa.shape[1] % 16 == 0 and K * cin + K <= wa.shape[1] < K * cin + K + 16
    colsum = A.numpy().astype(np.float64).sum(axis=1)                            # [K, V(w)]
    tail = np.zeros((2, 3, V, wa.shape[1] - K * cin))
    tail[..., :K] = colsum.T[None, None]
    got_aug = np.concatenate([agg, tail], axis=-1) @ wa.T
    np.testing.assert_allclose(got_aug.transpose(0, 3, 1, 2), want, rtol=1e-6, atol=1e-6)


def test_conv_as_gemm_is_tap_major():
    w = torch.arange(2 * 3 * 5, dtype=torch.float32).reshape(2, 3, 5, 1)         # [Cout, Cin, taps, 1]
    g = packing._conv_as_gemm(w)
    assert g.shape == (2, 15)
    for tap in range(5):
        for ci in range(3):
            assert float(g[1, tap * 3 + ci]) == float(w[1, ci, tap, 0])
