"""Host side of MC dropout (no GPU): the AUROC and ECE helpers, the dropout-id contract of the sample rows and the
workspace the library asks for."""
import ctypes as C

import numpy as np
import pytest

from oracle import dropout_stream as ds


def _desc(batch, T=3840, C_=6, nc=2, H=64, layers=2, training=0, need_grad=0):
    from multimodalsignal_b200._ext import CnnGruDesc
    d = CnnGruDesc()
    d.batch, d.in_channels, d.seq_len, d.num_classes = batch, C_, T, nc
    d.cnn_out, d.hidden, d.layers = 32, H, layers
    d.training, d.attention, d.need_grad, d.dropout_p = training, 1, need_grad, 0.5
    return d


def test_auroc_matches_sklearn_with_ties():
    from sklearn.metrics import roc_auc_score
    from multimodalsignal_b200.uncertainty import auroc
    rng = np.random.default_rng(0)
    for n, levels in ((50, 4), (200, 1000), (31, 2), (7, 1)):
        scores = rng.integers(0, levels, n).astype(np.float64) * 0.25      # few levels: many ties
        pos = rng.random(n) < 0.4
        pos[0], pos[1] = True, False
        assert auroc(scores, pos) == pytest.approx(roc_auc_score(pos, scores), abs=1e-12)


def test_auroc_single_class_is_nan():
    from multimodalsignal_b200.uncertainty import auroc
    assert np.isnan(auroc([0.1, 0.5, 0.2], [True, True, True]))
    assert np.isnan(auroc([0.1, 0.5, 0.2], [False, False, False]))
    assert np.isnan(auroc([], []))


def test_expected_calibration_error_against_a_loop():
    from multimodalsignal_b200.uncertainty import expected_calibration_error
    rng = np.random.default_rng(1)
    for n, nc, bins in ((500, 2, 10), (97, 4, 7), (1, 3, 10)):
        logits = rng.normal(size=(n, nc)) * 2
        probs = np.exp(logits) / np.exp(logits).sum(axis=1, keepdims=True)
        probs[0] = 1.0 / nc                                                 # a confidence on a bin edge
        labels = rng.integers(0, nc, n)
        ece = 0.0
        for k in range(bins):
            lo, hi = k / bins, (k + 1) / bins
            rows = [i for i in range(n) if lo <= probs[i].max() < hi or (k == bins - 1 and probs[i].max() == 1.0)]
            if rows:
                acc = np.mean([probs[i].argmax() == labels[i] for i in rows])
                conf = np.mean([probs[i].max() for i in rows])
                ece += len(rows) / n * abs(acc - conf)
        assert expected_calibration_error(probs, labels, bins=bins) == pytest.approx(ece, abs=1e-12)
    assert expected_calibration_error(np.array([[0.0, 1.0]]), [1]) == 0.0


@pytest.mark.parametrize("T,H", [(3840, 64), (3840, 128), (336, 32), (16384, 128)])
def test_site0_ids_of_the_largest_accepted_call_stay_below_the_head_site(T, H):
    """The library and mc_dropout accept R sample rows while R * L * 2H < 2^38: the largest site-0 id is then below the
    head site's first id, so the two sets of ids are disjoint; one more row is refused."""
    from multimodalsignal_b200 import _ext
    from multimodalsignal_b200.uncertainty import SITE0_LIMIT, gru_seq_len
    L = ds.gru_seq_len(T)
    assert gru_seq_len(T) == L and SITE0_LIMIT == ds.HEAD_BASE
    row = L * 2 * H
    r_max = (ds.HEAD_BASE - 1) // row                           # the most sample rows one call may hold
    last_site0 = r_max * row - 1                                # id of the last element of row r_max - 1, site 0
    assert last_site0 < ds.HEAD_BASE
    assert (r_max + 1) * row >= ds.HEAD_BASE                    # one more row reaches the bound
    ids = ds.gru_site_ids(0, 2, L, H)                           # the formula: row r starts at r * L * 2H
    assert int(ids[1, 0, 0]) == row and int(ids[-1, -1, -1]) == 2 * row - 1
    head_first = int(ds.head_site_ids(1)[0, 0])
    assert head_first == ds.HEAD_BASE > last_site0
    assert int(ds.gru_site_ids(1, 1, L, H)[0, 0, 0]) == ds.LAYER_STRIDE > ds.HEAD_BASE + r_max * ds.HEAD_HID
    lib = _ext.load_library()
    if r_max * L < 2 ** 31 - 1:                                 # rows x steps must also fit the GEMMs' int row count
        assert lib.mms_cnngru_mc_workspace_bytes(C.byref(_desc(r_max, T=T, H=H)), 1) > 0
    assert lib.mms_cnngru_mc_workspace_bytes(C.byref(_desc(r_max + 1, T=T, H=H)), 1) == -1


def test_mc_workspace_is_sized_for_the_windows():
    """64 windows x 32 samples need less workspace than an eval forward of the 2048 replicated rows: the encoder and
    layer-0 buffers are per window."""
    from multimodalsignal_b200 import _ext
    lib = _ext.load_library()
    for H in (64, 128):
        mc = lib.mms_cnngru_mc_workspace_bytes(C.byref(_desc(64, H=H)), 32)
        ev = lib.mms_cnngru_workspace_bytes(C.byref(_desc(2048, H=H)))
        assert 0 < mc < ev, (H, mc, ev)
    assert lib.mms_cnngru_mc_workspace_bytes(C.byref(_desc(64)), 0) == -1                   # samples < 1
    assert lib.mms_cnngru_mc_workspace_bytes(C.byref(_desc(64, training=1)), 4) == -1       # eval only
    assert lib.mms_cnngru_mc_workspace_bytes(C.byref(_desc(64, need_grad=1)), 4) == -1      # no gradients
