"""
Screen-and-refine arg-max (``gpso_set_screen_mode``) on the GPU: the record returned by the screened call must be
bit-identical -- index, mean, variance and UCB -- to the unscreened full-precision call on the same inputs, on every path
(device / host candidates, one / many windows, leaf batches), for every screening digit count, with ties, near-ties, NaNs and
plateaus among the candidates.
"""
import numpy as np
import pytest

from oracle import gpr_oracle as go
from pygpso_b200 import backend
from tests.test_gpu_parity import VARSIGMA, open_session, synthetic, theta_of

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cuda():
    return backend.default_backend()


def both(s, Xc, theta, mode, varsigma=VARSIGMA):
    """(unscreened record, screened record, screen info) for the same factor and candidates."""
    s.set_screen_mode(0)
    s.factorize(theta)
    ref = s.ucb_argmax(Xc, varsigma)
    assert s.screen_info()["path"] == "unscreened"
    s.set_screen_mode(mode)
    s.factorize(theta)
    got = s.ucb_argmax(Xc, varsigma)
    return ref, got, s.screen_info()


def same_record(a, b):
    # NaN == NaN for the purpose of "the same bits"
    return a[0] == b[0] and all(np.array([x]).tobytes() == np.array([y]).tobytes() for x, y in zip(a[1:], b[1:]))


@pytest.mark.parametrize("kernel", ["Matern52", "SquaredExponential", "Matern32", "Matern12"])
@pytest.mark.parametrize("N,d,M", [(1100, 4, 70_000), (2100, 6, 150_000)])
@pytest.mark.parametrize("mode", [1, 2, 3, 4, 5, 6])
def test_screened_argmax_is_bit_identical(cuda, kernel, N, d, M, mode):
    X, y = synthetic(N, d, seed=N)
    h = go.Hyper(0.25 * np.sqrt(d), 1.0, 1e-3, 0.05)
    Xc = np.random.default_rng(M + mode).random((M, d))
    s = open_session(cuda, kernel, X, y)
    ref, got, info = both(s, Xc, theta_of(h), mode)
    s.close()
    assert same_record(ref, got), (ref, got, info)
    assert info["path"] != "unscreened", info
    if info["path"] in ("screened", "mean-bound"):
        assert info["max_observed_deviation"] <= 0.25 * info["error_bound"]
        assert 1 <= info["survivors"] <= M // 16
    if mode in (1, 3, 4):  # the ladder and the 3/4-digit screens need no full pass here
        assert info["path"] == "screened", info
    if mode == 6:  # forced 2-digit all-pairs screen: too coarse for these UCB spreads, the call must notice
        assert info["digits"] == 2 and info["all_pairs"], info


def test_screened_matches_oracle_winner(cuda):
    """... and the common answer is the oracle's arg-max (sample small enough for the CPU)."""
    N, d, M = 1100, 5, 66_000
    X, y = synthetic(N, d, seed=4)
    h = go.Hyper(0.5, 1.2, 1e-3, 0.0)
    Xc = np.random.default_rng(7).random((M, d))
    s = open_session(cuda, "Matern52", X, y)
    s.set_screen_mode(1)  # automatic (the default), ladder restarted for this matrix size
    s.factorize(theta_of(h))
    got = s.ucb_argmax(Xc, VARSIGMA)
    info = s.screen_info()
    s.close()
    assert info["path"] == "screened", info
    mean, var = go.predict_y("Matern52", X, y, h, Xc)
    assert got[0] == go.ucb_argmax(mean, var, VARSIGMA)[0]


@pytest.mark.parametrize("mode", [1, 2, 3, 5, 6])
def test_ties_near_ties_and_nan(cuda, mode):
    N, d, M = 1100, 4, 80_000
    X, y = synthetic(N, d, seed=12)
    h = go.Hyper(0.5, 1.0, 1e-3, 0.0)
    theta = theta_of(h)
    rng = np.random.default_rng(3)
    Xc = rng.random((M, d))
    s = open_session(cuda, "Matern52", X, y)
    s.set_screen_mode(0)
    s.factorize(theta)
    w = s.ucb_argmax(Xc, VARSIGMA)[0]
    # exact duplicates of the winner before and after it, and near-duplicates whose UCB differs far below the screen's
    # resolution: the refine pass has to decide, with the lowest index on exact ties
    Xt = Xc.copy()
    dup_lo, dup_hi = max(w - 1234, 0), min(w + 4321, M - 1)
    Xt[dup_hi] = Xc[w]
    if dup_lo != w:
        Xt[dup_lo] = Xc[w]
    ref, got, info = both(s, Xt, theta, mode)
    assert ref[0] == min(dup_lo, w)
    assert same_record(ref, got), (ref, got, info)
    assert info["survivors"] >= 3
    # near-ties: perturbed copies of the winner (their UCB may come out above or below it, by far less than the screen resolves)
    for k, eps in enumerate((1e-13, 1e-11, 1e-9, 1e-7)):
        Xt[(w + 17 * (k + 1)) % M] = Xc[w] + eps * rng.standard_normal(d)
    ref, got, info = both(s, Xt, theta, mode)
    assert same_record(ref, got), (ref, got, info)
    assert info["survivors"] >= 7
    # a NaN candidate wins (first NaN, numpy semantics), screened or not; one with a huge coordinate is refined, not trusted
    Xn = Xt.copy()
    Xn[60_000, 1] = np.nan
    Xn[65_000, 2] = 1e300
    Xn[70_000, 0] = np.nan
    ref, got, info = both(s, Xn, theta, mode)
    assert ref[0] == 60_000 and np.isnan(ref[3])
    assert same_record(ref, got), (ref, got, info)
    s.close()


def test_plateau_falls_back_to_full_pass(cuda):
    """Far from the data every candidate has the prior variance and mean: no screen can separate them; the call must notice
    (survivors above the cap) and return the full pass's record."""
    N, d, M = 1100, 3, 70_000
    X, y = synthetic(N, d, seed=2)
    h = go.Hyper(0.05, 1.0, 1e-3, 0.0)
    rng = np.random.default_rng(5)
    Xc = 50.0 + rng.random((M, d))  # all far outside the unit cube of the training data
    s = open_session(cuda, "Matern52", X, y)
    for mode in (1, 5):
        ref, got, info = both(s, Xc, theta_of(h), mode)
        assert same_record(ref, got), (ref, got, info)
        assert info["path"].startswith("full pass"), info
    s.close()


def test_ladder_verdict_survives_the_handle(cuda):
    """The optimiser opens a new session for every fit.  The rung the ladder ended on is kept per matrix size for the process:
    after a call no rung could separate, a NEW session of the same size goes straight to the full pass (same record), and an
    explicit gpso_set_screen_mode restarts the ladder."""
    N, d, M = 1100, 3, 70_000
    X, y = synthetic(N, d, seed=2)
    theta = theta_of(go.Hyper(0.05, 1.0, 1e-3, 0.0))
    Xc = 50.0 + np.random.default_rng(5).random((M, d))  # plateau: prior mean and variance everywhere
    s = open_session(cuda, "Matern52", X, y)
    ref, got, info = both(s, Xc, theta, 1)
    s.close()
    assert same_record(ref, got) and info["path"].startswith("full pass"), info
    s = open_session(cuda, "Matern52", X, y)  # default mode, no explicit call: inherits the verdict
    s.factorize(theta)
    got2 = s.ucb_argmax(Xc, VARSIGMA)
    info2 = s.screen_info()
    assert same_record(ref, got2) and info2["path"] == "unscreened", info2
    s.set_screen_mode(1)
    s.factorize(theta)
    got3 = s.ucb_argmax(Xc, VARSIGMA)
    info3 = s.screen_info()
    s.close()
    assert same_record(ref, got3) and info3["path"].startswith("full pass"), info3
    # leave the ladder of this matrix size restarted for the tests that follow
    s = open_session(cuda, "Matern52", X, y)
    s.set_screen_mode(1)
    s.close()


@pytest.mark.parametrize("host", [True, False])
def test_windows_and_device_path(cuda, host):
    import torch

    N, d, M = 1100, 4, 90_000
    X, y = synthetic(N, d, seed=8)
    h = go.Hyper(0.5, 1.0, 1e-3, 0.0)
    Xc = np.random.default_rng(9).random((M, d))
    s = open_session(cuda, "Matern52", X, y)
    s.set_screen_mode(0)
    s.factorize(theta_of(h))
    ref = s.ucb_argmax(Xc, VARSIGMA)
    s.set_screen_mode(1)
    s.factorize(theta_of(h))
    s.set_window(16_384)  # six screening windows, double-buffered, side-stream overlap
    if host:
        got = s.ucb_argmax(Xc, VARSIGMA)
    else:
        xd = torch.from_numpy(Xc).cuda()
        got = s.ucb_argmax_dev(xd.data_ptr(), M, VARSIGMA, torch.cuda.current_stream().cuda_stream)
    info = s.screen_info()
    s.close()
    assert same_record(ref, got), (ref, got, info)
    assert info["path"] == "screened" and info["screen_windows"] >= 5, info


def test_leaf_batch_screened(cuda):
    """grow(12) leaf batch (265 720 candidates, one third duplicated centres) through the screened call."""
    N, d = 1100, 10
    X, y = synthetic(N, d, seed=21)
    h = go.Hyper(0.25 * np.sqrt(d), 1.0, 1e-3, 0.0)
    bounds = np.array([[0.0, 1.0 / 3.0]] + [[0.0, 1.0]] * (d - 1))
    s = open_session(cuda, "Matern52", X, y)
    s.set_screen_mode(0)
    s.factorize(theta_of(h))
    ref = s.grow_ucb_argmax(bounds, 12, VARSIGMA)
    s.set_screen_mode(1)
    s.factorize(theta_of(h))
    got = s.grow_ucb_argmax(bounds, 12, VARSIGMA)
    info = s.screen_info()
    s.close()
    assert same_record(ref, got), (ref, got, info)
    assert info["path"] != "unscreened"


def test_c3_shape_screened_vs_full(cuda):
    """Config C3's model (N = 4096, d = 10) on 400 000 of its candidates: screened == full pass == FP64 DMMA engine index."""
    import bench

    N, d, M, _ = bench.WORKLOADS["c3"]
    X, y = bench.synthetic_training(N, d)
    theta = bench.fixed_theta(d)
    m = 400_000
    Xc = np.empty((m, d))
    bench.fill_candidates(Xc, 0, m, M, d)
    s = open_session(cuda, "Matern52", X, y)
    ref, got, info = both(s, Xc, theta, 1)
    assert same_record(ref, got), (ref, got, info)
    assert info["path"] == "screened" and info["survivors"] < 2000, info
    assert info["digits"] == 2 and info["all_pairs"], info  # first rung of the ladder is enough on this model
    ref6, got6, info6 = both(s, Xc, theta, 6)
    assert same_record(ref, got6) and info6["path"] == "screened", (ref, got6, info6)
    ref3, got3, info3 = both(s, Xc, theta, 3)
    assert same_record(ref, got3) and info3["path"] == "screened" and info3["survivors"] <= info6["survivors"], (info3, info6)
    ref5, got5, info5 = both(s, Xc, theta, 5)
    assert same_record(ref, got5), (ref, got5, info5)
    assert info5["path"] == "mean-bound" and info5["survivors"] < 20000, info5
    s.set_screen_mode(0)
    s.set_predict_mode(1, 0)
    s.factorize(theta)
    dm = s.ucb_argmax(Xc, VARSIGMA)
    s.close()
    assert dm[0] == ref[0]
    assert abs(dm[3] - ref[3]) <= 1e-8 * max(abs(ref[3]), 1.0)
