"""CPU: the C restatement of the fused reinforce loop (tests/reinforce_oracle.c) against the reference's reinforce goldens,
and the coin helpers of the fused path (draw_coins / settle_coins) against the step loop's single draws."""
import numpy as np
import pytest
import torch

from pdp_solver_b200.nn import pdp_decimate
from tests.helpers import golden, load, maxdiff, name
from tests.reinforce_oracle import ReinforceOracle


@pytest.mark.parametrize("path", golden("reinforce_*.npz"), ids=name)
def test_restatement_vs_reference(path):
    """merged prediction of every iteration, the iteration count and the active masks exact; final messages within 1e-4"""
    z = load(path)
    o = ReinforceOracle(z["graph_map"], z["bvm"], z["bfm"], z["ef"])
    n_coins = z["coins"].shape[0]
    coins = np.concatenate([z["coins"], np.ones(int(z["T"]), np.float32)]).astype(np.float32)
    n, merged, freeze, q, f = o.reinforce_run((z["init_p0"], z["init_p1"]), (z["init_d0"], z["init_d1"]), int(z["T"]),
                                              float(z["pi"]), float(z["p_dec"]), coins)
    assert n == z["preds"].shape[0] == n_coins
    for it in range(n):
        assert maxdiff(merged[it], z["preds"][it]) == 0, "prediction differs at iteration %d" % (it + 1)
    assert maxdiff(merged[-1], z["pred"]) == 0
    # active mask after every iteration, from the freeze iterations
    act = np.stack([(freeze < 0) | (freeze > it + 1) for it in range(n)]).astype(np.float32)
    assert maxdiff(act, z["actives"].reshape(n, -1)) == 0
    assert maxdiff(q, z["final_q"]) < 1e-4 and maxdiff(f, z["final_f"]) < 1e-4


@pytest.mark.parametrize("done", ["zero", "one", "all"])
def test_coin_helpers_leave_the_generator_where_the_step_loop_does(done):
    """save, draw T, restore, redraw `done`: the same coins and the same generator state as `done` single draws"""
    T = 7
    k = {"zero": 0, "one": 1, "all": T}[done]
    torch.manual_seed(1234)
    ref = [float(torch.rand(1).item()) for _ in range(k)]
    after_ref = torch.rand(5)
    torch.manual_seed(1234)
    coins, state = pdp_decimate.draw_coins(T, "cpu")
    assert coins.shape == (T,) and coins.dtype == torch.float32
    assert coins[:k].tolist() == ref
    pdp_decimate.settle_coins(state, k, "cpu")
    assert torch.equal(torch.rand(5), after_ref)
