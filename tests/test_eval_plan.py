"""CPU: packing of a node set into the evaluation plan of runtime.GraphedEvalPass (one upload, fixed-width entries)."""
import numpy as np
import pytest

from pcgnn_b200.runtime import pack_eval_plan


@pytest.mark.parametrize("n,B", [(1, 4), (3, 4), (5, 2), (8, 4), (4096, 1024), (27572, 1024), (5184, 1024)])
def test_plan_holds_the_nodes_in_order_and_pads_with_the_last_entry_first_id(n, B):
    nodes = np.random.default_rng(n).permutation(10 * n)[:n]
    plan = pack_eval_plan(nodes.tolist(), B)
    k = -(-n // B)
    assert plan.dtype == np.int32 and plan.shape == (k, B)
    flat = plan.reshape(-1)
    assert np.array_equal(flat[:n], nodes)
    assert (flat[n:] == nodes[(k - 1) * B]).all()          # padding repeats the last entry's own first id
    if n % B == 0:
        assert flat.shape[0] == n                           # n = k*B: no padding at all


def test_plan_of_fewer_nodes_than_a_batch_is_one_entry():
    plan = pack_eval_plan(np.array([7, 3, 9]), 128)
    assert plan.shape == (1, 128) and plan[0, :3].tolist() == [7, 3, 9] and (plan[0, 3:] == 7).all()


def test_empty_set_and_bad_input_raise():
    with pytest.raises(ValueError, match="at least one node"):
        pack_eval_plan([], 64)
    with pytest.raises(ValueError):
        pack_eval_plan([1, 2], 0)
    with pytest.raises(ValueError):
        pack_eval_plan([1, -2], 4)
