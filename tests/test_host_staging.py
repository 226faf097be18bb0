"""Host staging: a queue job (mpcb200_solve_stream) has device arrays and an upload description of its own, so solving a queue
on a handle leaves the handle's resident batch as it was."""
import numpy as np
import pytest

from mpc_local_planner_b200 import capi, configs

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("cid,queue_uprev_dt", [(4, 0.2), (2, 0.0)])
def test_queue_job_leaves_resident_batch_alone(cuda_lib, cid, queue_uprev_dt):
    """cfg 4: the queue has no via-points, the batch has.  cfg 2 (finite control-rate rows): the queue has another u_prev_dt.
    Both use obstacle lists of the same length as the batch."""
    B = 8
    data = configs.generate(cid, B)
    queue = configs.generate(cid, 3 * B, first=B)
    s = capi.BatchSolver(configs.config_for(cid), B, device=0)
    s.upload(data["x0"], data["xf"], data["u_prev"], data["u_prev_dt"], data["obstacles"], data["viapoints"])
    s.solve_resident(cold=True)
    before = s.fetch()
    s.solve_stream(queue["x0"], queue["xf"], queue["u_prev"], queue_uprev_dt, queue["obstacles"], None)
    s.solve_resident(cold=True)
    after = s.fetch()
    s.close()
    for key in ("status", "iters", "u_seq", "x_seq", "dt", "kkt_err"):
        np.testing.assert_array_equal(after[key], before[key], err_msg=key)
