"""CPU: the UniPC sampling-loop glue (SURVEY.md 8f.1) -- host coefficients of wan2gp_b200.pipeline.UniPCSchedule + the linear update
the fused kernel applies -- against the UNMODIFIED reference schedulers, whose runs on this module's cases and inputs are recorded in
tests/golden/schedulers.npz, unipc.npz and dpmpp.npz (oracle/gen_golden.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import wan_oracle
from tests.helpers import GOLDEN, rel_l2
from wan2gp_b200.pipeline import DPMppSchedule, UniPCSchedule, causvid_timesteps, euler_timesteps, flow_match_timesteps, lcm_timesteps

CASES = [(6, 5.0), (20, 3.0), (30, 12.0), (2, 1.0), (1, 5.0)]


def run_ours(steps, shift, x, vs, cls=UniPCSchedule):
    sch = cls(steps, shift)
    x = x.clone()
    x_last, m0, m1 = torch.zeros_like(x), torch.zeros_like(x), torch.zeros_like(x)
    traj = []
    for i in range(steps):
        x, xc, x0 = wan_oracle.unipc_step(x, vs[i], x_last, m0, m1, sch.coefficients(i))
        x_last, m0, m1 = xc, x0, m0
        traj.append(x.clone())
    return sch, traj


def reference_run(prefix):
    """The reference scheduler's arrays stored under `<prefix>_*` in tests/golden/schedulers.npz."""
    g = np.load(os.path.join(GOLDEN, "schedulers.npz"))
    return {k[len(prefix) + 1:]: g[k] for k in g.files if k.startswith(prefix + "_")}


def inputs(steps, seed=0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(1, 4, 2, 3, 5, generator=g, dtype=torch.float64), [torch.randn(1, 4, 2, 3, 5, generator=g, dtype=torch.float64) for _ in range(steps)]


@pytest.mark.parametrize("steps,shift", CASES)
def test_unipc_matches_reference_scheduler(steps, shift):
    """Timesteps, sigmas and trajectory of the reference FlowUniPCMultistepScheduler (set_timesteps as any2video.py:519-520)."""
    ref = reference_run(f"unipc_{steps}_{shift:g}")
    x, vs = inputs(steps)
    sch, traj = run_ours(steps, shift, x, vs)
    assert sch.timesteps == [int(t) for t in ref["timesteps"]]
    assert np.allclose(sch.sigmas, ref["sigmas"].astype(np.float64), rtol=0, atol=0)
    for i, xr in enumerate(torch.from_numpy(ref["traj"])):
        # the reference keeps its scalars in fp32; ours are fp64
        assert rel_l2(traj[i], xr) < 2e-5, (i, rel_l2(traj[i], xr))


def test_unipc_matches_fixture():
    """tests/golden/unipc.npz = trajectory of the reference scheduler (oracle/gen_golden.py unipc): 20 steps, shift 3."""
    g = np.load(os.path.join(GOLDEN, "unipc.npz"))
    steps, shift = int(g["steps"]), float(g["shift"])
    x, vs = inputs(steps)
    sch, traj = run_ours(steps, shift, x, vs)
    assert sch.timesteps == [int(t) for t in g["timesteps"]]
    for i in range(steps):
        assert rel_l2(traj[i], torch.from_numpy(g["traj"][i])) < 2e-5


def test_unipc_orders():
    """order 1 on the first step, order 2 afterwards, order 1 again on the last step (lower_order_final); last step returns x0."""
    sch = UniPCSchedule(5, 5.0)
    cs = [sch.coefficients(i) for i in range(5)]
    assert cs[0]["pr"] == 0 and not cs[0]["use_corrector"] and all(c["use_corrector"] for c in cs[1:])
    assert all(c["pr"] != 0 for c in cs[1:4]) and cs[4]["pr"] == 0
    assert cs[4]["pp"] == 0 and abs(cs[4]["pq"] - 1.0) < 1e-12            # sigma_next = 0: x_next = x0
    assert all(np.isfinite(list(c.values())).all() for c in cs)


@pytest.mark.parametrize("steps,shift", CASES)
def test_dpmpp_matches_reference_scheduler(steps, shift):
    """sample_solver="dpm++" (any2video.py:523-532): host coefficients + the same fused update vs FlowDPMSolverMultistepScheduler."""
    ref = reference_run(f"dpmpp_{steps}_{shift:g}")
    x, vs = inputs(steps)
    sch, traj = run_ours(steps, shift, x, vs, DPMppSchedule)
    assert sch.timesteps == [int(t) for t in ref["timesteps"]]
    for i, xr in enumerate(torch.from_numpy(ref["traj"])):
        assert rel_l2(traj[i], xr) < 2e-5, (i, rel_l2(traj[i], xr))


def test_dpmpp_matches_fixture():
    g = np.load(os.path.join(GOLDEN, "dpmpp.npz"))
    steps, shift = int(g["steps"]), float(g["shift"])
    x, vs = inputs(steps)
    sch, traj = run_ours(steps, shift, x, vs, DPMppSchedule)
    assert sch.timesteps == [int(t) for t in g["timesteps"]]
    for i in range(steps):
        assert rel_l2(traj[i], torch.from_numpy(g["traj"][i])) < 2e-5


def test_single_step_solver_tables_match_reference():
    """euler / lcm / causvid are the same Euler kernel with different sigma tables: tables and whole trajectories vs the reference
    EulerScheduler-free restatement, LCMScheduler and FlowMatchScheduler (any2video.py:506-517, 533-543)."""
    def ours(ts, steps):
        x, vs = inputs(steps)
        for i in range(steps):
            x = wan_oracle.euler_step(x, vs[i], ts[i] / 1000.0, ts[i + 1] / 1000.0)
        return x
    for steps, shift in ((4, 5.0), (8, 3.0), (12, 7.0)):
        ref = reference_run(f"lcm_{steps}_{shift:g}")
        ts = lcm_timesteps(steps, shift)
        assert len(ts) == min(steps, 8) + 1 and np.allclose(ts[:-1], ref["timesteps"], rtol=1e-6)
        assert rel_l2(ours(ts, len(ts) - 1), torch.from_numpy(ref["out"]).double()) < 1e-5
    for steps in (4, 9):
        ref = reference_run(f"causvid_{steps}")
        assert rel_l2(ours(causvid_timesteps(steps), steps), torch.from_numpy(ref["out"]).double()) < 1e-5
    # Wan EulerScheduler (shared/utils/euler_scheduler.py)
    for steps, shift in ((50, 12.0), (20, 5.0), (1, 3.0)):
        ref = reference_run(f"euler_{steps}_{shift:g}")
        ts = euler_timesteps(steps, shift)
        assert len(ts) == steps + 1 and ts[-1] == 0.0 and np.allclose(ts[:-1], ref["timesteps"], rtol=1e-6)
        assert rel_l2(ours(ts, steps), torch.from_numpy(ref["out"])) < 1e-6


def test_denoiser_solver_selection():
    from wan2gp_b200.pipeline import WanDenoiser
    n = {s: WanDenoiser(None, num_steps=12, shift=5.0, sample_solver=s, device="cpu").num_steps for s in ("euler", "unipc", "", "dpm++", "lcm", "causvid")}
    assert n == {"euler": 12, "unipc": 12, "": 12, "dpm++": 12, "lcm": 8, "causvid": 9}      # lcm caps at 8 steps, causvid's table has 9
    with pytest.raises(NotImplementedError):
        WanDenoiser(None, sample_solver="heun", device="cpu")


def test_hunyuan_flow_match_table_matches_reference():
    """HunyuanDenoiser's sigma grid == FlowMatchDiscreteScheduler(shift, reverse=True, solver="euler") and its step is the Euler update."""
    for steps, shift in ((30, 7.0), (50, 9.0), (4, 6.0)):
        ref = reference_run(f"flow_match_{steps}_{shift:g}")
        ts = flow_match_timesteps(steps, shift)
        assert len(ts) == steps + 1 and ts[-1] == 0.0 and np.allclose(ts[:-1], ref["timesteps"], rtol=1e-6)
        xo, vs = inputs(steps)
        for i in range(steps):
            xo = wan_oracle.euler_step(xo, vs[i], ts[i] / 1000.0, ts[i + 1] / 1000.0)
        assert rel_l2(xo, torch.from_numpy(ref["out"]).double()) < 1e-5
