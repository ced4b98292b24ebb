"""Memory-safety net for the pointer-heavy kernels (compute-sanitizer is closed on the GPU pool): every buffer the
library writes -- state, observations, results -- is carved out of its own allocation between two 4 KB canary bands
(BatchedScotlandYardEnv(guard_bytes=...)); after resets, plain / deferred / host-buffer steps and rollouts at ragged
batch sizes, odd node counts (unaligned rows: the byte heads / tails of warp_copy_bytes and warp_write_node_features),
1 to 15 police, both node_features dtypes and every step variant, no canary byte may have changed.  A write past the
end of a tensor lands in a band instead of in a neighbouring allocation, where the parity tests would not see it."""
import itertools

import pytest

pytestmark = pytest.mark.gpu

SHAPES = [  # (N, E, P, B, belief, reveal, tolls)
    (10, 14, 1, 1, True, 0, 0),
    (13, 20, 2, 33, True, 3, 1),
    (15, 20, 2, 97, False, 0, 0),
    (37, 70, 5, 70, True, 2, 1),
    (50, 110, 3, 1024 + 5, False, 5, 0),
    (101, 190, 15, 45, True, 4, 1),
    (200, 400, 6, 4096 + 19, True, 5, 1),
    (333, 600, 4, 300, True, 5, 1),
    (1000, 2000, 6, 330 * 32 - 21, True, 5, 1),
]
VARIANTS = ["default", "bulk", "fused", "two_kernels", "lagged"]


def _configure(env, variant):
    if variant == "bulk":
        env.set_option("step_kernel", "two_kernels")
        env.set_option("writer_path", "bulk")
    elif variant == "fused":
        env.set_option("step_kernel", "fused")
    elif variant == "two_kernels":
        env.set_option("step_kernel", "two_kernels")
    elif variant == "lagged":
        env.set_option("step_kernel", "two_kernels")
        env.set_option("lagged_kernel", "on")


@pytest.mark.parametrize("shape,variant", [(s, v) for s, v in itertools.product(SHAPES, VARIANTS)
                                           if v == "default" or s[0] in (13, 200, 333)])
def test_no_write_outside_any_buffer(shape, variant):
    import torch

    import student_mechanism_design_b200 as pkg

    N, E, P, B, belief, reveal, tolls = shape
    for nf_dtype in (torch.float32, torch.uint8):
        env = pkg.BatchedScotlandYardEnv(B, P, 9, graph_nodes=N, graph_edges=E, num_graphs=3, seed=5, auto_reset=True, tolls=tolls,
                                         belief=belief, reveal_interval=reveal, keep_reward64=True, node_features_dtype=nf_dtype,
                                         guard_bytes=4096)
        _configure(env, variant)
        env.reset()
        env.check_guards()
        for s in range(6):
            acts = env.sample_actions(step_counter=s)
            if variant == "lagged":
                env.step_deferred(acts)
            else:
                env.step(acts)
        env.flush_observations()
        env.check_guards()
        env.rollout_random(5, step_counter=100)
        env.check_guards()
        env.step_host(env.sample_actions_host(step_counter=200))
        mask = (torch.arange(B, device=env.device) % 3 == 0)
        env.reset(reset_mask=mask)
        torch.cuda.synchronize()
        env.check_guards()
        assert bool(env.action_mask.any()) and int(env.timestep.max()) >= 0
        env.close()


def test_guard_bands_detect_a_stray_write():
    """The checker itself: one byte written right behind (or right in front of) a buffer is reported."""
    import student_mechanism_design_b200 as pkg

    for where in ("above", "below"):
        env = pkg.BatchedScotlandYardEnv(40, 2, 9, graph_nodes=15, graph_edges=20, seed=1, belief=True, guard_bytes=4096)
        env.reset()
        env.check_guards()
        raw, guard, nbytes = env._guards[3]
        raw[guard + nbytes if where == "above" else guard - 1] = 0
        with pytest.raises(pkg.SyError, match="guard band"):
            env.check_guards()
        env.close()
