"""Two B200s, NCCL: the ray-sharded data-parallel step of emernerf_b200.distributed (flat-bucket all-reduce, and
reduce-scatter -> sharded FusedAdam -> all-gather) equals the one-GPU full-batch step.  Needs >= 2 GPUs;
skipped otherwise."""
import pytest
import torch

from test_distributed_cpu import _run_dp

pytestmark = pytest.mark.gpu


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_nccl_steps_equal_the_full_batch_step(tmp_path):
    single = _run_dp("cuda", "single", 1, str(tmp_path / "single.pt"))
    for mode in ("allreduce", "sharded", "sharded_defer"):
        got = _run_dp("cuda", mode, 2, str(tmp_path / f"{mode}.pt"))
        for k, v in single.items():
            if "sky_head" in k:
                continue
            denom = v.abs().max().clamp_min(1e-12)
            assert ((got[k] - v).abs().max() / denom).item() < 1e-4, (mode, k, ((got[k] - v).abs().max() / denom).item())
