"""pb254_timing_* reports the stages of the last call on a context (include/pb254.h): a call that records no stage
leaves an empty list, not the stages of the call before it."""
import numpy as np
import pytest

from util import rand_field


@pytest.mark.parametrize("call", ["poseidon_permute", "lde_batch"])
def test_call_without_stages_clears_the_timings(hostsim_ctx, call):
    rng = np.random.default_rng(11)
    values = rand_field(rng, (3, 1 << 6))
    hostsim_ctx.commit(values, 1, 2)
    assert [name for name, _ in hostsim_ctx.timings()] == ["lde", "merkle"]
    if call == "poseidon_permute":
        hostsim_ctx.poseidon_permute(rand_field(rng, (4, 12)))
    else:
        hostsim_ctx.lde_batch(values, 1)
    assert hostsim_ctx.timings() == []
