"""-m gpu: the one native kernel the reference owns, pinned against ITSELF (SURVEY.md §8 row a6, §8c).

tests/golden/softsplat_ref.pt holds outputs of the reference's own CUDA-C `softsplat_out`
(/root/reference/MOFA-Video-Traj/models/softsplat.py:285-335), templated by the reference's own `cuda_kernel()`,
compiled with nvcc and launched on a B200, then normalised by the reference's own `softsplat(..., 'avg')` wrapper
(recipe: oracle/make_softsplat_ref.py).  Here: `mofa_softsplat_avg` through the reference-signature entry point
models.softsplat.softsplat must reproduce it (fp16 feature storage: <= 2e-3 * max|ref| + 1e-3), on collisions,
out-of-bounds targets, non-finite flow, zero flow and integer shifts.  The reference kernel's raw outputs are also held
against oracle/softsplat.py (fp32 atomics: <= 1e-5): re-run live when oracle/_ref/libsoftsplat_ref.so was built,
otherwise as recorded in the fixture."""
import os

import pytest
import torch

from oracle import make_softsplat_ref as ref
from oracle.softsplat import softsplat as oracle_softsplat
from oracle.softsplat import softsplat_out as oracle_softsplat_out

pytestmark = pytest.mark.gpu


@pytest.mark.skipif(not os.path.exists(ref.GOLDEN), reason="tests/golden/softsplat_ref.pt not generated yet")
def test_engine_softsplat_matches_reference_kernel_golden():
    from mofa_video_b200.models.softsplat import softsplat
    gold = torch.load(ref.GOLDEN)
    for i, c in enumerate(gold["cases"]):
        x, fl, want = c["x"].float(), c["flow"].float(), c["out_avg"]
        got = softsplat(x.cuda(), fl.cuda(), None, "avg").float().cpu()
        assert got.shape == want.shape
        tol = 2e-3 * want.abs().max().item() + 1e-3
        err = (got - want).abs().max().item()
        assert err <= tol, f"case {i} ({gold['kinds'][i]}): {err} > {tol}"


def test_reference_kernel_live_vs_oracle():
    """The reference kernel is re-run when oracle/_ref/libsoftsplat_ref.so was built (it needs the reference's source);
    otherwise its raw outputs recorded in tests/golden/softsplat_ref.pt on the same seeded inputs stand in."""
    gold = None if os.path.exists(ref.LIB) else torch.load(ref.GOLDEN)
    for i in range(len(ref.CASES)):
        x, fl = ref.make_case(i)
        raw = ref.run_reference_kernel(i, x, fl) if gold is None else gold["cases"][i]["out_sum"]
        ones = torch.cat([x, x.new_ones(x.shape[0], 1, x.shape[2], x.shape[3])], 1)
        want = oracle_softsplat_out(ones, fl)
        assert (raw - want).abs().max().item() <= 1e-5 * max(1.0, want.abs().max().item()), i
        avg = raw[:, :-1] / (raw[:, -1:] + 0.0000001)
        assert (avg - oracle_softsplat(x, fl, None, "avg")).abs().max().item() <= 1e-4 * max(1.0, avg.abs().max().item())
