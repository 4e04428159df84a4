"""CPU: MADE's plan (models/maf.py, _MadePlan), everything a degree assignment fixes: the k-block skip ranges of the
masked GEMMs and the job tables of the resident inverse and of its reverse solve. The job planners are host code in
libnfk, so a module built on the CPU plans the same tables a CUDA module does."""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def counts(deg, D):
    """cnt[d] = number of hidden units with degree <= d, d = 0..D."""
    return (deg.long()[None, :] <= torch.arange(D + 1)[:, None]).sum(1)


@pytest.mark.parametrize("flip", [True, False])
@pytest.mark.parametrize("H", [64, 512])
@pytest.mark.parametrize("D", [1, 2, 6, 63])
def test_plan_equals_the_planners(D, H, flip):
    """For the constructor's degrees, with push_inverse on and off: the ranges, kb2_end_half0, job tables, push flag
    and stream byte counts equal what _kb_ranges, _kb_ranges_t, ops.made_inverse_jobs and ops.made_inverse_bwd_jobs
    return for the same degrees. The push kernel is chosen exactly when requested and the degrees change on whole
    8-unit tiles with 2D <= 128."""
    from nf_distillation_b200 import ops
    from nf_distillation_b200.models.maf import MADE, _kb_ranges, _kb_ranges_t
    made = MADE(D, H, flip=flip)
    d1, d2 = made.deg1.long(), made.deg2.long()
    c1, c2 = counts(d1, D), counts(d2, D)
    for push in (True, False):
        made.push_inverse = push
        plan = made._plan()
        assert plan.sorted and plan.resident_ok
        assert plan.ranges == _kb_ranges(d2, d1, made.bn) and plan.ranges_t == _kb_ranges_t(d2, d1, made.bn)
        assert plan.kb2_end_half0 == (_kb_ranges(d2, d1, 256)[1][0] if H == 512 else H // 64)
        aligned = D == 1 or H // 8 >= D - 1
        assert plan.push == (push and aligned and 2 * D <= 128), push
        if plan.push:
            ref = ops.made_inverse_jobs(c1, c2, D, H, made.Dp, made.N3p, push=True)
        else:
            ref = ops.made_inverse_jobs(c1, c2, D, H, made.Dp)
        assert torch.equal(plan.jobs, ref) and plan.nbytes == int(ref[:, 5].sum()) * 16
        bwd = ops.made_inverse_bwd_jobs(c1, c2, D, H, made.N3p)
        assert torch.equal(plan.bwd_jobs, bwd) and plan.bwd_nbytes == int(bwd[:, 5].sum()) * 16


def test_unsorted_degrees_get_full_ranges_and_no_job_tables():
    from nf_distillation_b200.models.maf import MADE
    made = MADE(63, 512, flip=True)
    with torch.no_grad():
        made.deg2.copy_(made.deg2.flip(0))
    plan = made._plan()
    nt = 512 // made.bn
    assert not plan.sorted and not plan.resident_ok
    assert plan.ranges == plan.ranges_t == ([0] * nt, [8] * nt) and plan.kb2_end_half0 == 8
    assert plan.jobs is None and not plan.push and plan.bwd_jobs is None


def test_sorted_degrees_with_a_zero_skip_blocks_but_get_no_job_tables():
    """Degree 0 keeps the block-triangular structure the ranged GEMMs skip, but the resident inverse and the reverse
    solve need every degree >= 1."""
    from nf_distillation_b200.models.maf import MADE, _kb_ranges, _kb_ranges_t
    made = MADE(63, 512, flip=True)
    with torch.no_grad():
        made.deg1.sub_(1)
    d1, d2 = made.deg1.long(), made.deg2.long()
    plan = made._plan()
    assert plan.sorted and not plan.resident_ok
    assert plan.ranges == _kb_ranges(d2, d1, made.bn) and plan.ranges_t == _kb_ranges_t(d2, d1, made.bn)
    assert sum(e - b for b, e in zip(*plan.ranges)) < len(plan.ranges[0]) * 8       # something is skipped
    assert plan.jobs is None and not plan.push and plan.bwd_jobs is None


def test_shapes_the_resident_kernels_do_not_take_get_no_job_tables():
    """Hidden width 2048 leaves no shared memory for the resident kernels' weight ring: no tables, so the inverse and
    its gradients run the D-pass GEMMs."""
    from nf_distillation_b200 import ops
    from nf_distillation_b200.models.maf import MADE
    made = MADE(63, 2048, flip=True)
    assert not ops.made_inverse_resident_supported(63, 2048, made.Dp)
    plan = made._plan()
    assert plan.resident_ok and plan.jobs is None and not plan.push and plan.bwd_jobs is None


def test_a_new_plan_after_a_degree_write_or_a_push_toggle():
    from nf_distillation_b200.models.maf import MADE
    D, H = 6, 512
    made = MADE(D, H, flip=True)
    p0 = made._plan()
    assert made._plan() is p0 and p0.push
    made.push_inverse = False
    p1 = made._plan()
    assert p1 is not p0 and not p1.push
    made.push_inverse = True
    assert made._plan() is not p1 and made._plan().push
    p2 = made._plan()
    with torch.no_grad():
        made.deg1.copy_(torch.arange(H) * (D - 1) // H + 1)     # per-unit degrees: not on whole 8-unit tiles
    p3 = made._plan()
    assert p3 is not p2 and not p3.push and not torch.equal(p3.bwd_jobs, p2.bwd_jobs)
    made.load_state_dict(made.state_dict())                    # copied in place: a new version, the same degrees
    p4 = made._plan()
    assert p4 is not p3 and torch.equal(p4.jobs, p3.jobs)
