"""CPU checks of the work distribution of the time-tiled sweep (wafer_tb2_plan, pure host arithmetic): every
(tile, plane) of the launch is covered exactly once, the in-order bulk is a whole number of rounds, the static tail is
balanced, and no segment is a stub that would be all pipeline fill."""
import numpy as np
import pytest

TY, TZ = 30, 60  # output tile of sweep_tb.cuh


def _check(ny, nz, xb, xe, slots):
    import wafer_b200
    plan = wafer_b200.tb2_plan(ny, nz, xb, xe, slots)
    nty, ntz, P = -(-ny // TY), -(-nz // TZ), xe - xb
    cover = np.zeros((nty, ntz, P), dtype=np.int32)
    for owner, y0, z0, xa, xz in plan:
        assert y0 % TY == 0 and z0 % TZ == 0 and 0 <= y0 < ny and 0 <= z0 < nz
        assert xb <= xa < xz <= xe and -1 <= owner < slots
        cover[y0 // TY, z0 // TZ, xa - xb:xz - xb] += 1
    assert (cover == 1).all(), "every tile column plane exactly once"
    bulk = plan[plan[:, 0] < 0]
    tail = plan[plan[:, 0] >= 0]
    ncta = min(slots, max(1, (nty * ntz * P + 7) // 8))
    if 3 * ncta <= 4 * nty * ntz < 4 * ncta:
        ncta = nty * ntz  # nearly one column per CTA: the spare SMs stay idle
    assert len(bulk) % ncta == 0, "the dispatcher hands out whole rounds"
    if len(tail):
        work = np.zeros(ncta)
        for owner, _, _, xa, xz in tail:
            work[owner] += xz - xa
        assert work.max() - work.min() <= 12, "static shares are balanced to within the snapping"
        lens = tail[:, 4] - tail[:, 3]
        assert (lens >= min(6, P)).all(), "no stubs"
    # whole columns in the bulk, in tile order within each chunk
    if len(bulk):
        lens = bulk[:, 4] - bulk[:, 3]
        assert lens.min() >= min(P, 32) or P < 32
    return plan


@pytest.mark.parametrize("ny,nz,xb,xe,slots", [
    (1024, 1024, 0, 1024, 148),   # C4 on one GPU: 630 columns
    (1024, 1024, 0, 128, 148),    # one rank's slab at N = 8
    (1024, 1024, 0, 2, 148),      # a boundary launch of the NCCL-overlap path
    (512, 512, 0, 512, 148),      # 162 columns: one round + 14 columns cut 148 ways
    (2048, 2048, 0, 256, 148),    # C5
    (50, 50, 0, 50, 148), (33, 64, 0, 7, 148), (9, 10, 0, 12, 148), (3, 2, 0, 7, 148), (700, 61, 3, 90, 148),
    (512, 512, 2, 510, 132), (100, 100, 0, 1001, 7), (64, 64, 0, 5000, 148), (480, 512, 0, 512, 148), (300, 512, 0, 600, 148),
    # thin slabs of wide planes: the tail holds fewer than 6 planes per CTA, so only some CTAs get a share
    (512, 512, 0, 40, 148),
    (512, 512, 2, 62, 148),       # interior launch of the NCCL-overlap path at 512^3 on 8 GPUs
    (900, 1200, 0, 70, 148),
])
def test_plan_covers_every_plane_once_and_is_balanced(ny, nz, xb, xe, slots):
    _check(ny, nz, xb, xe, slots)


def test_plan_of_the_512_cubed_case_is_one_round_plus_a_cut_tail():
    plan = _check(512, 512, 0, 512, 148)
    bulk = plan[plan[:, 0] < 0]
    assert len(bulk) == 148 and ((bulk[:, 4] - bulk[:, 3]) == 512).all()
    tail = plan[plan[:, 0] >= 0]
    assert set(tail[:, 0]) == set(range(148)) and (tail[:, 4] - tail[:, 3]).sum() == 14 * 512


def test_plan_rejects_nonsense():
    import wafer_b200
    with pytest.raises(wafer_b200.WaferError):
        wafer_b200.tb2_plan(0, 10, 0, 10)
    with pytest.raises(wafer_b200.WaferError):
        wafer_b200.tb2_plan(10, 10, 5, 5)
