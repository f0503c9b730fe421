"""GPU: the chained-sampling records (tie_iter, vals) of the bucket sampler's multi-pick rounds equal those of one
pick per barrier on tie-heavy clouds.  A record whose maximum a point with different coordinates shares must not keep
saying so once that point has been lowered, or tie_iter comes out early and the next level loses its shortcut."""
import pytest
from conftest import knob_setenv
import torch

import synth

pytestmark = pytest.mark.gpu

CLOUDS = [
    ("lattice16384", lambda b: synth.cloud_lattice(b, 16384, 92), 1500),
    ("lattice12000", lambda b: synth.cloud_lattice(b, 12000, 94, step=1.0), 1200),
    ("dup16384", lambda b: synth.cloud_dup_padded(b, 16384, 90), 4096),
    ("obj16384", lambda b: synth.cloud_ground_objects(b, 16384, 91), 4096),
]


def _chain(xyz, m, k, monkeypatch):
    from tsmdet_b200 import pointnet2_utils as pu

    knob_setenv(monkeypatch, "TSMDET_FPS_ALGO", "bucket")
    knob_setenv(monkeypatch, "TSMDET_FPSB_K", str(k))
    idx, state = pu.farthest_point_sample_chained(xyz, m)
    torch.cuda.synchronize()
    return idx.cpu(), state.tie_iter.cpu(), state.vals.cpu().view(torch.int32)


@pytest.mark.parametrize("b", [16, 148])
@pytest.mark.parametrize("name,gen,m", CLOUDS, ids=[c[0] for c in CLOUDS])
def test_multi_pick_chain_records_equal_one_pick(name, gen, m, b, monkeypatch):
    xyz = torch.from_numpy(gen(b)).cuda()
    got, want = _chain(xyz, m, 8, monkeypatch), _chain(xyz, m, 1, monkeypatch)
    assert torch.equal(got[0], want[0]), name
    assert torch.equal(got[1], want[1]), f"{name}: tie_iter {got[1][got[1] != want[1]][:4]} vs {want[1][got[1] != want[1]][:4]}"
    assert torch.equal(got[2], want[2]), name
