"""Image completion on the CPU: the grid <-> raster code layouts, the hq_run_args layout (prefix_len took the place of the
trailing reserved field: same size, same offsets) and the Python-side validation of prefix codes."""
import ctypes

import pytest
import torch

from hqtransformer_b200 import _lib
from hqtransformer_b200.sampling import codes_to_grids, grids_to_codes, prefix_rows


@pytest.mark.parametrize("B,H,W", [(1, 8, 8), (3, 8, 8), (2, 4, 6), (5, 1, 3)])
def test_grids_to_codes_inverts_codes_to_grids(B, H, W):
    g = torch.Generator().manual_seed(B * 100 + H * 10 + W)
    ct = torch.randint(0, 1 << 20, (B, H * W), generator=g)
    cb = torch.randint(0, 1 << 20, (B, H * W, 4), generator=g)
    t, b = codes_to_grids(ct, cb, H=H)
    assert tuple(t.shape) == (B, H, W) and tuple(b.shape) == (B, 2 * H, 2 * W)
    ct2, cb2 = grids_to_codes(t, b)
    assert torch.equal(ct2, ct) and torch.equal(cb2, cb)
    # and the other way round, from grids
    gt = torch.randint(0, 1 << 20, (B, H, W), generator=g)
    gb = torch.randint(0, 1 << 20, (B, 2 * H, 2 * W), generator=g)
    t2, b2 = codes_to_grids(*grids_to_codes(gt, gb), H=H)
    assert torch.equal(t2, gt) and torch.equal(b2, gb)


def test_grids_to_codes_stack_order():
    """Bottom code j of top position (r, c) is grid cell (2r + j // 2, 2c + j % 2): within-stack order kh * 2 + kw."""
    gb = torch.arange(16 * 16).reshape(1, 16, 16)
    _, cb = grids_to_codes(torch.zeros(1, 8, 8, dtype=torch.int64), gb)
    for r, c in ((0, 0), (3, 5), (7, 7)):
        for j in range(4):
            assert int(cb[0, r * 8 + c, j]) == int(gb[0, 2 * r + j // 2, 2 * c + j % 2])


def test_grids_to_codes_rejects_bad_shapes():
    with pytest.raises(ValueError):
        grids_to_codes(torch.zeros(2, 8, 8, dtype=torch.int64), torch.zeros(2, 16, 15, dtype=torch.int64))
    with pytest.raises(ValueError):
        grids_to_codes(torch.zeros(2, 8, 8, dtype=torch.int64), torch.zeros(3, 16, 16, dtype=torch.int64))
    with pytest.raises(ValueError):
        grids_to_codes(torch.zeros(64, dtype=torch.int64), torch.zeros(2, 16, 16, dtype=torch.int64))


def test_run_args_layout_unchanged():
    assert ctypes.sizeof(_lib.HQRunArgs) == 16 + 7 * 8 + 56 + 2 * 8 + 8
    assert _lib.HQRunArgs.shared_prefix.offset == 16 + 7 * 8 + 56 + 2 * 8
    assert _lib.HQRunArgs.prefix_len.offset == 16 + 7 * 8 + 56 + 2 * 8 + 4
    assert [f for f, _ in _lib.HQRunArgs._fields_][-2:] == ["shared_prefix", "prefix_len"]


def test_header_names_the_field():
    import os
    import re
    header = open(os.path.join(os.path.dirname(_lib.PKG_DIR), "include", "hqgraft.h")).read()
    body = re.search(r"typedef struct hq_run_args \{(.*?)\} hq_run_args;", header, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = re.findall(r"^\s*(?:const\s+)?[\w]+\*?\s+\*?(\w+);", body, re.M)
    assert fields[-2:] == ["shared_prefix", "prefix_len"]
    assert "reserved" not in fields
    assert "hq_debug_attention_prefix" in _lib.PROTOTYPES and "hq_debug_attention_prefix" in header


def _parts(top, bot):
    return [(top, "prefix_code_top", 10, ()), (bot, "prefix_code_bot", 12, (4,))]


def test_prefix_rows_broadcast_and_dtype():
    t = torch.tensor([[1, 2, 3]], dtype=torch.int32)
    b = torch.randint(0, 12, (4, 3, 4))
    pt, pb = prefix_rows(_parts(t, b), 4, 8, "cpu")
    assert pt.dtype == torch.int64 and tuple(pt.shape) == (4, 3) and bool((pt == pt[:1]).all())
    assert torch.equal(pb, b)
    pt, pb = prefix_rows(_parts([[0, 9]], torch.zeros(1, 2, 4, dtype=torch.int64)), 1, 3, "cpu")
    assert tuple(pt.shape) == (1, 2)


@pytest.mark.parametrize("top,bot,err,match", [
    (torch.zeros(4, 3, 1, dtype=torch.int64), torch.zeros(4, 3, 4, dtype=torch.int64), ValueError, "must be"),
    (torch.zeros(2, 3, dtype=torch.int64), torch.zeros(2, 3, 4, dtype=torch.int64), ValueError, "must be"),
    (torch.zeros(4, 3, dtype=torch.int64), torch.zeros(4, 3, 2, dtype=torch.int64), ValueError, "must be"),
    (torch.zeros(4, 3, dtype=torch.int64), torch.zeros(4, 2, 4, dtype=torch.int64), ValueError, "positions"),
    (torch.zeros(4, 0, dtype=torch.int64), torch.zeros(4, 0, 4, dtype=torch.int64), ValueError, "outside"),
    (torch.zeros(4, 8, dtype=torch.int64), torch.zeros(4, 8, 4, dtype=torch.int64), ValueError, "outside"),
    (torch.zeros(4, 3), torch.zeros(4, 3, 4, dtype=torch.int64), ValueError, "integer"),
    (torch.full((4, 3), 10), torch.zeros(4, 3, 4, dtype=torch.int64), IndexError, "prefix_code_top"),
    (torch.zeros(4, 3, dtype=torch.int64), torch.full((4, 3, 4), -1), IndexError, "prefix_code_bot"),
])
def test_prefix_rows_validation(top, bot, err, match):
    with pytest.raises(err, match=match):
        prefix_rows(_parts(top, bot), 4, 8, "cpu")
