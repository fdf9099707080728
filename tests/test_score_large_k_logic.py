"""CPU tests of the k bounds of the ranking entry points: the "auto" scorer choice, the header's bound, and the
argument checks of the C ABI for k above ETPGT_SCORE_MAX_K (these calls return before touching a device)."""

import re
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]
HEADER = ROOT / "include" / "etpgt_b200.h"


def _parent_choice(batch, dim, k):
    """The choice made before k > 32 reached the tensor cores (model/base.py and parallel.sharded_predict)."""
    return "bf16" if batch >= 64 and dim in (64, 128, 192, 256) and 1 <= k <= 32 else "fp32"


def test_header_bound():
    from etpgt_b200 import ops

    m = re.search(r"#define ETPGT_SCORE_MAX_K (\d+)", HEADER.read_text())
    assert m and int(m.group(1)) == ops.SCORE_MAX_K == 256


@pytest.mark.parametrize("dim", [32, 64, 128, 192, 256])
@pytest.mark.parametrize("batch", [1, 63, 64, 1000])
def test_auto_choice_unchanged_up_to_64(dim, batch):
    from etpgt_b200 import ops

    for k in range(1, 65):
        assert ops.auto_score_precision(batch, dim, k) == _parent_choice(batch, dim, k), (batch, dim, k)


@pytest.mark.parametrize("batch", [1, 63, 64, 1000])
def test_auto_choice_above_64_is_tensor_cores(batch):
    from etpgt_b200 import ops

    for dim in (64, 128, 192, 256):
        for k in (65, 100, 128, 129, 200, 256):
            assert ops.auto_score_precision(batch, dim, k) == "bf16"
    assert ops.tensor_core_scoring_supported(256, 256)
    assert not ops.tensor_core_scoring_supported(256, 257)
    assert not ops.tensor_core_scoring_supported(256, 0)
    assert not ops.tensor_core_scoring_supported(32, 100)


@pytest.fixture(scope="module")
def lib():
    from etpgt_b200 import _lib

    if not _lib.lib_path().exists():
        pytest.skip("library not built")
    return _lib


def _rc_and_message(lib, name, *args):
    rc = getattr(lib.load(), name)(*args)
    return rc, lib.last_error()


def test_abi_rejects_k_257(lib):
    einval = -1
    rc, msg = _rc_and_message(lib, "etpgt_score_topk_bf16_eval", None, None, 10, 1000, 256, 257, 0, None, None, None,
                              None, None, 0, None)
    assert rc == einval and "256" in msg, msg
    rc, msg = _rc_and_message(lib, "etpgt_score_topk_bf16_exclude", None, None, 10, 1000, 256, 257, 0, None, None,
                              None, None, None, 0, None, 0, None)
    assert rc == einval and "256" in msg, msg
    rc, msg = _rc_and_message(lib, "etpgt_topk_merge", None, None, 10, 2, 257, None, None, None)
    assert rc == einval and "256" in msg, msg
    rc, msg = _rc_and_message(lib, "etpgt_topk_merge_parts", None, 2, 1 << 20, 1 << 16, 10, 257, 0, 10, None, None,
                              None, None, None)
    assert rc == einval and "256" in msg, msg
    # the fp32 scorer keeps its bound of 64 and names the tensor-core bound
    rc, msg = _rc_and_message(lib, "etpgt_score_topk_f32", None, None, 10, 1000, 256, 65, 0, None, None, None, 0, None)
    assert rc == einval and "64" in msg and "256" in msg, msg



@pytest.mark.parametrize("batch,items", [(2049, 1_000_000), (37889, 82174), (24582, 100_000), (8195, 300_000),
                                         (23861, 82174), (256, 10_000_000), (1, 100), (0, 100)])
def test_row_chunks_cover_every_chunk(lib, batch, items):
    """The workspace ops.score_topk allocates for k > 32 is enough for every chunk it scores, including a shorter
    last chunk whose split plan needs more (the library's sizing is not monotone in the row count)."""
    from etpgt_b200 import ops

    for k in (33, 100, 256):
        rows, ws = ops.score_row_chunks(batch, items, k)
        chunks = {min(rows, batch - r) for r in range(0, batch, rows)} if batch else {0}
        for n in chunks:
            assert ws >= ops.size("etpgt_score_topk_bf16_workspace_bytes", n, items, k), (batch, items, k, n)
        if rows > 1:
            assert ops.size("etpgt_score_topk_bf16_workspace_bytes", rows, items, k) <= 4 << 30
    # k <= 32: one call, the workspace of the whole batch, as before
    assert ops.score_row_chunks(batch, items, 20) == (batch, ops.size("etpgt_score_topk_bf16_workspace_bytes", batch,
                                                                       items, 20))
