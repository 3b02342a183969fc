"""More than 65535 (b, h) rows through the generic-score path. The keys kernel, the selection pass and the compaction
grid decode (row, tile) from a 1-D grid, so the row count is not capped by gridDim.y. Needs a B200: `pytest -m gpu`."""
import pytest
import torch

from oracle import press_oracle as O

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _native():
    from kvpress_b200 import native
    native.load()
    return native


@pytest.mark.parametrize("kind", ["random", "ties"])
def test_selection_and_compaction_beyond_65535_rows(kind):
    nat = _native()
    B, H, S, D, n_kept = 3, 22000, 300, 16, 77  # 66000 rows, two tiles per row (the second one partial)
    g = torch.Generator().manual_seed(66000)
    scores = torch.randn(B, H, S, generator=g)
    if kind == "ties":
        scores = (scores * 2).round() / 2
    scores = scores.to(torch.bfloat16)
    canon = O.select_lowest_index_ties(scores, n_kept)

    idx = nat.scores_select(scores.to(DEV), n_kept)
    assert torch.equal(idx.long().cpu(), canon)

    k = torch.randn(B, H, S, D, generator=g).to(torch.bfloat16)
    v = torch.randn(B, H, S, D, generator=g).to(torch.bfloat16)
    k_out, v_out, idx2 = nat.scores_compress(scores.to(DEV), k.to(DEV), v.to(DEV), n_kept, return_indices=True)
    assert torch.equal(idx2.long().cpu(), canon)
    assert torch.equal(k_out.cpu(), O.gather_rows(k, canon))
    assert torch.equal(v_out.cpu(), O.gather_rows(v, canon))
