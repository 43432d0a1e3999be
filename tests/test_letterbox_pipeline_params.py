"""Host side of the letterbox tables the pipelined processors upload (no device needed): engine.letterbox_rows, which
ShardedPostProcessor.submit / submit_tta and PipelinedPostProcessor.submit call before anything is set up or enqueued,
and the float32 rounding of the staging buffer's fill."""
import numpy as np
import pytest
import torch

from yoloseries_b200.engine import letterbox_rows, letterbox_table

INFO = [dict(scale=0.731, pad_top=3, pad_left=0, org_shape=(167, 219)),
        dict(scale=0.25, pad_top=0, pad_left=21, org_shape=(512, 470)),
        dict(scale=1.0, pad_top=0, pad_left=0, org_shape=[128, 160])]


def test_rows_are_the_table_in_image_order():
    rows = letterbox_rows(INFO, 3)
    assert rows == letterbox_table(INFO)
    assert rows[0] == [0.731, 3.0, 0.0, 167.0, 219.0] and rows[2][3:] == [128.0, 160.0]   # (org_h, org_w)


@pytest.mark.parametrize("n", [0, 2, 4])
def test_one_dict_per_image(n):
    info = (INFO * 2)[:n]
    with pytest.raises(ValueError, match=f"need one info dict per image: {n} != 3"):
        letterbox_rows(info, 3)


def test_staging_fill_rounds_like_the_table_upload_of_run():
    """LetterboxStaging writes the rows through a numpy view of its pinned float32 buffer; PostProcessor.run uploads
    torch.tensor(rows, dtype=float32).  Both must give the same bits, or the pipelined rows would differ from run's."""
    rng = np.random.default_rng(5)
    vals = [0.1, 1 / 3, 0.731, 1.6, 2.0 ** -149, 2.0 ** -126 * 0.75, 16777217.0, 3.4028235e38, 1e-45, 0.0]
    vals += list(rng.uniform(0.01, 4.0, 40)) + [int(x) for x in rng.integers(0, 1 << 25, 40)]
    rows = [vals[i:i + 5] for i in range(0, len(vals), 5)]
    buf = np.empty((len(rows), 5), dtype=np.float32)
    buf[...] = rows
    np.testing.assert_array_equal(buf.view(np.uint32), torch.tensor(rows, dtype=torch.float32).numpy().view(np.uint32))
