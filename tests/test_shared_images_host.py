"""CPU tier: the host side of ``AttentionDecoder.forward(..., image_index=)`` — validation of the index and the per-image row
lists (CSR) the indexed kernels sum over, and the C descriptor it is handed to the library in."""
import ctypes

import numpy as np
import pytest
import torch


def _build(idx, B=None, n_img=None):
    from icd_b200.models.attention import build_image_index
    idx = torch.as_tensor(idx)
    return build_image_index(idx, idx.shape[0] if B is None and idx.dim() == 1 else B, n_img)


def test_csr_lists_each_images_rows_in_ascending_order():
    idx = [3, 0, 3, 1, 3, 0, 5, 3]                      # images 2 and 4 have no rows, image 3 has four
    img, ptr, rows = _build(idx, n_img=7)
    assert img.dtype == ptr.dtype == rows.dtype == np.int32
    assert img.tolist() == idx
    assert ptr.tolist() == [0, 2, 3, 3, 7, 7, 8, 8]
    for i in range(7):
        mine = rows[ptr[i]:ptr[i + 1]].tolist()
        assert mine == [r for r, v in enumerate(idx) if v == i], i      # ascending, complete
    assert sorted(rows.tolist()) == list(range(len(idx)))


@pytest.mark.parametrize("dtype", [torch.int64, torch.int32, torch.int16, torch.uint8])
def test_every_integer_dtype_is_accepted(dtype):
    img, ptr, rows = _build(torch.tensor([1, 0, 1], dtype=dtype), n_img=2)
    assert img.tolist() == [1, 0, 1] and ptr.tolist() == [0, 1, 3] and rows.tolist() == [1, 0, 2]


def test_random_indices_against_a_plain_grouping():
    g = np.random.default_rng(3)
    for n_img in (1, 2, 17, 300):
        for B in (1, 5, 640):
            idx = g.integers(0, n_img, B)
            _, ptr, rows = _build(idx, n_img=n_img)
            assert ptr[0] == 0 and ptr[-1] == B and np.all(np.diff(ptr) >= 0)
            want = np.concatenate([np.flatnonzero(idx == i) for i in range(n_img)])
            assert np.array_equal(rows, want)


@pytest.mark.parametrize("bad,B,n_img,what", [
    (torch.tensor([0.0, 1.0]), 2, 2, "integer dtype"),
    (torch.tensor([True, False]), 2, 2, "integer dtype"),
    (torch.tensor([[0, 1]]), 2, 2, "1-D"),
    (torch.tensor(0), 1, 2, "1-D"),
    (torch.tensor([0, 1, 1]), 2, 2, "entries"),
    (torch.tensor([0, 2]), 2, 2, "values"),
    (torch.tensor([-1, 0]), 2, 2, "values"),
    ([0, 1], 2, 2, "torch tensor"),
    (torch.tensor([0, 0]), 2, 0, "images"),
])
def test_bad_indices_raise_value_error(bad, B, n_img, what):
    from icd_b200.models.attention import build_image_index
    with pytest.raises(ValueError, match=what):
        build_image_index(bad, B, n_img)


def test_descriptor_layout_and_device_packing():
    """icd_att_index_t as the header declares it (checked against the library's sizeof at load time), filled from one
    packed int32 tensor: img_index, then row_ptr, then rows."""
    from icd_b200 import _lib
    from icd_b200.models.attention import ImageIndex
    assert [f for f, _ in _lib.AttIndex._fields_] == ["n_img", "img_index", "img_row_ptr", "img_rows"]
    assert _lib.lib().icd_sizeof_att_index() == ctypes.sizeof(_lib.AttIndex)
    ix = ImageIndex(torch.tensor([2, 0, 2]), 3, 4)
    desc, packed, _ = ix.device(torch.device("cpu"))
    assert packed.dtype == torch.int32 and packed.tolist() == [2, 0, 2, 0, 1, 1, 3, 3, 1, 0, 2]
    base = packed.data_ptr()
    assert desc.n_img == 4 and desc.img_index == base
    assert desc.img_row_ptr == base + 3 * 4 and desc.img_rows == base + (3 + 5) * 4
