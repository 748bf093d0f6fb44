"""CPU checks behind colour host-frame detection: the colour example frames convert to the gray goldens, and the
sd_host_frame record keeps its layout now that its last field holds the channel count."""
import ctypes as C

import numpy as np

import colour_examples


def test_bgr_examples_convert_to_the_gray_goldens(oracle, golden):
    bgr = colour_examples.load(golden.dir)
    for i in range(5):
        assert bgr[i].shape == golden.examples[f"gray{i}"].shape + (3,)
        assert np.array_equal(oracle.bgr2gray_u8(bgr[i]), golden.examples[f"gray{i}"]), i
        # real colour: the three channels differ on most pixels, so the conversion weights matter
        assert np.mean(bgr[i][:, :, 0] != bgr[i][:, :, 1]) > 0.5 and np.mean(bgr[i][:, :, 2] != bgr[i][:, :, 1]) > 0.5, i


def test_host_frame_layout_is_unchanged():
    from superviseddescent_b200 import _capi, api
    hf = _capi.HostFrameC
    assert C.sizeof(hf) == 24
    assert [(name, getattr(hf, name).offset) for name, _ in hf._fields_] == \
        [("h_data", 0), ("width", 8), ("height", 12), ("row_stride", 16), ("channels", 20)]
    assert api._HOST_FRAME_DTYPE.itemsize == 24
    assert [api._HOST_FRAME_DTYPE.fields[n][1] for n in api._HOST_FRAME_DTYPE.names] == [0, 8, 12, 16, 20]


def test_host_frame_table_describes_colour_frames():
    from superviseddescent_b200 import api
    batch = np.zeros((3, 20, 30, 3), dtype=np.uint8)
    table, _ = api._host_frame_table(batch)
    assert list(table["w"]) == [30] * 3 and list(table["h"]) == [20] * 3 and list(table["s"]) == [90] * 3
    assert list(table["channels"]) == [3] * 3
    assert list(table["p"] - table["p"][0]) == [0, 1800, 3600]
    padded = np.zeros((20, 100), dtype=np.uint8)
    view = np.lib.stride_tricks.as_strided(padded, (20, 30, 3), (100, 3, 1))     # B,G,R rows with a 100-byte pitch, read in place
    table, keep = api._host_frame_table([np.zeros((5, 7), dtype=np.uint8), view])
    assert list(table["channels"]) == [1, 3] and list(table["s"]) == [7, 100] and list(table["w"]) == [7, 30]
    assert table["p"][1] == padded.ctypes.data
