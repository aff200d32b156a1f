"""CPU premise of the seeded-key sweep in test_gpu_seeded.py: on every shape the GPU tests load, the reference decompression
(orc_decompress_seeded_ksk / _bsk) puts the AES-CTR stream words (orc_csprng_mask_words) in each row's mask and the bodies after them,
and the stream is n_rows * mask_len words long, as upload_seeded sizes it."""
import ctypes as C
import time

import numpy as np
import pytest

from seeded_shapes import SHAPES, all_sets, bsk_stream, distinct_shapes, ksk_stream, probe_rows, seeded_key, shape_key, stream_rows


def test_shape_selection_covers_every_set():
    """36 classic + 6 multi-bit sets, each mapped to a kept shape; the 30 shapes are distinct"""
    sets = all_sets()
    assert len(sets) == 42
    kept = distinct_shapes()
    assert all(shape_key(q) in kept for q in sets.values())
    assert len(SHAPES) == len(kept) == 30
    assert {"1_0", "1_1", "2_2", "1_5", "1_6", "1_7", "multibit_2_2_g3", "multibit_1_1_g2"} <= set(SHAPES)


@pytest.mark.parametrize("name", SHAPES)
def test_decompression_is_the_stream(orc, name):
    L = orc.lib()
    key = seeded_key(orc, name)
    p = key.p
    t0 = time.time()
    for label, (n_rows, mask_len, body_len), seed, bodies, decompress, std_len in (
            ("KSK", ksk_stream(p), key.ksk_seed, key.ksk_bodies, key.ksk, L.orc_ksk_len(C.byref(p))),
            ("BSK", bsk_stream(p), key.bsk_seed, key.bsk_bodies, key.bsk, L.orc_bsk_len(C.byref(p)))):
        assert bodies.size == n_rows * body_len
        assert std_len == n_rows * (mask_len + body_len)
        rows = probe_rows(n_rows, mask_len)
        full = decompress().reshape(n_rows, mask_len + body_len)
        assert np.array_equal(full[rows, :mask_len], stream_rows(orc, seed, rows, mask_len)), (label, rows)
        assert np.array_equal(full[:, mask_len:], bodies.reshape(n_rows, body_len)), label
        assert (full[rows, :mask_len] != 0).mean() > 0.99
        last = np.zeros(1, dtype=np.uint64)
        L.orc_csprng_mask_words(seed, n_rows * mask_len - 1, last, 1)
        assert full[-1, mask_len - 1] == last[0], f"{label}: the last stream word is the last row's last mask word"
        del full
    print(f"{name}: KSK rows {ksk_stream(p)}, BSK rows {bsk_stream(p)}; probe rows {probe_rows(*ksk_stream(p)[:2])} / "
          f"{probe_rows(*bsk_stream(p)[:2])}; {time.time() - t0:.1f} s")
