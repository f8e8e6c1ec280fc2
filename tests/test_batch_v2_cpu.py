"""Host side of the version-2 batch decoder (gauspcc_b200/batch.py v2_stage_tables): the chunk tables of one stage of a union level,
built from the member scenes' streams, against a hand-built restatement of the format; malformed streams raise naming the scene."""
import numpy as np
import pytest

from gauspcc_b200.batch import v2_stage_tables


def _stream(rng, n, chunk):
    """a version-2 stream of n symbols under the file's chunk size: u16 byte count per chunk, then the chunks' bytes (random)"""
    cl = max(1, min(chunk, max(64, -(-n // 64))))                   # bitstream.py: chunk_len(n, chunk_size), restated
    chunks = -(-n // cl)
    cnt = rng.integers(0, 12, chunks).astype("<u2")
    return cnt.tobytes() + rng.integers(0, 256, int(cnt.sum()), dtype=np.uint8).tobytes()


def _restated(members, row0):
    """rows / offsets / payload written out chunk by chunk"""
    rows, offs, payload, r, o = [row0], [0], b"", row0, 0
    for _, n, chunk, sb in members:
        cl = max(1, min(chunk, max(64, -(-n // 64))))
        chunks = -(-n // cl)
        for w in range(chunks):
            rows.append(r + min((w + 1) * cl, n))
            o += int.from_bytes(sb[2 * w:2 * w + 2], "little")
            offs.append(o)
        payload += sb[2 * chunks:]
        r += n
    return rows, offs, payload


# (rows, file chunk size): chunk lengths 32 / 64 / 2048 / 16384 and others, last chunks of 1 row, and members whose chunk length
# (the 64-chunk rule) falls below their file's chunk size
MEMBERS = [
    (97, 32),                 # 32, 32, 32, 1
    (2049, 2048),             # chunk_len 64 < 2048: 32 chunks of 64 and one of 1 row
    (5000, 2048),             # chunk_len 80
    (2048 * 64 + 5, 2048),    # chunk_len 2048, last chunk 5 rows
    (16384 * 64 + 1, 16384),  # chunk_len 16384, last chunk 1 row
    (1, 16384),               # one row
    (64 * 64, 64),            # chunk_len 64, 64 full chunks
]


@pytest.mark.parametrize("row0", [0, 1000])
def test_tables_match_restatement(row0):
    rng = np.random.default_rng(7)
    members = [(f"scene-{j}", n, c, _stream(rng, n, c)) for j, (n, c) in enumerate(MEMBERS)]
    rows, offs, payload = v2_stage_tables(members, row0=row0)
    r_rows, r_offs, r_payload = _restated(members, row0)
    assert rows.dtype == np.uint32 and offs.dtype == np.uint32
    assert rows.tolist() == r_rows
    assert offs.tolist() == r_offs
    assert payload == r_payload
    assert rows.shape == offs.shape and int(offs[-1]) == len(payload)
    assert int(rows[-1]) == row0 + sum(n for n, _ in MEMBERS)


def test_known_chunk_boundaries():
    rng = np.random.default_rng(1)
    rows, _, _ = v2_stage_tables([("a", 97, 32, _stream(rng, 97, 32)), ("b", 2049, 2048, _stream(rng, 2049, 2048))])
    assert rows[:5].tolist() == [0, 32, 64, 96, 97]
    assert rows[5:].tolist() == [97 + 64 * (w + 1) for w in range(32)] + [97 + 2049]
    big = 16384 * 64 + 1
    rows, _, _ = v2_stage_tables([("c", big, 16384, _stream(rng, big, 16384))])
    assert rows.tolist() == [16384 * w for w in range(65)] + [big]


def test_members_with_different_chunk_sizes_and_empty():
    rng = np.random.default_rng(3)
    rows, offs, payload = v2_stage_tables([])
    assert rows.tolist() == [0] and offs.tolist() == [0] and payload == b""
    a, b = _stream(rng, 300, 32), _stream(rng, 300, 2048)             # same rows, different files' chunk sizes: 32 vs 64
    rows, _, _ = v2_stage_tables([("a", 300, 32, a), ("b", 300, 2048, b)])
    assert np.diff(rows[:11]).tolist() == [32] * 9 + [12]
    assert np.diff(rows[10:]).tolist() == [64] * 4 + [44]


def test_truncated_stream_names_the_scene():
    rng = np.random.default_rng(5)
    good = _stream(rng, 5000, 2048)
    bad = _stream(rng, 2049, 2048)[:20]                              # 33 chunks need 66 header bytes
    with pytest.raises(ValueError, match=r"scene-b\.bin: truncated version-2 stream"):
        v2_stage_tables([("scene-a.bin", 5000, 2048, good), ("scene-b.bin", 2049, 2048, bad)])


def test_counts_that_do_not_sum_name_the_scene():
    rng = np.random.default_rng(6)
    good = _stream(rng, 97, 32)
    for bad in (_stream(rng, 5000, 2048)[:-1], _stream(rng, 5000, 2048) + b"\0"):   # one byte short / one byte too many
        with pytest.raises(ValueError, match=r"scene 1: corrupt version-2 stream"):
            v2_stage_tables([("scene 0", 97, 32, good), ("scene 1", 5000, 2048, bad)])


def test_chunk_size_is_range_checked_without_a_device():
    from gauspcc_b200 import pcc_utils
    for bad in (16, 31, 16385):
        with pytest.raises(ValueError, match="32..16384"):
            pcc_utils.compress_point_clouds([np.zeros((1, 3), np.int32)], "unused.pt", ["unused.bin"], gpu_coder_chunk=bad)
