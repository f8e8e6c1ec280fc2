"""Host half of the GPU text parser (gauspcc_b200/plyio.py): the lines the kernel leaves to the host, given as the byte spans it
reports, are read with cli.read_points' own per-line rule and spliced back between the GPU's rows in line order."""
import numpy as np
import torch

from gauspcc_b200 import cli, plyio


def _spans(text: bytes, host_line_numbers, gpu_rows_before):
    lines, pos = [], 0
    for raw in text.splitlines(keepends=True):
        body = raw.rstrip(b"\r\n")
        lines.append((pos, pos + len(body)))
        pos += len(raw)
    return np.array([(*lines[k], r) for k, r in zip(host_line_numbers, gpu_rows_before)], dtype=np.uint32)


def test_host_rows_follow_read_points_rule(tmp_path):
    text = (b"ply\n1 2 3\nnan 1 2\n4 5 6 7\n-Infinity\t0 1\r\n1_0 2 3\nx 1 2\n"
            b"7 8 9\n\xc2\xa01\xe2\x80\x835 6\n1\x0b2 3\n\xff\n")
    # the GPU decides lines 0, 1, 3, 6, 7 (rows "1 2 3", "4 5 6", "7 8 9") and hands over 2, 4, 5, 8, 9, 10
    spans = _spans(text, [2, 4, 5, 8, 9, 10], [1, 2, 2, 3, 3, 3])
    before, extra = plyio.host_rows(text, spans)
    assert before.tolist() == [1, 2, 2, 3, 3]                      # the lone "\xff" line has no row
    raw_lines = text.splitlines()                                  # bytes split at "\n", "\r\n" and "\r" only
    want = [plyio.xyz_of_line(raw_lines[k].decode(plyio._TEXT_ENCODING, errors="ignore")) for k in (2, 4, 5, 8, 9)]
    assert np.array_equal(extra, np.array(want), equal_nan=True)
    gpu = torch.tensor([[1.0, 2, 3], [4, 5, 6], [7, 8, 9]], dtype=torch.float64)
    got = plyio.splice_rows(gpu, before, torch.from_numpy(extra)).numpy()
    p = tmp_path / "t.ply"
    p.write_bytes(text)
    ref = cli.read_points(str(p))
    assert got.shape == ref.shape == (8, 3)
    assert np.array_equal(got.view(np.uint64), ref.view(np.uint64))


def test_splice_edges():
    gpu = torch.arange(6, dtype=torch.float64).reshape(2, 3)
    extra = torch.full((3, 3), -1.0, dtype=torch.float64)
    got = plyio.splice_rows(gpu, [0, 0, 2], extra)                 # before the first row, twice, and after the last
    assert got[:, 0].tolist() == [-1, -1, 0, 3, -1]
    assert plyio.splice_rows(gpu, [], extra[:0]) is gpu
    only = plyio.splice_rows(gpu[:0], [0, 0], extra[:2])
    assert only.shape == (2, 3) and (only == -1).all()


def test_xyz_of_line_is_read_points_rule():
    assert plyio.xyz_of_line("1 2 3 4\n") == [1.0, 2.0, 3.0]
    assert plyio.xyz_of_line("1 2\n") is None
    assert plyio.xyz_of_line("1 2 z\n") is None
    assert plyio.xyz_of_line("1_0 +inf 2e3") == [10.0, float("inf"), 2000.0]
    assert plyio.xyz_of_line(" 1 2 3") == [1.0, 2.0, 3.0]   # Unicode whitespace splits as str.split does
