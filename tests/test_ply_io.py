"""The PLY text kernels (csrc/textio.cu via gauspcc_b200/plyio.py) against the Python they replace: the row formatter byte for
byte against Python's float repr, the parser row for row against float() / cli.read_points, the file tools end to end."""
import csv
import ctypes as C
import os
import random

import numpy as np
import pytest
import torch

from gauspcc_b200 import _lib, cli, pcc_utils, plyio
from gauspcc_b200.synth import hac_like_cloud

pytestmark = pytest.mark.gpu


def _save_ply_ascii_geo(coords: np.ndarray, path: str) -> None:
    """The writer decompress_point_cloud used before rows were formatted on the GPU (kit/io.py:36-49)."""
    coords = coords.astype(np.float32)
    with open(path, 'w') as f:
        f.write('ply\nformat ascii 1.0\n')
        f.write(f'element vertex {coords.shape[0]}\n')
        f.write('property float x\nproperty float y\nproperty float z\nend_header\n')
        for p in coords:
            f.write(f'{p[0]} {p[1]} {p[2]}\n')


@pytest.fixture(scope="module")
def ckpt(tmp_path_factory):
    from gauspcc_b200.weights import save_synthetic_checkpoint
    return save_synthetic_checkpoint(str(tmp_path_factory.mktemp("w") / "GausPcgc" / "best_model_ue_4stage_conv.pt"))


def _rows_text(v: np.ndarray) -> bytes:
    rows = v.astype(np.float32).reshape(-1, 3)
    return "".join(f"{p[0]} {p[1]} {p[2]}\n" for p in rows).encode()


def _format(v: np.ndarray) -> bytes:
    t = torch.from_numpy(np.ascontiguousarray(v.astype(np.float32).reshape(-1, 3))).cuda()
    return plyio.format_rows(t).cpu().numpy().tobytes()


def _pad3(v):
    v = np.asarray(v, dtype=np.float32).ravel()
    return np.concatenate([v, np.zeros((-len(v)) % 3, np.float32)])


def _special_values() -> np.ndarray:
    parts = [np.array([2.0 ** k for k in range(-149, 128)], np.float32)]               # every power of two
    sub = [1, 2, 3, 5, 7, 0x155555, 0x2AAAAA, 0x3FFFFF, 0x400000, 0x400001, 0x7FFFFE, 0x7FFFFF]
    sub += [(1 << k) - 1 for k in range(1, 24)] + [(1 << k) + 1 for k in range(1, 23)]
    parts.append(np.array(sub, np.uint32).view(np.float32))                               # subnormals of every bit length
    around = []
    for e in range(-6, 18):                                                               # +-1 ulp around every decade
        b = int(np.float32(10.0 ** e).view(np.uint32))
        around += [b + d for d in (-2, -1, 0, 1, 2)]
    around += [int(np.float32(x).view(np.uint32)) + d for x in (1e-4, 1e16, 9.999e-5, 9.999999e15) for d in (-1, 0, 1)]
    parts.append(np.array(around, np.uint32).view(np.float32))
    parts.append(np.array([0.0, -0.0, np.inf, -np.inf, np.nan, -65.04, 1e-5, 1e17], np.float32))
    return np.concatenate(parts)


def test_formatter_special_classes():
    v = _pad3(np.concatenate([_special_values(), -_special_values()]))
    assert _format(v) == _rows_text(v)


def test_formatter_integers():
    v = _pad3(np.concatenate([np.arange(0, 1 << 24, 1, dtype=np.float32)[::3], [2.0 ** 24], -np.arange(0, 1 << 24, 7)]))
    assert _format(v) == _rows_text(v)


def test_formatter_random_bit_patterns():
    bits = np.random.default_rng(0).integers(0, 1 << 32, 4_200_000, dtype=np.uint64).astype(np.uint32)
    v = _pad3(bits.view(np.float32))
    got, want = _format(v), _rows_text(v)
    if got != want:
        g, w = got.split(b"\n"), want.split(b"\n")
        bad = next(i for i in range(len(w)) if g[i] != w[i])
        pytest.fail(f"row {bad}: GPU {g[bad]!r}, Python {w[bad]!r}")


def test_formatter_buffer_too_small():
    lib = _lib.load()
    pts = torch.full((10, 3), -65.04, dtype=torch.float32, device="cuda")
    text = plyio.format_rows(pts)
    n = text.numel()
    out = torch.empty(n, dtype=torch.uint8, device="cuda")
    ws_b = lib.gpc_ply_format_workspace_bytes(10)
    ws = torch.empty(ws_b, dtype=torch.uint8, device="cuda")
    length = C.c_uint64(0)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    args = (C.c_void_p(pts.data_ptr()), 10, C.c_void_p(out.data_ptr()))
    assert lib.gpc_ply_format_f32(*args, n - 1, C.byref(length), C.c_void_p(ws.data_ptr()), ws_b, st) == -1   # GPC_EINVAL
    assert length.value == n
    assert lib.gpc_ply_format_f32(*args, n, C.byref(length), C.c_void_p(ws.data_ptr()), ws_b, st) == 0
    assert out.cpu().numpy().tobytes() == text.cpu().numpy().tobytes()


# ---------------------------------------------------------------- parser

def _same(a: np.ndarray, b: np.ndarray) -> bool:
    return a.shape == b.shape and np.array_equal(np.ascontiguousarray(a).view(np.uint64), np.ascontiguousarray(b).view(np.uint64))


def _check_file(path) -> torch.Tensor:
    got = plyio.read_points_device(str(path))
    ref = cli.read_points(str(path))
    assert got.is_cuda and got.dtype == torch.float64
    g = got.cpu().numpy()
    assert _same(g, ref), (g.shape, ref.shape, np.nonzero(g.view(np.uint64) != ref.view(np.uint64)) if g.shape == ref.shape else None)
    return got


def test_parser_reads_formatter_output(tmp_path):
    """The round trip: the GPU writer's text read back by the GPU parser is the float32 input, exactly."""
    rng = np.random.default_rng(1)
    bits = rng.integers(0, 1 << 32, 600_000, dtype=np.uint64).astype(np.uint32).view(np.float32)
    v = _pad3(np.concatenate([bits[np.isfinite(bits)], _special_values()])).reshape(-1, 3)
    p = tmp_path / "r.ply"
    plyio.write_ply_ascii(torch.from_numpy(v).cuda(), str(p))
    got = _check_file(p).cpu().numpy()
    assert _same(got, v.astype(np.float64))


def _random_decimal(r: random.Random) -> str:
    nd = r.randint(1, 25)
    digs = "".join(r.choice("0123456789") for _ in range(nd))
    k = r.randint(0, nd)
    dot = "." if r.random() < 0.7 else ""
    return r.choice(["", "-", "+"]) + digs[:k] + dot + digs[k:] + r.choice(["e", "E"]) + str(r.randint(-330, 310))


def test_parser_random_decimals(tmp_path):
    r = random.Random(2)
    lines = [" ".join(_random_decimal(r) for _ in range(3)) for _ in range(200_000)]
    p = tmp_path / "d.txt"
    p.write_text("\n".join(lines) + "\n")
    got = _check_file(p)
    assert got.shape[0] > 190_000


EDGE_TOKENS = [
    "+1", ".5", "5.", "1E5", "1e+5", "-1e-5", "007", "000.000120", "-0", "+0.0e0", "0e999999999", "1e-999999999", "1e999999999",
    "9007199254740993", "9007199254740992.5", "9007199254740993.000000000000000000001", "1.00000000000000011102230246251565404236316680908203125",
    "2.4703282292062327e-324", "2.4703282292062328e-324", "4.9406564584124654e-324", "2.2250738585072011e-308",
    "2.2250738585072012e-308", "2.225073858507201136057409796709131975934819546351645648e-308", "1.7976931348623157e308",
    "1.7976931348623158e308", "1.7976931348623159e308", "1.797693134862315807937289714053034150799e308", "1e5000", "-1e-5000",
    "123456789012345678901234567890", "0.000000000000000000000000000000000001", "1" + "0" * 40, "9" * 40 + "e-350",
    "3.4028235677973366e38", "1.401298464324817e-45", "7.006492321624085e-46",
]
BAD_TOKENS = ["abc", "1e", "e5", ".", "+", "-.e1", "0x10", "1.5.3", "--1", "1e5.5", "inf5", "nana", "1,5", "1d5"]


def test_parser_forms_and_edges(tmp_path):
    toks = EDGE_TOKENS + [t.upper() for t in EDGE_TOKENS]
    lines = [f"{a} {b} {c}" for a, b, c in zip(toks, toks[1:] + toks[:1], toks[2:] + toks[:2])]
    lines += [f"1 2 {b}" for b in BAD_TOKENS] + [f"{b} 1 2" for b in BAD_TOKENS]
    p = tmp_path / "e.txt"
    p.write_text("\n".join(lines) + "\n")
    got = _check_file(p)
    assert got.shape[0] == len(toks)


def test_parser_layout(tmp_path):
    cases = {
        "header": b"ply\nformat ascii 1.0\nelement vertex 2\nproperty float x\nproperty float y\nproperty float z\nend_header\n1 2 3\n4 5 6\n",
        "short_and_extra": b"1 2\n1\n\n1 2 3 4 5\n  7\t8 9   extra words\n\t\n1 2 3",
        "crlf": b"1 2 3\r\n4 5 6\r\n\r\n7 8 9\r\n",
        "lone_cr": b"1 2 3\r4 5 6\r\r7 8 9",
        "mixed": b"1 2 3\r\n4 5 6\r7 8 9\n\r\n10 11 12",
        "no_trailing_newline": b"1.5 -2.5 3e2",
        "blank_lines": b"\n\n\n1 2 3\n\n\n",
        "empty": b"",
        "only_newlines": b"\r\n\n\r",
        "tabs": b"1\t2\t3\n\t1\t\t2 \t3\t\n",
    }
    for name, text in cases.items():
        p = tmp_path / f"{name}.ply"
        p.write_bytes(text)
        _check_file(p)


def test_parser_host_fallback(tmp_path, monkeypatch):
    """Lines the GPU must not decide go to the host, and only those."""
    host_lines = [b"nan 1 2", b"-Infinity 1 2", b"1_0 2 3", b"1 2 \xc3\xa9", b"\xc2\xa01 2 3", b"1\x0b2 3", b"1 2 3\x0c",
                  b"1 2\x1c3", b"INF -inf +nan", b"1 2 1_000.5e-1_0", b"\xff\xfe1 2 3"]
    gpu_lines = [b"1 2 3", b"4 5 6 7", b"x y z", b"1e400 -1e-400 0"]
    order = [gpu_lines[0], host_lines[0], host_lines[1], gpu_lines[1], host_lines[2], host_lines[3], gpu_lines[2], host_lines[4],
             host_lines[5], host_lines[6], gpu_lines[3], host_lines[7], host_lines[8], host_lines[9], host_lines[10], gpu_lines[0]]
    text = b"\r\n".join(order) + b"\n"
    seen = []
    real = plyio.host_rows

    def spy(t, spans):
        seen.extend(t[b:e] for b, e, _ in np.asarray(spans, dtype=np.int64).reshape(-1, 3))
        return real(t, spans)

    monkeypatch.setattr(plyio, "host_rows", spy)
    p = tmp_path / "h.ply"
    p.write_bytes(text)
    _check_file(p)
    assert seen == [l for l in order if l in host_lines]
    # a file the GPU decides alone never calls the host
    seen.clear()
    p.write_bytes(b"\n".join(gpu_lines))
    _check_file(p)
    assert seen == []


def test_parser_refuses_4gib():
    with pytest.raises(ValueError):
        plyio.parse_text(np.lib.stride_tricks.as_strided(np.zeros(1, np.uint8), shape=(1 << 32,), strides=(0,)))


# ---------------------------------------------------------------- end to end

@pytest.mark.parametrize("pre_quantized", [True, False])
@pytest.mark.parametrize("sorted_output", [False, True])
def test_decompress_writes_the_python_writers_bytes(tmp_path, ckpt, pre_quantized, sorted_output):
    xyz = hac_like_cloud(30000, seed=7, extent_log2=14)
    b = str(tmp_path / "s.bin")
    pcc_utils.compress_point_cloud(xyz, ckpt, b)
    out = str(tmp_path / "s.ply")
    r = pcc_utils.decompress_point_cloud(b, ckpt, out, is_data_pre_quantized=pre_quantized, sorted_output=sorted_output)
    ref = str(tmp_path / "ref.ply")
    _save_ply_ascii_geo(r["point_cloud"].cpu().numpy(), ref)
    assert open(out, "rb").read() == open(ref, "rb").read()


def test_batch_decompress_writes_the_single_calls_files(tmp_path, ckpt):
    bins = []
    for i, (n, e) in enumerate([(20000, 14), (900, 10), (40000, 15)]):
        bins.append(str(tmp_path / f"{i}.bin"))
        pcc_utils.compress_point_cloud(hac_like_cloud(n, seed=20 + i, extent_log2=e), ckpt, bins[-1])
    outs = [str(tmp_path / "batch" / f"{i}.ply") for i in range(3)]
    rs = pcc_utils.decompress_point_clouds(bins, ckpt, is_data_pre_quantized=False, output_paths=outs)
    for b, o, r in zip(bins, outs, rs):
        single = str(tmp_path / "single" / (os.path.basename(b) + ".ply"))
        pcc_utils.decompress_point_cloud(b, ckpt, single, is_data_pre_quantized=False)
        assert r["output_path"] == o
        assert open(o, "rb").read() == open(single, "rb").read()
    with pytest.raises(ValueError):
        pcc_utils.decompress_point_clouds(bins, ckpt, output_paths=outs[:2])


def test_cli_batch_matches_per_file(tmp_path, ckpt):
    src = tmp_path / "in"
    (src / "sub").mkdir(parents=True)
    scale = lambda c: ((c * 16 - 131072) * 0.001)
    clouds = [hac_like_cloud(n, seed=40 + i, extent_log2=e) for i, (n, e) in enumerate([(3000, 11), (500, 9), (8000, 13), (2000, 12),
                                                                                      (6000, 12), (1000, 10)])]
    kitti = np.concatenate([scale(clouds[0]).astype(np.float32), np.ones((len(clouds[0]), 1), np.float32)], axis=1)
    kitti.tofile(src / "a.bin")
    np.save(src / "b.npy", scale(clouds[1]))
    _save_ply_ascii_geo(scale(clouds[2]), str(src / "c.ply"))
    with open(src / "sub" / "d.ply", "wb") as f:                    # CRLF, a header, a line left to the host
        f.write(b"ply\r\nformat ascii 1.0\r\n" + b"".join(f"{float(x)!r} {float(y)!r} {float(z)!r}\r\n".encode() for x, y, z in scale(clouds[3]))
                + b"-0.5\xc2\xa01 2\r\n")
    np.save(src / "e.npy", scale(clouds[4]).astype(np.float32))
    _save_ply_ascii_geo(scale(clouds[5]), str(src / "sub" / "f.ply"))
    (src / "g.txt").write_text("1 2 3\n")                          # not a listed suffix: ignored, as before
    res = {}
    for batch in (1, 4):
        enc, dec, rep = tmp_path / f"enc{batch}", tmp_path / f"dec{batch}", tmp_path / f"rep{batch}"
        common = ["--ckpt", ckpt, "--kernel_size", "5", "--resultdir", str(rep), "--batch", str(batch)]
        assert cli.main(["compress", "--input_glob", str(src), "--output_folder", str(enc)] + common) == 0
        assert cli.main(["decompress", "--input_glob", str(enc), "--output_folder", str(dec)] + common) == 0
        files = {os.path.relpath(os.path.join(d, f), tmp_path / f"{kind}{batch}"): open(os.path.join(d, f), "rb").read()
                 for kind in ("enc", "dec") for d, _, fs in os.walk(tmp_path / f"{kind}{batch}") for f in fs}
        res[batch] = files
        for name in ("ue_4stage_conv_data6.csv", "ue_4stage_conv_dec_data6.csv"):
            rows = list(csv.DictReader(open(rep / name)))
            assert [r["filedir"] for r in rows][-1] == "avg" and len(rows) == 7
    assert sorted(res[1]) == sorted(res[4]) and len(res[1]) == 12
    for k in res[1]:
        assert res[1][k] == res[4][k], k


def test_quantise_device_matches_host():
    rng = np.random.default_rng(3)
    xyz = np.concatenate([rng.uniform(-300, 300, (100_000, 3)), np.round(rng.uniform(-300, 300, (1000, 3)), 3)])
    for posQ in (1, 16):
        for pre in (False, True):
            v = np.round(xyz * 100) if pre else xyz
            assert torch.equal(cli.quantise_device(torch.from_numpy(v).cuda(), posQ, pre).cpu(), cli.quantise(v, posQ, pre))
