"""Device-side driver of the GausPcgc geometry codec: the level loop of
compress_point_cloud / decompress_point_cloud (reference: src/gs_compress/HAC/utils/pcc_utils.py:73-203
and :271-381) over the C-ABI kernels of libgpcgc.so.

PyTorch is used for device memory, streams and events only; every arithmetic step is a call into
the hand-written sm_100a library.  There is no CPU fallback: construction raises without CUDA.

HBM layout of one octree level (rows in ascending key order == the reference's (z,y,x) order):
    keys  int64[n]      packed voxel key (see include/gpcgc.h)
    occ   uint8[n]      occupancy byte (children present)
    feats float32[n,32] 128 B rows
    kmap  per-tile pair lists grouped by conv offset (seg / pair_nbr / pair_row)
"""
from __future__ import annotations

import contextlib
import ctypes as C
import os
import queue
import time
from concurrent.futures import ThreadPoolExecutor
from dataclasses import dataclass
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch

from . import _lib
from . import weights as W

STAGE_SHIFT = (7, 6, 4, 0)       # sym_i = (occ >> shift) & mask   (pcc_utils.py:112-115)
STAGE_MASK = (1, 1, 3, 15)
CTX_SHIFT = (None, 7, 6, 4)      # ctx_i = occ >> shift            (pcc_utils.py:122,129,137)
BASE_ROWS = 64                   # FOG loop stops when a level has < 64 rows (pcc_utils.py:87)
UM_TILE_ROWS = 512               # output rows per CTA of the tcgen05 conv: the one tile height spconv_um.cu builds (DESIGN.md 5)


def _ptr(t: Optional[torch.Tensor]):
    """device address as a plain int (None = NULL): ctypes converts it for the c_void_p argtypes without an intermediate object"""
    return None if t is None else t.data_ptr()


COORD_LIMIT = (1 << 20) - 16           # |voxel coordinate| the 21-bit key fields hold with room for the 5^3 neighbourhood


@dataclass
class KMap:
    """Kernel map of one coordinate set (built once, shared by every conv on the set), in the form its conv kernel consumes."""
    seg: torch.Tensor                         # first stream entry of every (tile, offset) segment
    pairs: Optional[torch.Tensor]             # mma.sync / sparse conv: combined stream nbr | row << 32 | k << 48
    n_pairs: int                              # stream entries (padded)
    tile_rows: int
    n_real: int = 0                           # true (row, neighbour) pairs
    v6_variant: int = 42                      # mma.sync conv: 42 one warp per tile, 46 / 47 offsets split over 8 / 16 warps, 48 = v6d
    um_rows: int = 0                          # > 0: tcgen05 conv (spconv_um.cu) with tiles of um_rows output rows; activations are split rows
    pair_nbr: Optional[torch.Tensor] = None   # um: input row of every stream entry (0xFFFFFFFF = padding)
    pair_off: Optional[torch.Tensor] = None   # um: byte offset of every entry's accumulator row
    sparse: bool = False                      # sparse big level: centre product + offset-sorted stragglers (spconv_sparse.cu)
    rowptr: Optional[torch.Tensor] = None     # sparse: first contribution of every row
    contrib: Optional[torch.Tensor] = None    # sparse: scratch [stragglers, 32] fp32, rewritten by every conv on the level
    tile_order: Optional[torch.Tensor] = None # um: the level's tiles, heaviest (most stream entries) first


@dataclass
class Level:
    keys: torch.Tensor
    occ: Optional[torch.Tensor]
    n: int
    kmap: Optional[KMap] = None


class DeviceWeights:
    """state_dict (reference key layout, gauspcc_b200/weights.py) resident in HBM."""

    def __init__(self, sd: Dict[str, torch.Tensor], device: torch.device, channels: int = 32, kernel_size: int = 5):
        if channels != 32 or kernel_size not in (3, 5):
            raise NotImplementedError("libgpcgc is built for channels=32 and kernel_size 5 (HAC call sites) or 3 (the reference CLI default)")
        W.validate_state_dict(sd, channels, kernel_size)
        self.kernel_size = kernel_size
        f = lambda k: sd[k].detach().to(device=device, dtype=torch.float32).contiguous()
        self.prior_emb = f("prior_embedding.weight")
        self.target_emb = f("target_embedding.target_res_embedding.weight")
        self.convs = torch.stack([f(k) for k in W.CONV_KEYS]).contiguous()           # [18,K^3,32,32]
        if kernel_size == 3:       # the 27 matrices at their K = 5 offset indices ((dz+2)*5 + (dy+2))*5 + (dx+2); the kernel map drops the rest
            k5 = [((dz + 2) * 5 + (dy + 2)) * 5 + (dx + 2) for dz in (-1, 0, 1) for dy in (-1, 0, 1) for dx in (-1, 0, 1)]
            full = torch.zeros((len(W.CONV_KEYS), 125, 32, 32), dtype=torch.float32, device=device)
            full[:, torch.tensor(k5, device=device)] = self.convs
            self.convs = full.contiguous()
        lib = _lib.load()
        st = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
        self.convs_frag = torch.empty_like(self.convs)       # [18,125,2,2,2,32] uint4: mma.sync A fragments of W^T (bf16 hi / lo)
        _lib.check(lib.gpc_spconv_pack_weights_frag(_ptr(self.convs), len(W.CONV_KEYS), _ptr(self.convs_frag), st), "gpc_spconv_pack_weights_frag")
        self.convs_um = torch.empty_like(self.convs)         # [18,125,8,32,16 B]: tcgen05 A operand (W^T bf16 hi | lo), one TMEM lane per channel
        _lib.check(lib.gpc_spconv_pack_weights_um(_ptr(self.convs), len(W.CONV_KEYS), _ptr(self.convs_um), st), "gpc_spconv_pack_weights_um")
        self.stage_emb = [None] + [f(f"pred_head_s{i}_emb.weight") for i in (1, 2, 3)]
        self.head = [tuple(f(f"pred_head_s{i}.{j}.{p}") for j, p in ((0, "weight"), (0, "bias"), (2, "weight"), (2, "bias")))
                     for i in range(4)]


class GausPcgcCodec:
    def __init__(self, weights: DeviceWeights, device: Optional[torch.device] = None, tile_rows: Optional[int] = None,
                 ac_threads: Optional[int] = None):
        if not torch.cuda.is_available():
            raise _lib.GpcError("GausPcgcCodec needs a CUDA device; there is no CPU fallback")
        self.lib = _lib.load()
        self.dev = torch.device(device if device is not None else "cuda")
        self.w = weights
        # Which conv kernel a level runs is a function of the LEVEL ONLY (rows, pairs per row): encoder and decoder must take the
        # same decision, because each kernel has its own fp32 summation order and the range coder needs bit-identical CDFs on both
        # sides.  The thresholds are therefore constants of the bitstream format, not tunables; tools/ and tests/ may override the
        # attributes on a codec object they use for BOTH directions (A/B timing, kernel-family parity).
        #   rows >= UM_MIN_ROWS and >= SPARSE_MAX_DENSITY pairs per row: tcgen05 conv (spconv_um.cu), split-row activations
        #   rows >= SPARSE_MIN_ROWS and  < SPARSE_MAX_DENSITY pairs per row: centre product + sorted stragglers (spconv_sparse.cu)
        #   otherwise: the mma.sync conv, tile shape by level size (_v6_config)
        self.um_min_rows = 150_000
        self.sparse_max_density = 4.5
        self.sparse_min_rows = 150_000
        self.adaptive_tiles = tile_rows is None       # tests: a fixed tile height / kernel variant of the mma.sync conv on every level
        self.tile_rows = int(tile_rows or 64)
        self.v6_variant = 42
        self._fns: Dict[str, object] = {}
        self._stream_h = None
        n_thr = ac_threads or int(os.environ.get("GPC_AC_THREADS", min(16, len(os.sched_getaffinity(0)))))
        self.pool = ThreadPoolExecutor(max_workers=max(1, n_thr))
        self._pinned: Optional[torch.Tensor] = None
        self._pinned_dec: Optional[torch.Tensor] = None
        # decoder wavefront (stages of a level overlap chunk by chunk): levels with >= wave_min_rows rows, chunks of wave_chunk_rows
        # rows (a multiple of 8192 = the sparse conv's row blocks and of the v6d tile heights)
        # (how the decoder ORDERS its work -- wavefront or stage by stage -- does not change a single bit of any CDF: the row-range
        # launches compute the same sums; tests/test_gpu_parity.py::test_decoder_wavefront)
        self.wave_decode = True
        self.wave_min_rows = 150_000
        self.wave_chunk_rows = 32768
        self._wave_side: Optional[list] = None
        self._wave_buf: Optional[torch.Tensor] = None
        self._enc_side = None                         # encoder: levels run on the main stream and this one (encode())
        self._dec_side = None                         # decoder: children + their kernel map beside the prior stack (level_features())
        self._coder_arena = None                      # (c_low, c_high) words of all streams of a scene (container version 2)
        self.wave_log: Optional[list] = None          # tools/wave_times.py: per-level record of the wavefront
        self.debug_dec_cdfs: Optional[dict] = None    # tests: (level, stage) -> CDF rows the stage-by-stage decoder computed
        self._launch_base = 0
        self.last_stats: Dict[str, float] = {}
        self._segments: List[Tuple[torch.cuda.Event, torch.cuda.Event]] = []
        self._seg_open: Optional[torch.cuda.Event] = None
        self.conv_profile: Optional[list] = None       # bench.py: [(ev0, ev1, algorithmic bytes, flops, launches)] per group of convs
        self._prof_group = None
        self._prof_single = None

    # ------------------------------------------------------------------ plumbing
    def _stream(self):
        """raw handle of torch's current stream; inside encode() / decode() it is looked up once (the host issues ~1 500 launches per
        step and must stay ahead of the GPU on the coarse levels, where a kernel is shorter than a careless Python call)"""
        if self._stream_h is not None:
            return self._stream_h
        return torch.cuda.current_stream(self.dev).cuda_stream

    def _empty(self, shape, dtype):
        return torch.empty(shape, dtype=dtype, device=self.dev)

    def _ws(self, nbytes: int):
        return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=self.dev)

    def _pin(self, nbytes: int) -> torch.Tensor:
        if self._pinned is None or self._pinned.numel() < nbytes:
            self._pinned = torch.empty(int(nbytes * 1.25) + 4096, dtype=torch.uint8, pin_memory=True)
        return self._pinned

    def _seg_begin(self):
        ev = torch.cuda.Event(enable_timing=True)
        ev.record(torch.cuda.current_stream(self.dev))
        self._seg_open = ev

    def _seg_end(self):
        ev = torch.cuda.Event(enable_timing=True)
        ev.record(torch.cuda.current_stream(self.dev))
        self._segments.append((self._seg_open, ev))
        self._seg_open = None

    def _seg_total_ms(self) -> float:
        torch.cuda.synchronize(self.dev)
        ms = sum(a.elapsed_time(b) for a, b in self._segments)
        self._segments = []
        return ms

    def _profile_events(self):
        """timing events come from a pool that is created once: cudaEventCreate inside the timed region is not free"""
        if not hasattr(self, "_ev_pool"):
            self._ev_pool, self._ev_next = [], 0
        if self._ev_next + 2 > len(self._ev_pool):
            self._ev_pool += [torch.cuda.Event(enable_timing=True) for _ in range(4096)]
        e0, e1 = self._ev_pool[self._ev_next], self._ev_pool[self._ev_next + 1]
        self._ev_next += 2
        return e0, e1

    def prewarm_profile_events(self, n_events: int):
        """bench.py: torch creates a CUDA event lazily at its first record(); do that for every event the timed region will use
        BEFORE the timed region (each creation is tens of microseconds of host time between two launches)."""
        if not hasattr(self, "_ev_pool"):
            self._ev_pool, self._ev_next = [], 0
        while len(self._ev_pool) < n_events:
            self._ev_pool.append(torch.cuda.Event(enable_timing=True))
        st = torch.cuda.current_stream(self.dev)
        for e in self._ev_pool[:n_events]:
            e.record(st)
        torch.cuda.synchronize(self.dev)
        self._ev_next = 0

    def _popcount(self, occ: torch.Tensor) -> int:
        """number of children of a level = set bits of its occupancy bytes, counted on the device (8 B back instead of the level)"""
        if not hasattr(self, "_pop8"):
            self._pop8 = torch.tensor([bin(i).count("1") for i in range(256)], dtype=torch.int32, device=self.dev)
        return int(self._pop8[occ.long()].sum().item()) if occ.numel() else 0

    def _call(self, name, *args):
        fn = self._fns.get(name)
        if fn is None:
            fn = self._fns[name] = getattr(self.lib, name)
        rc = fn(*args)
        if rc:
            _lib.check(rc, name)

    @property
    def launches(self) -> int:
        """kernels launched by libgpcgc since the current encode()/decode() call started"""
        return int(self.lib.gpc_launch_count()) - self._launch_base

    # ------------------------------------------------------------------ keys / pyramid
    def pack_keys(self, xyz: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """[n,3] float32/int32 CUDA -> (keys int64[n], meta int32[8] = status, pad, min xyz, max xyz)."""
        n = xyz.shape[0]
        keys = self._empty((n,), torch.int64)
        meta = torch.zeros(8, dtype=torch.int32, device=self.dev)
        if xyz.dtype == torch.float32:
            self._call("gpc_pack_keys_f32", _ptr(xyz), n, _ptr(keys), _ptr(meta), self._stream())
        elif xyz.dtype == torch.int32:
            self._call("gpc_pack_keys_i32", _ptr(xyz), n, _ptr(keys), _ptr(meta), self._stream())
        else:
            raise TypeError(f"xyz must be float32 or int32, got {xyz.dtype}")
        self._call("gpc_key_minmax", _ptr(keys), n, C.c_void_p(meta.data_ptr() + 8), self._stream())
        return keys, meta

    def _xform(self, mm: np.ndarray) -> _lib.KeyXform:
        xf = _lib.KeyXform()
        arr = np.ascontiguousarray(mm, dtype=np.uint32)
        _lib.check(self.lib.gpc_make_xform_h(arr.ctypes.data_as(C.c_void_p), C.byref(xf)), "gpc_make_xform_h")
        return xf

    def sort_unique(self, keys: torch.Tensor, mm: np.ndarray) -> torch.Tensor:
        n = keys.shape[0]
        xf = self._xform(mm)
        skeys = self._empty((n,), torch.int64)
        svals = self._empty((n,), torch.int32)
        ws_b = self.lib.gpc_sort_workspace_bytes(n)
        ws = self._ws(ws_b)
        self._call("gpc_sort_pairs", _ptr(keys), _ptr(None), _ptr(skeys), _ptr(svals), n, xf, _ptr(ws), ws_b, self._stream())
        out = self._empty((n,), torch.int64)
        cnt = torch.zeros(1, dtype=torch.int32, device=self.dev)
        ws_b = self.lib.gpc_pyramid_workspace_bytes(n)
        ws = self._ws(ws_b)
        self._call("gpc_unique_sorted", _ptr(skeys), n, _ptr(out), _ptr(cnt), _ptr(ws), ws_b, self._stream())
        m = int(cnt.item())
        return out[:m]

    def build_pyramid(self, leaf_keys: torch.Tensor, mm: np.ndarray) -> List[Level]:
        """FOG loop (pcc_utils.py:83-89): returns levels coarsest -> finest (finest = parents of the points)."""
        levels: List[Level] = []
        cur = leaf_keys
        mm = mm.astype(np.int64).copy()
        while True:
            n = cur.shape[0]
            mm = (mm >> 1) + (1 << 19)                       # parent field = (f >> 1) + 2^19
            xf = self._xform(mm)
            pk = self._empty((max(n, 1),), torch.int64)
            po = self._empty((max(n, 1),), torch.uint8)
            cnt = torch.zeros(1, dtype=torch.int32, device=self.dev)
            ws_b = self.lib.gpc_pyramid_workspace_bytes(n)
            ws = self._ws(ws_b)
            self._call("gpc_pyramid_down", _ptr(cur), n, xf, _ptr(pk), _ptr(po), _ptr(cnt), _ptr(ws), ws_b, self._stream())
            m = int(cnt.item())
            levels.append(Level(pk[:m], po[:m], m))
            cur = pk[:m]
            if m < BASE_ROWS:
                break
        return levels[::-1]

    def expand(self, lvl: Level, n_child: int) -> Tuple[torch.Tensor, torch.Tensor]:
        ck = self._empty((n_child,), torch.int64)
        cp = self._empty((n_child,), torch.int32)
        ws_b = self.lib.gpc_expand_workspace_bytes(lvl.n)
        ws = self._ws(ws_b)
        self._call("gpc_expand_children", _ptr(lvl.keys), _ptr(lvl.occ), lvl.n, n_child, _ptr(ck), _ptr(cp), _ptr(ws), ws_b,
                   self._stream())
        return ck, cp

    # ------------------------------------------------------------------ kernel map / conv
    def _v6_config(self, n: int) -> Tuple[int, int]:
        """(rows per CTA, kernel variant) of the mma.sync conv for a level of n rows:
        128 / 64 rows per warp on big levels (W^T reuse, v6d); fewer rows on the coarse levels so that they still fill the 148 SMs;
        on the coarse levels the 125 offsets of a tile are additionally split over 8 / 16 warps (variants 46 / 47): those
        launches are bound by one warp's chain of dependent 8-pair tiles, ~63 us each before, 15-30 us now."""
        if not self.adaptive_tiles:
            return self.tile_rows, self.v6_variant
        if n >= 150_000:
            return 128, 48          # v6d: rows straight into the MMA fragments, 128-row tiles halve the W^T traffic per pair
        if n >= 40_000:
            return 64, 48
        if n >= 20_000:
            return 32, 46
        if n >= 1_500:
            return 16, 46
        return 8, 47

    def _recentre(self, xyz: torch.Tensor):
        """xyz - shift with shift a per-axis multiple of 2^(bits of the extent + 1) (>= 2^levels: floor(c / 2^l) commutes with it on
        every level) that centres the scene on the origin; ValueError if the extent itself exceeds the key fields."""
        lo = xyz.amin(0).to(torch.int64).cpu().numpy()
        hi = xyz.amax(0).to(torch.int64).cpu().numpy()
        G = 1 << (int((hi - lo).max()).bit_length() + 1)
        shift = ((lo + hi) // 2 + G // 2) // G * G
        if max(int(np.abs(hi - shift).max()), int(np.abs(lo - shift).max())) > COORD_LIMIT:
            raise ValueError(f"voxel coordinates must lie within +-{COORD_LIMIT}, or span less than ~{COORD_LIMIT * 2 // 5} voxels anywhere")
        return xyz - torch.tensor(shift, dtype=xyz.dtype, device=xyz.device), shift

    def _count_pairs(self, dense: torch.Tensor, n: int, tr: int, pad: int):
        """first pass over the dense map: seg (exclusive scan of the padded per-(tile, offset) counts), entries, true pairs"""
        tiles = (n + tr - 1) // tr
        seg = self._empty((tiles * 126 + 1,), torch.int32)
        cnt = torch.zeros(2, dtype=torch.int32, device=self.dev)
        ws_b = self.lib.gpc_kmap_pairs_workspace_bytes(n, tr)
        ws = self._ws(ws_b)
        self._call("gpc_kmap_pairs_count", _ptr(dense), n, tr, pad, _ptr(seg), _ptr(cnt), _ptr(ws), ws_b, self._stream())
        n_pairs, n_real = (int(v) for v in cnt.tolist())
        return seg, n_pairs, n_real

    def _v6_map(self, dense: torch.Tensor, n: int, tr: int, v6v: int, counted=None) -> KMap:
        seg, n_pairs, n_real = counted if counted is not None else self._count_pairs(dense, n, tr, 8)
        pairs = self._empty((max(n_pairs, 1),), torch.int64)
        self._call("gpc_kmap_pairs_fill", _ptr(dense), n, tr, _ptr(seg), None, None, _ptr(pairs), n_pairs, self._stream())
        return KMap(seg, pairs, n_pairs, tr, n_real=n_real, v6_variant=v6v)

    def _count_um(self, dense: torch.Tensor, n: int, tr: int):
        """the tcgen05 conv's tiling of the level: seg, stream entries (padded to 16 per (tile, offset)), true pairs"""
        tiles = (n + tr - 1) // tr
        seg = self._empty((tiles * 126 + 1,), torch.int32)
        tot = torch.zeros(2, dtype=torch.int64, device=self.dev)
        ws_b = self.lib.gpc_kmap_um_workspace_bytes(n, tr)
        ws = self._ws(ws_b)
        self._call("gpc_kmap_um_count", _ptr(dense), n, tr, _ptr(seg), _ptr(tot), _ptr(ws), ws_b, self._stream())
        n_pairs, n_real = (int(v) for v in tot.tolist())
        return seg, n_pairs, n_real

    def _um_map(self, dense: torch.Tensor, n: int, tr: int, counted=None) -> KMap:
        """pair stream of the tcgen05 conv: tiles of tr rows, segments padded to 16 entries, input rows + accumulator-row offsets"""
        seg, n_pairs, n_real = counted if counted is not None else self._count_um(dense, n, tr)
        nbr = self._empty((max(n_pairs, 1),), torch.int32)
        off = self._empty((max(n_pairs, 1),), torch.int32)
        self._call("gpc_kmap_um_fill", _ptr(dense), n, tr, _ptr(seg), _ptr(nbr), _ptr(off), self._stream())
        km = KMap(seg, None, n_pairs, tr, n_real=n_real, um_rows=tr, pair_nbr=nbr, pair_off=off)
        # CTAs take the level's tiles heaviest first (shorter tail)
        starts = seg[::126].to(torch.int64)                      # first stream entry of every tile (+ the end of the last)
        km.tile_order = torch.argsort(starts[1:] - starts[:-1], descending=True, stable=True).to(torch.int32)
        return km

    def _sparse_map(self, dense: torch.Tensor, n: int) -> KMap:
        m = int(self.lib.gpc_kmap_sparse_segments(n))
        seg = self._empty((m + 1,), torch.int32)
        rowptr = self._empty((n + 1,), torch.int32)
        tot = torch.zeros(2, dtype=torch.int32, device=self.dev)
        ws_b = self.lib.gpc_kmap_sparse_workspace_bytes(n)
        ws = self._ws(ws_b)
        self._call("gpc_kmap_sparse_count", _ptr(dense), n, _ptr(seg), _ptr(rowptr), _ptr(tot), _ptr(ws), ws_b, self._stream())
        n_entries, n_strag = (int(v) for v in tot.tolist())
        pairs = self._empty((max(n_entries, 1),), torch.int64)
        self._call("gpc_kmap_sparse_fill", _ptr(dense), n, _ptr(seg), _ptr(rowptr), _ptr(ws), _ptr(pairs), n_entries, self._stream())
        km = KMap(seg, pairs, n_entries, 0, n_real=n + n_strag, sparse=True, rowptr=rowptr)
        km.contrib = self._empty((max(n_strag, 1), 32), torch.float32)
        return km

    @staticmethod
    def _kmap_bytes(n: int) -> int:
        """SURVEY.md 8(d): hash build n*12 + cap*12 (cap = 2n), probes n*K^3*8; the pair stream adds pairs*12 (not known here)"""
        return n * 12 + 2 * n * 12 + n * 125 * 8

    def dense_map(self, keys: torch.Tensor, count_tile: int = 0):
        """hash table of the level + the offset-major [125][n] map of input rows (-1 = absent); with count_tile also the number of
        present neighbours per (tile of count_tile rows, offset), counted from the probes: returns (map, cell_counts)"""
        n = keys.shape[0]
        cap = self.lib.gpc_hash_capacity(n)
        table = self._ws(cap * 16)
        self._call("gpc_hash_build", _ptr(keys), n, _ptr(table), cap, self._stream())
        dense = self._empty((125, n), torch.int32)
        cells = self._empty((((n + count_tile - 1) // count_tile) * 126,), torch.int32) if count_tile else None
        self._call("gpc_kmap_dense", _ptr(table), cap, _ptr(keys), n, _ptr(dense), self.w.kernel_size, count_tile, _ptr(cells),
                   self._stream())
        return (dense, cells) if count_tile else dense

    def _scan_um(self, cells: torch.Tensor, n: int, tr: int):
        """_count_um from the cell counts the dense-map kernel produced"""
        seg = self._empty((((n + tr - 1) // tr) * 126 + 1,), torch.int32)
        tot = torch.zeros(2, dtype=torch.int64, device=self.dev)
        ws_b = self.lib.gpc_kmap_um_workspace_bytes(n, tr)
        ws = self._ws(ws_b)
        self._call("gpc_kmap_um_scan", _ptr(cells), n, tr, _ptr(seg), _ptr(tot), _ptr(ws), ws_b, self._stream())
        n_pairs, n_real = (int(v) for v in tot.tolist())
        return seg, n_pairs, n_real

    def build_kmap(self, keys: torch.Tensor, family: Optional[str] = None) -> KMap:
        """Kernel map of a coordinate set in the form of the conv kernel the level runs.  The family is a function of the level only
        (rows, pairs per row -- see __init__); `family` ("v6" | "um" | "sparse") forces one (tests / tools, both directions alike)."""
        n = keys.shape[0]
        big = n >= min(self.um_min_rows, self.sparse_min_rows)
        if family is None and not big:
            family = "v6"
        if family == "v6":
            tr, v6v = self._v6_config(n)
            return self._v6_map(self.dense_map(keys), n, tr, v6v)
        if family == "sparse":
            return self._sparse_map(self.dense_map(keys), n)
        # big level: the probes count the pairs per (tile of the tcgen05 conv, offset): density (pairs per row, centre included) and
        # the first pass of the pair stream in one
        tr = UM_TILE_ROWS
        dense, cells = self.dense_map(keys, tr)
        counted = self._scan_um(cells, n, tr)
        density = counted[2] / max(n, 1)
        if family is None:
            if n >= self.sparse_min_rows and 0 < self.sparse_max_density and density < self.sparse_max_density and n < 30_000_000:
                return self._sparse_map(dense, n)            # 32-bit straggler indices: n * 124 < 2^32
            if n < self.um_min_rows:
                tr6, v6v = self._v6_config(n)
                return self._v6_map(dense, n, tr6, v6v)
        return self._um_map(dense, n, tr, counted)

    def split_rows(self, x: torch.Tensor) -> torch.Tensor:
        """fp32 rows [n,32] -> split rows (int32 [n,32]: 16 words of bf16x2 hi | 16 words of bf16x2 lo)."""
        xs = self._empty(x.shape, torch.int32)
        self._call("gpc_rows_split", _ptr(x), x.shape[0], _ptr(xs), self._stream())
        return xs

    def conv(self, x: torch.Tensor, widx: int, km: KMap, residual: Optional[torch.Tensor] = None, relu: bool = False,
             out: Optional[torch.Tensor] = None, fmt: str = "f32", rows: Optional[Tuple[int, int]] = None):
        """One sparse conv.  Activations are fp32 rows (float32 tensors) or split rows (int32 tensors: the tcgen05 levels);
        fmt = "f32" | "split" | "both" selects what a tcgen05 level writes ("both" returns (f32, split)); out = the fp32 output
        buffer, or for fmt == "split" the split output buffer.
        rows = (r0, r1): only the output rows [r0, r1) are computed (whole tiles / blocks; decoder wavefront)."""
        n = x.shape[0]
        r0, r1 = rows if rows is not None else (0, 0)
        flags = 1 if relu else 0
        if km.um_rows:
            xs = x if x.dtype == torch.int32 else self.split_rows(x)
            y = ys = None
            if fmt in ("f32", "both"):
                y = out if (out is not None and fmt == "f32") else self._empty((n, 32), torch.float32)
            if fmt in ("split", "both"):
                ys = out if (out is not None and fmt == "split") else self._empty((n, 32), torch.int32)
            if residual is not None and residual.dtype == torch.int32:
                flags |= 2
            if rows is None:
                self._prof_conv_begin()
            self._call("gpc_spconv_fwd_um", _ptr(xs), _ptr(self.w.convs_um[widx]), _ptr(km.seg), _ptr(km.pair_nbr), _ptr(km.pair_off), n,
                       km.um_rows, _ptr(km.tile_order), _ptr(residual), flags, _ptr(y), _ptr(ys), r0, r1, self._stream())
            if rows is None:
                self._prof_conv_end(n, km)
            return y if fmt == "f32" else (ys if fmt == "split" else (y, ys))
        assert fmt == "f32" and x.dtype == torch.float32
        y = out if out is not None else self._empty((n, 32), torch.float32)
        if rows is not None:
            if km.sparse:
                self._call("gpc_spconv_sparse_fwd_rows", _ptr(x), _ptr(self.w.convs_frag[widx]), _ptr(km.seg), _ptr(km.pairs),
                           _ptr(km.rowptr), n, km.n_pairs, _ptr(km.contrib), _ptr(residual), flags, _ptr(y), r0, r1, self._stream())
            else:
                self._call("gpc_spconv_fwd_v6_rows", _ptr(x), _ptr(self.w.convs_frag[widx]), _ptr(km.seg), _ptr(km.pairs), n,
                           km.tile_rows, _ptr(residual), flags, _ptr(y), km.v6_variant, r0, r1, self._stream())
            return y
        self._prof_conv_begin()
        if km.sparse:
            self._call("gpc_spconv_sparse_fwd", _ptr(x), _ptr(self.w.convs_frag[widx]), _ptr(km.seg), _ptr(km.pairs), _ptr(km.rowptr), n,
                       km.n_pairs, _ptr(km.contrib), _ptr(residual), flags, _ptr(y), self._stream())
        else:
            self._call("gpc_spconv_fwd_v6", _ptr(x), _ptr(self.w.convs_frag[widx]), _ptr(km.seg), _ptr(km.pairs), n, km.tile_rows,
                       _ptr(residual), flags, _ptr(y), km.v6_variant, self._stream())
        self._prof_conv_end(n, km)
        return y

    # ---- bench.py's conv timing.  One CUDA-event pair per GROUP of convs on the same level (a 5-conv stack, a 2-conv stage):
    # an event pair around every conv launch (936 records per step) cost 10-50 ms per step and made the step time jitter
    # (tools/jitter.py: 134.6 +- 0.1 ms unprofiled against 146-185 ms with per-conv events).
    def _prof_open(self):
        if self.conv_profile is None or self._prof_group is not None:
            return None
        e0, e1 = self._profile_events()
        e0.record(torch.cuda.current_stream(self.dev))
        self._prof_group = [e0, e1, 0, 0, 0, "conv"]
        return self._prof_group

    def _prof_close(self, grp):
        if grp is None:
            return
        grp[1].record(torch.cuda.current_stream(self.dev))
        self.conv_profile.append(tuple(grp))
        self._prof_group = None

    def _stage(self, name: str, nbytes: int = 0):
        """bench.py's per-stage profile: one CUDA-event pair around a non-conv stage (algorithmic bytes per SURVEY.md 8(d))"""
        codec = self

        class _Ctx:
            def __enter__(self_):
                self_.g = None
                if codec.conv_profile is not None and codec._prof_group is None:
                    e0, e1 = codec._profile_events()
                    e0.record(torch.cuda.current_stream(codec.dev))
                    self_.g = (e0, e1)
                return self_

            def __exit__(self_, *a):
                if self_.g is not None:
                    self_.g[1].record(torch.cuda.current_stream(codec.dev))
                    codec.conv_profile.append((self_.g[0], self_.g[1], int(nbytes), 0, 0, name))
                return False
        return _Ctx()

    def _prof_conv_begin(self):
        self._prof_single = self._prof_open()          # None inside a group (or when not profiling)

    def _prof_conv_end(self, n: int, km: KMap):
        g = self._prof_group
        if g is not None:
            # SURVEY.md 8(d): per layer n*C*4*2 + pairs*8 + K^3*C^2*4 bytes and 2*pairs*C^2 FLOP
            g[2] += n * 32 * 4 * 2 + km.n_real * 8 + 125 * 32 * 32 * 4
            g[3] += 2 * km.n_real * 32 * 32
            g[4] += 1
            g[5] = "conv_um" if km.um_rows else ("conv_sparse" if km.sparse else "conv_v6")
        self._prof_close(self._prof_single)
        self._prof_single = None

    def res_stack(self, x: torch.Tensor, ids, km: KMap, final: str = "f32"):
        """Conv3d, ReLU, ResNet, ResNet (network_ue_4stage_conv.py:17-22; ResNet kit/nn.py:18-22)."""
        grp = self._prof_open()
        try:
            return self._res_stack(x, ids, km, final)
        finally:
            self._prof_close(grp)

    def _res_stack(self, x: torch.Tensor, ids, km: KMap, final: str):
        if km.um_rows:             # tcgen05 level: everything between the first and the last conv stays in split rows
            x = self.conv(x, ids[0], km, relu=True, fmt="split")
            t = self.conv(x, ids[1], km, relu=True, fmt="split")
            x = self.conv(t, ids[2], km, residual=x, relu=True, fmt="split")
            t = self.conv(x, ids[3], km, relu=True, fmt="split")
            return self.conv(t, ids[4], km, residual=x, relu=True, fmt=final)
        x = self.conv(x, ids[0], km, relu=True)
        for a, b in ((ids[1], ids[2]), (ids[3], ids[4])):
            t = self.conv(x, a, km, relu=True)
            x = self.conv(t, b, km, residual=x, relu=True)
        return x

    def level_features(self, parent: Level, n_child: int, child_kmap: Optional[KMap] = None):
        """pcc_utils.py:99-109 == :300-311: prior stack on S_d, expand, target embedding, target stack.
        child_kmap: the kernel map of the child set if the caller has built it already (encoder).
        Returns (child level, u): u = fp32 rows, or (fp32 rows, split rows) on a tcgen05 level."""
        if parent.kmap is None:
            with self._stage("kmap", self._kmap_bytes(parent.n)):
                parent.kmap = self.build_kmap(parent.keys)
        pum = bool(parent.kmap.um_rows)
        f = self._empty((parent.n, 32), torch.int32 if pum else torch.float32)
        with self._stage("embed", parent.n * 129):
            self._call("gpc_embed_rows", _ptr(parent.occ), parent.n, _ptr(self.w.prior_emb), None if pum else _ptr(f), _ptr(f) if pum else None,
                       self._stream())
        if child_kmap is None and self.conv_profile is None and n_child >= 20_000:
            # decoder: the children and their kernel map depend on the parents' occupancy only, not on the prior features --
            # they are built on a side stream (incl. the host round trip of the pair counts) while the prior stack runs
            main = torch.cuda.current_stream(self.dev)
            ready = torch.cuda.Event()
            ready.record(main)                                       # parent.keys / parent.occ are complete
            f = self.res_stack(f, W.PRIOR_CONVS, parent.kmap)        # enqueued on main; the host goes on
            if self._dec_side is None:
                self._dec_side = torch.cuda.Stream(self.dev)
            side, main_h = self._dec_side, self._stream_h
            with torch.cuda.stream(side):
                side.wait_event(ready)
                self._stream_h = side.cuda_stream
                ck, cp = self.expand(parent, n_child)
                child_kmap = self.build_kmap(ck)
            self._stream_h = main_h
            main.wait_stream(side)
            for t in (ck, cp, child_kmap.seg, child_kmap.pairs, child_kmap.pair_nbr, child_kmap.pair_off, child_kmap.rowptr,
                      child_kmap.contrib, child_kmap.tile_order):
                if t is not None:
                    t.record_stream(main)                            # allocated under the side stream, used on main from here on
        else:
            f = self.res_stack(f, W.PRIOR_CONVS, parent.kmap)        # fp32 rows (the children gather them)
            with self._stage("expand", parent.n * 33 + n_child * 12):
                ck, cp = self.expand(parent, n_child)
            if child_kmap is None:
                with self._stage("kmap", self._kmap_bytes(n_child)):
                    child_kmap = self.build_kmap(ck)
        child = Level(ck, None, n_child, child_kmap)
        cum = bool(child.kmap.um_rows)
        u0 = self._empty((n_child, 32), torch.int32 if cum else torch.float32)
        with self._stage("embed", n_child * (12 + 4 + 256)):
            self._call("gpc_gather_parent_add_octant", _ptr(f), _ptr(cp), _ptr(ck), n_child, _ptr(self.w.target_emb), None if cum else _ptr(u0),
                       _ptr(u0) if cum else None, self._stream())
        # tcgen05 level: u is needed as fp32 rows (context embeddings) and as split rows (stage 0 conv input)
        u = self.res_stack(u0, W.TARGET_CONVS, child.kmap, final="both" if cum else "f32")
        return child, u

    def stage_cdf(self, u: torch.Tensor, occ_partial: Optional[torch.Tensor], i: int, km: KMap, cdf_out: Optional[torch.Tensor],
                  prob_out: Optional[torch.Tensor] = None, lohi_out: Optional[torch.Tensor] = None):
        """stage i: (+ context embedding) -> spatial_conv_s{i} -> pred_head_s{i} -> uint16 CDF rows.
        Encoder: lohi_out given => occ_partial is the TRUE occupancy, the stage's symbol is split off inside the head kernel
        and only (c_low, c_high) of that symbol is written (4 B per row for the host coder)."""
        u, u_split = u if isinstance(u, tuple) else (u, None)
        n = u.shape[0]
        um = bool(km.um_rows)
        if i == 0:
            f = u_split if um else u
        else:
            f = self._empty((n, 32), torch.int32 if um else torch.float32)
            with self._stage("embed", n * 257):
                self._call("gpc_add_ctx_embed", _ptr(u), _ptr(occ_partial), CTX_SHIFT[i], _ptr(self.w.stage_emb[i]), n, None if um else _ptr(f),
                           _ptr(f) if um else None, self._stream())
        c0, c1 = W.stage_convs(i)
        grp = self._prof_open()
        t = self.conv(f, c0, km, relu=True, fmt="split" if um else "f32")
        t = self.conv(t, c1, km)
        self._prof_close(grp)
        w1, b1, w2, b2 = self.w.head[i]
        with self._stage("head", n * (128 + 2 * (W.STAGE_ALPHABETS[i] + 1))):
            if lohi_out is not None:
                self._call("gpc_head_cdf_sym", _ptr(t), n, _ptr(w1), _ptr(b1), _ptr(w2), _ptr(b2), W.STAGE_ALPHABETS[i], _ptr(occ_partial),
                           STAGE_SHIFT[i], _ptr(lohi_out), _ptr(cdf_out), _ptr(prob_out), self._stream())
            else:
                self._call("gpc_head_cdf", _ptr(t), n, _ptr(w1), _ptr(b1), _ptr(w2), _ptr(b2), W.STAGE_ALPHABETS[i], _ptr(cdf_out),
                           _ptr(prob_out), self._stream())

    # ------------------------------------------------------------------ GPU chunk coder (container version 2)
    @staticmethod
    def chunk_len(n: int, chunk: int) -> int:
        """Symbols per chunk of a version-2 stream of n symbols under the file's chunk size: the file's size, but at least 64 chunks
        per stream where 64-symbol chunks allow -- a chunk is a serial chain on one warp, and a coarse level decoded as one or two
        chunks would take as long as a 1M-row level.  (Every chunk costs ~4 bytes: shorter chunks on the big levels are the file's
        choice, not this rule's.)"""
        return max(1, min(chunk, max(64, (n + 63) // 64)))

    def _chunk_begin(self, stream_rows: List[int], chunk: int):
        """Version-2 encode: ONE device array holds the (c_low, c_high) words of every stream of the scene, one after the other;
        the head kernels write their words straight into it, and at the end ONE launch codes all chunks of all streams at once (a
        chunk is one warp walking a serial chain: ten thousand of them side by side take as long as one)."""
        starts, cstarts, total = [], [0], 0
        for n in stream_rows:
            starts.append(total)
            cl = self.chunk_len(n, chunk)
            for o in range(0, n, cl):
                cstarts.append(total + min(o + cl, n))
            total += n
        if self._coder_arena is None or self._coder_arena.numel() < total:
            self._coder_arena = torch.empty(int(total * 1.25) + 64, dtype=torch.int32, device=self.dev)
        self._coder_starts, self._coder_total, self._coder_rows = starts, total, list(stream_rows)
        self._coder_cstarts = np.array(cstarts, dtype=np.uint32)

    def _chunk_slot(self, k: int) -> torch.Tensor:
        return self._coder_arena[self._coder_starts[k]:self._coder_starts[k] + self._coder_rows[k]]

    def _chunk_finish(self, chunk: int) -> List[bytes]:
        """code every chunk of every stream in one launch, bring counts and bytes to the host in one staging copy each"""
        chunks = int(self._coder_cstarts.shape[0]) - 1
        if chunks <= 0:
            return [b""] * len(self._coder_rows)
        cstarts = torch.from_numpy(self._coder_cstarts.view(np.int32)).to(self.dev)
        cnt = self._empty((chunks,), torch.int32)
        offs = self._empty((chunks + 1,), torch.int32)
        ws_b = self.lib.gpc_chunk_workspace_bytes(chunks, chunk)
        ws = self._ws(ws_b)
        self._call("gpc_chunk_encode_lohi", _ptr(self._coder_arena), _ptr(cstarts), chunks, chunk, _ptr(cnt), _ptr(offs), _ptr(ws), ws_b,
                   self._stream())
        cnt_h = cnt.cpu().numpy()                                               # synchronises; offsets on the host from the counts
        if cnt_h.size and int(cnt_h.max()) > 0xFFFF:
            raise ValueError("chunk too long for the u16 byte counts of container version 2")
        offs_h = np.concatenate([[0], np.cumsum(cnt_h, dtype=np.int64)])
        nbytes = int(offs_h[-1])
        out = self._empty((nbytes + 64,), torch.uint8)
        self._call("gpc_chunk_merge", _ptr(ws), chunks, chunk, _ptr(offs), _ptr(out), self._stream())
        pin = self._pin(nbytes + 64)
        pin[:nbytes].copy_(out[:nbytes], non_blocking=True)
        torch.cuda.current_stream(self.dev).synchronize()
        host = pin.numpy()
        streams, c0 = [], 0
        for n in self._coder_rows:
            cl = self.chunk_len(n, chunk)
            c1 = c0 + (n + cl - 1) // cl
            streams.append(cnt_h[c0:c1].astype("<u2").tobytes() + host[int(offs_h[c0]):int(offs_h[c1])].tobytes())
            c0 = c1
        return streams

    def _chunk_upload(self, streams: List[bytes]):
        """all version-2 streams of a file -> device in ONE staging copy (a 1M-anchor scene is ~9 MB); per stream its offset.
        Behind them room for the chunks' byte offsets, which the levels fill in as their sizes become known."""
        torch.cuda.current_stream(self.dev).synchronize()        # nothing of an earlier call still reads the staging buffer
        offs, total = [], 0
        for sb in streams:
            offs.append(total)
            total += (len(sb) + 255) // 256 * 256
        room = 2 * sum(len(sb) for sb in streams) + 64 * len(streams) + 4096          # a chunk has a 2-byte count in its stream: <= len / 2 chunks, 4 B each
        pin = self._pin(total + room)
        host = pin.numpy()
        for o, sb in zip(offs, streams):
            host[o:o + len(sb)] = np.frombuffer(sb, dtype=np.uint8)
        dev = torch.empty(total + room, dtype=torch.uint8, device=self.dev)
        dev[:total].copy_(pin[:total], non_blocking=True)
        torch.cuda.current_stream(self.dev).synchronize()        # the staging buffer is free again (the GPU is idle here anyway)
        self._v2_cursor, self._v2_end = total, total + room
        return dev, offs

    def _chunk_decode(self, cdf_d: torch.Tensor, stream: bytes, dev_bytes: torch.Tensor, off: int, n: int, Lp: int, chunk: int) -> torch.Tensor:
        chunk = self.chunk_len(n, chunk)
        chunks = (n + chunk - 1) // chunk
        if len(stream) < 2 * chunks:
            raise ValueError("truncated version-2 stream")
        cnt_h = np.frombuffer(stream, dtype="<u2", count=chunks)
        offs_h = np.zeros(chunks + 1, dtype=np.uint32)
        np.cumsum(cnt_h, dtype=np.uint32, out=offs_h[1:])
        if int(offs_h[-1]) != len(stream) - 2 * chunks:
            raise ValueError("corrupt version-2 stream (chunk byte counts)")
        # the chunks' byte offsets: host prefix sums, into their own (never reused) piece of the staging buffer and the device array
        a = (self._v2_cursor + 15) // 16 * 16
        b = a + 4 * (chunks + 1)
        if b > self._v2_end:
            raise ValueError("corrupt version-2 file (more chunks than its streams can hold)")
        self._v2_cursor = b
        self._pinned.numpy()[a:b] = offs_h.view(np.uint8)
        dev_bytes[a:b].copy_(self._pinned[a:b], non_blocking=True)
        sym = self._empty((n,), torch.uint8)
        self._call("gpc_chunk_decode_u16", _ptr(cdf_d), C.c_void_p(dev_bytes.data_ptr() + off + 2 * chunks), C.c_void_p(dev_bytes.data_ptr() + a),
                   n, Lp, chunk, _ptr(sym), self._stream())
        return sym

    # ------------------------------------------------------------------ host range coder
    def _ac_encode_lohi(self, lohi: np.ndarray, ready: Optional[torch.cuda.Event] = None) -> bytes:
        if ready is not None:
            ready.synchronize()                        # the level's D2H copies have landed (GPU keeps running later levels)
        n = lohi.shape[0]
        cap = 4 * n + 64
        out = np.empty(cap, dtype=np.uint8)
        ln = C.c_int64(0)
        _lib.check(self.lib.gpc_ac_encode_lohi_h(lohi.ctypes.data_as(C.c_void_p), n, out.ctypes.data_as(C.c_void_p), cap,
                                                 C.byref(ln)), "gpc_ac_encode_lohi_h")
        return out[:ln.value].tobytes()

    def _ac_decode(self, cdf: np.ndarray, stream: bytes, sym_out: np.ndarray):
        n, Lp = cdf.shape
        buf = (C.c_char * max(len(stream), 1)).from_buffer_copy(stream if len(stream) else b"\0")
        _lib.check(self.lib.gpc_ac_decode_h(cdf.ctypes.data_as(C.c_void_p), C.cast(buf, C.c_void_p), len(stream), n, Lp,
                                            sym_out.ctypes.data_as(C.c_void_p)), "gpc_ac_decode_h")

    # ------------------------------------------------------------------ encode
    def _encode_level(self, d: int, parent: Level, gt: Level, collect: bool, download: bool, gpu_chunk: int, keep_lohi: bool, aux, carve,
                      level_futs):
        """one octree level of the encoder on the current stream: features, four stages, (c_low, c_high) words on their way to the coder"""
        child, u = self.level_features(parent, gt.n, child_kmap=gt.kmap)      # same coordinate set, same row order
        if collect:
            aux["child_keys"][d] = child.keys
        level_jobs = []
        for i in range(4):
            A = W.STAGE_ALPHABETS[i]
            cdf_d = self._empty((gt.n, A + 1), torch.int16) if collect else None
            prob_d = self._empty((gt.n, A), torch.float32) if collect else None
            lohi_d = self._chunk_slot(4 * d + i) if (download and gpu_chunk) else self._empty((gt.n,), torch.int32)
            self.stage_cdf(u, gt.occ, i, child.kmap, cdf_d, prob_d, lohi_out=lohi_d)
            if download and gpu_chunk:
                pass                                                        # coded with all other streams at the end (_chunk_finish)
            elif download:
                lohi_h = carve(gt.n * 4, torch.int32, (gt.n,))
                lohi_h.copy_(lohi_d, non_blocking=True)
                level_jobs.append(lohi_h)
            elif keep_lohi:
                aux["lohi"][4 * d + i] = lohi_d
            if collect:
                aux["probs"][4 * d + i] = prob_d
                aux["cdfs"][4 * d + i] = cdf_d
        if download and not gpu_chunk:
            ready = torch.cuda.Event(blocking=True)          # the coder threads sleep on it instead of spinning
            ready.record(torch.cuda.current_stream(self.dev))
            # host range coding of this level overlaps the GPU work of the coarser levels
            level_futs[d] = [self.pool.submit(self._ac_encode_lohi, h.numpy().view(np.uint32), ready) for h in level_jobs]

    def encode(self, xyz: torch.Tensor, collect: bool = False, download: bool = True, gpu_chunk: int = 0, keep_lohi: bool = False):
        """[N,3] CUDA float32/int32 voxel indices -> (base_xyz int32 [n0,3], base_occ u8 [n0], streams, aux).

        download=False (bench, device-timed number): the CDF rows and symbols stay in HBM, nothing is copied to
        the host and the range coder does not run (streams is None); the device work is unchanged.
        keep_lohi (download=False only): aux["lohi"][4 * d + i] holds what the range coder would take for stage i of level d, one
        int32 c_low | c_high << 16 per row; otherwise each stage's buffer is released as soon as its level is done.
        gpu_chunk > 0 (container version 2, SURVEY 8f-3; NOT the reference bitstream): the streams are coded on the GPU in chunks
        of gpu_chunk symbols (csrc/attr_ac.cu: one warp per chunk) -- no host range coder, only compressed bytes cross PCIe.
        A stream is then `u16 bytes_of_chunk[chunks]` followed by the chunks' bytes.
        """
        if keep_lohi and download:
            raise ValueError("keep_lohi needs download=False: a downloading encode hands the words to the range coder")
        self._launch_base = int(self.lib.gpc_launch_count())
        self._segments = []
        self._stream_h = torch.cuda.current_stream(self.dev).cuda_stream
        self._seg_begin()
        xyz = xyz.contiguous()
        n_in = int(xyz.shape[0])
        with self._stage("order", n_in * 20 + 6 * n_in * 24):            # pack + 6-pass radix sort + unique (SURVEY 8d radix model)
            keys, meta = self.pack_keys(xyz)
        meta_h = meta.cpu().numpy()
        if meta_h[0] & 1:
            raise ValueError("compress_point_cloud expects voxelised (integral) coordinates")
        shift = None
        if meta_h[0] & 2:
            # outside the 21-bit key fields: code the scene translated towards the origin (the pyramid is translation-invariant for
            # offsets that are multiples of 2^levels; the base level is written in the caller's coordinates again at the end)
            xyz, shift = self._recentre(xyz)
            with self._stage("order", 0):
                keys, meta = self.pack_keys(xyz)
            meta_h = meta.cpu().numpy()
            assert not (meta_h[0] & 2)
        mm = meta_h[2:8].astype(np.uint32)
        with self._stage("order", 0):
            leaf = self.sort_unique(keys, mm)
        with self._stage("pyramid", int(leaf.shape[0]) * (25 + 6 * 24) * 8 // 7):   # geometric sum over the levels: n_l*12 + n_(l+1)*13 + one sort of n_l pairs
            levels = self.build_pyramid(leaf, mm.astype(np.int64))
        L = len(levels) - 1
        rows = sum(l.n for l in levels[1:])
        arena = self._pin(rows * 16 + 64 * 4 * max(L, 1) + 4096) if download else None
        cursor = 0
        futs = []
        aux = {"levels": levels, "probs": [], "cdfs": []} if (collect or not download) else None
        if keep_lohi:
            aux["lohi"] = [None] * (4 * L)

        def carve(nbytes, dtype, shape):
            nonlocal cursor
            start = (cursor + 63) // 64 * 64
            cursor = start + nbytes
            t = arena[start:start + nbytes]
            return t.view(dtype).view(shape)

        # Kernel maps of all levels first, coarse -> fine: the order in which the decoder meets them, so that both sides take the same
        # per-level kernel decisions (build_kmap's sparse switch is sticky along that order).  The levels themselves are then coded
        # FINE -> COARSE: every level's CDFs depend on the ground truth only, and with the big levels first their host range coding
        # (10 ms per stream at 1M rows) overlaps the GPU work of the remaining levels instead of trailing the last kernel.
        if L:
            for lv in levels:
                if lv.kmap is None:
                    with self._stage("kmap", self._kmap_bytes(lv.n)):
                        lv.kmap = self.build_kmap(lv.keys)
        level_futs = [[] for _ in range(L)]
        if download and gpu_chunk:
            self._chunk_begin([levels[k // 4 + 1].n for k in range(4 * L)], gpu_chunk)
        if collect:
            aux["child_keys"], aux["probs"], aux["cdfs"] = [None] * L, [None] * (4 * L), [None] * (4 * L)
        # Every level of the encoder is independent work: the levels are spread over the main stream and one side stream, so that
        # one level's launch tails, pipeline ramps and small kernels (embeddings, heads, the 15-180 us launches of the coarse levels)
        # run beside another level's convs (0 / 1 / 2-6 side streams: 61.8 / 56.4 / 56.5-57.8 ms per 1M-anchor encode).  Not while
        # bench.py's per-stage profile is on (its event pairs assume one stream).
        side = None
        main = torch.cuda.current_stream(self.dev)
        if self.conv_profile is None and not collect and L > 1:
            if self._enc_side is None:
                self._enc_side = torch.cuda.Stream(self.dev)
            side = self._enc_side
            side.wait_stream(main)                                             # pyramid and kernel maps are complete
        main_h = self._stream_h
        for d in range(L - 1, -1, -1):
            parent, gt = levels[d], levels[d + 1]
            # big levels alternate main, side, main, ... (finest first); the coarse levels all go to the side stream
            st = side if side is not None and (gt.n < self.um_min_rows or (L - 1 - d) % 2) else None
            with (torch.cuda.stream(st) if st is not None else contextlib.nullcontext()):
                self._stream_h = st.cuda_stream if st is not None else main_h
                self._encode_level(d, parent, gt, collect, download, gpu_chunk, keep_lohi, aux, carve, level_futs)
        self._stream_h = main_h
        if side is not None:
            main.wait_stream(side)
        futs = [f for lf in level_futs for f in lf]            # stream order of the container: level-major coarse -> fine
        base = levels[0]
        base_xyz = self._empty((base.n, 3), torch.int32)
        self._call("gpc_unpack_keys_i32", _ptr(base.keys), base.n, _ptr(base_xyz), self._stream())
        base_xyz_h = base_xyz.cpu().numpy()
        if shift is not None:
            depth = L + 1                              # the base level is the leaves' ancestors depth levels up
            assert not np.any(shift % (1 << depth)), "translation must be a multiple of 2^depth"
            moved = base_xyz_h.astype(np.int64) + (shift >> depth)
            if np.abs(moved).max(initial=0) >= (1 << 31):
                raise ValueError("base coordinates do not fit int32")
            base_xyz_h = moved.astype(np.int32)
        base_occ_h = base.occ.cpu().numpy()
        self._seg_end()
        gpu_ms = self._seg_total_ms()                  # synchronises: all D2H copies have landed
        streams = [f.result() for f in futs] if download else None
        if download and gpu_chunk:
            streams = self._chunk_finish(gpu_chunk)
        self._stream_h = None
        self.last_stats = {"gpu_ms": gpu_ms, "launches": self.launches, "rows": rows, "levels": L,
                           "d2h_bytes": cursor, "n_unique": int(leaf.shape[0])}
        return base_xyz_h, base_occ_h, streams, aux

    # ------------------------------------------------------------------ decoder: the four stages of a level as a wavefront
    # pcc_utils.py:319-366 decodes a level stage by stage: CDFs of stage i for ALL rows -> range decoder (one serial stream) -> symbols
    # -> stage i+1.  The dependency is local, though: stage i+1 of a row needs the stage-i symbols of the rows within two 5^3 convs
    # of it, and rows are sorted by (z, y, x).  So stage 0 is handed to its decoder in chunks of rows; whenever decoder i reports a
    # piece, the GPU computes the stage-(i+1) CDFs of every row whose neighbourhood is now decoded (_wave_plan: a lag of a few
    # z planes), and the four stage streams decode on four host threads, one piece behind each other.  Same kernels, same sums,
    # same bitstream; the serial range decoder (0.28 s of a 0.35 s decode at 1M anchors) overlaps with itself.
    def _wave_ok(self, child: Level, n: int) -> bool:
        km = child.kmap
        if not self.wave_decode or n < self.wave_min_rows:
            return False
        if km.sparse:
            tile = 8192                     # the sparse conv's row blocks
        elif km.um_rows or km.v6_variant == 48:
            tile = km.tile_rows
        else:
            return False
        # the plan (_wave_plan) is valid for any geometry; it degenerates to stage by stage at worst
        return self.wave_chunk_rows % tile == 0 and len(self._wave_chunks(n)) >= 2

    def _wave_plan(self, keys: torch.Tensor, n: int, chunks: List[Tuple[int, int]], tile: int):
        """Row ranges of the wavefront: each stage lags the previous one by a few z PLANES.  Rows are sorted by (z, y, x); if stage i is known for
        the rows < e, the first conv of stage i+1 is exact for every row whose 5^3 neighbours are all < e: the planes z <= z[e] - 3,
        i.e. the rows before the first row of plane z[e] - 2 (rounded down to the conv's tile height); the second conv, likewise, for
        the rows two more planes back; those rows' CDFs go to decoder i+1.  Returns per stage the piece ends E[i][c] (stage 0: the
        chunks) and the first-conv ends CA[i][c], as Python ints; piece c of stage i+1 is released by piece c of stage i."""
        dev = self.dev
        nn = torch.tensor(n, device=dev)

        def lag(end: torch.Tensor) -> torch.Tensor:
            zf = keys[end.clamp(max=n - 1)] >> 42                                  # plane of the first row that is not valid yet
            out = torch.searchsorted(keys, (zf - 2) << 42) // tile * tile          # smallest key of plane zf - 2 -> its first row
            return torch.where(end >= n, nn, out)

        E = [torch.tensor([r1 for _, r1 in chunks], device=dev, dtype=torch.int64)]
        CA = [E[0]]
        for _ in range(3):
            ca = lag(E[-1])
            CA.append(ca)
            E.append(lag(ca))
        flat = torch.stack(E + CA).cpu().tolist()
        return flat[:4], flat[4:]

    def _wave_chunks(self, n: int) -> List[Tuple[int, int]]:
        """Row chunks of a wavefront level: wave_chunk_rows each, the last one ragged"""
        ch = self.wave_chunk_rows
        return [(r, min(r + ch, n)) for r in range(0, n, ch)]

    def _decode_level_wavefront(self, u, child: Level, n: int, streams: List[bytes], occ: torch.Tensor):
        km = child.kmap
        chunks = self._wave_chunks(n)
        nc = len(chunks)
        u, u_split = u if isinstance(u, tuple) else (u, None)
        um = bool(km.um_rows)                  # tcgen05 level: conv inputs (context-embedded rows, first-conv outputs) are split rows
        Lps = [a + 1 for a in W.STAGE_ALPHABETS]
        # pinned staging: the four stages' CDF rows and symbols live at the same time
        need = n * (2 * sum(Lps) + 4) + 4096
        if self._pinned_dec is None or self._pinned_dec.numel() < need:
            self._pinned_dec = torch.empty(int(need * 1.5), dtype=torch.uint8, pin_memory=True)
        pin, off = self._pinned_dec, 0
        cdf_h, sym_h = [], []
        for Lp in Lps:
            cdf_h.append(pin[off:off + n * Lp * 2].view(torch.int16).view(n, Lp))
            off += (n * Lp * 2 + 63) // 64 * 64
        for _ in range(4):
            sym_h.append(pin[off:off + n])
            off += (n + 63) // 64 * 64
        cdf_d = [self._empty((n, Lp), torch.int16) for Lp in Lps]
        sym_d = [self._empty((n,), torch.uint8) for _ in range(4)]
        # eleven level-sized feature arrays, carved from one buffer the codec keeps (grown geometrically): scenes of other sizes reuse it
        # instead of sending the caching allocator back to cudaMalloc, and no block returns to the allocator while side streams use it
        if self._wave_buf is None or self._wave_buf.numel() < 11 * n * 32:
            self._wave_buf = None
            self._wave_buf = torch.empty(int(11 * n * 32 * 1.3) + 1024, dtype=torch.float32, device=self.dev)
        carve = [self._wave_buf[k * n * 32:(k + 1) * n * 32].view(n, 32) for k in range(11)]
        as_in = (lambda t: t.view(torch.int32)) if um else (lambda t: t)
        f = [None] + [as_in(t) for t in carve[0:3]]
        t0 = [as_in(t) for t in carve[3:7]]
        t1 = carve[7:11]
        cfmt = "split" if um else "f32"
        stream = torch.cuda.current_stream(self.dev)
        ev_q = [queue.Queue() for _ in range(4)]
        done_q: "queue.Queue" = queue.Queue()
        ac_s = [0.0] * 4
        state_bytes = int(self.lib.gpc_ac_decode_state_bytes())

        def worker(i: int):
            try:
                st = C.create_string_buffer(state_bytes)
                data = streams[i]
                buf = (C.c_char * max(len(data), 1)).from_buffer_copy(data if len(data) else b"\0")
                _lib.check(self.lib.gpc_ac_decode_begin_h(C.cast(st, C.c_void_p), C.cast(buf, C.c_void_p), len(data)), "gpc_ac_decode_begin_h")
                cdf_np, sym_np = cdf_h[i].numpy().view(np.uint16), sym_h[i].numpy()
                for c, (r0, r1) in enumerate(P[i]):
                    if r1 <= r0:                       # empty piece (plane lag): nothing to decode, but the next stage's step c is due
                        done_q.put((i, c, None))
                        continue
                    ev = ev_q[i].get()
                    if ev is None:
                        return
                    ev.synchronize()
                    tb = time.perf_counter()
                    _lib.check(self.lib.gpc_ac_decode_more_h(C.cast(st, C.c_void_p), cdf_np[r0:r1].ctypes.data_as(C.c_void_p), r1 - r0,
                                                             Lps[i], sym_np[r0:r1].ctypes.data_as(C.c_void_p)), "gpc_ac_decode_more_h")
                    ac_s[i] += time.perf_counter() - tb
                    done_q.put((i, c, None))
            except BaseException as e:          # noqa: BLE001 -- handed to the main thread, which re-raises
                done_q.put((i, -1, e))

        # One CUDA stream per stage on the dense levels: a 32 K-row chunk is 256 one-warp CTAs, a seventh of the GPU, and a chunk's conv
        # lasts as long as its slowest warp's chain of tiles, so on one stream the three stages' chunk work (0.9 ms per chunk index at
        # 442 K rows) outlasted the decoders (0.55 ms).  Stage j's work runs on stream j; what it reads from other stages (symbols,
        # occupancy bits) has reached the host before it is enqueued, and at any moment the stages work on disjoint chunks.  The
        # sparse levels (decoder-bound, and their convs share the level's contribution scratch) stay on the one stream.
        multi = not km.sparse
        if multi and self._wave_side is None:
            self._wave_side = [torch.cuda.Stream(device=self.dev) for _ in range(3)]
        S = [stream] + (self._wave_side if multi else [stream] * 3)
        SH = [st_.cuda_stream for st_ in S]
        # the per-completion work below runs ~100 times per level: plain integer addresses instead of tensor views
        call = self._call
        p_u, p_occ = u.data_ptr(), occ.data_ptr()
        p_f = [0] + [t.data_ptr() for t in f[1:]]
        p_t1 = [t.data_ptr() for t in t1]
        p_cdf_d, p_cdf_h = [t.data_ptr() for t in cdf_d], [t.data_ptr() for t in cdf_h]
        p_sym_d, p_sym_h = [t.data_ptr() for t in sym_d], [t.data_ptr() for t in sym_h]
        heads = [tuple(_ptr(t) for t in self.w.head[i]) for i in range(4)]
        embs = [0] + [_ptr(self.w.stage_emb[j]) for j in range(1, 4)]

        def emit_cdf(i: int, c: int, rng: Optional[Tuple[int, int]] = None):
            """head of stage i on chunk c (or the row range rng) -> D2H -> event for decoder thread i"""
            r0, r1 = chunks[c] if rng is None else rng
            w1, b1, w2, b2 = heads[i]
            call("gpc_head_cdf", p_t1[i] + r0 * 128, r1 - r0, w1, b1, w2, b2, W.STAGE_ALPHABETS[i], p_cdf_d[i] + r0 * Lps[i] * 2, None, SH[i])
            call("gpc_copy_async", p_cdf_h[i] + r0 * Lps[i] * 2, p_cdf_d[i] + r0 * Lps[i] * 2, (r1 - r0) * Lps[i] * 2, SH[i])
            ev = torch.cuda.Event(blocking=True)               # decoder thread i sleeps on it (a spinning waiter per stage stole the cores
            ev.record(S[i])                                    # the launch thread needs)
            ev_q[i].put(ev)

        E, CA = self._wave_plan(child.keys, n, chunks, 8192 if km.sparse else km.tile_rows)
        P = [[(E[i][c - 1] if c else 0, E[i][c]) for c in range(nc)] for i in range(4)]
        workers = [self.pool.submit(worker, i) for i in range(4)]
        t_wait = 0.0
        try:
            # stage 0 needs no symbols: whole level at once, CDFs handed over chunk by chunk
            c0, c1 = W.stage_convs(0)
            self.conv(u_split if um else u, c0, km, relu=True, out=t0[0], fmt=cfmt)
            self.conv(t0[0], c1, km, out=t1[0])
            for c in range(nc):
                emit_cdf(0, c)
            if multi:
                ready = torch.cuda.Event()
                ready.record(stream)               # u, the kernel map, the zeroed occupancy: all produced on the main stream
                for st_ in S[1:]:
                    st_.wait_event(ready)
            pending = 4 * nc
            while pending:
                tb = time.perf_counter()
                i, c, err = done_q.get()
                t_wait += time.perf_counter() - tb
                if err is not None:
                    raise err
                pending -= 1
                j = min(i + 1, 3)
                sh = self._stream_h = SH[j]           # everything this completion triggers goes to the next stage's stream
                r0, r1 = P[i][c]
                if r1 > r0:
                    call("gpc_copy_async", p_sym_d[i] + r0, p_sym_h[i] + r0, r1 - r0, sh)
                    call("gpc_merge_symbol", p_occ + r0, r1 - r0, STAGE_SHIFT[i], p_sym_d[i] + r0, sh)
                if i == 3:
                    continue
                k0, k1 = W.stage_convs(j)
                if r1 > r0:
                    call("gpc_add_ctx_embed", p_u + r0 * 128, p_occ + r0, CTX_SHIFT[j], embs[j], r1 - r0,
                         None if um else p_f[j] + r0 * 128, p_f[j] + r0 * 128 if um else None, sh)
                a0, a1 = (CA[j][c - 1] if c else 0), CA[j][c]
                if a1 > a0:
                    self.conv(f[j], k0, km, relu=True, out=t0[j], rows=(a0, a1), fmt=cfmt)
                q0, q1 = P[j][c]
                if q1 > q0:
                    self.conv(t0[j], k1, km, out=t1[j], rows=(q0, q1))
                    emit_cdf(j, c, (q0, q1))
        except BaseException:
            for q in ev_q:
                q.put(None)                       # let the decoder threads go
            raise
        finally:
            self._stream_h = SH[0]
            if multi:
                for st_ in S[1:]:                 # the level's buffers go back to the main stream's allocator only after the side streams
                    done = torch.cuda.Event()
                    done.record(st_)
                    stream.wait_event(done)
            for w_ in workers:
                try:
                    w_.result()
                except BaseException:             # noqa: BLE001 -- the first error is already on its way up
                    pass
        if self.wave_log is not None:
            self.wave_log.append({"rows": n, "chunks": nc, "sparse": bool(km.sparse), "ac_s": [round(v, 4) for v in ac_s]})
        return t_wait, max(ac_s)

    def decode(self, base_xyz: np.ndarray, base_occ: np.ndarray, streams: List[bytes], scale: float = 1.0,
               forced_occ: Optional[List[torch.Tensor]] = None, sorted_rows: bool = False, gpu_chunk: int = 0) -> torch.Tensor:
        """-> float32 [N,3] CUDA, rows in the reference's order (children of (z,y,x)-sorted parents, octant ascending), or,
        with sorted_rows, in ascending (z,y,x) == calculate_morton_order order (SURVEY 8f-1: the caller's re-sort,
        HAC/scene/gaussian_model.py:1253-1255, becomes the identity).

        forced_occ (bench only): per-level ground-truth occupancy already on the device; the GPU work is
        then identical to a real decode but the host range decoder is skipped ("device-timed" number).
        """
        self._launch_base = int(self.lib.gpc_launch_count())
        self._segments = []
        self._stream_h = torch.cuda.current_stream(self.dev).cuda_stream
        if len(streams) % 4:
            raise ValueError("stream count must be a multiple of 4 (one group per octree level)")
        self._seg_begin()
        bx_h = np.array(base_xyz, dtype=np.int32).reshape(-1, 3)
        L = len(streams) // 4 + 1                      # leaves are 2^L base voxels wide: one level per stream group + the base's own occupancy
        shift = None
        if bx_h.size and (int(np.abs(bx_h.astype(np.int64)).max()) + 1) << L > COORD_LIMIT:
            # some leaf of the base voxels may lie outside the 21-bit key fields: decode translated (children are 2c + b, so any base
            # translation t is a leaf translation t * 2^L) and add it back on the decoded rows.  If even the centred scene does not
            # fit, the encoder cannot have translated either (it would have refused): the file is of a scene near the origin that
            # spans nearly the whole range, and decodes as it is.
            b64 = bx_h.astype(np.int64)
            t = (b64.min(axis=0) + b64.max(axis=0) + 1) // 2
            if max(int(-(b64.min(axis=0) - t).min()) << L, ((int((b64.max(axis=0) - t).max()) + 1) << L) - 1) <= COORD_LIMIT:
                bx_h = (b64 - t).astype(np.int32)
                shift = t << L
        bx = torch.from_numpy(bx_h).to(self.dev)
        bo = torch.from_numpy(np.array(base_occ, dtype=np.uint8).reshape(-1)).to(self.dev)
        keys, meta = self.pack_keys(bx)
        meta_h = meta.cpu().numpy()
        if meta_h[0] & 2:
            raise ValueError("corrupt base coordinates")
        n0 = keys.shape[0]
        # the reference stores the base level in torchsparse's emission order; canonicalise to (z,y,x)
        xf = self._xform(meta_h[2:8].astype(np.uint32))
        skeys = self._empty((n0,), torch.int64)
        perm = self._empty((n0,), torch.int32)
        ws_b = self.lib.gpc_sort_workspace_bytes(n0)
        ws = self._ws(ws_b)
        self._call("gpc_sort_pairs", _ptr(keys), _ptr(None), _ptr(skeys), _ptr(perm), n0, xf, _ptr(ws), ws_b, self._stream())
        cur = Level(skeys, bo[perm.long()] if n0 else bo, n0)
        pin = self._pinned_dec                     # staging for CDF rows / symbols, kept across calls (grown geometrically)
        if gpu_chunk and forced_occ is None:
            v2_dev, v2_off = self._chunk_upload(streams)
        t_wait = t_ac = 0.0
        n_wave = 0
        for g in range(0, len(streams), 4):
            n_child = self._popcount(cur.occ) if forced_occ is None else int(forced_occ[g // 4].shape[0])
            child, u = self.level_features(cur, n_child)
            occ = torch.zeros(n_child, dtype=torch.uint8, device=self.dev)
            if forced_occ is None and (pin is None or pin.numel() < n_child * 40):
                pin = self._pinned_dec = torch.empty(int(n_child * 40 * 1.5) + 4096, dtype=torch.uint8, pin_memory=True)
            if forced_occ is None and gpu_chunk:
                # container version 2: the stage's symbols are decoded on the GPU from the CDF rows where they lie; nothing crosses
                # PCIe but the compressed bytes, no host coder, no wavefront needed
                for i in range(4):
                    A = W.STAGE_ALPHABETS[i]
                    cdf_d = self._empty((n_child, A + 1), torch.int16)
                    self.stage_cdf(u, occ, i, child.kmap, cdf_d)
                    sym_d = self._chunk_decode(cdf_d, streams[g + i], v2_dev, v2_off[g + i], n_child, A + 1, gpu_chunk)
                    self._call("gpc_merge_symbol", _ptr(occ), n_child, STAGE_SHIFT[i], _ptr(sym_d), self._stream())
                child.occ = occ
                cur = child
                continue
            if forced_occ is None and self._wave_ok(child, n_child):
                dw, da = self._decode_level_wavefront(u, child, n_child, streams[g:g + 4], occ)
                t_wait += dw
                t_ac += da
                n_wave += 1
                pin = self._pinned_dec                 # the wavefront may have grown the staging buffer
                child.occ = occ
                cur = child
                continue
            for i in range(4):
                A = W.STAGE_ALPHABETS[i]
                cdf_d = self._empty((n_child, A + 1), torch.int16)
                self.stage_cdf(u, occ, i, child.kmap, cdf_d)
                if self.debug_dec_cdfs is not None:            # tests: the decoder's CDF rows of every (level, stage)
                    self.debug_dec_cdfs[(g // 4, i)] = cdf_d
                if forced_occ is not None:
                    sym_d = self._empty((n_child,), torch.uint8)
                    self._call("gpc_split_symbol", _ptr(forced_occ[g // 4]), n_child, STAGE_SHIFT[i], STAGE_MASK[i], _ptr(sym_d),
                               self._stream())
                else:
                    cdf_h = pin[:n_child * (A + 1) * 2].view(torch.int16).view(n_child, A + 1)
                    cdf_h.copy_(cdf_d, non_blocking=True)
                    self._seg_end()
                    t0 = time.perf_counter()
                    torch.cuda.current_stream(self.dev).synchronize()
                    t1 = time.perf_counter()
                    sym_h = pin[n_child * 36:n_child * 37]
                    self._ac_decode(cdf_h.numpy().view(np.uint16), streams[g + i], sym_h.numpy())
                    t_wait += t1 - t0
                    t_ac += time.perf_counter() - t1
                    self._seg_begin()
                    sym_d = sym_h.to(self.dev, non_blocking=True)
                self._call("gpc_merge_symbol", _ptr(occ), n_child, STAGE_SHIFT[i], _ptr(sym_d), self._stream())
            child.occ = occ
            cur = child
        n_pts = self._popcount(cur.occ)
        out = self._empty((n_pts, 3), torch.float32)
        k_scale = float(scale) if shift is None else 1.0
        if sorted_rows:
            ck, _ = self.expand(cur, n_pts)            # child keys already in (z,y,x) order: closed-form ranks, no sort
            self._call("gpc_unpack_keys_f32", _ptr(ck), n_pts, k_scale, _ptr(out), self._stream())
        else:
            ws_b = self.lib.gpc_expand_workspace_bytes(cur.n)
            ws = self._ws(ws_b)
            self._call("gpc_expand_leaves_f32", _ptr(cur.keys), _ptr(cur.occ), cur.n, n_pts, k_scale, _ptr(out), _ptr(ws), ws_b,
                       self._stream())
        if shift is not None:                          # integers below 2^24 add exactly in fp32, as in the reference's own float rows
            out += torch.tensor(shift, dtype=torch.float32, device=self.dev)
            if float(scale) != 1.0:
                out *= float(scale)
        self._seg_end()
        self._stream_h = None
        # host_ac_s: seconds inside the range decoder on the critical path (wavefront levels: the slowest of the four concurrent
        # streams); gpu_ms: CUDA-event time of the GPU segments (wavefront levels: first launch to last, idle gaps included)
        self.last_stats = {"gpu_ms": self._seg_total_ms(), "launches": self.launches, "host_ac_s": t_ac, "gpu_wait_s": t_wait,
                           "wave_levels": n_wave}
        return out


_WEIGHT_CACHE: Dict[tuple, DeviceWeights] = {}


def load_weights(ckpt_path: str, device: torch.device, channels: int = 32, kernel_size: int = 5) -> DeviceWeights:
    """torch.load the checkpoint once per (path, mtime, device); the reference reloads on every call
    (pcc_utils.py:65-67).  Missing file -> FileNotFoundError, bad layout -> RuntimeError, as there."""
    key = (os.path.abspath(ckpt_path), os.path.getmtime(ckpt_path), str(device), channels, kernel_size)
    if key not in _WEIGHT_CACHE:
        sd = torch.load(ckpt_path, map_location="cpu")
        _WEIGHT_CACHE[key] = DeviceWeights(sd, device, channels, kernel_size)
    return _WEIGHT_CACHE[key]
