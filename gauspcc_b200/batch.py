"""Many point clouds per call: the scenes of a batch are coded as ONE octree, level by level, and every file stays exactly what the
single-scene codec (codec.GausPcgcCodec.encode / decode) writes and reads for that scene alone.

Why the bytes do not change.  Translating a scene by a multiple of 2^(depth + 1) changes none of its octree levels, kernel maps or
streams (codec.GausPcgcCodec._recentre relies on the same fact).  The planner (plan_unions) stacks the scenes of a union along z, each
translated by (0, 0, T_s) with T_s a multiple of 2^(D+1) (D = the deepest base level of the batch) and a z gap of at least 4 * 2^D
voxels between neighbours, so at every coded scale
  * no 5^3 neighbourhood and no parent reaches into another scene (they stay >= 4 voxels apart),
  * keys sort scene-major: scene s is one contiguous row range [r0_s, r1_s) of every union level.
Scenes are stacked deepest first, so at every scale the scenes that still have children form a prefix of the union level, and the
base levels of shallower scenes join at its end.

What runs once per union level: hash build, dense map, children expansion, embeddings, context embeddings, heads, symbol merge, one
D2H and one H2D copy per stage.  What stays per scene: the conv family and its tiling (build_kmap's rule on the scene's own rows and
pairs, _v6_config on its own row count), run by the *_range kernels (csrc/kmap.cu, spconv.cu, spconv_sparse.cu, spconv_um.cu) whose
tiles start at r0_s while neighbour indices address the whole level -- so every row is summed exactly as in the scene's own level --
and the range coder streams, coded on the codec's thread pool, one task per (scene, stage).

Container version 2 (files of compress_point_cloud(..., gpu_coder_chunk=c)): a version-2 stream is cut into chunks by a rule on
that stream's own row count (GausPcgcCodec.chunk_len), and a scene's rows of a union level are its own level's rows, so the streams
of all members are coded side by side on the GPU.  Encode: the head kernels write every (scene, level, stage) stream's words into
one arena, a union level's stage as one contiguous slot, and one chunk-coder launch codes all chunks at the end.  Decode: per union
level one H2D copy of the four stages' chunk tables and payloads (v2_stage_tables), then per stage the head, one chunk decoder
launch over all members' rows and the symbol merge -- no CDF row leaves the GPU and no host coder runs.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import bitstream
from . import weights as W
from .codec import COORD_LIMIT, CTX_SHIFT, STAGE_SHIFT, UM_TILE_ROWS, GausPcgcCodec, KMap, Level, _ptr

Z_SHIFT = 42                      # z field of a voxel key (include/gpcgc.h)


def v2_stage_tables(streams: Sequence[Tuple[str, int, int, bytes]], row0: int = 0) -> Tuple[np.ndarray, np.ndarray, bytes]:
    """The chunk tables of one stage of a union level for gpc_chunk_decode_u16_ranges.  streams: per member scene, in union row
    order, (name, rows n at this level, the file's chunk size, its version-2 stream of this level and stage); the members' rows
    follow one another from row0.  Returns
      rows    u32[chunks + 1]  chunk boundaries: every member's rows cut by chunk_len(n, its chunk size), offset by its first row
      offsets u32[chunks + 1]  prefix sums of the chunks' u16 byte counts
      payload                  the members' chunk bytes without their u16 count headers, one after the other.
    A stream shorter than its count header, or whose counts do not sum to its length, raises ValueError naming the scene."""
    rows = [np.array([row0], dtype=np.int64)]
    cnts = [np.zeros(1, dtype=np.int64)]
    payload = []
    r = int(row0)
    for name, n, chunk, sb in streams:
        n = int(n)
        cl = GausPcgcCodec.chunk_len(n, int(chunk))
        chunks = (n + cl - 1) // cl
        if len(sb) < 2 * chunks:
            raise ValueError(f"{name}: truncated version-2 stream")
        cnt = np.frombuffer(sb, dtype="<u2", count=chunks).astype(np.int64)
        if int(cnt.sum()) != len(sb) - 2 * chunks:
            raise ValueError(f"{name}: corrupt version-2 stream (chunk byte counts)")
        rows.append(r + np.minimum(np.arange(1, chunks + 1, dtype=np.int64) * cl, n))
        cnts.append(cnt)
        payload.append(memoryview(sb)[2 * chunks:])
        r += n
    rows_a = np.concatenate(rows)
    offs = np.cumsum(np.concatenate(cnts))
    if int(rows_a[-1]) > 0xFFFFFFFF or int(offs[-1]) > 0xFFFFFFFF:
        raise ValueError("a union level's version-2 chunk table exceeds u32 rows or bytes")
    return rows_a.astype(np.uint32), offs.astype(np.uint32), b"".join(payload)


# ---------------------------------------------------------------------------------------------------------------- planner
@dataclass
class UnionPlan:
    scenes: List[int]                             # input indices, in z order (deepest scene first)
    tz: List[int]                                 # z translation of each, in leaf voxels (a multiple of 2^(D+1))
    rows: int = 0


def plan_unions(z_lo: Sequence[int], z_hi: Sequence[int], depths: Sequence[int], rows: Sequence[int], max_rows: int,
                limit: int = COORD_LIMIT) -> Tuple[List[UnionPlan], List[int]]:
    """Pure function of the scenes' leaf-voxel z extents, depths (the scale of the base level: its voxels are 2^depth leaves wide) and
    row counts.  Returns (unions, singles): every scene is in exactly one union or in `singles` (coded alone by the single-scene
    path: a scene whose translated extent or rows do not fit a union by itself).

    Within a union the scenes are stacked in order of decreasing depth (ties: input order); translations are multiples of 2^(D+1),
    consecutive scenes are more than 4 * 2^D voxels apart, every translated z lies in [-limit, limit], and the rows of a union sum to
    at most max_rows.  A new union starts when the next scene would overflow either."""
    n = len(depths)
    if not (len(z_lo) == len(z_hi) == len(rows) == n):
        raise ValueError("plan_unions: per-scene inputs differ in length")
    if n == 0:
        return [], []
    D = max(int(d) for d in depths)
    G = 1 << (D + 1)
    gap = 4 << D
    order = sorted(range(n), key=lambda s: (-int(depths[s]), s))
    unions: List[UnionPlan] = []
    singles: List[int] = []
    cur: Optional[UnionPlan] = None
    cursor = -limit

    def place(s: int, c: int) -> int:
        return -((int(z_lo[s]) - c) // G) * G                      # smallest multiple of G with z_lo + T >= c

    for s in order:
        lo, hi, r = int(z_lo[s]), int(z_hi[s]), int(rows[s])
        if cur is not None:
            t = place(s, cursor)
            if hi + t <= limit and cur.rows + r <= max_rows:
                cur.scenes.append(s)
                cur.tz.append(t)
                cur.rows += r
                cursor = hi + t + gap + 1
                continue
        t = place(s, -limit)
        if hi + t > limit or r > max_rows:
            singles.append(s)
            continue
        cur = UnionPlan([s], [t], r)
        unions.append(cur)
        cursor = hi + t + gap + 1
    return unions, singles


# ---------------------------------------------------------------------------------------------------------------- union levels
@dataclass
class ULevel:
    """one level of a union: the member scenes' rows one after the other (union order), per member its row range and kernel map"""
    keys: torch.Tensor
    occ: Optional[torch.Tensor]
    members: List[int]                            # positions in the union's scene list
    ranges: List[Tuple[int, int]]
    kmaps: Optional[List[KMap]] = None

    @property
    def n(self) -> int:
        return int(self.keys.shape[0])


def union_levels(levels: Sequence[Sequence[Level]], tz: Sequence[int]) -> Tuple[Dict[int, ULevel], Dict[int, int], Dict[int, int]]:
    """The union levels of the members of one union (plan_unions order, deepest first).  levels[j]: member j's pyramid, coarsest
    first (its base voxels are 2^len(levels[j]) leaves wide); tz[j]: its z translation in leaf voxels.  Returns (U, K, M):
      U[sg]  for sg = 1 .. D (1 = parents of the leaves): the members' levels at scale sg, keys translated by tz >> sg, one after the
             other, with each member's row range (kernel maps not built)
      K[sg]  for sg = 1 .. D - 1: the members with a level at scale sg + 1, i.e. those whose rows at scale sg are children (a prefix)
      M[sg]  their rows: the first M[sg] rows of U[sg]."""
    depths = [len(lv) for lv in levels]
    D = max(depths)
    U: Dict[int, ULevel] = {}
    for sg in range(1, D + 1):
        part = [j for j, d in enumerate(depths) if d >= sg]
        keys, occs, ranges, r = [], [], [], 0
        for j in part:
            lvl = levels[j][depths[j] - sg]
            keys.append(BatchCodec._translate(lvl.keys, tz[j] >> sg))
            occs.append(lvl.occ)
            ranges.append((r, r + lvl.n))
            r += lvl.n
        U[sg] = ULevel(torch.cat(keys), torch.cat(occs), part, ranges)
    K = {sg: sum(1 for d in depths if d >= sg + 1) for sg in range(1, D)}
    M = {sg: U[sg].ranges[K[sg] - 1][1] for sg in range(1, D)}
    return U, K, M


@dataclass
class Act:
    """activations of a union level: per scene fp32 rows (mma.sync / sparse families) or split rows (tcgen05 family).  f and s may be
    the same memory (an intermediate: each scene keeps its own format in its own rows)"""
    f: Optional[torch.Tensor]
    s: Optional[torch.Tensor]
    alias: bool = False


@dataclass
class _Scene:
    idx: int                                      # input position
    depth: int = 0
    levels: list = field(default_factory=list)    # encoder: the scene's own pyramid (single-scene frame), coarsest first
    shift: Optional[np.ndarray] = None            # encoder: _recentre's translation; decoder: decode()'s leaf translation
    base_xyz: Optional[np.ndarray] = None         # decoder: base voxels in the single-scene frame
    base_occ: Optional[np.ndarray] = None
    streams: Optional[List[bytes]] = None
    scale: float = 1.0
    tz: int = 0
    n_unique: int = 0                             # encoder: distinct voxels (the version-2 trailer's count)
    chunk: int = 0                                # decoder: the file's version-2 chunk size (0: version 1)
    name: str = ""                                # decoder: how errors name the scene


class BatchCodec:
    """Batched encode / decode over a GausPcgcCodec (its weights, kernel-family thresholds, thread pool and helpers)."""

    def __init__(self, codec: GausPcgcCodec):
        self.c = codec
        # rows of the largest level of a union (encoder: the scenes' finest coded levels; decoder: estimated as one row per stream
        # byte, since the rows are not known before they are decoded).  ~32 M rows keep a union's dense map and feature arrays
        # within ~70 GB.
        self.max_rows = 32_000_000
        self.last_stats: dict = {}
        self._v2_pin: Optional[torch.Tensor] = None   # decoder: pinned staging of a union level's version-2 chunk tables

    # ------------------------------------------------------------------ kernel maps of the scenes of a level
    def _kmaps(self, lv: ULevel) -> List[KMap]:
        """build_kmap's decision and pair stream for every member's row range, over one dense map of the whole level; the host reads
        the counts of all members at once (one synchronisation per pass instead of one per scene)"""
        c = self.c
        k = len(lv.ranges)
        n_level = lv.n
        dense = c.dense_map(lv.keys)
        big_rows = min(c.um_min_rows, c.sparse_min_rows)
        fam: List[Optional[str]] = []
        cnt32 = torch.zeros((max(k, 1), 2), dtype=torch.int32, device=c.dev)
        cnt64 = torch.zeros((max(k, 1), 2), dtype=torch.int64, device=c.dev)
        seg: List[Optional[torch.Tensor]] = [None] * k
        ws: List[Optional[torch.Tensor]] = [None] * k
        rowptr: List[Optional[torch.Tensor]] = [None] * k

        def count(j: int, f: str):
            r0, r1 = lv.ranges[j]
            n = r1 - r0
            if f == "v6":
                tr, _ = c._v6_config(n)
                seg[j] = c._empty((((n + tr - 1) // tr) * 126 + 1,), torch.int32)
                wb = c.lib.gpc_kmap_pairs_workspace_bytes(n, tr)
                ws[j] = c._ws(wb)
                c._call("gpc_kmap_pairs_count_range", _ptr(dense), n_level, r0, r1, tr, 8, _ptr(seg[j]), _ptr(cnt32[j]), _ptr(ws[j]), wb,
                        c._stream())
            elif f == "sparse":
                seg[j] = c._empty((int(c.lib.gpc_kmap_sparse_segments(n)) + 1,), torch.int32)
                rowptr[j] = c._empty((n + 1,), torch.int32)
                wb = c.lib.gpc_kmap_sparse_workspace_bytes(n)
                ws[j] = c._ws(wb)
                c._call("gpc_kmap_sparse_count_range", _ptr(dense), n_level, r0, r1, _ptr(seg[j]), _ptr(rowptr[j]), _ptr(cnt32[j]),
                        _ptr(ws[j]), wb, c._stream())
            else:
                tr = UM_TILE_ROWS
                seg[j] = c._empty((((n + tr - 1) // tr) * 126 + 1,), torch.int32)
                wb = c.lib.gpc_kmap_um_workspace_bytes(n, tr)
                ws[j] = c._ws(wb)
                c._call("gpc_kmap_um_count_range", _ptr(dense), n_level, r0, r1, tr, _ptr(seg[j]), _ptr(cnt64[j]), _ptr(ws[j]), wb,
                        c._stream())

        for j in range(k):
            r0, r1 = lv.ranges[j]
            f = "v6" if r1 - r0 < big_rows else None            # build_kmap: levels below both thresholds take the mma.sync conv
            fam.append(f)
            count(j, f or "um")
        c32, c64 = cnt32.tolist(), cnt64.tolist()
        again = []
        for j in range(k):
            if fam[j] is not None:
                continue
            r0, r1 = lv.ranges[j]
            n = r1 - r0
            density = c64[j][1] / max(n, 1)
            if n >= c.sparse_min_rows and 0 < c.sparse_max_density and density < c.sparse_max_density and n < 30_000_000:
                fam[j] = "sparse"
            elif n < c.um_min_rows:
                fam[j] = "v6"
            else:
                fam[j] = "um"
                continue
            count(j, fam[j])
            again.append(j)
        if again:
            c32 = cnt32.tolist()
        kms: List[KMap] = []
        for j in range(k):
            r0, r1 = lv.ranges[j]
            n = r1 - r0
            if fam[j] == "v6":
                tr, v6v = c._v6_config(n)
                n_pairs, n_real = c32[j]
                pairs = c._empty((max(n_pairs, 1),), torch.int64)
                c._call("gpc_kmap_pairs_fill_range", _ptr(dense), n_level, r0, r1, tr, _ptr(seg[j]), _ptr(pairs), n_pairs, c._stream())
                kms.append(KMap(seg[j], pairs, n_pairs, tr, n_real=n_real, v6_variant=v6v))
            elif fam[j] == "sparse":
                n_entries, n_strag = c32[j]
                pairs = c._empty((max(n_entries, 1),), torch.int64)
                c._call("gpc_kmap_sparse_fill_range", _ptr(dense), n_level, r0, r1, _ptr(seg[j]), _ptr(rowptr[j]), _ptr(ws[j]),
                        _ptr(pairs), n_entries, c._stream())
                km = KMap(seg[j], pairs, n_entries, 0, n_real=n + n_strag, sparse=True, rowptr=rowptr[j])
                km.contrib = c._empty((max(n_strag, 1), 32), torch.float32)
                kms.append(km)
            else:
                tr = UM_TILE_ROWS
                n_pairs, n_real = c64[j]
                nbr = c._empty((max(n_pairs, 1),), torch.int32)
                off = c._empty((max(n_pairs, 1),), torch.int32)
                c._call("gpc_kmap_um_fill_range", _ptr(dense), n_level, r0, r1, tr, _ptr(seg[j]), _ptr(nbr), _ptr(off), c._stream())
                km = KMap(seg[j], None, n_pairs, tr, n_real=n_real, um_rows=tr, pair_nbr=nbr, pair_off=off)
                starts = seg[j][::126].to(torch.int64)
                km.tile_order = torch.argsort(starts[1:] - starts[:-1], descending=True, stable=True).to(torch.int32)
                kms.append(km)
        return kms

    # ------------------------------------------------------------------ per-scene convs over union buffers
    def _new_act(self, n: int, kms: List[KMap], both: bool = False) -> Act:
        """an intermediate (each scene's own format in one buffer) or, with both, fp32 rows for all scenes + split rows for the
        tcgen05 scenes"""
        c = self.c
        if both:
            return Act(c._empty((n, 32), torch.float32), c._empty((n, 32), torch.int32) if any(k.um_rows for k in kms) else None)
        buf = c._empty((n, 32), torch.float32)
        return Act(buf, buf.view(torch.int32), alias=True)

    def _conv(self, x: Act, widx: int, lv: ULevel, n: int, k: int, out: Act, residual: Optional[Act] = None, relu: bool = False):
        """one conv on the first k members of lv, whose rows are the first n of the buffers"""
        c = self.c
        st = c._stream()
        for j in range(k):
            km = lv.kmaps[j]
            r0, r1 = lv.ranges[j]
            flags = 1 if relu else 0
            if km.um_rows:
                y = None if (out.alias or out.f is None) else out.f
                ys = out.s
                res = None
                if residual is not None:
                    res, flags = residual.s, flags | 2
                c._call("gpc_spconv_fwd_um_range", _ptr(x.s), _ptr(c.w.convs_um[widx]), _ptr(km.seg), _ptr(km.pair_nbr), _ptr(km.pair_off),
                        n, r0, r1, _ptr(km.tile_order), _ptr(res), flags, _ptr(y), _ptr(ys), st)
            elif km.sparse:
                c._call("gpc_spconv_sparse_fwd_range", _ptr(x.f), _ptr(c.w.convs_frag[widx]), _ptr(km.seg), _ptr(km.pairs), _ptr(km.rowptr),
                        n, r0, r1, km.n_pairs, _ptr(km.contrib), _ptr(residual.f if residual is not None else None), flags, _ptr(out.f), st)
            else:
                c._call("gpc_spconv_fwd_v6_range", _ptr(x.f), _ptr(c.w.convs_frag[widx]), _ptr(km.seg), _ptr(km.pairs), n, r0, r1,
                        km.tile_rows, _ptr(residual.f if residual is not None else None), flags, _ptr(out.f), km.v6_variant, st)

    def _stack(self, x: Act, ids, lv: ULevel, n: int, k: int, both: bool) -> Act:
        """Conv3d, ReLU, ResNet, ResNet (codec.GausPcgcCodec._res_stack) on the first k members of lv"""
        a = self._new_act(n, lv.kmaps)
        self._conv(x, ids[0], lv, n, k, a, relu=True)
        t = self._new_act(n, lv.kmaps)
        self._conv(a, ids[1], lv, n, k, t, relu=True)
        b = self._new_act(n, lv.kmaps)
        self._conv(t, ids[2], lv, n, k, b, residual=a, relu=True)
        self._conv(b, ids[3], lv, n, k, t, relu=True)
        out = self._new_act(n, lv.kmaps[:k], both=True) if both else Act(self.c._empty((n, 32), torch.float32), None)
        self._conv(t, ids[4], lv, n, k, out, residual=b, relu=True)
        return out

    @staticmethod
    def _runs(lv: ULevel, k: int):
        """maximal row ranges of consecutive members with the same activation format: (r0, r1, split?)"""
        runs = []
        for j in range(k):
            r0, r1 = lv.ranges[j]
            um = bool(lv.kmaps[j].um_rows)
            if runs and runs[-1][2] == um and runs[-1][1] == r0:
                runs[-1][1] = r1
            else:
                runs.append([r0, r1, um])
        return [tuple(r) for r in runs if r[1] > r[0]]

    def _level_features(self, parent: ULevel, child: ULevel, m: int, k: int, ck: torch.Tensor, cp: torch.Tensor):
        """prior stack on the parent level, target embedding and target stack on the first m rows (k members) of the child level;
        -> Act(fp32 rows, split rows of the tcgen05 scenes)"""
        c = self.c
        st = c._stream()
        f = self._new_act(parent.n, parent.kmaps)
        for r0, r1, um in self._runs(parent, len(parent.ranges)):
            c._call("gpc_embed_rows", _ptr(parent.occ) + r0, r1 - r0, _ptr(c.w.prior_emb), None if um else _ptr(f.f) + r0 * 128,
                    _ptr(f.s) + r0 * 128 if um else None, st)
        fp = self._stack(f, W.PRIOR_CONVS, parent, parent.n, len(parent.ranges), both=False)
        u0 = self._new_act(m, child.kmaps)
        for r0, r1, um in self._runs(child, k):
            c._call("gpc_gather_parent_add_octant", _ptr(fp.f), _ptr(cp) + r0 * 4, _ptr(ck) + r0 * 8, r1 - r0, _ptr(c.w.target_emb),
                    None if um else _ptr(u0.f) + r0 * 128, _ptr(u0.s) + r0 * 128 if um else None, st)
        return self._stack(u0, W.TARGET_CONVS, child, m, k, both=True)

    def _stage(self, u: Act, occ: torch.Tensor, i: int, child: ULevel, m: int, k: int) -> torch.Tensor:
        """context embedding + spatial_conv_s{i} of stage i -> fp32 rows for the head"""
        c = self.c
        if i == 0:
            f = Act(u.f, u.s)
        else:
            f = self._new_act(m, child.kmaps)
            for r0, r1, um in self._runs(child, k):
                c._call("gpc_add_ctx_embed", _ptr(u.f) + r0 * 128, _ptr(occ) + r0, CTX_SHIFT[i], _ptr(c.w.stage_emb[i]), r1 - r0,
                        None if um else _ptr(f.f) + r0 * 128, _ptr(f.s) + r0 * 128 if um else None, c._stream())
        c0, c1 = W.stage_convs(i)
        t = self._new_act(m, child.kmaps)
        self._conv(f, c0, child, m, k, t, relu=True)
        out = Act(c._empty((m, 32), torch.float32), None)
        self._conv(t, c1, child, m, k, out)
        return out.f

    def _begin(self):
        c = self.c
        self._launch0 = int(c.lib.gpc_launch_count())
        c._stream_h = torch.cuda.current_stream(c.dev).cuda_stream

    def _end(self, **stats):
        c = self.c
        c._stream_h = None
        self.last_stats = dict(stats, launches=int(c.lib.gpc_launch_count()) - self._launch0)

    @staticmethod
    def _translate(keys: torch.Tensor, dz: int) -> torch.Tensor:
        return keys + (dz << Z_SHIFT) if dz else keys

    # ------------------------------------------------------------------ encode
    def encode(self, xyz_list: List[torch.Tensor], gpu_chunk: int = 0) -> List[Tuple[np.ndarray, np.ndarray, List[bytes]]]:
        """-> per scene (base_xyz, base_occ, streams), exactly GausPcgcCodec.encode's for that scene alone.  gpu_chunk > 0: container
        version 2 -- the streams are compress_point_cloud(..., gpu_coder_chunk=gpu_chunk)'s, its trailer (bitstream.v2_trailer)
        included"""
        c = self.c
        results: List[Optional[tuple]] = [None] * len(xyz_list)

        def trail(streams: List[bytes], n_unique: int) -> List[bytes]:
            return streams + [bitstream.v2_trailer(gpu_chunk, n_unique)] if gpu_chunk else streams
        n_unions = 0
        self._begin()
        try:
            scenes = []
            for s, xyz in enumerate(xyz_list):
                sc = _Scene(s)
                xyz = xyz.contiguous()
                keys, meta = c.pack_keys(xyz)
                meta_h = meta.cpu().numpy()
                if meta_h[0] & 1:
                    raise ValueError(f"compress_point_clouds: scene {s} is not voxelised (integral) coordinates")
                if meta_h[0] & 2:
                    xyz, sc.shift = c._recentre(xyz)
                    keys, meta = c.pack_keys(xyz)
                    meta_h = meta.cpu().numpy()
                mm = meta_h[2:8].astype(np.uint32)
                leaf = c.sort_unique(keys, mm)
                sc.n_unique = int(leaf.shape[0])
                sc.levels = c.build_pyramid(leaf, mm.astype(np.int64))
                sc.depth = len(sc.levels)                     # the base voxels are 2^depth leaves wide
                sc.zr = (int(mm[2]) - (1 << 20), int(mm[5]) - (1 << 20))
                scenes.append(sc)
            multi = [sc for sc in scenes if sc.depth >= 2]
            unions, singles = plan_unions([sc.zr[0] for sc in multi], [sc.zr[1] for sc in multi], [sc.depth for sc in multi],
                                          [sc.levels[-1].n for sc in multi], self.max_rows)
            for sc in scenes:
                if sc.depth < 2:
                    results[sc.idx] = self._finish_base(sc, trail([], sc.n_unique))
            for j in singles:                              # a scene that fits no union: the single-scene path
                sc = multi[j]
                bx, bo, streams, _ = c.encode(xyz_list[sc.idx], gpu_chunk=gpu_chunk)
                self._begin_again()
                results[sc.idx] = (bx, bo, trail(streams, c.last_stats["n_unique"]))
            for up in unions:
                members = [multi[j] for j in up.scenes]
                for sc, t in zip(members, up.tz):
                    sc.tz = t
                for sc, streams in zip(members, self._encode_union(members, gpu_chunk)):
                    results[sc.idx] = self._finish_base(sc, trail(streams, sc.n_unique))
            n_unions = len(unions)
        finally:
            self._end(unions=n_unions)
        return results

    def _begin_again(self):
        """the single-scene path resets the codec's stream handle"""
        self.c._stream_h = torch.cuda.current_stream(self.c.dev).cuda_stream

    def _finish_base(self, sc: _Scene, streams: List[bytes]):
        """base level in the caller's coordinates (GausPcgcCodec.encode, end)"""
        c = self.c
        base = sc.levels[0]
        base_xyz = c._empty((base.n, 3), torch.int32)
        c._call("gpc_unpack_keys_i32", _ptr(base.keys), base.n, _ptr(base_xyz), c._stream())
        base_xyz_h = base_xyz.cpu().numpy()
        if sc.shift is not None:
            depth = sc.depth
            assert not np.any(sc.shift % (1 << depth)), "translation must be a multiple of 2^depth"
            moved = base_xyz_h.astype(np.int64) + (sc.shift >> depth)
            if np.abs(moved).max(initial=0) >= (1 << 31):
                raise ValueError("base coordinates do not fit int32")
            base_xyz_h = moved.astype(np.int32)
        return base_xyz_h, base.occ.cpu().numpy(), streams

    def _encode_union(self, members: List[_Scene], gpu_chunk: int = 0) -> List[List[bytes]]:
        c = self.c
        D = max(sc.depth for sc in members)
        U, K, M = union_levels([sc.levels for sc in members], [sc.tz for sc in members])
        for sg in range(1, D + 1):
            # scale 1 is only ever a child level: the members with deeper levels (all of them: base-only scenes are not in unions)
            U[sg].kmaps = self._kmaps(U[sg])
        streams: List[List[Optional[bytes]]] = [[None] * (4 * (sc.depth - 1)) for sc in members]
        futs = []
        if gpu_chunk:
            # version 2: the (scene, level, stage) streams in the order (union level, stage, member) in the codec's coder arena, so
            # that the words of one stage of a union level (its first M rows, member after member) are one contiguous slot
            first = {}
            seg_rows: List[int] = []
            for sg in range(1, D):
                for i in range(4):
                    first[sg, i] = len(seg_rows)
                    seg_rows += [r1 - r0 for r0, r1 in U[sg].ranges[:K[sg]]]
            c._chunk_begin(seg_rows, gpu_chunk)
        else:
            pin = c._pin(sum(M.values()) * 16 + 4096 * 4 * D)
        cursor = 0
        for sg in range(1, D):                              # finest first: its range coding overlaps the coarser levels' GPU work
            parent, child = U[sg + 1], U[sg]
            k, m = K[sg], M[sg]
            ck, cp = c.expand(parent, m)
            u = self._level_features(parent, child, m, k, ck, cp)
            occ = child.occ
            hosts = []
            for i in range(4):
                t = self._stage(u, occ, i, child, m, k)
                if gpu_chunk:
                    a = c._coder_starts[first[sg, i]]
                    lohi_d = c._coder_arena[a:a + m]
                else:
                    lohi_d = c._empty((m,), torch.int32)
                w1, b1, w2, b2 = c.w.head[i]
                c._call("gpc_head_cdf_sym", _ptr(t), m, _ptr(w1), _ptr(b1), _ptr(w2), _ptr(b2), W.STAGE_ALPHABETS[i], _ptr(occ),
                        STAGE_SHIFT[i], _ptr(lohi_d), None, None, c._stream())
                if gpu_chunk:
                    continue                               # coded with every other stream of the union at the end
                start = (cursor + 63) // 64 * 64
                cursor = start + m * 4
                h = pin[start:start + m * 4].view(torch.int32)
                h.copy_(lohi_d, non_blocking=True)
                hosts.append(h)
            if gpu_chunk:
                continue
            ready = torch.cuda.Event(blocking=True)
            ready.record(torch.cuda.current_stream(c.dev))
            for j in range(k):
                sc = members[child.members[j]]
                r0, r1 = child.ranges[j]
                g = sc.depth - 1 - sg
                for i in range(4):
                    futs.append((child.members[j], 4 * g + i,
                                 c.pool.submit(c._ac_encode_lohi, hosts[i].numpy()[r0:r1].view(np.uint32), ready)))
        if gpu_chunk:
            coded = c._chunk_finish(gpu_chunk)             # one launch codes every chunk of every scene's streams
            for sg in range(1, D):
                child = U[sg]
                for i in range(4):
                    for j in range(K[sg]):
                        sc = members[child.members[j]]
                        streams[child.members[j]][4 * (sc.depth - 1 - sg) + i] = coded[first[sg, i] + j]
        for j, q, f in futs:
            streams[j][q] = f.result()
        return streams

    # ------------------------------------------------------------------ decode
    def decode(self, files: List[tuple], sorted_rows: bool = False, names: Optional[Sequence[str]] = None) -> List[torch.Tensor]:
        """files: per scene (posQ, base_xyz, base_occ, streams) of container version 1, or (posQ, base_xyz, base_occ, streams, chunk)
        with the streams of a version-2 file (trailer removed, bitstream.split_v2) and its chunk size; all files of one call are of
        one container version.  -> per scene GausPcgcCodec.decode's rows.  names: how errors name the scenes (default "scene i")."""
        c = self.c
        out: List[Optional[torch.Tensor]] = [None] * len(files)
        chunks = [int(f[4]) if len(f) > 4 else 0 for f in files]
        if any(chunks) and not all(chunks):
            raise ValueError("container version 1 and version 2 files cannot be decoded in one call")
        self._begin()
        n_unions = 0
        self._round_trips = 0
        try:
            scenes = []
            for s, (posQ, bx, bo, streams) in enumerate(f[:4] for f in files):
                if len(streams) % 4:
                    raise ValueError("stream count must be a multiple of 4 (one group per octree level)")
                sc = _Scene(s, streams=streams, scale=float(posQ), chunk=chunks[s], name=names[s] if names else f"scene {s}")
                sc.depth = L = len(streams) // 4 + 1
                bx_h = np.array(bx, dtype=np.int32).reshape(-1, 3)
                sc.base_occ = np.array(bo, dtype=np.uint8).reshape(-1)
                if bx_h.shape[0] != sc.base_occ.shape[0]:
                    raise ValueError(f"scene {s}: base coordinates and occupancy differ in length")
                # the single-scene decoder's frame (GausPcgcCodec.decode): translated when some leaf would leave the key fields
                if bx_h.size and (int(np.abs(bx_h.astype(np.int64)).max()) + 1) << L > COORD_LIMIT:
                    b64 = bx_h.astype(np.int64)
                    t = (b64.min(axis=0) + b64.max(axis=0) + 1) // 2
                    if max(int(-(b64.min(axis=0) - t).min()) << L, ((int((b64.max(axis=0) - t).max()) + 1) << L) - 1) <= COORD_LIMIT:
                        bx_h = (b64 - t).astype(np.int32)
                        sc.shift = t << L
                sc.base_xyz = bx_h
                scenes.append(sc)
            multi, zlo, zhi, est = [], [], [], []
            for sc in scenes:
                b = sc.base_xyz.astype(np.int64)
                fits = b.size and (max(int(-b.min()) << sc.depth, ((int(b.max()) + 1) << sc.depth) - 1) <= COORD_LIMIT)
                if sc.depth >= 2 and fits:
                    multi.append(sc)
                    zlo.append(int(b[:, 2].min()) << sc.depth)
                    zhi.append(((int(b[:, 2].max()) + 1) << sc.depth) - 1)
                    est.append(sum(len(x) for x in sc.streams))
                else:
                    out[sc.idx] = self._single_decode(files[sc.idx], sorted_rows, sc.name)
            unions, singles = plan_unions(zlo, zhi, [sc.depth for sc in multi], est, self.max_rows)
            for j in singles:
                out[multi[j].idx] = self._single_decode(files[multi[j].idx], sorted_rows, multi[j].name)
            for up in unions:
                members = [multi[j] for j in up.scenes]
                for sc, t in zip(members, up.tz):
                    sc.tz = t
                for sc, rows in zip(members, self._decode_union(members, sorted_rows)):
                    out[sc.idx] = rows
            n_unions = len(unions)
        finally:
            # stage_round_trips: how often the union decoder waited for a stage's CDF rows on the host (version 1: four per union
            # level; version 2 decodes on the GPU: none).  Child counts and kernel-map sizes are read back either way.
            self._end(unions=n_unions, stage_round_trips=self._round_trips)
        return out

    def _single_decode(self, f, sorted_rows: bool, name: str) -> torch.Tensor:
        posQ, bx, bo, streams = f[:4]
        chunk = int(f[4]) if len(f) > 4 else 0
        try:
            rows = self.c.decode(bx, bo, streams, scale=float(posQ), sorted_rows=sorted_rows, gpu_chunk=chunk)
        except ValueError as e:
            if not chunk:
                raise
            raise ValueError(f"{name}: {e}") from e                # a corrupt version-2 stream, named as the union decoder names it
        finally:
            self._begin_again()
        return rows

    def _base_level(self, sc: _Scene) -> Tuple[torch.Tensor, torch.Tensor]:
        """the scene's base voxels as keys in (z,y,x) order, translated to its union slot, and their occupancy in that order (the
        reference stores the base level in torchsparse's emission order; decode() sorts it the same way)"""
        b = sc.base_xyz.astype(np.int64) + (1 << 20)
        b[:, 2] += sc.tz >> sc.depth
        keys = (b[:, 2] << 42) | (b[:, 1] << 21) | b[:, 0]
        order = np.argsort(keys, kind="stable")
        return (torch.from_numpy(keys[order]).to(self.c.dev),
                torch.from_numpy(np.ascontiguousarray(sc.base_occ[order])).to(self.c.dev))

    def _counts(self, lv: ULevel) -> List[int]:
        """children of every member of a level: one read-back of the cumulative set-bit counts at the members' boundaries"""
        c = self.c
        if not hasattr(c, "_pop8"):
            c._popcount(lv.occ[:1])
        cum = torch.cumsum(c._pop8[lv.occ.long()], 0)
        ends = torch.tensor([r1 - 1 for _, r1 in lv.ranges], dtype=torch.int64, device=c.dev)
        e = cum[ends].tolist()
        return [int(a - b) for a, b in zip(e, [0] + e[:-1])]

    def _v2_upload(self, tabs: List[Tuple[np.ndarray, np.ndarray, bytes]]) -> Tuple[torch.Tensor, List[tuple]]:
        """the four stages' chunk tables and payloads of a union level -> device, in ONE copy from pinned staging.  Returns the
        device buffer (the caller keeps it until the level's decoder launches are enqueued) and per stage the device addresses
        (payload, offsets, rows) and its chunk count for gpc_chunk_decode_u16_ranges.

        The staging buffer is rewritten once per level.  That is safe because the decoder calls this right after _counts, whose
        read-back synchronises the stream: the previous level's copy out of this buffer has completed by then."""
        c = self.c
        place, total = [], 0
        for rows, offs, payload in tabs:
            p = []
            for nbytes in (len(payload), offs.nbytes, rows.nbytes):
                p.append(total)
                total = (total + nbytes + 15) // 16 * 16
            place.append(p)
        if self._v2_pin is None or self._v2_pin.numel() < total:
            self._v2_pin = torch.empty(int(total * 1.5) + 4096, dtype=torch.uint8, pin_memory=True)
        host = self._v2_pin.numpy()
        for (rows, offs, payload), (a, b, r) in zip(tabs, place):
            host[a:a + len(payload)] = np.frombuffer(payload, dtype=np.uint8)
            host[b:b + offs.nbytes] = offs.view(np.uint8)
            host[r:r + rows.nbytes] = rows.view(np.uint8)
        dev = c._empty((max(total, 16),), torch.uint8)
        dev[:total].copy_(self._v2_pin[:total], non_blocking=True)
        base = dev.data_ptr()
        return dev, [(base + a, base + b, base + r, int(rows.shape[0]) - 1) for (rows, _, _), (a, b, r) in zip(tabs, place)]

    def _decode_union(self, members: List[_Scene], sorted_rows: bool) -> List[torch.Tensor]:
        c = self.c
        D = max(sc.depth for sc in members)
        bases = [self._base_level(sc) for sc in members]

        def with_bases(keys, occ, ranges, mem, sg):
            """append the members whose base level is at scale sg (they come after the deeper members' rows)"""
            ks, os_, r = [keys] if keys is not None else [], [occ] if occ is not None else [], ranges[-1][1] if ranges else 0
            ranges, mem = list(ranges), list(mem)
            for j, sc in enumerate(members):
                if sc.depth == sg:
                    bk, bo = bases[j]
                    ks.append(bk)
                    os_.append(bo)
                    ranges.append((r, r + bk.shape[0]))
                    mem.append(j)
                    r += bk.shape[0]
            return ULevel(torch.cat(ks), torch.cat(os_) if os_ else None, mem, ranges)

        cur = with_bases(None, None, [], [], D)
        cur.kmaps = self._kmaps(cur)
        Lps = [a + 1 for a in W.STAGE_ALPHABETS]
        v2 = members[0].chunk > 0                            # decode() admits one container version per call
        for sg in range(D - 1, 0, -1):
            cnt = self._counts(cur)                          # synchronises the stream: see _v2_upload
            m = sum(cnt)
            k = len(cur.ranges)
            if v2:
                # every member of cur has children; their rows of the child level follow one another from 0.  v2_dev holds the
                # uploaded tables until the next level replaces it, after the stream has passed this level's decoder launches
                own = [members[j] for j in cur.members]
                v2_dev, tabs = self._v2_upload([v2_stage_tables([(sc.name, n_, sc.chunk, sc.streams[4 * (sc.depth - 1 - sg) + i])
                                                                 for sc, n_ in zip(own, cnt)]) for i in range(4)])
            ck, cp = c.expand(cur, m)
            ranges, r = [], 0
            for n_ in cnt:
                ranges.append((r, r + n_))
                r += n_
            child = with_bases(ck, None, ranges, cur.members, sg)
            child.kmaps = self._kmaps(child)
            u = self._level_features(cur, child, m, k, ck, cp)
            occ = torch.zeros(m, dtype=torch.uint8, device=c.dev)
            if v2:
                for i in range(4):
                    t = self._stage(u, occ, i, child, m, k)
                    cdf_d = c._empty((m, Lps[i]), torch.int16)
                    w1, b1, w2, b2 = c.w.head[i]
                    c._call("gpc_head_cdf", _ptr(t), m, _ptr(w1), _ptr(b1), _ptr(w2), _ptr(b2), W.STAGE_ALPHABETS[i], _ptr(cdf_d), None,
                            c._stream())
                    sym_d = c._empty((m,), torch.uint8)
                    in_p, offs_p, rows_p, n_chunks = tabs[i]
                    c._call("gpc_chunk_decode_u16_ranges", _ptr(cdf_d), Lps[i], in_p, offs_p, rows_p, n_chunks, m, _ptr(sym_d), c._stream())
                    c._call("gpc_merge_symbol", _ptr(occ), m, STAGE_SHIFT[i], _ptr(sym_d), c._stream())
                child.occ = torch.cat([occ] + [bases[j][1] for j in child.members[k:]]) if child.n > m else occ
                cur = child
                continue
            if c._pinned_dec is None or c._pinned_dec.numel() < m * 40:
                c._pinned_dec = torch.empty(int(m * 40 * 1.5) + 4096, dtype=torch.uint8, pin_memory=True)
            pin = c._pinned_dec
            for i in range(4):
                t = self._stage(u, occ, i, child, m, k)
                cdf_d = c._empty((m, Lps[i]), torch.int16)
                w1, b1, w2, b2 = c.w.head[i]
                c._call("gpc_head_cdf", _ptr(t), m, _ptr(w1), _ptr(b1), _ptr(w2), _ptr(b2), W.STAGE_ALPHABETS[i], _ptr(cdf_d), None,
                        c._stream())
                cdf_h = pin[:m * Lps[i] * 2].view(torch.int16).view(m, Lps[i])
                cdf_h.copy_(cdf_d, non_blocking=True)
                torch.cuda.current_stream(c.dev).synchronize()
                self._round_trips += 1
                sym_h = pin[m * 36:m * 37]
                cdf_np, sym_np = cdf_h.numpy().view(np.uint16), sym_h.numpy()
                jobs = []
                for j in range(k):
                    sc = members[child.members[j]]
                    r0, r1 = child.ranges[j]
                    if r1 > r0:
                        g = sc.depth - 1 - sg
                        jobs.append(c.pool.submit(c._ac_decode, cdf_np[r0:r1], sc.streams[4 * g + i], sym_np[r0:r1]))
                for f in jobs:
                    f.result()
                sym_d = sym_h.to(c.dev, non_blocking=True)
                c._call("gpc_merge_symbol", _ptr(occ), m, STAGE_SHIFT[i], _ptr(sym_d), c._stream())
            child.occ = torch.cat([occ] + [bases[j][1] for j in child.members[k:]]) if child.n > m else occ
            cur = child
        # leaves: per scene, its rows back in the single-scene frame, then decode()'s output arithmetic
        cnt = self._counts(cur)
        outs: List[Optional[torch.Tensor]] = [None] * len(members)
        for j, (r0, r1) in enumerate(cur.ranges):
            sc = members[cur.members[j]]
            keys = self._translate(cur.keys[r0:r1], -(sc.tz >> 1))
            n_pts = cnt[j]
            rows = c._empty((n_pts, 3), torch.float32)
            k_scale = sc.scale if sc.shift is None else 1.0
            if sorted_rows:
                ckk, _ = c.expand(Level(keys, cur.occ[r0:r1], r1 - r0), n_pts)
                c._call("gpc_unpack_keys_f32", _ptr(ckk), n_pts, k_scale, _ptr(rows), c._stream())
            else:
                ws_b = c.lib.gpc_expand_workspace_bytes(r1 - r0)
                ws = c._ws(ws_b)
                c._call("gpc_expand_leaves_f32", _ptr(keys), _ptr(cur.occ[r0:r1]), r1 - r0, n_pts, k_scale, _ptr(rows), _ptr(ws), ws_b,
                        c._stream())
            if sc.shift is not None:
                rows += torch.tensor(sc.shift, dtype=torch.float32, device=c.dev)
                if sc.scale != 1.0:
                    rows *= sc.scale
            outs[cur.members[j]] = rows
        return outs
