"""Training of GausPcgc checkpoints on the GPU, on the codec's own geometry and conv kernels.

    SparseConvFn   autograd of one 5^3 sparse conv on any of the codec's three conv families (the KMap's): forward the family's
                   kernel, input gradient the same kernel with the mirrored, transposed weights W'[k] = W[124 - k]^T (a submanifold
                   map is symmetric: nbr_k(o) = i exactly when nbr_{124-k}(i) = o), weight gradient the family's (csrc/spconv_grad.cu):
                     mma.sync  gpc_spconv_fwd_v6, gpc_spconv_wgrad_v6 (or gpc_spconv_wgrad_v6_balanced on levels of at least
                               GausPcgcNet.wgrad_balanced_min_rows rows)
                     sparse    gpc_spconv_sparse_fwd, gpc_spconv_wgrad_sparse
                     tcgen05   gpc_spconv_fwd_um on split rows (gpc_rows_split), gpc_spconv_wgrad_um
    WeightPack     one conv weight's packs (mma.sync fragments, tcgen05 operand, and their mirrors), built once per forward pass
                   and shared by every conv on every level
    GausPcgcNet    the model of SURVEY.md Appendix A as an nn.Module whose state_dict() is the reference layout
                   (weights.reference_layout); forward(xyz) returns the code length of the file's occupancy streams under the
                   coder's probabilities; forward_batch(patches) the same for many patches, run as union octrees (batch.py)
    partition      kd-tree patches (median split along the longest axis), the patching of the reference's dataset.py
    train          Adam over minibatches of patches, checkpoints in the reference layout

The geometry (pyramid, children, kernel maps) comes from GausPcgcCodec exactly as the encoder builds it, so a checkpoint trained here
is trained on the voxels, row orders and conv offsets it is later coded with: it loads with pcc_utils.compress_point_cloud unchanged.
GausPcgcNet.conv_families picks the conv kernels: "v6" (the default) runs every level on the mma.sync family, "codec" runs every
level on the family the codec codes it with (GausPcgcCodec.build_kmap's rule: mma.sync below 150 K rows, the sparse conv or the
tcgen05 conv above), so a network trains on the very kernels and summation orders that will code its levels.

Determinism: the same seed, inputs and initial weights give a bit-identical checkpoint.  The convs sum in an order fixed by the map,
and the torch backward steps that would accumulate with atomics (embedding rows, the children -> parent gather) are written as
fixed-order sums instead.  No process-wide torch flag is touched.
"""
from __future__ import annotations

import time
from typing import Callable, Dict, Iterator, List, Optional, Sequence, Tuple, Union

import numpy as np
import torch
from torch import nn

from . import _lib
from . import weights as W
from .batch import plan_unions, union_levels
from .codec import CTX_SHIFT, STAGE_MASK, STAGE_SHIFT, GausPcgcCodec, KMap, Level, _ptr

# the 27 offsets of a 3^3 kernel at their K = 5 indices ((dz+2)*5 + (dy+2))*5 + (dx+2), as DeviceWeights places them
K5_OF_K3 = tuple(((dz + 2) * 5 + (dy + 2)) * 5 + (dx + 2) for dz in (-1, 0, 1) for dy in (-1, 0, 1) for dx in (-1, 0, 1))


def _stream(dev: torch.device):
    return torch.cuda.current_stream(dev).cuda_stream


def pack_frag(W125: torch.Tensor) -> torch.Tensor:
    """W [125,32,32] fp32 -> the mma.sync A fragments of W^T (gpc_spconv_pack_weights_frag, 512 000 bytes)"""
    Wa = torch.empty_like(W125)
    _lib.check(_lib.load().gpc_spconv_pack_weights_frag(_ptr(W125), 1, _ptr(Wa), _stream(W125.device)), "gpc_spconv_pack_weights_frag")
    return Wa


def conv_v6(x: torch.Tensor, Wa: torch.Tensor, km: KMap) -> torch.Tensor:
    """y = sum_k x[nbr_k(o)] . W[k] over the level's mma.sync pair stream (no residual, no activation)"""
    y = torch.empty_like(x)
    _lib.check(_lib.load().gpc_spconv_fwd_v6(_ptr(x), _ptr(Wa), _ptr(km.seg), _ptr(km.pairs), x.shape[0], km.tile_rows, None, 0, _ptr(y),
                                             km.v6_variant, _stream(x.device)), "gpc_spconv_fwd_v6")
    return y


def pack_um(W125: torch.Tensor) -> torch.Tensor:
    """W [125,32,32] fp32 -> the tcgen05 conv's A operand of W^T (gpc_spconv_pack_weights_um, 512 000 bytes)"""
    Wp = torch.empty_like(W125)
    _lib.check(_lib.load().gpc_spconv_pack_weights_um(_ptr(W125), 1, _ptr(Wp), _stream(W125.device)), "gpc_spconv_pack_weights_um")
    return Wp


def conv_sparse(x: torch.Tensor, Wa: torch.Tensor, km: KMap) -> torch.Tensor:
    """the same conv on a sparse level's map (gpc_spconv_sparse_fwd).  The stragglers' products go through km.contrib, the one
    scratch every conv on the level shares, forward and backward alike: that is safe only because they all run in order on one
    stream (the current one), each rewriting contrib completely before it reads it back."""
    y = torch.empty_like(x)
    _lib.check(_lib.load().gpc_spconv_sparse_fwd(_ptr(x), _ptr(Wa), _ptr(km.seg), _ptr(km.pairs), _ptr(km.rowptr), x.shape[0], km.n_pairs,
                                                 _ptr(km.contrib), None, 0, _ptr(y), _stream(x.device)), "gpc_spconv_sparse_fwd")
    return y


def conv_um(x: torch.Tensor, Wp: torch.Tensor, km: KMap) -> torch.Tensor:
    """the same conv on a tcgen05 level's map (gpc_spconv_fwd_um): x fp32 is split into bf16 hi / lo rows first, y is fp32"""
    lib, st, n = _lib.load(), _stream(x.device), x.shape[0]
    xs = torch.empty((n, 32), dtype=torch.int32, device=x.device)
    _lib.check(lib.gpc_rows_split(_ptr(x), n, _ptr(xs), st), "gpc_rows_split")
    y = torch.empty_like(x)
    _lib.check(lib.gpc_spconv_fwd_um(_ptr(xs), _ptr(Wp), _ptr(km.seg), _ptr(km.pair_nbr), _ptr(km.pair_off), n, km.um_rows,
                                     _ptr(km.tile_order), None, 0, _ptr(y), None, 0, 0, st), "gpc_spconv_fwd_um")
    return y


def kmap_family(km: KMap) -> str:
    """"v6" (mma.sync), "sparse" or "um" (tcgen05): the conv family a kernel map was built for"""
    return "um" if km.um_rows else ("sparse" if km.sparse else "v6")


def conv_dgrad(dy: torch.Tensor, W125: torch.Tensor, km: KMap) -> torch.Tensor:
    """dx = sum_k dy[nbr_{124-k}(i)] . W[124-k]^T: the family's forward conv with W'[k] = W[124 - k]^T"""
    Wm = W125.flip(0).transpose(1, 2).contiguous()
    if km.um_rows:
        return conv_um(dy, pack_um(Wm), km)
    if km.sparse:
        return conv_sparse(dy, pack_frag(Wm), km)
    return conv_v6(dy, pack_frag(Wm), km)


def conv_wgrad(x: torch.Tensor, dy: torch.Tensor, km: KMap, balanced: bool = False) -> torch.Tensor:
    """dW[k] = sum over the pairs (o, i) of offset k of x[i]^T dy[o]  ->  fp32 [125,32,32], by the map's family: gpc_spconv_wgrad_um
    and gpc_spconv_wgrad_sparse on tcgen05 and sparse maps; on mma.sync maps gpc_spconv_wgrad_v6 (split by tiles), or with
    balanced gpc_spconv_wgrad_v6_balanced (the work split by pairs, for big levels)"""
    lib = _lib.load()
    n = x.shape[0]
    dW = torch.empty((125, 32, 32), dtype=torch.float32, device=x.device)
    if km.um_rows:
        ws_b = int(lib.gpc_spconv_wgrad_um_workspace_bytes(n, km.um_rows, km.n_pairs))
        ws = torch.empty(max(ws_b, 256), dtype=torch.uint8, device=x.device)
        _lib.check(lib.gpc_spconv_wgrad_um(_ptr(x), _ptr(dy), _ptr(km.seg), _ptr(km.pair_nbr), _ptr(km.pair_off), n, km.um_rows,
                                           km.n_pairs, _ptr(dW), _ptr(ws), ws_b, _stream(x.device)), "gpc_spconv_wgrad_um")
        return dW
    if km.sparse:
        ws_b = int(lib.gpc_spconv_wgrad_sparse_workspace_bytes(n, km.n_pairs))
        ws = torch.empty(max(ws_b, 256), dtype=torch.uint8, device=x.device)
        _lib.check(lib.gpc_spconv_wgrad_sparse(_ptr(x), _ptr(dy), _ptr(km.seg), _ptr(km.pairs), _ptr(km.rowptr), n, km.n_pairs,
                                               _ptr(dW), _ptr(ws), ws_b, _stream(x.device)), "gpc_spconv_wgrad_sparse")
        return dW
    if balanced:
        ws_b = int(lib.gpc_spconv_wgrad_balanced_workspace_bytes(n, km.tile_rows, km.n_pairs))
        ws = torch.empty(max(ws_b, 256), dtype=torch.uint8, device=x.device)
        _lib.check(lib.gpc_spconv_wgrad_v6_balanced(_ptr(x), _ptr(dy), _ptr(km.seg), _ptr(km.pairs), n, km.tile_rows, km.n_pairs, _ptr(dW),
                                                    _ptr(ws), ws_b, _stream(x.device)), "gpc_spconv_wgrad_v6_balanced")
        return dW
    ws_b = int(lib.gpc_spconv_wgrad_workspace_bytes(n, km.tile_rows))
    ws = torch.empty(max(ws_b, 256), dtype=torch.uint8, device=x.device)
    _lib.check(lib.gpc_spconv_wgrad_v6(_ptr(x), _ptr(dy), _ptr(km.seg), _ptr(km.pairs), n, km.tile_rows, _ptr(dW), _ptr(ws), ws_b,
                                       _stream(x.device)), "gpc_spconv_wgrad_v6")
    return dW


class WeightPack:
    """One conv weight (a [125|27,32,32] parameter) prepared for the kernels: W125, its forward fragment pack (mma.sync and sparse
    convs), and, each built on first use, the tcgen05 operand pack and the packs of the mirrored weights W125.flip(0).transpose(1, 2)
    that the backward passes use.  Built once per forward pass of the network, so every conv on every level reuses the same bytes
    the per-call packs would have been."""

    def __init__(self, Wk: torch.Tensor, wgrad_balanced_min_rows: Optional[int] = None):
        self.W125 = _to125(Wk.detach())
        self.fwd = pack_frag(self.W125)
        self._mirror: Optional[torch.Tensor] = None
        self._um: Optional[torch.Tensor] = None
        self._mirror_um: Optional[torch.Tensor] = None
        self.wgrad_balanced_min_rows = wgrad_balanced_min_rows     # None: every level takes gpc_spconv_wgrad_v6

    def mirror(self) -> torch.Tensor:
        if self._mirror is None:
            self._mirror = pack_frag(self.W125.flip(0).transpose(1, 2).contiguous())
        return self._mirror

    def um(self) -> torch.Tensor:
        if self._um is None:
            self._um = pack_um(self.W125)
        return self._um

    def mirror_um(self) -> torch.Tensor:
        if self._mirror_um is None:
            self._mirror_um = pack_um(self.W125.flip(0).transpose(1, 2).contiguous())
        return self._mirror_um

    def conv(self, x: torch.Tensor, km: KMap, mirrored: bool = False) -> torch.Tensor:
        """x through the conv of km's family with these weights (mirrored: with W'[k] = W[124 - k]^T, the input gradient)"""
        if km.um_rows:
            return conv_um(x, self.mirror_um() if mirrored else self.um(), km)
        Wa = self.mirror() if mirrored else self.fwd
        return conv_sparse(x, Wa, km) if km.sparse else conv_v6(x, Wa, km)


class SparseConvFn(torch.autograd.Function):
    """y = conv(x, W) on the kernel map km (a KMap of any family: mma.sync, sparse or tcgen05, fp32 rows in and out); W is
    [125,32,32] or [27,32,32] (kernel_size 3: the 27 matrices go to their K = 5 offsets, where the map holds the only present
    neighbours, and their gradient is gathered back).  pack: W's WeightPack (built from W when not given)."""

    @staticmethod
    def forward(ctx, x: torch.Tensor, Wk: torch.Tensor, km: KMap, pack: Optional[WeightPack] = None):
        if (km.pairs is None) == (km.um_rows == 0):
            raise _lib.GpcError("SparseConvFn needs a kernel map from GausPcgcCodec.build_kmap")
        x = x.contiguous()
        pack = pack if pack is not None else WeightPack(Wk)
        ctx.km, ctx.k3, ctx.pack = km, Wk.shape[0] == 27, pack
        ctx.save_for_backward(x)
        return pack.conv(x, km)

    @staticmethod
    def backward(ctx, dy: torch.Tensor):
        (x,) = ctx.saved_tensors
        pack, km = ctx.pack, ctx.km
        dy = dy.contiguous()
        dx = pack.conv(dy, km, mirrored=True) if ctx.needs_input_grad[0] else None
        dW = None
        if ctx.needs_input_grad[1]:
            lim = pack.wgrad_balanced_min_rows
            dW = conv_wgrad(x, dy, km, balanced=lim is not None and x.shape[0] >= lim)      # (balanced: mma.sync maps only)
            if ctx.k3:
                dW = dW[torch.tensor(K5_OF_K3, device=dW.device)]
        return dx, dW, None, None


def _to125(Wk: torch.Tensor) -> torch.Tensor:
    if Wk.shape[0] == 125:
        return Wk.contiguous()
    full = torch.zeros((125, 32, 32), dtype=Wk.dtype, device=Wk.device)
    full[torch.tensor(K5_OF_K3, device=Wk.device)] = Wk
    return full


class EmbedFn(torch.autograd.Function):
    """table[idx]; the table's gradient is one_hot(idx)^T @ grad as one fp64 matrix product (a fixed summation order, where
    torch's embedding backward accumulates rows with atomics)"""

    @staticmethod
    def forward(ctx, table: torch.Tensor, idx: torch.Tensor):
        ctx.save_for_backward(idx)
        ctx.rows = table.shape[0]
        return table[idx]

    @staticmethod
    def backward(ctx, g: torch.Tensor):
        (idx,) = ctx.saved_tensors
        oh = (idx[:, None] == torch.arange(ctx.rows, device=idx.device)[None, :]).to(torch.float64)
        return (oh.t() @ g.to(torch.float64)).to(g.dtype), None


class ChildGatherFn(torch.autograd.Function):
    """children's rows of the parents' features, F[parent]; the gradient of a parent is the sum of its <= 8 children's, added in
    octant order (torch's index_select backward is an atomic index_add_)"""

    @staticmethod
    def forward(ctx, f: torch.Tensor, parent: torch.Tensor, octant: torch.Tensor):
        n_child = parent.shape[0]
        slot = torch.full((f.shape[0] * 8,), n_child, dtype=torch.int64, device=f.device)
        slot[parent * 8 + octant] = torch.arange(n_child, device=f.device)
        ctx.save_for_backward(slot.view(-1, 8))
        return f[parent]

    @staticmethod
    def backward(ctx, g: torch.Tensor):
        (slot,) = ctx.saved_tensors
        gp = torch.cat([g, g.new_zeros((1, g.shape[1]))])
        acc = gp[slot[:, 0]]
        for o in range(1, 8):
            acc = acc + gp[slot[:, o]]
        return acc, None, None


class _Geometry:
    """what GausPcgcCodec reads of its weights when it only builds geometry: the kernel size of the map"""

    def __init__(self, kernel_size: int):
        self.kernel_size = kernel_size


def _octant(keys: torch.Tensor) -> torch.Tensor:
    return (keys & 1) | (((keys >> 21) & 1) << 1) | (((keys >> 42) & 1) << 2)


# Levels of at least this many rows take the balanced weight gradient (gpc_spconv_wgrad_v6_balanced): the crossover measured on
# sparse finest levels (profiles/r07_train_batch.md), and above 150 000 in any case: a patch of at most 150 000 points has no level
# that large, so single-patch training keeps gpc_spconv_wgrad_v6 and its bits.
WGRAD_BALANCED_MIN_ROWS = 600_000

# GausPcgcNet.conv_families: "v6" every level on the mma.sync conv; "codec" every level on the family the codec codes it with
CONV_FAMILIES = ("v6", "codec")


def check_conv_families(conv_families: str) -> str:
    if conv_families not in CONV_FAMILIES:
        raise ValueError(f"conv_families must be one of {CONV_FAMILIES}, got {conv_families!r}")
    return conv_families


class GausPcgcNet(nn.Module):
    """The GausPcgc network with the reference's state_dict layout (weights.reference_layout(32, kernel_size)).  Starts from
    `state_dict` (a checkpoint in that layout) or from make_synthetic_state_dict(seed).  fog.conv.kernel is a constant buffer.
    conv_families: "v6" runs every level on the mma.sync conv; "codec" runs every level on the conv family the codec picks for it
    (GausPcgcCodec.build_kmap with its own thresholds; in forward_batch the rule sees each union level as a whole)."""

    def __init__(self, kernel_size: int = 5, state_dict: Optional[Dict[str, torch.Tensor]] = None, seed: int = 5,
                 conv_families: str = "v6"):
        super().__init__()
        if kernel_size not in (3, 5):
            raise ValueError("kernel_size must be 3 or 5")
        self.conv_families = check_conv_families(conv_families)
        self.kernel_size = kernel_size
        sd = state_dict if state_dict is not None else W.make_synthetic_state_dict(seed, 32, kernel_size)
        W.validate_state_dict(sd, 32, kernel_size)
        for name in W.reference_layout(32, kernel_size):
            *path, leaf = name.split(".")
            mod = self
            for p in path:
                if not hasattr(mod, p):
                    mod.add_module(p, nn.Module())
                mod = getattr(mod, p)
            t = sd[name].detach().to(torch.float32).clone()
            if name == "fog.conv.kernel":
                mod.register_buffer(leaf, t)
            else:
                mod.register_parameter(leaf, nn.Parameter(t))
        self._codec: Optional[GausPcgcCodec] = None
        self.wgrad_balanced_min_rows = WGRAD_BALANCED_MIN_ROWS
        # rows of the finest level of one union in forward_batch (plan_unions' row cap); a bigger batch runs as several unions
        self.union_max_rows = 4_000_000

    def codec(self, dev: torch.device) -> GausPcgcCodec:
        if self._codec is None or self._codec.dev != dev:
            self._codec = GausPcgcCodec(_Geometry(self.kernel_size), dev, ac_threads=1)
        return self._codec

    def _pyramid(self, xyz: torch.Tensor) -> Tuple[List[Level], Tuple[int, int]]:
        """the encoder's octree levels (no kernel maps) and the z extent of the leaves in the key frame (after _recentre)"""
        dev = next(self.parameters()).device
        codec = self.codec(dev)
        with torch.no_grad():
            xyz = xyz.to(device=dev, dtype=torch.int32).contiguous()
            keys, meta = codec.pack_keys(xyz)
            meta_h = meta.cpu().numpy()
            if meta_h[0] & 2:
                xyz, _ = codec._recentre(xyz)
                keys, meta = codec.pack_keys(xyz)
                meta_h = meta.cpu().numpy()
            mm = meta_h[2:8].astype(np.uint32)
            levels = codec.build_pyramid(codec.sort_unique(keys, mm), mm.astype(np.int64))
        return levels, (int(mm[2]) - (1 << 20), int(mm[5]) - (1 << 20))

    def kmap(self, keys: torch.Tensor) -> KMap:
        """the kernel map a level of these keys runs on: the mma.sync family ("v6"), or the codec's own choice ("codec")"""
        family = "v6" if check_conv_families(self.conv_families) == "v6" else None
        codec = self.codec(keys.device)
        with torch.no_grad():
            return codec.build_kmap(keys, family=family)

    def geometry(self, xyz: torch.Tensor) -> List[Level]:
        """the encoder's octree of a voxel cloud (GausPcgcCodec.encode): levels coarsest -> finest, each with its kernel map
        (self.kmap); levels[d + 1] are the children of levels[d] in (z, y, x) order"""
        levels, _ = self._pyramid(xyz)
        for lv in levels:
            lv.kmap = self.kmap(lv.keys)
        return levels

    def _packs(self, P: Dict[str, torch.Tensor]) -> Dict[str, WeightPack]:
        return {k: WeightPack(P[k], self.wgrad_balanced_min_rows) for k in W.CONV_KEYS}

    def _stack(self, x: torch.Tensor, P: Dict[str, torch.Tensor], packs: Dict[str, WeightPack], ids: Sequence[int],
               km: KMap) -> torch.Tensor:
        conv = lambda t, i: SparseConvFn.apply(t, P[W.CONV_KEYS[i]], km, packs[W.CONV_KEYS[i]])
        x = torch.relu(conv(x, ids[0]))
        for a, b in ((ids[1], ids[2]), (ids[3], ids[4])):
            t = torch.relu(conv(x, a))
            x = torch.relu(conv(t, b) + x)
        return x

    def _level_bits(self, parent: Level, gt: Level, P: Dict[str, torch.Tensor], packs: Dict[str, WeightPack], bits: torch.Tensor,
                    probs: Optional[List[torch.Tensor]]) -> torch.Tensor:
        """bits + the code length of gt's four stages given its parent level (each with its kernel map); the stages'
        probability rows are appended to probs when it is a list"""
        codec = self.codec(gt.keys.device)
        dev = gt.keys.device
        with torch.no_grad():
            _, cp = codec.expand(parent, gt.n)                         # children == gt.keys row for row
            cp = cp.to(torch.int64)
            occ = gt.occ.to(torch.int64)
        f = EmbedFn.apply(P["prior_embedding.weight"], parent.occ.to(torch.int64))
        f = self._stack(f, P, packs, W.PRIOR_CONVS, parent.kmap)
        u = ChildGatherFn.apply(f, cp, _octant(gt.keys)) + EmbedFn.apply(P["target_embedding.target_res_embedding.weight"], _octant(gt.keys))
        u = self._stack(u, P, packs, W.TARGET_CONVS, gt.kmap)
        for i in range(4):
            f = u if i == 0 else u + EmbedFn.apply(P[f"pred_head_s{i}_emb.weight"], occ >> CTX_SHIFT[i])
            c0, c1 = W.stage_convs(i)
            t = torch.relu(SparseConvFn.apply(f, P[W.CONV_KEYS[c0]], gt.kmap, packs[W.CONV_KEYS[c0]]))
            t = SparseConvFn.apply(t, P[W.CONV_KEYS[c1]], gt.kmap, packs[W.CONV_KEYS[c1]])
            h = torch.relu(nn.functional.linear(t, P[f"pred_head_s{i}.0.weight"], P[f"pred_head_s{i}.0.bias"]))
            logits = nn.functional.linear(h, P[f"pred_head_s{i}.2.weight"], P[f"pred_head_s{i}.2.bias"])
            p = torch.softmax(logits, dim=1)
            A = W.STAGE_ALPHABETS[i]
            sym = (occ >> STAGE_SHIFT[i]) & STAGE_MASK[i]
            hot = sym[:, None] == torch.arange(A, device=dev)[None, :]
            # the coder's probability of the symbol: q[k] = round(cdf[k] * (65536 - A)) + k (kit/op.py) gives it
            # (p * (65536 - A) + 1) / 65536 up to rounding, so a symbol never costs more than 16 bits
            bits = bits - torch.log2(((p * hot).sum(1) * (65536 - A) + 1) / 65536).sum()
            if probs is not None:
                probs.append(p.detach())
        return bits

    def forward(self, xyz: torch.Tensor, collect: bool = False) -> Dict[str, object]:
        """xyz int [N,3] voxel coordinates -> {"bits": code length of the occupancy streams, sum of -log2 of the coder's
        probability of every true symbol, (p * (65536 - A) + 1) / 65536 (fp32 scalar, differentiable),
        "bpp": bits / N, "points": N, "levels": coded levels, "families": {"v6" | "sparse" | "um": levels whose kernel map is of
        that conv family}}; collect=True adds "probs": the softmax rows of every (level, stage) in the codec's stream order
        (encode(..., collect=True)'s aux["probs"])."""
        levels = self.geometry(xyz)
        P = dict(self.named_parameters())
        packs = self._packs(P)
        bits = torch.zeros((), dtype=torch.float32, device=levels[0].keys.device)
        probs: List[torch.Tensor] = []
        for d in range(len(levels) - 1):
            bits = self._level_bits(levels[d], levels[d + 1], P, packs, bits, probs if collect else None)
        n = int(xyz.shape[0])
        out = {"bits": bits, "bpp": bits / max(n, 1), "points": n, "levels": len(levels) - 1,
               "families": _family_counts(lv.kmap for lv in levels)}
        if collect:
            out["probs"] = probs
        return out

    def forward_batch(self, patches: Sequence[torch.Tensor], collect: bool = False) -> Dict[str, object]:
        """The code length of many voxel clouds (int [N,3] each), run as union octrees (batch.py): each patch's pyramid is built as
        geometry() builds it, plan_unions stacks them along z with at most union_max_rows rows in a union's finest level, and every
        union runs the network once per union level, so one launch per conv serves all its patches.  No 5^3 neighbourhood and no
        parent spans two patches, so every patch's rows see exactly what they see alone; only the conv tilings (which depend on the
        level's size) and the summation order of the bits differ.  A parent runs on its whole union level, a child on the level's
        first M rows (the patches with parents at that scale).  Patches that fit no union run alone.
        Returns {"bits": summed over the patches (fp32 scalar, differentiable), "bpp": bits / total points, "points", "patches",
        "unions", "families": {"v6" | "sparse" | "um": kernel maps of that conv family the step ran (one per union level and row
        count, one per level of a patch run alone)}}; collect=True adds "probs": per patch, its rows of every (level, stage) in the
        order forward(xyz, collect=True) gives them."""
        if not patches:
            raise ValueError("forward_batch needs at least one patch")
        P = dict(self.named_parameters())
        packs = self._packs(P)
        dev = next(self.parameters()).device
        geo = [self._pyramid(xyz) for xyz in patches]
        bits = torch.zeros((), dtype=torch.float32, device=dev)
        probs: List[List[torch.Tensor]] = [[] for _ in patches]
        ran: List[KMap] = []
        multi = [s for s, (lv, _) in enumerate(geo) if len(lv) >= 2]
        unions, singles = plan_unions([geo[s][1][0] for s in multi], [geo[s][1][1] for s in multi], [len(geo[s][0]) for s in multi],
                                      [geo[s][0][-1].n for s in multi], self.union_max_rows)
        for j in singles:
            s = multi[j]
            levels = geo[s][0]
            for lv in levels:
                lv.kmap = self.kmap(lv.keys)
                ran.append(lv.kmap)
            for d in range(len(levels) - 1):
                bits = self._level_bits(levels[d], levels[d + 1], P, packs, bits, probs[s] if collect else None)
        for up in unions:
            members = [multi[j] for j in up.scenes]
            U, K, M = union_levels([geo[s][0] for s in members], up.tz)
            D = max(len(geo[s][0]) for s in members)
            maps: Dict[Tuple[int, int], KMap] = {}

            def level(sg: int, rows: int) -> Level:
                ul = U[sg]
                if (sg, rows) not in maps:
                    maps[sg, rows] = self.kmap(ul.keys[:rows])
                    ran.append(maps[sg, rows])
                return Level(ul.keys[:rows], ul.occ[:rows], rows, maps[sg, rows])

            for sg in range(D - 1, 0, -1):                     # coarsest first, as forward() runs a patch's levels
                got: Optional[List[torch.Tensor]] = [] if collect else None
                bits = self._level_bits(level(sg + 1, U[sg + 1].n), level(sg, M[sg]), P, packs, bits, got)
                if collect:
                    for j in range(K[sg]):
                        r0, r1 = U[sg].ranges[j]
                        probs[members[U[sg].members[j]]] += [q[r0:r1] for q in got]
        n = sum(int(xyz.shape[0]) for xyz in patches)
        out = {"bits": bits, "bpp": bits / max(n, 1), "points": n, "patches": len(patches), "unions": len(unions),
               "families": _family_counts(ran)}
        if collect:
            out["probs"] = probs
        return out

    def checkpoint(self) -> Dict[str, torch.Tensor]:
        """state_dict in the reference layout, on the CPU (what torch.save writes and compress_point_cloud loads)"""
        return {k: v.detach().to("cpu").clone() for k, v in self.state_dict().items()}


def _family_counts(kmaps) -> Dict[str, int]:
    counts = {"v6": 0, "sparse": 0, "um": 0}
    for km in kmaps:
        counts[kmap_family(km)] += 1
    return counts


def partition(xyz: torch.Tensor, max_points: int = 150_000) -> List[torch.Tensor]:
    """kd-tree patches of a cloud: a patch of more than max_points points is split at its median along its longest axis (the first
    such axis on ties), points of equal coordinate in input order.  Returns the row indices (int64, on xyz's device) of every patch,
    left before right; every row is in exactly one patch.  Device-agnostic and deterministic."""
    if max_points < 1:
        raise ValueError("max_points must be >= 1")
    n = int(xyz.shape[0])
    out: List[torch.Tensor] = []
    todo = [torch.arange(n, device=xyz.device)]
    while todo:
        idx = todo.pop()
        if idx.numel() <= max_points:
            if idx.numel():
                out.append(idx)
            continue
        p = xyz[idx]
        ext = (p.amax(0) - p.amin(0)).tolist()
        axis = ext.index(max(ext))
        srt = idx[torch.sort(p[:, axis], stable=True).indices]
        half = idx.numel() // 2
        todo.append(srt[half:])
        todo.append(srt[:half])
    return out


def _load_init(init) -> Optional[Dict[str, torch.Tensor]]:
    if init is None or isinstance(init, dict):
        return init
    return torch.load(init, map_location="cpu")


def batches(n_patches: int, batch_size: int, seed: int) -> Iterator[List[int]]:
    """The patch indices of every step: consecutive batch_size entries of one stream of permutations of range(n_patches), a new
    permutation drawn from `seed` whenever the last one is used up (so every patch is seen once per pass, and a batch may straddle
    two passes).  batch_size 1 gives the order single-patch training has always used."""
    if batch_size < 1:
        raise ValueError(f"batch_size must be >= 1, got {batch_size}")
    if batch_size > n_patches:
        raise ValueError(f"batch_size {batch_size} exceeds the {n_patches} patches to train on")

    def stream() -> Iterator[List[int]]:
        gen = torch.Generator().manual_seed(int(seed))
        order: List[int] = []
        while True:
            batch = []
            while len(batch) < batch_size:
                if not order:
                    order = torch.randperm(n_patches, generator=gen).tolist()
                batch.append(order.pop(0))
            yield batch
    return stream()


def train(clouds: Sequence[torch.Tensor], ckpt_out: Optional[str] = None, init: Union[None, str, Dict[str, torch.Tensor]] = None,
          steps: int = 1000, lr: float = 5e-4, seed: int = 0, kernel_size: int = 5, max_points: int = 150_000, save_every: int = 0,
          synthetic_seed: int = 5, log: Optional[Callable[[Dict[str, float]], None]] = None, batch_size: int = 1,
          conv_families: str = "v6"):
    """Train on voxel clouds (int [N,3] each): the clouds are cut into kd-tree patches of at most max_points points, and every
    step codes batch_size patches (batches(): the order a permutation per pass, drawn from `seed`) and takes one Adam step (lr 5e-4
    as the reference) on their bits per point.  batch_size 1 runs GausPcgcNet.forward on the patch; larger batches run
    forward_batch (union octrees).  conv_families: "v6" (every level on the mma.sync conv) or "codec" (every level on the conv
    family the codec codes it with; GausPcgcNet).  Starts from `init` (checkpoint path or state_dict) or make_synthetic_state_dict(synthetic_seed).
    Saves torch.save(state_dict) in the reference layout to ckpt_out every save_every steps (0: never) and at the end.
    Returns (state_dict, rows) with one row {"step", "points" (of the step's patches), "bpp", "time"} per step; `log` is called
    with each row."""
    check_conv_families(conv_families)
    if not torch.cuda.is_available():
        raise _lib.GpcError("training needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    dev = torch.device("cuda", torch.cuda.current_device())
    patches: List[torch.Tensor] = []
    for c in clouds:
        xyz = c.to(device=dev, dtype=torch.int32)
        patches += [xyz[i].contiguous() for i in partition(xyz, max_points)]
    if not patches:
        raise ValueError("no points to train on")
    order = batches(len(patches), batch_size, seed)
    net = GausPcgcNet(kernel_size, _load_init(init), synthetic_seed, conv_families=conv_families).to(dev)
    opt = torch.optim.Adam(net.parameters(), lr=lr)
    rows: List[Dict[str, float]] = []
    t0 = time.time()
    for step in range(1, steps + 1):
        batch = [patches[i] for i in next(order)]
        opt.zero_grad(set_to_none=True)
        out = net(batch[0]) if batch_size == 1 else net.forward_batch(batch)
        if out["bpp"].requires_grad:
            out["bpp"].backward()
            opt.step()
        row = {"step": step, "points": int(out["points"]), "bpp": float(out["bpp"].detach()), "time": time.time() - t0}
        rows.append(row)
        if log is not None:
            log(row)
        if ckpt_out and save_every and step % save_every == 0 and step < steps:
            torch.save(net.checkpoint(), ckpt_out)
    sd = net.checkpoint()
    if ckpt_out:
        torch.save(sd, ckpt_out)
    return sd, rows
