"""Per-image cached vision K/V for autoregressive caption decode.

In the reference decode loop (full_model.py:241-363) every step calls the bridge on the whole token
prefix and re-projects the unchanged image through w_k / w_v of every block
(bridge_module.py:99-100) -- 155 GFLOP per step at batch 32 that depend only on the image. Because the
bridge self-attention is non-causal and unmasked (:138,236) the text side cannot be cached exactly,
but the vision K/V can: they are computed once per image here and every decode step reads them.

The cache is two plain torch tensors owned by this object: `kv` (bf16, [B*Nv, num_blocks*2*D]; block
i's K at columns [2iD, 2iD+D), V in the next D columns -- the projection output, used for steps of more
than 64 positions), `kv_packed` (the same values as [B][num_blocks][heads][2][Nv][d+8], the layout
the mma.sync decode kernel streams with one bulk copy per 16-key tile; steps of up to 32 positions) and
`kv_tc` (32-key tiles as the swizzled operand images of the tcgen05 decode kernel; steps of 33..64). The CUDA library only ever sees their
pointers for the duration of a call.

Position rows (`x1`, fp32 [B, max_positions, D]): block 0's cross-attention sub-layer
(bridge_module.py:316-323) maps text row (b, j) to x1[b, j] = x + W_o * SDPA(W_q * LN(x), K_b, V_b),
which involves no other text position, so a decode loop that appends tokens computes it once per
position (`BridgeLite.forward(..., kv_cache=cache, cached_positions=k)`) instead of once per position
per step. Everything after it (block 0's non-causal self-attention onwards) mixes positions and is
recomputed on the whole prefix, as in the reference.

Beam search (`beams=K`): the K beams of an image attend to the same image K/V, so the K/V buffers stay per image
(B images) and only the position rows grow to one per beam (`x1` [B*K, max_positions, D], row b*K + k).
`BridgeLite` runs the cross-attention of the B*K text rows as B query blocks of K*s rows over the image's cache and
the rest of each block per beam; `reorder_beams(parents)` follows the beams chosen by a step.
"""
from __future__ import annotations

import torch

__all__ = ["VisionKVCache"]


class VisionKVCache:
    """`precision="bf16"` (default): bf16 K/V read by the tensor-core decode kernels (the reference's
    autocast numerics). `precision="fp32"`: fp32 K/V (`kv32`) from the fp32 master weights, read by the fp32
    inference path (csrc/exact_fp32.cu) -- the numerics of the reference's own decode, which runs without
    autocast (full_model.py:221-261); greedy token ids then equal the fp32 reference's on every step."""

    def __init__(self, bridge, vision_features: torch.Tensor, max_positions: int = 64, precision: str = "bf16",
                 beams: int = 1):
        if vision_features.dim() != 3:
            raise RuntimeError("vision_features must be [B, Nv, vision_dim]")
        if precision not in ("bf16", "fp32"):
            raise ValueError("precision must be 'bf16' or 'fp32'")
        if not 1 <= int(beams) <= 8:
            raise ValueError(f"beams must be in [1, 8], got {beams}")
        self.precision = precision
        self.beams = int(beams)
        self._bridge = bridge
        self.max_positions = int(max_positions)
        self.batch, self.len_vision = int(vision_features.shape[0]), int(vision_features.shape[1])
        self.kv = self.kv_packed = self.kv_tc = self.kv32 = self.vision_bf16 = None
        self.x1 = None
        self.refill(vision_features)

    def refill(self, vision_features: torch.Tensor) -> "VisionKVCache":
        """(Re)compute the cache for a new batch of images of the same shape, IN PLACE: every buffer keeps
        its address, so CUDA graphs captured over this cache (`DecodeStepGraphs`) stay valid and a
        captioning loop pays the K/V projection + packing per batch but no re-capture. Also resets the
        position rows and re-reads the bridge weights' versions."""
        bridge = self._bridge
        if vision_features.dim() != 3 or (int(vision_features.shape[0]), int(vision_features.shape[1])) != (self.batch, self.len_vision):
            raise RuntimeError(f"refill needs vision_features [{self.batch}, {self.len_vision}, vision_dim] (the shape the "
                               "cache was built for)")
        with torch.no_grad():
            if self.precision == "fp32":
                kv32 = bridge.project_vision_kv_fp32(vision_features)
                self.kv32 = kv32 if self.kv32 is None else self.kv32.copy_(kv32)
            else:
                self._fill_bf16(bridge, vision_features)
        self._versions = tuple(p._version for p in bridge.parameters())
        dev = self.kv32.device if self.precision == "fp32" else self.kv.device
        if self.x1 is None and self.max_positions > 0:
            self.x1 = torch.empty((self.batch * self.beams, self.max_positions, bridge.language_dim), device=dev,
                                  dtype=torch.float32)
        self.positions_filled = 0
        return self

    def _fill_bf16(self, bridge, vision_features: torch.Tensor) -> None:
        d = bridge.language_dim // bridge.num_heads_cross
        if self.kv is None:
            self.vision_bf16, self.kv = bridge.project_vision_kv(vision_features)
            # decode layout (per image / block / head: padded K rows then V rows), read by the K/V-streaming
            # cross-attention kernel whenever a step has <= 64 text positions
            self.kv_packed = bridge.pack_vision_kv(self.kv, self.batch, self.len_vision)
            # tcgen05 decode layout, read by steps of 33..64 positions (where the mma.sync kernel is bound by the
            # legacy tensor pipe); only built for the head dims that kernel is instantiated for
            self.kv_tc = bridge.pack_vision_kv_tc(self.kv, self.batch, self.len_vision) if d in (64, 128, 288) else None
        else:   # same buffers, new contents
            bridge.project_vision_kv(vision_features, out=(self.vision_bf16, self.kv))
            bridge.pack_vision_kv(self.kv, self.batch, self.len_vision, out=self.kv_packed)
            if self.kv_tc is not None:
                bridge.pack_vision_kv_tc(self.kv, self.batch, self.len_vision, out=self.kv_tc)

    def position_rows(self, length: int, cached_positions: int, device, dim: int):
        """The row store for a forward over `length` text positions of which the first
        `cached_positions` are reused, or None when the prefix is longer than the store (the caller then
        computes every row). Raises if rows are asked for that were never written."""
        if self.x1 is None or length > self.max_positions:
            return None
        k = int(cached_positions)
        if not 0 <= k < length:
            raise RuntimeError(f"cached_positions must be in [0, {length}) for a prefix of {length} positions, got {k}")
        if k > self.positions_filled:
            raise RuntimeError(f"cached_positions={k} but only {self.positions_filled} positions are cached")
        if self.x1.device != device or self.x1.shape[-1] != dim:
            raise RuntimeError("position rows live on another device / have another width than the text")
        self.positions_filled = length
        return self.x1

    def reorder_beams(self, parents: torch.Tensor) -> None:
        """Beam search: position-row store row r takes the filled rows of row parents[r], in place (the buffer
        keeps its address, so captured graphs stay valid). `parents` int64 [batch * beams] is what
        `ops.beam_step` wrote: b * beams + (a beam of image b), in range by construction."""
        if parents.dtype != torch.int64 or parents.shape != (self.batch * self.beams,):
            raise RuntimeError(f"parents must be int64 [{self.batch * self.beams}]")
        if self.x1 is None or self.positions_filled == 0:
            return
        rows = self.x1[:, :self.positions_filled]
        rows.copy_(rows.index_select(0, parents))

    @property
    def nbytes(self) -> int:
        """bytes of the decode-layout cache (what a decode step reads)"""
        t = self.kv32 if self.precision == "fp32" else self.kv_packed
        return t.numel() * t.element_size()

    def is_current(self) -> bool:
        """False once the bridge weights were updated after the cache was filled."""
        return self._versions == tuple(p._version for p in self._bridge.parameters())
