"""Host-buffer front end of the fused ISP (SURVEY 8f rank 1: rig ingestion + output stage).

The reference's rig driver reads raw bytes on the host, copies them to the device, runs the ISP and
copies the RGB back for display / JPEG (scripts/tonemap_scan.py:63-100, :151-179), one step at a time.
``RigPipeline`` keeps that contract -- packed12 frames in host memory in, tone-mapped frames in host
memory out -- but overlaps the three legs on separate CUDA streams with ``depth`` slots of pinned
staging buffers: H2D of step k+1 and D2H of step k-1 run while step k is in the ISP kernels.  The ISP
state (``isp.metrics``) advances in submission order, exactly as if the steps ran back to back.
"""
from __future__ import annotations

from typing import List, Sequence

import numpy as np
import torch

from .dtypes import as_dtype, u8


class _Slot:
    def __init__(self, n, h, w, out_shape, out_dtype, device):
        self.d_in = [torch.empty((h, w * 3 // 2), dtype=torch.uint8, device=device) for _ in range(n)]
        self.d_out = [torch.empty(out_shape, dtype=out_dtype.torch, device=device) for _ in range(n)]
        self.h_out = [torch.empty(out_shape, dtype=out_dtype.torch, pin_memory=True) for _ in range(n)]
        self.copied_in = torch.cuda.Event()
        self.computed = torch.cuda.Event()
        self.copied_out = torch.cuda.Event()
        self.busy = False


class RigPipeline:
    def __init__(self, isp, n_frames: int, height: int, width: int, tonemap: str = "reinhard", dtype=u8,
                 depth: int = 2, yuv420: bool = False, ids_format: bool = False, **tonemap_args):
        """``isp`` may resize (outputs are then the resized images) and ``yuv420=True`` selects the planar YUV 4:2:0
        output of ``process_packed12`` (1.5 instead of 3 bytes per pixel over PCIe).  The ISP's flips are applied by the sweep's
        store, so the result still lands in the slot; the transposing transforms (rotate_90, the rig script's default) are
        applied by the normalise pass of the one-sweep Reinhard -> u8 forms, which also writes the slot, and elsewhere by the
        transform kernel behind the sweep, whose result is copied into the slot.  No transform with resize / YUV."""
        assert width % 8 == 0 and height % 2 == 0, "fused path needs width % 8 == 0 and even height"
        base = getattr(isp, "isp", isp)
        tname = base.transform.value
        transposing = tname in ("rotate_90", "rotate_270", "transpose", "transverse")
        assert tname == "none" or not (base._resizes or yuv420 or base.demosaic != "malvar"), \
            "RigPipeline writes straight into its slots: transforms need the plain Malvar RGB sweep"
        self.isp, self.n, self.h, self.w = isp, n_frames, height, width
        self.tonemap, self.out_dtype, self.tm = tonemap, as_dtype(dtype), tonemap_args
        self.yuv420 = bool(yuv420)
        self.ids_format = bool(ids_format)
        self.device = isp.device
        plan = base._resize_plan(height, width)
        ho, wo = (height, width) if plan is None else (plan[0][1], plan[0][0])
        self.out_shape = (ho * 3 // 2, wo) if self.yuv420 else ((wo, ho, 3) if transposing else (ho, wo, 3))
        with torch.cuda.device(self.device):
            self.s_in, self.s_isp, self.s_out = (torch.cuda.Stream(self.device) for _ in range(3))
            self.slots = [_Slot(n_frames, height, width, self.out_shape, self.out_dtype, self.device) for _ in range(depth)]
        self._next = 0
        self.h2d_bytes_per_step = n_frames * height * width * 3 // 2
        self.d2h_bytes_per_step = n_frames * int(np.prod(self.out_shape)) * self.out_dtype.itemsize

    @staticmethod
    def pin(frames: Sequence[np.ndarray]) -> List[torch.Tensor]:
        """Copy host frames into pinned memory once (what a capture driver's DMA buffers would be)."""
        return [torch.from_numpy(np.ascontiguousarray(f)).pin_memory() for f in frames]

    def submit(self, host_frames: Sequence[torch.Tensor]) -> int:
        """Enqueue one time step (n_frames packed12 host tensors).  Returns the slot index to pass to
        ``result``.  Blocks only if that slot's previous result was never collected in time."""
        assert len(host_frames) == self.n
        idx = self._next
        slot = self.slots[idx]
        self._next = (idx + 1) % len(self.slots)
        if slot.busy:
            slot.copied_out.synchronize()          # slot reuse: its previous D2H must be complete
        slot.busy = True
        with torch.cuda.device(self.device):
            with torch.cuda.stream(self.s_in):
                for d, hbuf in zip(slot.d_in, host_frames):
                    d.copy_(hbuf, non_blocking=True)
                slot.copied_in.record(self.s_in)
            with torch.cuda.stream(self.s_isp):
                self.s_isp.wait_event(slot.copied_in)
                self.isp.process_packed12(slot.d_in, tonemap=self.tonemap, dtype=self.out_dtype, out=slot.d_out,
                                          **(dict(yuv420=True) if self.yuv420 else {}),
                                          **(dict(ids_format=True) if self.ids_format else {}), **self.tm)
                slot.computed.record(self.s_isp)
            with torch.cuda.stream(self.s_out):
                self.s_out.wait_event(slot.computed)
                for hbuf, d in zip(slot.h_out, slot.d_out):
                    hbuf.copy_(d, non_blocking=True)
                slot.copied_out.record(self.s_out)
        return idx

    def result(self, idx: int) -> List[torch.Tensor]:
        """Wait for the step submitted into slot ``idx``; the returned pinned host tensors stay valid
        until that slot is reused (``depth`` submissions later)."""
        slot = self.slots[idx]
        slot.copied_out.synchronize()
        slot.busy = False
        return slot.h_out

    def process(self, host_frames: Sequence[torch.Tensor]) -> List[torch.Tensor]:
        return self.result(self.submit(host_frames))

    def drain(self):
        for s in self.slots:
            if s.busy:
                s.copied_out.synchronize()
                s.busy = False
