"""Host-buffer entry point: spectrograms of waveforms that live in (pinned) host
memory, with the PCIe copies overlapped with the kernels.

The batch is cut into chunks of clips; chunk i+1 is copied host->device on a
copy stream while chunk i is transformed on the compute stream and chunk i-1 is
copied device->host on a third stream (the two DMA directions are independent
engines), so a call costs ~max(H2D, compute, D2H) instead of their sum.  The
copy streams are NOT ordered after the caller's stream, so back-to-back calls
keep the host->device engine busy across call boundaries (the input of call
i+1 streams in while call i's last chunk is still being transformed / copied
out); buffer reuse is ordered by events that live across calls.

Pinned buffers should sit on the GPU's NUMA node (``alloc_pinned``): a remote
node costs up to half of the PCIe rate on multi-socket hosts.
"""
from __future__ import annotations

import os
from typing import List, Optional

import torch


def gpu_local_cpus(device_index: int) -> Optional[List[int]]:
    """CPUs of the NUMA node the GPU hangs off (NVML ideal affinity, sysfs as a fallback);
    ``None`` when neither source is available (single-node hosts do not care)."""
    try:
        avail = set(os.sched_getaffinity(0))
    except AttributeError:
        return None
    cpus: List[int] = []
    try:
        import pynvml

        pynvml.nvmlInit()
        uuid = str(torch.cuda.get_device_properties(device_index).uuid)
        try:
            h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
        except Exception:  # noqa: BLE001
            h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
        words = (max(avail | {os.cpu_count() or 1}) + 64) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        for w, bits in enumerate(mask):
            for b in range(64):
                if (int(bits) >> b) & 1:
                    cpus.append(64 * w + b)
    except Exception:  # noqa: BLE001
        cpus = []
    if not cpus:
        try:
            p = torch.cuda.get_device_properties(device_index)
            bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
            with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
                node = int(f.read().strip())
            if node >= 0:
                with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
                    for part in f.read().strip().split(","):
                        lo, _, hi = part.partition("-")
                        cpus.extend(range(int(lo), int(hi or lo) + 1))
        except Exception:  # noqa: BLE001
            cpus = []
    cpus = sorted(set(cpus) & avail)
    return cpus or None


def alloc_pinned(shape, dtype=torch.float32, device_index: int = 0, fill: Optional[str] = None):
    """Pinned host tensor whose pages are first-touched by a thread running on the GPU's NUMA node
    (Linux places pages on the node of the touching CPU).  ``fill='randn'`` fills it with white
    noise; default: zeros.  Returns ``(tensor, placement)``, placement = 'gpu-local node (n cpus)'
    or 'default policy'."""
    cpus = gpu_local_cpus(device_index)
    old = None
    if cpus:
        try:
            old = os.sched_getaffinity(0)
            os.sched_setaffinity(0, cpus)
        except OSError:
            old = None
    try:
        t = torch.empty(shape, dtype=dtype, pin_memory=True)
        if fill == "randn":
            t.normal_()
        else:
            t.zero_()
    finally:
        if old is not None:
            os.sched_setaffinity(0, old)
    return t, (f"gpu-local node ({len(cpus)} cpus)" if (cpus and old is not None) else "default policy")


_X_DTYPES = (torch.float32, torch.bfloat16, torch.float16)


class HostPipeline:
    def __init__(self, module: torch.nn.Module, chunk_clips: int = 8, copy_streams: int = 1,
                 **forward_kwargs):
        """``copy_streams`` > 1 splits each chunk's host->device copy over several streams
        (several DMA engines can then drive the PCIe link together)."""
        self.module = module
        self.chunk = int(chunk_clips)
        self.n_in = max(1, int(copy_streams))
        self.kw = forward_kwargs
        self._dev = None
        self._in = None
        self._streams = None
        self._done_compute = [None, None, None]
        self._count = 0

    N_BUF = 3  # input staging buffers: copy-in of chunk c+2 may start while chunk c is transformed

    def _setup(self, device, L, dtype):
        if self._dev != (device, L, dtype):
            self._in = [torch.empty((self.chunk, L), dtype=dtype, device=device)
                        for _ in range(self.N_BUF)]
            self._streams = (torch.cuda.Stream(device), torch.cuda.Stream(device))
            self._extra_in = [torch.cuda.Stream(device) for _ in range(self.n_in - 1)]
            self._done_compute = [None] * self.N_BUF
            self._count = 0
            self._dev = (device, L, dtype)

    @torch.no_grad()
    def __call__(self, x_host: torch.Tensor, out_host: Optional[torch.Tensor] = None,
                 device: Optional[torch.device] = None) -> torch.Tensor:
        """x_host: (B, L) pinned CPU tensor, float32, bfloat16 or float16 -> fp32 spectrograms in a
        pinned CPU tensor (allocated on first use if ``out_host`` is None).  16-bit audio is copied
        and transformed as is (half the bytes over the link of fp32); the result equals the
        module's on the fp32 copy of the same samples.  Asynchronous with
        respect to the host: the CURRENT stream waits for the last copy, so
        ``torch.cuda.current_stream().synchronize()`` (or an event recorded on it)
        marks completion.  ``x_host`` must hold its data when the call is made (it is read
        by the copy engine without waiting for work queued on the current stream)."""
        if x_host.is_cuda or x_host.dtype not in _X_DTYPES or x_host.dim() != 2:
            raise ValueError("x_host must be a (B, L) float32, bfloat16 or float16 CPU tensor")
        if not x_host.is_pinned():
            raise ValueError("x_host must be pinned (torch.Tensor.pin_memory()) for asynchronous copies")
        device = device or next(self.module.buffers()).device
        B, L = x_host.shape
        self._setup(device, L, x_host.dtype)
        s_in, s_out = self._streams
        cur = torch.cuda.current_stream(device)
        in_streams = [s_in] + self._extra_in
        n_chunks = (B + self.chunk - 1) // self.chunk
        for c in range(n_chunks):
            lo, hi = c * self.chunk, min(B, (c + 1) * self.chunk)
            slot = self._count % self.N_BUF
            self._count += 1
            buf = self._in[slot][: hi - lo]
            n_rows = hi - lo
            parts = min(len(in_streams), n_rows)
            for pi in range(parts):
                r0, r1 = (n_rows * pi) // parts, (n_rows * (pi + 1)) // parts
                st = in_streams[pi]
                with torch.cuda.stream(st):
                    if self._done_compute[slot] is not None:
                        st.wait_event(self._done_compute[slot])  # buffer still read by an older chunk
                    buf[r0:r1].copy_(x_host[lo + r0: lo + r1], non_blocking=True)
                    ev_in = torch.cuda.Event()
                    ev_in.record(st)
                cur.wait_event(ev_in)
            y = self.module(buf, **self.kw)
            ev_c = torch.cuda.Event()
            ev_c.record(cur)
            self._done_compute[slot] = ev_c
            if out_host is None:
                out_host = torch.empty((B,) + tuple(y.shape[1:]), dtype=y.dtype).pin_memory()
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev_c)
                out_host[lo:hi].copy_(y, non_blocking=True)
            y.record_stream(s_out)
        cur.wait_stream(s_out)
        return out_host
