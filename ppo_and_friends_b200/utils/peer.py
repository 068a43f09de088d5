"""
NVLink peer-memory group for the fused gradient all-reduce + clip + Adam (csrc/peer.cu).

Push exchange: each rank allocates ONE receive buffer `[2 parities][R source ranks][n_floats]` and one flag array
with cudaMalloc through the C ABI, exports CUDA IPC handles, and the handles are exchanged with
`torch.distributed.all_gather_object` (any backend).  Rank r's backward kernels write every gradient element into
slot `[parity][r]` of its own buffer AND of every peer's buffer (the `mirror_delta` byte offsets of
`ppoaf_update_bufs`), so the gradients cross NVLink while the backward pass runs; the fused kernel then only
exchanges flags and reads its R local slots.
"""
import ctypes as C

import torch
import torch.distributed as dist

from .._lib import check, load


class _RawCudaBuffer:
    """Exposes a raw device allocation to torch through __cuda_array_interface__ (no copy, no ownership)."""

    def __init__(self, ptr, n_floats):
        self.__cuda_array_interface__ = {"shape": (n_floats,), "typestr": "<f4", "data": (int(ptr), False), "version": 2}


class PeerGroup:
    def __init__(self, n_floats, device):
        assert dist.is_initialized() and dist.get_world_size() > 1
        lib = load()
        self.rank, self.world = dist.get_rank(), dist.get_world_size()
        self.n_floats = int(n_floats)
        self.device = torch.device(device)
        nbytes = (self.n_floats * 4 + 255) // 256 * 256
        self.slot_bytes = nbytes
        self._local = []
        for size in (2 * self.world * nbytes, 256):            # receive buffer [2][R][n], flags
            p = C.c_void_p()
            check(lib.ppoaf_peer_alloc(size, C.byref(p)), "ppoaf_peer_alloc")
            self._local.append(p.value)
        handles = []
        for p in self._local:
            buf = C.create_string_buffer(64)
            check(lib.ppoaf_peer_export(C.c_void_p(p), buf), "ppoaf_peer_export")
            handles.append(buf.raw)
        torch.cuda.synchronize(self.device)
        gathered = [None] * self.world
        dist.all_gather_object(gathered, handles)
        self._opened = []
        self.ptrs = []                                         # ptrs[r] = [recv, flags] of rank r, valid on this device
        for r in range(self.world):
            if r == self.rank:
                self.ptrs.append(list(self._local))
                continue
            mine = []
            for h in gathered[r]:
                p = C.c_void_p()
                check(lib.ppoaf_peer_import(h, C.byref(p)), "ppoaf_peer_import")
                mine.append(p.value)
                self._opened.append(p.value)
            self.ptrs.append(mine)
        def slot(base, parity, src):
            return base + (parity * self.world + src) * nbytes
        # this rank's gradient buffer for parity k = its own slot of its own receive buffer
        self.grads = [torch.as_tensor(_RawCudaBuffer(slot(self._local[0], k, self.rank), self.n_floats), device=self.device)
                      for k in range(2)]
        # byte offsets from a local gradient address to the same element of this rank's slot inside every peer
        self.mirror_delta = [self.ptrs[q][0] - self._local[0] for q in range(self.world) if q != self.rank]
        self.ctrl = torch.zeros(lib.ppoaf_peer_ctrl_bytes(), dtype=torch.uint8, device=self.device)
        self._grad_arrays = []                                 # the R LOCAL slots the fused kernel sums, per parity
        for k in range(2):
            arr = (C.c_void_p * self.world)(*[slot(self._local[0], k, r) for r in range(self.world)])
            self._grad_arrays.append(arr)
        self._flag_array = (C.c_void_p * self.world)(*[self.ptrs[r][1] for r in range(self.world)])
        dist.barrier()                                         # everyone has mapped everyone before first use

    def allreduce_adam(self, parity, nets, mb_cursor, hparams, stream_ptr):
        check(load().ppoaf_peer_allreduce_adam(
            self._grad_arrays[parity], self._flag_array, self.world, self.rank, C.c_void_p(nets.flat_params.data_ptr()),
            C.c_void_p(nets.adam_m.data_ptr()), C.c_void_p(nets.adam_v.data_ptr()), C.c_void_p(nets.adam_step.data_ptr()),
            C.c_void_p(mb_cursor.data_ptr()), C.c_void_p(hparams.data_ptr()), nets.n_actor, nets.n_critic,
            C.c_void_p(self.ctrl.data_ptr()), stream_ptr), "ppoaf_peer_allreduce_adam")

    def error_flag(self):
        off = load().ppoaf_peer_ctrl_bytes() - 256 + 16
        return int(self.ctrl[off:off + 4].view(torch.int32).item())

    def close(self):
        lib = load()
        torch.cuda.synchronize(self.device)
        if dist.is_initialized():
            dist.barrier()
        for p in self._opened:
            lib.ppoaf_peer_close(C.c_void_p(p))
        for p in self._local:
            lib.ppoaf_peer_free(C.c_void_p(p))
        self._opened, self._local = [], []


class NvlsGroup:
    """
    NVSwitch-multicast variant (csrc/peer.cu, nvls_allreduce_adam_kernel): the gradient buffers (two parities), a
    parameter staging buffer and a 256-byte flag block are ONE symmetric allocation made with
    `torch.distributed._symmetric_memory` (plumbing: VMM allocation, handle exchange, multicast binding).  Same interface
    as PeerGroup; `mirror_delta` is empty because nothing is pushed by the backward kernels.
    """

    @staticmethod
    def available():
        try:
            import torch.distributed._symmetric_memory  # noqa: F401
            return True
        except Exception:
            return False

    def __init__(self, n_floats, device):
        import torch.distributed._symmetric_memory as symm_mem
        assert dist.is_initialized() and dist.get_world_size() > 1
        lib = load()
        self.rank, self.world = dist.get_rank(), dist.get_world_size()
        self.n_floats = int(n_floats)
        self.device = torch.device(device)
        slot = (self.n_floats * 4 + 255) // 256 * 256 // 4          # floats per buffer, 256-byte aligned
        blk = lib.ppoaf_nvls_flag_block_bytes() // 4
        self._buf = symm_mem.empty(3 * slot + blk, dtype=torch.float32, device=self.device)
        self._buf.zero_()
        torch.cuda.synchronize(self.device)
        self._hdl = symm_mem.rendezvous(self._buf, group=dist.group.WORLD)
        mc = int(getattr(self._hdl, "multicast_ptr", 0) or 0)
        if mc == 0:
            raise RuntimeError("symmetric memory has no multicast mapping on this system")
        base = self._buf.data_ptr()
        self.grads = [self._buf[k * slot:k * slot + self.n_floats] for k in range(2)]
        self.mirror_delta = []
        self._g_mc = [mc + k * slot * 4 for k in range(2)]
        peers = [int(p) for p in self._hdl.buffer_ptrs]
        self._staging = (C.c_void_p * self.world)(*[peers[r] + 2 * slot * 4 for r in range(self.world)])
        self._blocks = (C.c_void_p * self.world)(*[peers[r] + 3 * slot * 4 for r in range(self.world)])
        self._ctrl_bytes = lib.ppoaf_nvls_ctrl_bytes()
        self.ctrl = torch.zeros(self._ctrl_bytes, dtype=torch.uint8, device=self.device)
        dist.barrier()

    def allreduce_adam(self, parity, nets, mb_cursor, hparams, stream_ptr):
        check(load().ppoaf_nvls_allreduce_adam(
            C.c_void_p(self._g_mc[parity]), self._staging, self._blocks, self.world,
            self.rank, C.c_void_p(nets.flat_params.data_ptr()), C.c_void_p(nets.adam_m.data_ptr()),
            C.c_void_p(nets.adam_v.data_ptr()), C.c_void_p(nets.adam_step.data_ptr()), C.c_void_p(mb_cursor.data_ptr()),
            C.c_void_p(hparams.data_ptr()), nets.n_actor, nets.n_critic, C.c_void_p(self.ctrl.data_ptr()), stream_ptr),
            "ppoaf_nvls_allreduce_adam")

    def error_flag(self):
        off = self._ctrl_bytes - 256 + 16
        return int(self.ctrl[off:off + 4].view(torch.int32).item())

    def gather_moments(self, nets):
        """The kernel keeps adam_m / adam_v current only on the float4 rows this rank owns, [r * slice, (r + 1) * slice)
        with slice = ceil(nv / R).  Gather every owner's rows, so each rank holds the full moments a torch.optim.Adam
        would (before a checkpoint).  Collective: every rank calls it."""
        nv = (nets.n_actor + nets.n_critic) // 4
        sl = -(-nv // self.world)
        lo, hi = min(nv, self.rank * sl), min(nv, (self.rank + 1) * sl)
        for buf in (nets.adam_m, nets.adam_v):
            rows = buf[:4 * nv].view(nv, 4)
            mine = torch.zeros(sl, 4, dtype=buf.dtype, device=buf.device)
            mine[:hi - lo] = rows[lo:hi]
            full = torch.empty(self.world * sl, 4, dtype=buf.dtype, device=buf.device)
            dist.all_gather_into_tensor(full, mine)
            rows.copy_(full[:nv])

    def close(self):
        torch.cuda.synchronize(self.device)
        if dist.is_initialized():
            dist.barrier()
        self._hdl = None
        self._buf = None


def make_exchange_group(n_floats, device):
    """The push exchange over CUDA IPC by default; PPOAF_NVLS=1 selects the NVSwitch-multicast two-shot exchange when
    the system offers a multicast mapping.  Measured on 8 x B200 (C4, us per minibatch step, push / NVLS):
    R=2 111 / 118, R=4 116 / 135, R=8 133 / 146 -- three cross-GPU barrier rounds cost more than the bytes they save at
    1.84 MB of gradients, so NVLS stays opt-in until the parameter count makes the exchange bandwidth-bound."""
    import os
    if os.environ.get("PPOAF_NVLS", "0") == "1" and NvlsGroup.available():
        ok = torch.zeros(1, dtype=torch.int32, device=device)
        grp = None
        try:
            grp = NvlsGroup(n_floats, device)
            ok += 1
        except Exception as e:                              # no multicast / no VMM support: every rank must agree
            if dist.get_rank() == 0:
                print(f"NVLS exchange unavailable ({type(e).__name__}: {e}); using the push exchange", flush=True)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 1:
            return grp
    return PeerGroup(n_floats, device)
