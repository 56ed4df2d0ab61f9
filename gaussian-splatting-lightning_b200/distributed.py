"""Gaussian-sharded multi-GPU renderer — the reference's exchange, on the b200gs kernels.

Mirrors ``internal/renderers/gsplat_distributed_renderer.py`` (SURVEY.md §3d, §8e):

* parameters are sharded by contiguous Gaussian index ranges (``:76-89``); there is no gradient all-reduce;
* every rank renders ONE camera per step; the W camera descriptions are all-gathered (``:319-335`` gathers ids and looks
  them up in the dataset — here the 40-float view itself is gathered, so no dataset object is needed);
* each rank projects its shard to all W cameras (K1, gsplat constants) and evaluates SH colours (``:252-311``);
* the VISIBLE projected splats — 11 floats (xy 2, depth 1, conic 3, compensation 1, opacity 1, rgb 3) + radius — are sent
  to the rank that owns the camera with an all-to-all (``:127-217``).  Here: ONE ``all_to_all_single`` of ``[V, 12]``
  fp32 rows (radius bit-cast into the 12th column) instead of the reference's two list-form all-to-alls — one message
  per peer, and it also runs on gloo for the CPU tests (gloo has no list-form all_to_all);
* the owner concatenates the rows in rank order (= global Gaussian-index order, so depth ties break exactly as in the
  single-GPU renderer), bins and blends its whole image locally (K2-K7);
* backward is the mirror image: blend backward on the owner, the ``[V,12]`` gradient rows travel back through the same
  all-to-all, K8 runs per camera on the shard's owner.

The distributed image is bit-identical to the single-GPU gsplat-mode render of the unsharded model
(tests/test_gpu_distributed.py).  A per-pixel reduce of partial images would NOT be (SURVEY §0.4).
"""
import os
import threading
import weakref
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import torch
import torch.distributed as dist

from .renderers import Renderer, RendererOutputInfo

ROW_FLOATS = 12  # xy(2) depth(1) conic(3) comp(1) opacity(1) rgb(3) radius-bits(1)
VIEW_FLOATS = 40  # width height fx fy cx cy | world_to_camera 16 | camera_center 3 | pad


def shard_range(n: int, world_size: int, rank: int) -> Tuple[int, int]:
    """Contiguous index shard of rank (gsplat_distributed_renderer.py:76-83): round(n/W) each, last takes the rest."""
    per = round(n / world_size)
    lo = per * rank
    hi = n if rank + 1 == world_size else lo + per
    return lo, min(hi, n)


class _AllToAllRows(torch.autograd.Function):
    """all_to_all_single of row blocks with uneven splits; the backward is the mirrored exchange."""

    @staticmethod
    def forward(ctx, rows: torch.Tensor, send_counts: List[int], recv_counts: List[int], group):
        rows = rows.contiguous()
        out = rows.new_empty((sum(recv_counts),) + tuple(rows.shape[1:]))
        dist.all_to_all_single(out, rows, output_split_sizes=list(recv_counts), input_split_sizes=list(send_counts), group=group)
        ctx.send_counts, ctx.recv_counts, ctx.group = list(send_counts), list(recv_counts), group
        return out

    @staticmethod
    def backward(ctx, g: torch.Tensor):
        g = g.contiguous()
        gin = g.new_empty((sum(ctx.send_counts),) + tuple(g.shape[1:]))
        dist.all_to_all_single(gin, g, output_split_sizes=ctx.send_counts, input_split_sizes=ctx.recv_counts, group=ctx.group)
        return gin, None, None, None


def exchange_counts(send_counts: Sequence[int], device, group=None) -> List[int]:
    """Tell every peer how many rows it will receive from me; returns how many I receive from each peer."""
    send = torch.tensor(list(send_counts), dtype=torch.int64, device=device)
    recv = torch.empty_like(send)
    dist.all_to_all_single(recv, send, group=group)
    return [int(x) for x in recv.tolist()]


def exchange_rows(rows_per_dest: Sequence[torch.Tensor], group=None) -> Tuple[torch.Tensor, List[int]]:
    """rows_per_dest[j]: [V_j, C] rows destined to rank j.  Returns (rows received, concatenated in source-rank order;
    per-source counts).  Differentiable w.r.t. the rows."""
    send_counts = [int(r.shape[0]) for r in rows_per_dest]
    recv_counts = exchange_counts(send_counts, rows_per_dest[0].device, group)
    rows = torch.cat(list(rows_per_dest), dim=0)
    return _AllToAllRows.apply(rows, send_counts, recv_counts, group), recv_counts


def pack_rows(xys, depths, conics, comp, opacities, rgbs, radii, visible) -> torch.Tensor:
    """[V, 12] fp32 rows of the visible splats (gsplat_distributed_renderer.py:167-178 + the int tensor of :177)."""
    radii_bits = radii.view(torch.float32) if radii.dtype == torch.int32 else radii.to(torch.int32).view(torch.float32)
    rows = torch.cat([xys, depths.unsqueeze(-1), conics, comp.unsqueeze(-1), opacities.reshape(-1, 1), rgbs,
                      radii_bits.unsqueeze(-1)], dim=-1)
    return rows[visible]


def unpack_rows(rows: torch.Tensor):
    xys, depths, conics, comp, opac, rgbs, rbits = torch.split(rows, [2, 1, 3, 1, 1, 3, 1], dim=-1)
    radii = rbits.detach().contiguous().view(torch.int32).squeeze(-1)
    return xys.contiguous(), depths.squeeze(-1).contiguous(), conics.contiguous(), comp.squeeze(-1), opac.squeeze(-1), rgbs.contiguous(), radii


def pack_view(camera) -> torch.Tensor:
    """The quantities K1 (gsplat constants) needs from a camera, as VIEW_FLOATS fp32 on the camera's device."""
    dev = camera.world_to_camera.device
    v = torch.zeros(VIEW_FLOATS, dtype=torch.float32, device=dev)
    head = torch.stack([camera.width.float(), camera.height.float(), camera.fx.float(), camera.fy.float(), camera.cx.float(),
                        camera.cy.float()]).to(dev)
    v[0:6] = head
    v[6:22] = camera.world_to_camera.reshape(-1)
    v[22:25] = camera.camera_center
    return v


def pack_view_host(camera, cache: bool = True) -> torch.Tensor:
    """pack_view on the host (pinned-free CPU tensor), cached on the camera object: reading a camera's device tensors costs a
    device sync, and a training set revisits the same camera objects every epoch."""
    v = getattr(camera, "_b200gs_packed_view", None) if cache else None
    if v is None:
        v = pack_view(camera).detach().cpu()
        if cache:
            try:
                setattr(camera, "_b200gs_packed_view", v)
            except Exception:
                pass
    return v


_HOST_GROUPS = {}


def _host_group(group):
    """A gloo twin of `group` for the per-step camera exchange: 40 floats per rank travel host to host, so the exchange
    neither waits for the GPU nor makes the GPU wait for the host (an NCCL all_gather followed by .cpu() drains the
    device queue at the start of every step).  Created collectively on first use."""
    key = id(group) if group is not None else None
    with _STATE_LOCK:
        g = _HOST_GROUPS.get(key)
    if g is None:
        if dist.get_backend(group) == "gloo":
            g = group if group is not None else dist.group.WORLD
        else:
            ranks = dist.get_process_group_ranks(group) if group is not None else None
            g = dist.new_group(ranks=ranks, backend="gloo")
        with _STATE_LOCK:
            _HOST_GROUPS[key] = g
    return g


class _ShmBoard:
    """Host-side all-gather of a few floats per rank and step through POSIX shared memory, for process groups whose ranks all live
    on one host (the NVSwitch box the peer exchange needs anyway).  A gloo all_gather of 8 x 160 bytes took ~0.8 ms of HOST time per
    step at 8 ranks (profiles/round2_timeline_n8.md) — with ~1.2 ms of other host work per step that made the host, not the GPUs, the
    bottleneck of the 8-GPU step.  Here every rank writes its record and a sequence number into its own slot of an mmap'ed file in
    /dev/shm and reads the others' once their sequence number has arrived: a few microseconds.  Slots are double-buffered by step
    parity: a rank can be at most one step ahead of the slowest reader (it cannot finish step s+1's gather before every rank has
    written its step s+1 record, which a rank does only after reading step s).  Stores and loads are in program order on x86 hosts
    (the sequence number is written after the record and read before it)."""

    SLOT_BYTES = 256 * ((VIEW_FLOATS * 4 + 8 + 255) // 256)

    def __init__(self, group):
        import mmap
        import numpy as np
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        hg = _host_group(group)
        size = 2 * self.world * self.SLOT_BYTES
        path = [None]
        if self.rank == 0:
            name = f"/dev/shm/b200gs_board_{os.getpid()}_{int.from_bytes(os.urandom(6), 'little'):x}"
            fd = os.open(name, os.O_CREAT | os.O_EXCL | os.O_RDWR, 0o600)
            os.ftruncate(fd, size)
            path[0] = name
        dist.broadcast_object_list(path, src=dist.get_global_rank(hg, 0), group=hg)
        if self.rank != 0:
            fd = os.open(path[0], os.O_RDWR)
        self._mm = mmap.mmap(fd, size)
        os.close(fd)
        dist.barrier(group=hg)            # everybody has mapped the file: its name can go (no leak if a rank dies later)
        if self.rank == 0:
            os.unlink(path[0])
        self._buf = np.frombuffer(self._mm, dtype=np.uint8)
        self._np = np
        self.seq = 0

    def _slot(self, parity, j):
        o = (parity * self.world + j) * self.SLOT_BYTES
        return self._buf[o:o + 8].view(self._np.int64), self._buf[o + 8:o + 8 + VIEW_FLOATS * 4].view(self._np.float32)

    def all_gather(self, mine: torch.Tensor) -> torch.Tensor:
        import time
        self.seq += 1
        p = self.seq & 1
        seq_w, rec_w = self._slot(p, self.rank)
        rec_w[:] = mine.numpy()
        seq_w[0] = self.seq
        out = torch.empty(self.world, VIEW_FLOATS, dtype=torch.float32)
        o = out.numpy()
        t0 = None
        for j in range(self.world):
            seq_r, rec_r = self._slot(p, j)
            spins = 0
            while int(seq_r[0]) != self.seq:
                spins += 1
                if spins % 2000 == 0:
                    time.sleep(0)
                    t0 = t0 or time.monotonic()
                    if time.monotonic() - t0 > 600.0:
                        raise RuntimeError(f"b200gs: rank {j} did not post its camera for step {self.seq} within 600 s")
            o[j] = rec_r
        return out


_BOARDS = {}


def _same_host(group) -> bool:
    import socket
    names = [None] * dist.get_world_size(group)
    dist.all_gather_object(names, socket.gethostname(), group=_host_group(group))
    return len(set(names)) == 1 and os.path.isdir("/dev/shm")


def _board(group):
    """The shared-memory board of `group`, or None when its ranks span several hosts (collective on first use)."""
    key = id(group) if group is not None else None
    with _STATE_LOCK:
        if key in _BOARDS:
            return _BOARDS[key]
    board = None
    if os.environ.get("B200GS_SHM_BOARD", "1") != "0":
        ok = _same_host(group)
        if ok:
            try:
                board = _ShmBoard(group)
            except OSError:
                board = None
            flags = [None] * dist.get_world_size(group)
            dist.all_gather_object(flags, board is not None, group=_host_group(group))
            if not all(flags):
                board = None
    with _STATE_LOCK:
        _BOARDS[key] = board
    return board


def gather_views_host(camera, group=None, cache: bool = True) -> torch.Tensor:
    """[world, VIEW_FLOATS] CPU tensor with every rank's camera, no device synchronisation (cache=False re-reads the camera's
    device tensors every call — one sync — for cameras whose pose is being optimised).  Ranks of one host exchange through shared
    memory (_ShmBoard), otherwise through the gloo twin of the group."""
    world = dist.get_world_size(group)
    mine = pack_view_host(camera, cache).contiguous()
    board = _board(group)
    if board is not None:
        return board.all_gather(mine)
    out = torch.empty(world * VIEW_FLOATS, dtype=torch.float32)
    dist.all_gather_into_tensor(out, mine, group=_host_group(group))
    return out.reshape(world, VIEW_FLOATS)


class GatheredView:
    """Host-side view of one gathered camera (what ``cameras`` in the return dict holds)."""

    def __init__(self, flat: torch.Tensor, device):
        f = flat.tolist()
        self.width, self.height = int(f[0]), int(f[1])
        self.fx, self.fy, self.cx, self.cy = f[2], f[3], f[4], f[5]
        self.world_to_camera = flat[6:22].reshape(4, 4)
        self.camera_center_host = flat[22:25]
        self.camera_center = flat[22:25].to(device, non_blocking=True)


_EXCHANGE_CAP = {}      # (group id, world) -> rows per fixed-size block, agreed by all ranks (from the previous step's GLOBAL max)
EXCHANGE_SLACK = 1.15
_STATE_LOCK = threading.RLock()   # guards _EXCHANGE_CAP / _HOST_GROUPS / _PEERS (a viewer thread may render beside the trainer)


def _group_key(group, world):
    return (id(group) if group is not None else None, world)


class _RawDevice:
    """Device memory that was not allocated by torch, exposed through __cuda_array_interface__ (fp32, 1-D)."""

    def __init__(self, ptr: int, n_floats: int):
        self.__cuda_array_interface__ = {"shape": (int(n_floats),), "typestr": "<f4", "data": (int(ptr), False), "version": 2}


class PeerExchange:
    """Exchange buffers every rank of the box can address: each rank owns two receive buffers for splat rows (alternating by
    step) and one for gradient rows, `world * rows_per_block` rows of 12 floats each, allocated with cudaMalloc and mapped into
    the peers with CUDA IPC (b200gs_ipc_*).  Producers store rows straight into the owner's buffer from their pack kernel
    (b200gs_project_pack_multi) and consumers pull gradient rows straight out of the owner's buffer in K8 — NVLink loads/stores from
    our own kernels, no all-to-all.  All methods are collective."""

    def __init__(self, group, device):
        self.group, self.device = group, device
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.rows_per_block = 0
        self.enabled = True
        self.own = {}          # name -> device pointer of my buffer
        self.peers = {}        # name -> [device pointer on rank j for j in range(world)] (own pointer at j == rank)
        self._opened = []
        self.step = 0

    NAMES = ("recv0", "recv1", "vrecv")

    def ensure(self, rows_per_block: int) -> bool:
        """Make room for `rows_per_block` rows per (source, destination) block.  Returns False (on every rank) when peer
        mapping is unavailable on any rank; the caller then keeps the NCCL all-to-all."""
        import ctypes
        from . import _lib
        if not self.enabled or self.world > 8:
            return False
        if rows_per_block <= self.rows_per_block:
            return True
        L = _lib.lib()
        # a peer may still be reading the old buffers (its backward of the previous step pulls gradient rows from here): every rank
        # drains its GPU, then all meet, and only then are the old mappings torn down
        torch.cuda.synchronize(self.device)
        dist.barrier(group=_host_group(self.group))
        self.release()
        want = int(rows_per_block * 1.25) + 4096
        nbytes = self.world * want * ROW_FLOATS * 4
        handles, ok = {}, True
        try:
            for name in self.NAMES:
                ptr_, h = ctypes.c_void_p(), ctypes.create_string_buffer(64)
                _lib.check(L.b200gs_ipc_alloc(nbytes, ctypes.byref(ptr_), h), "b200gs_ipc_alloc")
                self.own[name] = int(ptr_.value)
                handles[name] = bytes(h.raw)
        except Exception:
            ok = False
        gathered = [None] * self.world
        dist.all_gather_object(gathered, (ok, handles), group=_host_group(self.group))
        ok = all(g[0] for g in gathered)
        if ok:
            try:
                for name in self.NAMES:
                    ptrs = []
                    for j in range(self.world):
                        if j == self.rank:
                            ptrs.append(self.own[name])
                            continue
                        ptr_ = ctypes.c_void_p()
                        _lib.check(L.b200gs_ipc_open(gathered[j][1][name], ctypes.byref(ptr_)), "b200gs_ipc_open")
                        self._opened.append(int(ptr_.value))
                        ptrs.append(int(ptr_.value))
                    self.peers[name] = ptrs
            except Exception:
                ok = False
        flags = [None] * self.world
        dist.all_gather_object(flags, ok, group=_host_group(self.group))
        if not all(flags):
            self.release()
            self.enabled = False
            return False
        self.rows_per_block = want
        return True

    def tensor(self, name: str, rows: int) -> torch.Tensor:
        """My own buffer `name` as a [rows, 12] fp32 tensor."""
        return torch.as_tensor(_RawDevice(self.own[name], rows * ROW_FLOATS), device=self.device).view(rows, ROW_FLOATS)

    def peer_tensor(self, name: str, j: int, rows: int) -> torch.Tensor:
        return torch.as_tensor(_RawDevice(self.peers[name][j], rows * ROW_FLOATS), device=self.device).view(rows, ROW_FLOATS)

    def release(self):
        from . import _lib
        L = _lib.lib()
        torch.cuda.synchronize(self.device)
        for p in self._opened:
            L.b200gs_ipc_close(p)
        for p in self.own.values():
            L.b200gs_ipc_free(p)
        self._opened, self.own, self.peers, self.rows_per_block = [], {}, {}, 0


_PEERS = {}


def _peer_exchange(group, device) -> PeerExchange:
    key = (id(group) if group is not None else None, str(device))
    with _STATE_LOCK:
        pe = _PEERS.get(key)
        if pe is None:
            pe = _PEERS[key] = PeerExchange(group, device)
    return pe


class _ShardStep:
    """What the two autograd nodes of one sharded step share (buffers of the projection, the exchange and the raster)."""
    __slots__ = ("views", "cam_views", "rank", "world", "group", "n", "aa", "sh_degree", "peer", "xy", "depth", "conic", "rgb", "opac", "radii",
                 "clamped", "row_index", "fixed_cap", "counts", "recv", "binning", "final_T", "n_contrib", "hw", "v_rows", "v_send", "parity",
                 "peer_mode", "xys_refs", "want_xy", "plan_cap", "plan_peer", "d_count", "send_rows", "params")


def _project_shard(st: _ShardStep, means, log_scales, raw_quats, ol, shs_dc, shs_rest):
    """K1 of the shard for all cameras of the step: one multi-view launch (<= 8 cameras), else one launch per camera."""
    import ctypes
    from . import ops
    from ._lib import B200gsView, check, lib, ptr
    L = lib()
    dev, n, world = means.device, st.n, st.world
    wn = world * n
    f32 = dict(dtype=torch.float32, device=dev)
    st.xy, st.depth, st.conic = torch.empty(wn, 2, **f32), torch.empty(wn, **f32), torch.empty(wn, 3, **f32)
    st.rgb, st.opac = torch.empty(wn, 3, **f32), torch.empty(wn, **f32)
    st.radii = torch.empty(wn, dtype=torch.int32, device=dev)
    st.clamped = torch.empty(wn, dtype=torch.uint8, device=dev)
    st.cam_views = [ops._copy_view(v, sh_degree=int(st.sh_degree), sh_stride=int(shs_dc.shape[1] + shs_rest.shape[1])) for v in st.views]
    stream = ops._stream()
    with ops._stage("project_fwd"):
        if world <= 8:
            arr = (B200gsView * world)(*st.cam_views)
            check(L.b200gs_project_fwd_raw_multi(arr, world, n, ptr(means), ptr(log_scales), ptr(raw_quats), ptr(ol), ptr(shs_dc), ptr(shs_rest),
                                                 int(st.aa), ptr(st.xy), ptr(st.depth), ptr(st.radii), ptr(st.conic), ptr(st.rgb), ptr(st.clamped),
                                                 ptr(st.opac), stream), "b200gs_project_fwd_raw_multi")
        else:
            tiles = torch.empty(n, dtype=torch.int32, device=dev)
            comp = torch.empty(n, **f32)
            for j, v in enumerate(st.cam_views):
                o = j * n
                check(L.b200gs_project_fwd_raw(ctypes.byref(v), n, ptr(means), ptr(log_scales), ptr(raw_quats), ptr(ol), ptr(shs_dc),
                                               ptr(shs_rest), int(st.aa), st.xy.data_ptr() + 8 * o, st.depth.data_ptr() + 4 * o,
                                               st.radii.data_ptr() + 4 * o, st.conic.data_ptr() + 12 * o, ptr(comp), ptr(tiles),
                                               st.rgb.data_ptr() + 12 * o, st.clamped.data_ptr() + o, st.opac.data_ptr() + 4 * o, stream),
                      "b200gs_project_fwd_raw")


def _project_pack_shard(st: _ShardStep, means, log_scales, raw_quats, ol, shs_dc, shs_rest):
    """K1 of the shard for all cameras FUSED with the packing of the exchange (b200gs_project_pack_multi; fixed-capacity steps, <= 8
    cameras): camera j's visible splats go, as [.,12] rows in Gaussian-index order, straight into this rank's block of camera j's
    owner's receive buffer (peer memory over NVLink) or of a local send buffer (NCCL mode).  Kept locally: mean2D, radii, clamped,
    row_index, and d_count[j] = visible splats of camera j."""
    import ctypes
    from . import ops
    from ._lib import B200gsView, check, lib, ptr
    L = lib()
    dev, n, world, rank, cap = means.device, st.n, st.world, st.rank, st.plan_cap
    wn = world * n
    st.xy = torch.empty(wn, 2, dtype=torch.float32, device=dev)
    st.radii = torch.empty(wn, dtype=torch.int32, device=dev)
    st.clamped = torch.empty(wn, dtype=torch.uint8, device=dev)
    st.row_index = torch.empty(wn, dtype=torch.int32, device=dev)
    st.d_count = torch.empty(world, dtype=torch.int64, device=dev)
    st.depth = st.conic = st.rgb = st.opac = None
    st.cam_views = [ops._copy_view(v, sh_degree=int(st.sh_degree), sh_stride=int(shs_dc.shape[1] + shs_rest.shape[1])) for v in st.views]
    row_bytes = ROW_FLOATS * 4
    if st.plan_peer:
        pe = st.peer
        pe.step += 1
        st.parity = pe.step & 1
        name = "recv1" if st.parity else "recv0"
        dst = [pe.peers[name][j] + rank * cap * row_bytes for j in range(world)]      # my block in camera j's owner's buffer
        st.send_rows = None
    else:
        st.send_rows = torch.empty(world * cap, ROW_FLOATS, dtype=torch.float32, device=dev)
        dst = [st.send_rows.data_ptr() + j * cap * row_bytes for j in range(world)]
    ws = torch.empty(int(L.b200gs_project_pack_workspace_bytes(world, n)), dtype=torch.uint8, device=dev)
    arr = (B200gsView * world)(*st.cam_views)
    dst_arr = (ctypes.c_void_p * world)(*dst)
    with ops._stage("project_fwd"):
        check(L.b200gs_project_pack_multi(arr, world, n, ptr(means), ptr(log_scales), ptr(raw_quats), ptr(ol), ptr(shs_dc), ptr(shs_rest),
                                          int(st.aa), ptr(st.xy), ptr(st.radii), ptr(st.clamped), ptr(st.row_index), dst_arr, cap, ptr(ws),
                                          ws.numel(), ptr(st.d_count), ops._stream()), "b200gs_project_pack_multi")


class _ProjectShard(torch.autograd.Function):
    """Node A of a sharded step: raw shard parameters -> the mean2D of every (camera, Gaussian) pair, one [n,2] tensor per camera
    (graph tensors: the distributed density controller calls retain_grad() on them, distributed_vanilla_density_controller.py:
    16-22).  Everything else the projection produces travels to node B through the shared _ShardStep.  backward = K8 for all
    cameras in one launch, reading its cotangents straight from the gradient rows node B's backward obtained (local buffer
    after the return all-to-all, or the camera owners' buffers over NVLink)."""

    @staticmethod
    def forward(ctx, means, log_scales, raw_quats, opac_logits, shs_dc, shs_rest, st: _ShardStep):
        means, log_scales, raw_quats = means.contiguous(), log_scales.contiguous(), raw_quats.contiguous()
        ol = opac_logits.contiguous().reshape(-1)
        shs_dc, shs_rest = shs_dc.contiguous(), shs_rest.contiguous()
        if st.plan_cap:
            _project_pack_shard(st, means, log_scales, raw_quats, ol, shs_dc, shs_rest)
        else:
            _project_shard(st, means, log_scales, raw_quats, ol, shs_dc, shs_rest)
        st.params = (means, log_scales, raw_quats, ol, shs_dc, shs_rest)      # for node B's overflow fallback; dropped there
        ctx.st = st
        ctx.opac_shape = tuple(opac_logits.shape)
        ctx.save_for_backward(means, log_scales, raw_quats, ol, shs_dc, shs_rest)
        return tuple(st.xy[j * st.n:(j + 1) * st.n] for j in range(st.world))

    @staticmethod
    def backward(ctx, *_grad_xys):
        # the mean2D cotangents are columns 0..1 of the gradient rows already (node B handed them to autograd only so that
        # `.grad` of the per-camera tensors gets populated); K8 reads the full rows
        import ctypes
        from . import ops
        from ._lib import B200gsView, check, lib, ptr
        L = lib()
        st = ctx.st
        means, log_scales, raw_quats, ol, shs_dc, shs_rest = ctx.saved_tensors
        dev, n, world = means.device, st.n, st.world
        if st.v_rows is None:
            raise RuntimeError("b200gs sharded renderer: backward of the projection ran before the rasterization's backward")
        f32 = dict(dtype=torch.float32, device=dev)
        v_means, v_ls, v_q = torch.empty(n, 3, **f32), torch.empty(n, 3, **f32), torch.empty(n, 4, **f32)
        v_ol, v_dc, v_rest = torch.empty(n, **f32), torch.empty_like(shs_dc), torch.empty_like(shs_rest)
        stream = ops._stream()
        with ops._stage("project_bwd"):
            if world <= 8:
                arr = (B200gsView * world)(*st.cam_views)
                rows = (ctypes.c_void_p * world)(*[int(p) for p in st.v_rows])
                check(L.b200gs_project_bwd_rows_multi(arr, world, n, ptr(means), ptr(log_scales), ptr(raw_quats), ptr(ol), ptr(shs_dc), ptr(shs_rest),
                                                      int(st.aa), ptr(st.radii), ptr(st.clamped), ptr(st.row_index), rows, ptr(v_means), ptr(v_ls),
                                                      ptr(v_q), ptr(v_ol), ptr(v_dc), ptr(v_rest), stream), "b200gs_project_bwd_rows_multi")
            else:
                for j, view in enumerate(st.cam_views):
                    check(L.b200gs_project_bwd_rows(ctypes.byref(view), n, ptr(means), ptr(log_scales), ptr(raw_quats), ptr(ol), ptr(shs_dc),
                                                    ptr(shs_rest), int(st.aa), st.radii.data_ptr() + 4 * j * n, st.clamped.data_ptr() + j * n,
                                                    st.row_index.data_ptr() + 4 * j * n, int(st.v_rows[j]), 1 if j > 0 else 0, ptr(v_means),
                                                    ptr(v_ls), ptr(v_q), ptr(v_ol), ptr(v_dc), ptr(v_rest), None, 0, stream), "b200gs_project_bwd_rows")
        st.v_send = None
        return v_means, v_ls, v_q, v_ol.reshape(ctx.opac_shape), v_dc, v_rest, None


class _ExchangeRasterize(torch.autograd.Function):
    """Node B of a sharded step: (projected shard of every camera) -> this rank's image.
    forward : device-side stable compaction of the visible splats into [.,12] rows, written either into a local send buffer
              (-> ONE all_to_all_single) or — peer mode — straight into the camera owners' receive buffers over NVLink by the pack
              kernel itself; K2-K7 read the received rows in place, pair buffers sized lazily from the previous step.
              Steady state has NO host sync: every destination gets a fixed-size block of rows (capacity = 1.15 x the previous
              step's GLOBAL maximum, identical on all ranks; unused rows are zero = culled), so no size exchange is needed; this
              step's global maximum (one 8-byte all_reduce, which in peer mode is also the barrier that tells a rank its receive
              buffer is complete) is read back after the rest of the forward has been enqueued and, if it exceeded the capacity
              on ANY rank, ALL ranks redo the forward with the exact, synchronising exchange (first step, or a > 15 % jump).
    backward: K7 accumulates into a [R,12] gradient row buffer; the rows return through the mirrored all_to_all_single, or —
              peer mode — stay where they are and node A's K8 pulls them from the owners after one barrier."""

    @staticmethod
    def forward(ctx, bg, st: _ShardStep, *xys):
        from . import ops
        from ._lib import MODE_GSPLAT, check, lib, ptr
        import ctypes
        L = lib()
        dev = bg.device
        n, world, rank, group = st.n, st.world, st.rank, st.group
        wn = world * n
        stream = ops._stream()
        bg = bg.contiguous()
        f32 = dict(dtype=torch.float32, device=dev)
        gv = st.views[rank]
        W, H = gv.width, gv.height
        key = _group_key(group, world)

        def exact():
            """size exchange + host syncs: first step and overflow fallback (works from the separate arrays of the unfused K1)"""
            st.row_index = torch.empty(wn, dtype=torch.int32, device=dev)
            ws = torch.empty(max(int(L.b200gs_pack_rows_workspace_bytes(wn)), 256), dtype=torch.uint8, device=dev)
            rows = torch.empty(wn, ROW_FLOATS, **f32)          # upper bound; the first sum(V_j) rows are the send buffer
            d_count = torch.empty(1, dtype=torch.int64, device=dev)
            with ops._stage("pack"):
                check(L.b200gs_pack_rows(wn, n, 0, ptr(st.xy), ptr(st.depth), ptr(st.conic), None, ptr(st.opac), ptr(st.rgb), ptr(st.radii),
                                         ptr(ws), ws.numel(), ptr(st.row_index), ptr(rows), ptr(d_count), stream), "b200gs_pack_rows")
            last = torch.arange(1, world + 1, device=dev, dtype=torch.int64) * n - 1
            ends = st.row_index[last].to(torch.int64) + (st.radii[last] > 0).to(torch.int64)     # cumulative visible counts per camera
            counts = torch.empty(2 * world + 1, dtype=torch.int64, device=dev)                   # [send | recv | global max]
            counts[:world] = ends - torch.cat([ends.new_zeros(1), ends[:-1]])
            dist.all_to_all_single(counts[world:2 * world], counts[:world], group=group)
            counts[2 * world] = counts[:world].max()
            dist.all_reduce(counts[2 * world:], op=dist.ReduceOp.MAX, group=group)
            host_counts = counts.cpu().tolist()                                                  # host sync
            send_counts, recv_counts, gmax = host_counts[:world], host_counts[world:2 * world], host_counts[2 * world]
            recv = torch.empty(sum(recv_counts), ROW_FLOATS, **f32)
            dist.all_to_all_single(recv, rows[:sum(send_counts)], output_split_sizes=recv_counts, input_split_sizes=send_counts, group=group)
            binning, out = ops.bin_and_blend_rows(MODE_GSPLAT, W, H, recv, bg, True)
            cap = int(gmax * EXCHANGE_SLACK) + 1024
            with _STATE_LOCK:
                _EXCHANGE_CAP[key] = cap
            if st.peer is not None:
                st.peer.ensure(cap)                      # collective: every rank takes this branch in the same step
            return (send_counts, recv_counts), recv, binning, out

        cap = st.plan_cap
        result = None
        st.fixed_cap, st.peer_mode = 0, False
        if cap:
            # node A's fused kernel has already stored every rank's rows where they are consumed (peer mode) or into the send buffer.
            # ONE small collective: all-gather of the per-camera row counts -> the valid rows of each received block (no padding pass),
            # the global maximum (overflow check), and — peer mode — the barrier: when it completes here, every rank's K1 (which
            # precedes its all-gather in stream order) has finished storing into this rank's buffer.
            use_peer = st.plan_peer
            all_counts = torch.empty(world * world, dtype=torch.int64, device=dev)             # [source rank][camera]
            dist.all_gather_into_tensor(all_counts, st.d_count, group=group)
            gmax_dev = all_counts.max().reshape(1)
            gmax_host = ops._host_counts()
            check(L.b200gs_publish_i64(ptr(gmax_dev), gmax_host.data_ptr(), 1, stream), "b200gs_publish_i64")
            published = torch.cuda.Event()
            published.record()
            recv_counts = all_counts.view(world, world)[:, rank].clamp(max=cap).contiguous()
            if use_peer:
                recv = st.peer.tensor("recv1" if st.parity else "recv0", world * cap)
            else:
                recv = torch.empty(world * cap, ROW_FLOATS, **f32)
                dist.all_to_all_single(recv, st.send_rows, group=group)
                st.send_rows = None
            binning, out = ops.bin_and_blend_rows(MODE_GSPLAT, W, H, recv, bg, True, False, recv_counts, cap)
            published.synchronize()                           # long past: the blend has been enqueued behind it
            gmax = int(gmax_host[0])
            ops._return_host_counts(gmax_host)
            if gmax <= cap:                                   # same verdict on every rank: gmax is global
                with _STATE_LOCK:
                    _EXCHANGE_CAP[key] = int(gmax * EXCHANGE_SLACK) + 1024
                result = (None, recv, binning, out)
                st.fixed_cap, st.peer_mode = cap, use_peer
            else:                                             # a > 15 % jump: redo with the unfused projection and the exact exchange
                _project_shard(st, *st.params)
        if result is None:
            st.fixed_cap, st.peer_mode = 0, False             # the exact step exchanges through NCCL in both directions
            result = exact()
        st.params = None
        st.counts, st.recv, st.binning, (image, st.final_T, st.n_contrib) = result
        st.hw = (H, W)
        st.xy = st.depth = st.conic = st.rgb = st.opac = None      # consumed: the rows hold everything from here on
        st.v_rows = None
        ctx.st = st
        ctx.save_for_backward(bg)
        return image

    @staticmethod
    def backward(ctx, v_image):
        from ._lib import MODE_GSPLAT, check, lib, ptr
        from . import ops
        L = lib()
        st = ctx.st
        (bg,) = ctx.saved_tensors
        dev = bg.device
        n, world, rank, group = st.n, st.world, st.rank, st.group
        stream = ops._stream()
        H, W = st.hw
        v_image = v_image.contiguous()
        cap = st.fixed_cap
        peer_mode = st.peer_mode
        if peer_mode:
            v_recv = st.peer.tensor("vrecv", world * cap)
            v_recv.zero_()
        else:
            v_recv = torch.zeros_like(st.recv)
        with ops._stage("blend_bwd"):
            check(L.b200gs_blend_bwd_rows(MODE_GSPLAT, W, H, ptr(st.binning.tile_ranges), ptr(st.binning.sorted_ids), ptr(st.recv), ptr(bg),
                                          ptr(st.final_T), ptr(st.n_contrib), ptr(v_image), 3, 1, None, 1.0, 1.0, ptr(v_recv), stream), "b200gs_blend_bwd_rows")
        grads = []

        def xy_grad(j, rows, shift):
            """d loss / d mean2D of camera j's projections = columns 0..1 of their gradient rows.  Only materialised when somebody
            will read it (`retain_grad()` on the per-camera xys, as the distributed density controller does, or want_xy_grads): node
            A's K8 reads the full rows itself.  Gather without a host sync (no boolean-mask indexing)."""
            ref = st.xys_refs[j]() if st.xys_refs is not None else None
            if not st.want_xy and (ref is None or not ref.retains_grad):
                return None
            idx = st.row_index[j * n:(j + 1) * n]
            vis = (st.radii[j * n:(j + 1) * n] > 0) & (idx >= 0)
            k = (idx.long() + shift).clamp_(0, rows.shape[0] - 1)
            return rows[:, 0:2][k] * vis.unsqueeze(1)

        if peer_mode:
            # one barrier: every camera owner's K7 is done.  Entry (j, i) with row_index = j*cap + k lives at row rank*cap + k of owner
            # j's buffer: shift each base pointer so that K8 can index it with row_index directly.
            token = torch.zeros(1, dtype=torch.int32, device=dev)
            dist.all_reduce(token, group=group)
            pe = st.peer
            st.v_rows = [pe.peers["vrecv"][j] + (rank * cap - j * cap) * ROW_FLOATS * 4 for j in range(world)]
            st.v_send = v_recv
            for j in range(world):
                grads.append(xy_grad(j, pe.peer_tensor("vrecv", j, world * cap), rank * cap - j * cap))
        else:
            if cap:
                v_send = torch.empty_like(v_recv)
                dist.all_to_all_single(v_send, v_recv, group=group)
            else:
                send_counts, recv_counts = st.counts
                v_send = torch.empty(max(sum(send_counts), 1), ROW_FLOATS, dtype=torch.float32, device=dev)
                dist.all_to_all_single(v_send[:sum(send_counts)], v_recv, output_split_sizes=send_counts, input_split_sizes=recv_counts, group=group)
            st.v_send = v_send
            st.v_rows = [v_send.data_ptr()] * world
            for j in range(world):
                grads.append(xy_grad(j, v_send, 0))
        st.recv = st.binning = st.final_T = st.n_contrib = None
        return (None, None) + tuple(grads)


@dataclass
class B200DistributedRendererConfig:
    """YAML-selectable config, the fields of `GSplatDistributedRenderer` (gsplat_distributed_renderer.py:16-38)."""
    block_size: int = 16
    anti_aliased: bool = True
    filter_2d_kernel_size: float = 0.3
    tile_based_culling: bool = True
    redistribute_interval: int = 1000
    redistribute_until: int = 15_000
    redistribute_threshold: float = 1.1
    fused: bool = True
    peer_exchange: bool = True

    def instantiate(self, *args, **kwargs):
        return B200DistributedRenderer(config=self)


def replace_tensors_to_properties(tensors: Dict[str, torch.Tensor], optimizers) -> Dict[str, torch.nn.Parameter]:
    """New parameter tensors into the optimizers' single-tensor param groups, optimizer state reset; properties that no optimizer
    holds become frozen Parameters.  Same contract as DensityControllerUtils.replace_tensors_to_properties with selector=None
    (internal/density_controllers/density_controller.py:148-209), which the reference's training_setup uses for sharding."""
    new_parameters = {}
    for opt in optimizers:
        for group in opt.param_groups:
            tensor = tensors.get(group["name"], None)
            if tensor is None:
                continue
            assert len(group["params"]) == 1
            assert group["name"] not in new_parameters, "parameter `{}` appears in multiple optimizers".format(group["name"])
            stored_state = opt.state.get(group["params"][0], None)
            new_param = torch.nn.Parameter(tensor.requires_grad_(True))
            if stored_state is not None:
                stored_state["exp_avg"] = torch.zeros_like(tensor)
                stored_state["exp_avg_sq"] = torch.zeros_like(tensor)
                del opt.state[group["params"][0]]
                group["params"][0] = new_param
                opt.state[new_param] = stored_state
            else:
                group["params"][0] = new_param
            new_parameters[group["name"]] = new_param
    for k, v in tensors.items():
        if k not in new_parameters:
            new_parameters[k] = torch.nn.Parameter(v, requires_grad=False)
    return new_parameters


def all_to_all_rows_by_destination(local: torch.Tensor, destination: torch.Tensor, recv_counts: List[int], world: int, group=None) -> torch.Tensor:
    """Rows of `local` go to rank destination[i]; returns the rows this rank receives, concatenated in source-rank order
    (gsplat_distributed_renderer.py:464-479, with one all_to_all_single instead of the list form)."""
    order = torch.argsort(destination, stable=True)
    send = local[order].contiguous()
    send_counts = torch.bincount(destination, minlength=world).tolist()
    out = local.new_empty((int(sum(recv_counts)),) + tuple(local.shape[1:]))
    dist.all_to_all_single(out, send, output_split_sizes=[int(c) for c in recv_counts], input_split_sizes=[int(c) for c in send_counts], group=group)
    return out


class B200DistributedRenderer(Renderer):
    """Drop-in for ``GSplatDistributedRendererImpl`` (gsplat_distributed_renderer.py:41-516): `pc` holds THIS rank's shard;
    ``training_setup`` shards the model and its optimizers by contiguous index ranges (:63-118), ``forward`` returns this rank's
    image plus what the distributed density controller reads — ``projection_results_list`` (per camera: radii, xys (graph tensor:
    ``retain_grad()`` / ``.grad`` work), depths, conics, compensation), ``visible_mask_list``, ``cameras``,
    ``xys_grad_scale_required`` (:407-414; distributed_vanilla_density_controller.py:16-47) — and ``after_training_step``
    rebalances the shards incl. the Adam moments (:416-510)."""

    def __init__(self, anti_aliased: bool = True, group=None, fused: bool = True, want_xy_grads: bool = False, cache_cameras: bool = True,
                 config: Optional[B200DistributedRendererConfig] = None, peer_exchange: bool = True):
        """fused: when `pc` is the vanilla Gaussian model, run the step as two autograd nodes on the raw parameters (multi-view K1 /
        K8, device-side packing, rows consumed in place, no host sync in the steady state); otherwise the generic path below,
        built from the same ops the single-GPU renderers use.  peer_exchange: store / pull the rows through peer-mapped buffers
        over NVLink instead of NCCL all-to-alls (falls back to NCCL when CUDA IPC is unavailable or the group has > 8 ranks)."""
        super().__init__()
        self.config = config if config is not None else B200DistributedRendererConfig(anti_aliased=anti_aliased, fused=fused,
                                                                                        peer_exchange=peer_exchange)
        self.anti_aliased = self.config.anti_aliased
        self.group = group
        self.fused = self.config.fused
        # B200GS_PEER_EXCHANGE=0: measurement switch (NCCL all-to-alls instead of the peer-mapped buffers), same on every rank
        self.peer_exchange = self.config.peer_exchange and os.environ.get("B200GS_PEER_EXCHANGE", "1") != "0"
        self.want_xy_grads = want_xy_grads   # kept for callers of the previous interface: the per-camera gradients are `.grad` of the xys now
        self.cache_cameras = cache_cameras   # False when camera poses are optimised (the packed host view is cached on the camera)
        self.world_size, self.global_rank = 1, 0
        self.on_density_changed = None

    # ---- lifecycle (renderer.py:90-100; gaussian_splatting.py:657) ------------------------------------------------------
    def training_setup(self, module):
        self.world_size = module.trainer.world_size
        self.global_rank = module.trainer.global_rank
        n_gaussians = module.gaussian_model.n_gaussians
        lo, hi = shard_range(n_gaussians, self.world_size, self.global_rank)
        new_param_tensors = {name: value[lo:hi] for name, value in module.gaussian_model.properties.items()}
        module.gaussian_model.properties = replace_tensors_to_properties(new_param_tensors, module.gaussian_optimizers)
        self.on_density_changed = module.density_updated_by_renderer
        self.on_density_changed()
        print(f"rank={self.global_rank}, l={lo}, r={hi}")
        return None, None

    def after_training_step(self, step: int, module):
        c = self.config
        if c.redistribute_interval < 0 or step >= c.redistribute_until or step % c.redistribute_interval != 0:
            return
        self.redistribute(module)

    def redistribute(self, module):
        with torch.no_grad():
            counts = [0 for _ in range(self.world_size)]
            dist.all_gather_object(counts, int(module.gaussian_model.get_xyz.shape[0]), group=self.group)
            if min(counts) * self.config.redistribute_threshold >= max(counts):
                return
            self.random_redistribute(module)

    def random_redistribute(self, module):
        """Every Gaussian (parameters AND Adam moments) moves to a uniformly random rank (gsplat_distributed_renderer.py:447-510)."""
        model, optimizers = module.gaussian_model, module.gaussian_optimizers
        world = self.world_size
        dev = model.get_xyz.device
        destination = torch.randint(0, world, (model.get_xyz.shape[0],), device=dev)
        send_counts = torch.bincount(destination, minlength=world)
        recv_counts = torch.empty_like(send_counts)
        dist.all_to_all_single(recv_counts, send_counts, group=self.group)
        recv_counts = recv_counts.tolist()

        def move(t):
            return all_to_all_rows_by_destination(t, destination, recv_counts, world, self.group)

        new_tensors = {}
        for opt in optimizers:
            for group in opt.param_groups:
                assert len(group["params"]) == 1
                old = group["params"][0]
                state = opt.state.get(old, None)
                new_param = torch.nn.Parameter(move(old.detach()).requires_grad_(True))
                if state is not None:
                    state["exp_avg"] = move(state["exp_avg"])
                    state["exp_avg_sq"] = move(state["exp_avg_sq"])
                    del opt.state[old]
                    opt.state[new_param] = state
                group["params"][0] = new_param
                new_tensors[group["name"]] = new_param
        for name in model.get_property_names():
            if name not in new_tensors:
                new_tensors[name] = move(model.get_property(name))
        model.properties = new_tensors
        if self.on_density_changed is not None:
            self.on_density_changed()

    def get_available_outputs(self):
        return {"rgb": RendererOutputInfo("render")}

    # ---- forward ---------------------------------------------------------------------------------------------------------
    def _forward_fused(self, raw, viewpoint_camera, pc, bg_color, scaling_modifier):
        from . import ops
        from ._lib import MODE_GSPLAT
        world = dist.get_world_size(self.group)
        rank = dist.get_rank(self.group)
        dev = bg_color.device
        flat = gather_views_host(viewpoint_camera, self.group, self.cache_cameras)
        cams = [GatheredView(flat[j], dev) for j in range(world)]
        st = _ShardStep()
        st.views = [ops.make_view(MODE_GSPLAT, gv.width, gv.height, fx=gv.fx, fy=gv.fy, cx=gv.cx, cy=gv.cy, viewmatrix=gv.world_to_camera,
                                  campos=gv.camera_center_host, scale_modifier=scaling_modifier, eps2d=self.config.filter_2d_kernel_size)
                    for gv in cams]
        st.rank, st.world, st.group, st.n = rank, world, self.group, int(raw["means"].shape[0])
        st.aa, st.sh_degree = bool(self.anti_aliased), int(pc.active_sh_degree)
        st.peer = _peer_exchange(self.group, dev) if (self.peer_exchange and bg_color.is_cuda and dist.get_backend(self.group) == "nccl") else None
        st.v_rows = st.v_send = st.d_count = st.send_rows = st.params = None
        with _STATE_LOCK:
            cap = _EXCHANGE_CAP.get(_group_key(self.group, world))
        st.plan_cap = int(cap) if (cap and world <= 8 and bg_color.is_cuda) else 0        # fixed-capacity step: K1 fused with the packing
        st.plan_peer = bool(st.plan_cap and st.peer is not None and st.peer.ensure(st.plan_cap))
        st.xys_refs, st.want_xy = None, bool(self.want_xy_grads)
        xys = _ProjectShard.apply(raw["means"], raw["scales"], raw["rotations"], raw["opacities"], raw["shs_dc"], raw["shs_rest"], st)
        st.xys_refs = [weakref.ref(x) for x in xys]
        n = st.n
        # (radii, means2d, depths, conics, compensations) per camera like the reference; its consumers read [0] and [1] only
        # (distributed_vanilla_density_controller.py:28-37) — depths / conics live in the exchanged rows and are not duplicated here
        projection_results_list = [(st.radii[j * n:(j + 1) * n], xys[j], None, None, None) for j in range(world)]
        visible_mask_list = [r[0] > 0 for r in projection_results_list]
        img = _ExchangeRasterize.apply(bg_color, st, *xys)
        return {
            "render": img.permute(2, 0, 1),
            "cameras": cams,
            "projection_results_list": projection_results_list,
            "visible_mask_list": visible_mask_list,
            "xys_grad_scale_required": True,
        }

    def forward(self, viewpoint_camera, pc, bg_color: torch.Tensor, scaling_modifier=1.0, render_types: list = None, **kwargs):
        from . import ops
        from ._lib import MODE_GSPLAT
        if self.fused:
            from .renderers import _raw_parameters
            raw = _raw_parameters(pc)
            if raw is not None:
                return self._forward_fused(raw, viewpoint_camera, pc, bg_color, scaling_modifier)
        world = dist.get_world_size(self.group)
        rank = dist.get_rank(self.group)
        dev = bg_color.device

        # 1. every rank learns all W cameras
        flat = gather_views_host(viewpoint_camera, self.group, self.cache_cameras)
        views = [GatheredView(flat[j], dev) for j in range(world)]

        # 2. project my shard to every camera, colours for every camera
        means, scales, opacities = pc.get_xyz, pc.get_scaling, pc.get_opacity
        quats = pc.get_rotation
        quats = quats / quats.norm(dim=-1, keepdim=True)
        feats = pc.get_features
        rows_per_dest, projection_results_list, visible_mask_list = [], [], []
        for j, gv in enumerate(views):
            view = ops.make_view(MODE_GSPLAT, gv.width, gv.height, fx=gv.fx, fy=gv.fy, cx=gv.cx, cy=gv.cy,
                                 viewmatrix=gv.world_to_camera, scale_modifier=scaling_modifier)
            xys, depths, radii, conics, comp, tiles, _ = ops.project_gaussians(means, scales, scaling_modifier, quats, None, 0, 0, 0, 0,
                                                                              gv.height, gv.width, view=view)
            visible = radii > 0
            rgbs = torch.clamp(ops.spherical_harmonics(pc.active_sh_degree, means.detach() - gv.camera_center, feats) + 0.5, min=0.0)
            rows_per_dest.append(pack_rows(xys, depths, conics, comp, opacities, rgbs, radii, visible))
            projection_results_list.append((radii, xys, depths, conics, comp, visible))
            visible_mask_list.append(visible)

        # 3. all-to-all of the visible splats
        rows, recv_counts = exchange_rows(rows_per_dest, self.group)

        # 4. local rasterization of my camera
        xys, depths, conics, comp, opac, rgbs, radii = unpack_rows(rows)
        if self.anti_aliased:
            opac = opac * comp
        gv = views[rank]
        img = ops.rasterize_gaussians(xys, depths, radii, conics, None, rgbs, opac, gv.height, gv.width, 16, bg_color, False)
        return {
            "render": img.permute(2, 0, 1),
            "cameras": views,
            "projection_results_list": projection_results_list,
            "visible_mask_list": visible_mask_list,
            "xys_grad_scale_required": True,
            "n_received": recv_counts,
        }
