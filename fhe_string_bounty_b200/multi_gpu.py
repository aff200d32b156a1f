"""Multi-GPU execution of the string operations (SURVEY.md 8e): keys replicated, haystack windows / radix blocks
partitioned across ranks, and ONE exchange at the narrow end of the tree -- for the boolean trees (eq, contains) a sum of each
rank's boolean block; for the lexicographic comparisons a gather of each rank's sign block followed by the pairwise sign tree;
for find a gather of each rank's (found, first index) followed by a two-level first-rank selection; for the elementwise case
conversions an optional gather of the converted chars and nothing else.  u64 wrap-around addition of LWE words IS homomorphic
addition, so the summed block holds the count of ranks whose share matched (<= total_mod - 1) and one final LUT
(x != 0 / x == ranks) finishes the tree on every rank.  What crosses the link is 16 KiB per block.

The sharding logic is written once against a small `Comm` interface with two implementations:

* DeviceComm -- the product path.  A rank's share runs as a device-resident program (tfhe_b200_program_run_device), its result rows
  are written straight into the engine's symmetric exchange buffer, ONE engine kernel publishes / waits / pulls the peers' rows over
  NVLink peer memory (csrc/exchange.cu) and the finishing program consumes them -- no host round trip and no collective-library call
  between the input upload and the result download.  exchange="nccl" routes the same tensors through torch.distributed instead (used
  as the cross-check of the peer exchange and where CUDA IPC is unavailable).
* HostComm -- the CPU tests: `execute(program, inputs) -> outputs` is the oracle executor, the collectives are gloo.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch
import torch.distributed as dist

from ._native import Engine, NativeError
from .host import Program


def shard_range(n_items: int, rank: int, world: int) -> tuple[int, int]:
    """contiguous, balanced partition of n_items (first ranks get the remainder)"""
    base, rem = divmod(n_items, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


# ---- communication / execution back ends ----------------------------------------------------------------------------------------

class HostComm:
    """numpy blocks on the host; programs run through `execute(program, inputs)`; collectives on CPU tensors (gloo)."""

    def __init__(self, execute, rank: int | None = None, world: int | None = None):
        self.execute = execute
        self.min_shard_width = 0          # the CPU tests shard everything: they test the sharding logic, not its pay-off
        self.rank = dist.get_rank() if rank is None else rank
        self.world = dist.get_world_size() if world is None else world
        self._programs: dict = {}

    def program(self, op: str, args: tuple, params: dict) -> Program:
        key = (op, tuple(args), tuple(sorted(params.items())))
        if key not in self._programs:
            self._programs[key] = Program(op, args, params=params)
        return self._programs[key]

    def run(self, prog: Program, inputs):
        if isinstance(inputs, (list, tuple)):          # pieces of the input block array, in order
            inputs = np.concatenate([np.asarray(x, dtype=np.uint64).reshape(len(x), -1) for x in inputs])
        return self.execute(prog, np.ascontiguousarray(inputs, dtype=np.uint64))

    def zeros(self, rows: int, lwe_len: int):
        return np.zeros((rows, lwe_len), dtype=np.uint64)

    def padded(self, blocks, rows: int, lwe_len: int):
        out = np.zeros((rows, lwe_len), dtype=np.uint64)
        out[:len(blocks)] = blocks
        return out

    def all_reduce(self, blocks):
        """sum of LWE ciphertexts over ranks == homomorphic addition (wrapping u64 via two's-complement int64)"""
        if self.world == 1:
            return blocks
        t = torch.from_numpy(np.ascontiguousarray(blocks).view(np.int64).copy())
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return t.numpy().view(np.uint64)

    def all_gather(self, blocks):
        """every rank's (m, lwe_len) rows -> (world, m, lwe_len) on every rank"""
        t = torch.from_numpy(np.ascontiguousarray(blocks).view(np.int64).copy())
        out = torch.empty((self.world * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype)
        dist.all_gather_into_tensor(out, t)
        return out.numpy().view(np.uint64).reshape((self.world,) + tuple(t.shape))

    def rows(self, x, sel):
        return np.ascontiguousarray(x[sel])

    def to_host(self, x) -> np.ndarray:
        return x


class PeerExchange:
    """tfhe_b200_exchange_* (csrc/exchange.cu): the engine's own exchange over NVLink peer memory.  The 64-byte CUDA IPC handles are
    handed round with torch.distributed (any transport would do; this happens once, outside every timed path)."""

    def __init__(self, eng: Engine, rank: int, world: int, max_rows: int, group=None):
        self.eng, self.lib, self.rank, self.world, self.max_rows = eng, eng.lib, rank, world, max_rows
        h = C.c_void_p()
        eng._check(self.lib.tfhe_b200_exchange_create(eng.h, rank, world, max_rows, C.byref(h)))
        self.h = h
        if world > 1:
            mine = np.zeros(64, dtype=np.uint8)
            eng._check(self.lib.tfhe_b200_exchange_handle(self.h, mine.ctypes.data))
            t = torch.from_numpy(mine).to(f"cuda:{eng.device}") if dist.get_backend(group) == "nccl" else torch.from_numpy(mine)
            out = torch.empty(world * 64, dtype=torch.uint8, device=t.device)
            dist.all_gather_into_tensor(out, t, group=group)
            handles = np.ascontiguousarray(out.cpu().numpy())
            eng._check(self.lib.tfhe_b200_exchange_attach(self.h, handles.ctypes.data))

    @classmethod
    def local(cls, eng: Engine, rank: int, world: int, max_rows: int) -> "PeerExchange":
        """an exchange of a rank driven by this process; the caller attaches the group (tfhe_b200_exchange_attach_local)"""
        ex = cls.__new__(cls)
        ex.eng, ex.lib, ex.rank, ex.world, ex.max_rows = eng, eng.lib, rank, world, max_rows
        h = C.c_void_p()
        eng._check(eng.lib.tfhe_b200_exchange_create(eng.h, rank, world, max_rows, C.byref(h)))
        ex.h = h
        return ex

    def send_rows_ptr(self) -> int:
        p = C.c_void_p()
        self.eng._check(self.lib.tfhe_b200_exchange_send_rows(self.h, C.byref(p)))
        return p.value

    def gather_stride(self, rows: int) -> int:
        return int(self.lib.tfhe_b200_exchange_gather_stride(self.h, rows))

    def all_gather(self, rows: int, d_out: int, stream: int):
        self.eng._check(self.lib.tfhe_b200_exchange_all_gather(self.h, rows, d_out, stream))

    def all_reduce_sum(self, rows: int, d_out: int, stream: int):
        self.eng._check(self.lib.tfhe_b200_exchange_all_reduce_sum(self.h, rows, d_out, stream))

    def close(self):
        if getattr(self, "h", None):
            self.lib.tfhe_b200_exchange_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _on_own_stream(method):
    """run a DeviceComm method on the comm's own CUDA stream, ordered after whatever the caller's current stream has enqueued (the C ABI
    reads a NULL stream handle as "the context's stream", so torch's default stream must never be passed down)"""
    import functools

    @functools.wraps(method)
    def wrapper(self, *args, **kwargs):
        cur = torch.cuda.current_stream(self.dev)
        if cur != self.stream:
            self.stream.wait_stream(cur)
        with torch.cuda.stream(self.stream):
            return method(self, *args, **kwargs)
    return wrapper


class DeviceComm:
    """Device-resident execution on one Engine per rank.  Blocks are int64 CUDA tensors of shape (rows, k*N+1) (the bit pattern of the
    u64 words); everything is enqueued on the comm's own CUDA stream and nothing synchronises until to_host()."""

    def __init__(self, eng: Engine, rank: int | None = None, world: int | None = None, exchange: str = "peer", max_rows: int = 16):
        if exchange not in ("peer", "nccl"):
            raise ValueError("exchange must be 'peer' or 'nccl'")
        self.eng = eng
        self.dev = torch.device(f"cuda:{eng.device}")
        self.stream = torch.cuda.Stream(device=self.dev)
        # A tree whose widest level fits one ciphertext per SM is a chain of narrow-level launches whatever its width: splitting it
        # over ranks only adds the exchange and the finishing level (round 1: eq of 8-char strings 113 ops/s on one GPU, 84 on two).
        self.min_shard_width = torch.cuda.get_device_properties(self.dev).multi_processor_count
        self.rank = (dist.get_rank() if dist.is_initialized() else 0) if rank is None else rank
        self.world = (dist.get_world_size() if dist.is_initialized() else 1) if world is None else world
        self.exchange = exchange
        self.max_rows = max_rows
        self.L = eng.p.big_len
        self._programs: dict = {}
        self._pending_send: tuple | None = None     # (rows,) of the result just written into the exchange send area
        self._host_out: dict = {}                    # page-locked result buffers, by shape
        self._group = None                           # set by local_group(): several ranks of one process on one GPU
        self.peer = PeerExchange(eng, self.rank, self.world, max_rows) if (exchange == "peer" and self.world > 1) else None
        self._program_peer: PeerExchange | None = None   # the exchange of run_program_sharded, sized by the shard plan on first need

    @classmethod
    def local_group(cls, engines: list, max_rows: int = 16) -> list:
        """several ranks driven by ONE process on ONE GPU (one Engine per rank; the single-GPU tests): the exchange buffers are attached
        by pointer (tfhe_b200_exchange_attach_local) and every exchange runs as one cooperative launch over all ranks
        (tfhe_b200_exchange_group_run) -- kernels that wait on one another must never be separate launches on one device.  Each rank is
        driven from its own thread on its own CUDA stream; the threads meet at a host barrier around the group launch."""
        import threading
        world = len(engines)
        comms = [cls(e, rank=r, world=world, exchange="nccl", max_rows=max_rows) for r, e in enumerate(engines)]
        if world > 1:
            for c in comms:
                c.exchange = "peer"
                c.peer = PeerExchange.local(c.eng, c.rank, world, max_rows)
            arr = (C.c_void_p * world)(*[c.peer.h for c in comms])
            for c in comms:
                c.eng._check(c.eng.lib.tfhe_b200_exchange_attach_local(c.peer.h, arr))
            group = {"barrier": threading.Barrier(world), "handles": arr, "events": [None] * world, "outs": [None] * world, "done": None,
                     "error": None, "args": [None] * world}
            for c in comms:
                c._group = group
        return comms

    def _group_exchange(self, rows: int, out: torch.Tensor, reduce: bool):
        """single-GPU group: every rank's thread records "my rows are staged", all meet, rank 0 launches the one cooperative kernel after
        every rank's stream, all meet again and order their streams after it"""
        g = self._group
        stream = self.stream
        ev = torch.cuda.Event()
        ev.record(stream)
        g["events"][self.rank], g["outs"][self.rank] = ev, out
        g["barrier"].wait()
        if self.rank == 0:
            try:
                for e in g["events"]:
                    stream.wait_event(e)
                outs = (C.c_void_p * self.world)(*[o.data_ptr() for o in g["outs"]])
                self.eng._check(self.eng.lib.tfhe_b200_exchange_group_run(g["handles"], self.world, rows, outs, int(reduce), stream.cuda_stream))
                done = torch.cuda.Event()
                done.record(stream)
                g["done"], g["error"] = done, None
            except Exception as e:      # the other ranks' threads must not be left at the barrier
                g["error"] = e
        g["barrier"].wait()
        if g["error"] is not None:
            raise NativeError(f"group exchange failed: {g['error']}")
        stream.wait_event(g["done"])

    def program(self, op: str, args: tuple, params: dict) -> Program:
        key = (op, tuple(args), tuple(sorted(params.items())))      # per DeviceComm = per engine: a program is bound to one context
        if key not in self._programs:
            self._programs[key] = Program(op, args, params=params)
        return self._programs[key]

    def _stream(self) -> int:
        return self.stream.cuda_stream

    def _to_device(self, x):
        """host array (numpy, ideally a view of page-locked memory: the copy is then one asynchronous DMA) or tensor -> CUDA tensor.  A
        list of pieces is assembled on the device, piece by piece, without a host-side concatenation."""
        if isinstance(x, (list, tuple)):
            pieces = [self._as_tensor(q) for q in x]
            out = torch.empty((sum(q.shape[0] for q in pieces), self.L), dtype=torch.int64, device=self.dev)
            r = 0
            for q in pieces:
                out[r:r + q.shape[0]].copy_(q.reshape(-1, self.L), non_blocking=True)
                r += q.shape[0]
            return out
        t = self._as_tensor(x)
        return t if t.is_cuda else t.to(self.dev, non_blocking=True)

    @staticmethod
    def _as_tensor(x):
        if isinstance(x, torch.Tensor):
            return x
        x = np.asarray(x)
        if x.dtype != np.uint64 or not x.flags.c_contiguous:
            x = np.ascontiguousarray(x, dtype=np.uint64)
        return torch.from_numpy(x.view(np.int64))

    @_on_own_stream
    def run(self, prog: Program, inputs, to_send_area: bool = False):
        """rows of `inputs` (host numpy / pinned tensor: uploaded here; CUDA tensor: used in place) -> CUDA tensor of the outputs.  With
        to_send_area the rows are written straight into the exchange buffer (the collective that follows reads them there)."""
        d_in = self._to_device(inputs).reshape(-1, self.L) if prog.n_inputs else None
        if prog.n_inputs and d_in.shape[0] != prog.n_inputs:
            raise ValueError(f"{prog.op}: expected {prog.n_inputs} input blocks, got {d_in.shape[0]}")
        if to_send_area and self.peer is not None and prog.n_outputs <= self.max_rows:
            out_ptr, out = self.peer.send_rows_ptr(), None
            self._pending_send = (prog.n_outputs,)
        else:
            out = torch.empty((prog.n_outputs, self.L), dtype=torch.int64, device=self.dev)
            out_ptr = out.data_ptr()
        self.eng._check(self.eng.lib.tfhe_b200_program_run_device(self.eng.h, prog.h, d_in.data_ptr() if d_in is not None else None, out_ptr,
                                                                   self._stream()))
        self._keep = d_in          # the upload must outlive the enqueued copy
        return out

    @_on_own_stream
    def zeros(self, rows: int, lwe_len: int):
        return torch.zeros((rows, lwe_len), dtype=torch.int64, device=self.dev)

    @_on_own_stream
    def padded(self, blocks, rows: int, lwe_len: int):
        """`blocks` followed by zero rows up to `rows` (equal shares for an all-gather), enqueued on the comm's stream like the program
        that produces `blocks` (a slice assignment on torch's current stream would not wait for it)"""
        out = torch.zeros((rows, lwe_len), dtype=torch.int64, device=self.dev)
        if blocks.shape[0]:
            out[:blocks.shape[0]].copy_(blocks)
        return out

    def _stage_for_peer(self, blocks) -> int:
        """rows that are not already in the send area (a rank without a share contributes zeros) are copied there"""
        if blocks is None:
            rows = self._pending_send[0]
            self._pending_send = None
            return rows
        rows = blocks.shape[0]
        if rows > self.max_rows:
            raise NativeError(f"exchange buffer holds {self.max_rows} rows, {rows} requested")
        # device-to-device copy on the current stream: the raw send area wrapped as a tensor view
        _tensor_from_ptr(self.peer.send_rows_ptr(), rows * self.L, self.dev).copy_(blocks.reshape(-1))
        return rows

    @_on_own_stream
    def all_reduce(self, blocks):
        if self.world == 1:
            return blocks
        if self.peer is not None and (blocks is None or blocks.shape[0] <= self.max_rows):
            rows = self._stage_for_peer(blocks)
            out = torch.empty((rows * self.L + 1) // 2 * 2, dtype=torch.int64, device=self.dev)
            if self._group is not None:
                self._group_exchange(rows, out, True)
            else:
                self.peer.all_reduce_sum(rows, out.data_ptr(), self._stream())
            return out[: rows * self.L].reshape(rows, self.L)
        t = blocks.contiguous()
        dist.all_reduce(t, op=dist.ReduceOp.SUM)      # NCCL on the current stream; int64 wrap-around == u64 wrap-around
        return t

    @_on_own_stream
    def all_gather(self, blocks):
        if self.peer is not None and (blocks is None or blocks.shape[0] <= self.max_rows):
            rows = self._stage_for_peer(blocks)
            stride = self.peer.gather_stride(rows)
            out = torch.empty((self.world, stride), dtype=torch.int64, device=self.dev)
            if self._group is not None:
                self._group_exchange(rows, out, False)
            else:
                self.peer.all_gather(rows, out.data_ptr(), self._stream())
            # rows * L odd: every rank's part is padded to an even word count, so this slice is strided and reshape() would return a VIEW;
            # the copy a caller's later reshape then makes would run on whatever stream is current there.  Materialise it here.
            return out[:, : rows * self.L].reshape(self.world, rows, self.L).contiguous()
        t = blocks.contiguous()
        out = torch.empty((self.world * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=self.dev)
        dist.all_gather_into_tensor(out, t)
        return out.reshape((self.world,) + tuple(t.shape))

    @_on_own_stream
    def rows(self, x, sel):
        return x[sel].contiguous()

    @_on_own_stream
    def to_host(self, x) -> np.ndarray:
        """the one device -> host copy of an operation (synchronises the stream), through a page-locked buffer.  Results above 1 MiB are
        returned as a view of that buffer (valid until the next result of the same shape); small ones are copied out."""
        if x.dim() == 1:
            x = x[None, :]
        x = x.contiguous()
        key = tuple(x.shape)
        if key not in self._host_out:
            self._host_out[key] = torch.empty(x.shape, dtype=torch.int64).pin_memory()
        buf = self._host_out[key]
        buf.copy_(x, non_blocking=True)
        self.stream.synchronize()
        out = buf.numpy().view(np.uint64)
        return out if out.nbytes > (1 << 20) else out.copy()

    def _program_exchange(self, max_rows: int) -> PeerExchange:
        """the exchange of run_program_sharded, holding at least `max_rows` rows per rank.  Creating or replacing it is collective: every
        rank runs the same program at the same min_shard_width, so every rank arrives here with the same max_rows."""
        old = self._program_peer
        if old is not None and old.max_rows >= max_rows:
            return old
        g = self._group
        barrier = g["barrier"].wait if g is not None else dist.barrier
        if old is not None:
            # a peer may still be reading this rank's send area in its last scatter: free it once every rank's stream has drained
            self.stream.synchronize()
            barrier()
            old.close()
            self._program_peer = None
        if g is None:
            self._program_peer = PeerExchange(self.eng, self.rank, self.world, max_rows)
            return self._program_peer
        ex = PeerExchange.local(self.eng, self.rank, self.world, max_rows)
        g["args"][self.rank] = ex.h
        barrier()
        arr = (C.c_void_p * self.world)(*g["args"])
        self.eng._check(self.eng.lib.tfhe_b200_exchange_attach_local(ex.h, arr))
        barrier()                      # nobody reuses g["args"] before every rank has attached
        self._program_peer = ex
        return ex

    def _group_run_sharded(self, prog: Program, ex: PeerExchange, d_in, out: torch.Tensor):
        """single-GPU group: as _group_exchange, rank 0 issues the one tfhe_b200_program_run_sharded_group call for every rank"""
        g = self._group
        stream = self.stream
        ev = torch.cuda.Event()
        ev.record(stream)
        g["events"][self.rank] = ev
        g["args"][self.rank] = (self.eng.h, prog.h, ex.h, d_in.data_ptr() if d_in is not None else None, out.data_ptr() if out.numel() else None)
        g["barrier"].wait()
        if self.rank == 0:
            try:
                for e in g["events"]:
                    stream.wait_event(e)
                ptrs = lambda i: (C.c_void_p * self.world)(*[a[i] for a in g["args"]])
                self.eng._check(self.eng.lib.tfhe_b200_program_run_sharded_group(ptrs(0), ptrs(1), ptrs(2), self.world, ptrs(3), ptrs(4),
                                                                                 self.min_shard_width, stream.cuda_stream))
                done = torch.cuda.Event()
                done.record(stream)
                g["done"], g["error"] = done, None
            except Exception as e:      # the other ranks' threads must not be left at the barrier
                g["error"] = e
        g["barrier"].wait()
        if g["error"] is not None:
            raise NativeError(f"sharded group run failed: {g['error']}")
        stream.wait_event(g["done"])

    def close(self):
        if self._program_peer is not None:
            self._program_peer.close()
            self._program_peer = None
        if self.peer is not None:
            self.peer.close()
            self.peer = None
        for p in self._programs.values():
            p.close()
        self._programs.clear()


def _tensor_from_ptr(ptr: int, n_words: int, dev: torch.device) -> torch.Tensor:
    """int64 tensor view of raw device memory owned by the engine (no copy, no ownership)"""
    class _Iface:
        pass
    o = _Iface()
    o.__cuda_array_interface__ = {"shape": (n_words,), "typestr": "<i8", "data": (ptr, False), "version": 3}
    return torch.as_tensor(o, device=dev)


def _on_comm_stream(fn):
    """a sharded operation in full -- including the incidental tensor views / copies between the comm's calls -- with the comm's
    stream as torch's current stream (a copy enqueued on another stream would not wait for the kernels before it)"""
    import functools

    @functools.wraps(fn)
    def wrapper(comm, *args, **kwargs):
        comm = _comm(comm)
        if isinstance(comm, DeviceComm):
            cur = torch.cuda.current_stream(comm.dev)
            if cur != comm.stream:
                comm.stream.wait_stream(cur)
            with torch.cuda.stream(comm.stream):
                return fn(comm, *args, **kwargs)
        return fn(comm, *args, **kwargs)
    return wrapper


def _comm(x):
    """the CPU tests pass a bare `execute(program, inputs)` callable"""
    return x if isinstance(x, (HostComm, DeviceComm)) else HostComm(x)


def _share(comm, prog, inputs):
    """run a rank's share; on the device path the result rows land directly in the exchange send area (returns None then)"""
    if isinstance(comm, DeviceComm):
        return comm.run(prog, inputs, to_send_area=True)
    return comm.run(prog, inputs)


def _bpc(params: dict) -> int:
    """blocks per char: ceil(8 / log2(message_modulus)); 4 for the 2-bit sets"""
    bits = int(params["msg_mod"]).bit_length() - 1
    return -(-8 // bits)


def _worth_sharding(comm, first_level_width: int) -> bool:
    """shard only when the widest (first) level of the tree is wider than what one GPU runs as a single narrow-level launch"""
    return comm.world > 1 and first_level_width > comm.min_shard_width


# ---- the sharded operations -----------------------------------------------------------------------------------------------------
# `comm` is a DeviceComm / HostComm (or a bare execute callable -> HostComm).  hay / pat / a / b / s are the encrypted blocks, 4 per
# char, as host arrays (numpy or pinned tensors); only a rank's own share is uploaded.  The result is returned as a host array.

@_on_comm_stream
def sharded_contains(comm, params: dict, hay, pat, hay_len: int, pat_len: int, rank: int | None = None, world: int | None = None,
                     device: str | None = None) -> np.ndarray:
    """contains(hay, pat) with the windows split over the ranks.  Every rank returns the same boolean block."""
    comm = _comm(comm)
    rank, world = comm.rank, comm.world
    n_win = hay_len - pat_len + 1
    if n_win <= 0 or pat_len == 0 or not _worth_sharding(comm, n_win * _bpc(params) * pat_len):   # nothing to split: the plain single-GPU program
        return comm.to_host(comm.run(comm.program("string_contains", (hay_len, pat_len), params), [hay, pat]))[0]
    total_mod = params["msg_mod"] * params["carry_mod"]
    active = min(world, n_win, total_mod - 1)       # the summed flags must stay below the padding bit; surplus ranks contribute zero
    if rank < active:
        w0, w1 = shard_range(n_win, rank, active)
        # a rank only needs the haystack chars its windows touch: upload hay[w0 : w1 - 1 + pat_len] and the pattern
        lo, hi = w0, w1 - 1 + pat_len
        mine = _share(comm, comm.program("string_contains_windows", (hi - lo, pat_len, 0, w1 - w0), params), [hay[_bpc(params) * lo:_bpc(params) * hi], pat])
    else:
        mine = comm.zeros(1, hay.shape[1])
    total = comm.all_reduce(mine)
    return comm.to_host(comm.run(comm.program("bool_sum_finish", (active, 0), params), total))[0]


@_on_comm_stream
def sharded_eq(comm, params: dict, a, b, n_chars: int, rank: int | None = None, world: int | None = None,
               device: str | None = None) -> np.ndarray:
    """eq of two equal-length strings with the chars split over ranks: per-rank eq of its slice, sum, x == active."""
    comm = _comm(comm)
    rank, world = comm.rank, comm.world
    if n_chars == 0:
        return comm.to_host(comm.run(comm.program("string_eq", (0, 0), params), np.zeros((0, 1), dtype=np.uint64)))[0]
    if not _worth_sharding(comm, _bpc(params) * n_chars):
        return comm.to_host(comm.run(comm.program("string_eq", (n_chars, n_chars), params), [a, b]))[0]
    total_mod = params["msg_mod"] * params["carry_mod"]
    active = max(1, min(world, n_chars, total_mod - 1))
    if rank < active:
        c0, c1 = shard_range(n_chars, rank, active)
        mine = _share(comm, comm.program("string_eq", (c1 - c0, c1 - c0), params), [a[_bpc(params) * c0:_bpc(params) * c1], b[_bpc(params) * c0:_bpc(params) * c1]])
    else:
        mine = comm.zeros(1, a.shape[1])
    total = comm.all_reduce(mine)
    return comm.to_host(comm.run(comm.program("bool_sum_finish", (active, 1), params), total))[0]


_CMP = {"lt": (1, 0), "le": (1, 1), "gt": (0, 0), "ge": (0, 1)}     # (want_less, or_equal) of strings.h cmp()


@_on_comm_stream
def sharded_compare(comm, params: dict, op: str, a, b, n_chars: int, rank: int | None = None, world: int | None = None,
                    device: str | None = None) -> np.ndarray:
    """lt / le / gt / ge of two equal-length strings with the chars split over ranks (SURVEY 8e, lexicographic tree): every rank
    reduces its char range to one sign block (comparator.rs:389-464), the sign blocks are gathered (world x 16 KiB) and every
    rank finishes with the pairwise sign tree + map_sign_result (ceil(log2(world)) + 1 levels of at most world/2 PBS)."""
    comm = _comm(comm)
    rank, world = comm.rank, comm.world
    want_less, or_equal = _CMP[op]
    active = max(1, min(world, n_chars))
    if n_chars == 0 or not _worth_sharding(comm, 2 * n_chars):       # first level: one sign block per pair of blocks
        return comm.to_host(comm.run(comm.program("string_" + op, (n_chars, n_chars), params), [a, b]))[0]
    if rank < active:
        c0, c1 = shard_range(n_chars, rank, active)
        mine = _share(comm, comm.program("string_cmp_sign", (c1 - c0, c1 - c0), params), [a[_bpc(params) * c0:_bpc(params) * c1], b[_bpc(params) * c0:_bpc(params) * c1]])
    else:
        mine = comm.zeros(1, a.shape[1])
    signs = comm.all_gather(mine)[:active, 0]
    # char 0 is the most significant: the sign tree wants the least significant range first
    order = list(range(active - 1, -1, -1))
    return comm.to_host(comm.run(comm.program("signs_finish", (active, want_less, or_equal), params), comm.rows(signs, order)))[0]


@_on_comm_stream
def sharded_case(comm, params: dict, op: str, s, n_chars: int, rank: int | None = None, world: int | None = None,
                 device: str | None = None, gather: bool = True) -> np.ndarray:
    """to_lowercase / to_uppercase with the chars split over ranks: elementwise, so there is no exchange on the path.  With
    gather=True every rank returns the whole converted string (one gather of the converted blocks, 16 KiB per block -- for a
    1024-char string that is 67 MB and costs more than the conversion); with gather=False a rank returns its own chars
    [shard_range(n_chars, rank, world)] only (SURVEY 8e: "no exchange; optional all-gather")."""
    comm = _comm(comm)
    rank, world = comm.rank, comm.world
    if n_chars == 0 or not _worth_sharding(comm, 2 * n_chars):
        out = comm.to_host(comm.run(comm.program("string_" + op, (n_chars,), params), s))
        if gather or world == 1:
            return out
        c0, c1 = shard_range(n_chars, rank, min(world, n_chars)) if rank < min(world, n_chars) else (0, 0)
        return out[_bpc(params) * c0:_bpc(params) * c1]
    active = min(world, n_chars)
    per = -(-n_chars // active)                                  # padded share, in chars
    c0 = c1 = 0
    if rank < active:
        c0, c1 = shard_range(n_chars, rank, active)
    L = s.shape[1]
    conv = comm.run(comm.program("string_" + op, (c1 - c0,), params), s[_bpc(params) * c0:_bpc(params) * c1]) if c1 > c0 else comm.zeros(0, L)
    if not gather:
        return comm.to_host(conv) if c1 > c0 else np.zeros((0, L), dtype=np.uint64)
    mine = comm.padded(conv, _bpc(params) * per, L)      # on the comm's stream: `conv` is still being computed there
    parts = comm.to_host(comm.all_gather(mine).reshape(world * _bpc(params) * per, L)).reshape(world, _bpc(params) * per, L)
    out = []
    for r in range(active):
        r0, r1 = shard_range(n_chars, r, active)
        out.append(parts[r, :_bpc(params) * (r1 - r0)])
    return np.concatenate(out)


@_on_comm_stream
def sharded_find(comm, params: dict, hay, pat, hay_len: int, pat_len: int, rank: int | None = None, world: int | None = None,
                 device: str | None = None) -> np.ndarray:
    """find(hay, pat) with the windows split over ranks: every rank finds the first match inside its window range (reported as a
    global index), the (found, index) blocks are gathered and every rank selects the lowest rank that found (two PBS levels).
    Returns [found, index blocks...] like the single-GPU program."""
    comm = _comm(comm)
    rank, world = comm.rank, comm.world
    n_win = hay_len - pat_len + 1
    inputs = [hay, pat]
    if n_win <= 1 or pat_len == 0 or not _worth_sharding(comm, n_win * _bpc(params) * pat_len):
        return comm.to_host(comm.run(comm.program("string_find", (hay_len, pat_len), params), inputs))
    total_mod = params["msg_mod"] * params["carry_mod"]
    active = min(world, n_win, total_mod // 2)
    nb = 1
    while (1 << (2 * nb)) < n_win:
        nb += 1
    if rank < active:
        w0, w1 = shard_range(n_win, rank, active)
        mine = _share(comm, comm.program("string_find_windows", (hay_len, pat_len, w0, w1), params), inputs)
    else:
        mine = comm.zeros(1 + nb, hay.shape[1])
    parts = comm.all_gather(mine)[:active]
    return comm.to_host(comm.run(comm.program("find_combine", (active, nb), params), parts.reshape(active * (1 + nb), -1)))


# ---- any recorded program, its wide levels split across the ranks ------------------------------------------------------------------

@_on_comm_stream
def run_program_sharded(comm: DeviceComm, prog: Program, inputs) -> torch.Tensor:
    """Any recorded program across the ranks of `comm`; every rank calls it with the same program (under DeviceComm.local_group each rank
    with its own Program object, e.g. comm.program(...): a program binds to one context) and the same inputs, and gets all outputs as a
    CUDA tensor (n_outputs, k*N+1) of int64 words on the comm's stream.

    Levels wider than comm.min_shard_width are split: each rank keyswitches and bootstraps its shard_range share of the level and one
    scatter kernel hands every row to every rank over NVLink peer memory (tfhe_b200_program_run_sharded).  Narrower levels run in full on
    every rank, with no communication.

    The scatter uses an exchange of its own, created collectively on first need and sized by the shard plan; the `peer` exchange of the
    sharded_* operations stays as it is.  Its send area is double-buffered, so it takes 2 x (largest share) x (k*N+1) x 8 bytes per rank:
    string_eq_many {8, 8, 4096} at world 2 has a widest level of 131 072 PBS, so a share of 65 536 rows and about 2.1 GB per rank."""
    if not isinstance(comm, DeviceComm):
        raise TypeError("run_program_sharded runs on a DeviceComm")
    if comm.world == 1:
        return comm.run(prog, inputs)
    if comm.exchange != "peer":
        raise ValueError("run_program_sharded: exchange='nccl' is not supported; the per-level scatter runs over peer memory only "
                         "(DeviceComm(exchange='peer'))")
    _, max_rows, _ = prog.shard_plan(comm.world, comm.min_shard_width)
    ex = comm._program_exchange(max(1, max_rows))
    d_in = comm._to_device(inputs).reshape(-1, comm.L) if prog.n_inputs else None
    if prog.n_inputs and d_in.shape[0] != prog.n_inputs:
        raise ValueError(f"{prog.op}: expected {prog.n_inputs} input blocks, got {d_in.shape[0]}")
    out = torch.empty((prog.n_outputs, comm.L), dtype=torch.int64, device=comm.dev)
    if comm._group is not None:
        comm._group_run_sharded(prog, ex, d_in, out)
    else:
        comm.eng._check(comm.eng.lib.tfhe_b200_program_run_sharded(comm.eng.h, prog.h, ex.h, d_in.data_ptr() if d_in is not None else None,
                                                                   out.data_ptr() if out.numel() else None, comm.min_shard_width,
                                                                   comm._stream()))
    comm._keep = d_in          # the upload must outlive the enqueued copy
    return out
