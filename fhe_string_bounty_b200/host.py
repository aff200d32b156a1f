"""Python face of the host layer (csrc/host/*.h through the C ABI): record an integer / string operation as a
level-batched program, inspect it (no GPU needed), run it on an Engine.

The operation names and operand order are those of include/tfhe_b200.h (tfhe_b200_program_build)."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from ._native import Engine, NativeError, Params, PARAM_MESSAGE_2_CARRY_2_KS_PBS, load_native


@dataclass
class ProgramIR:
    """Flat copy of a recorded program (what tfhe_b200_program_copy returns)."""
    n_inputs: int
    n_slots: int
    level_lin_off: np.ndarray
    level_pbs_off: np.ndarray
    lin: np.ndarray          # [n_lin, 3] out_slot, term_begin, term_end
    lin_body: np.ndarray     # [n_lin]
    term_slot: np.ndarray
    term_coef: np.ndarray
    pbs: np.ndarray          # [n_pbs, 3] in_slot, out_slot, lut
    lut_tables: np.ndarray   # [n_luts, total_mod]
    lut_degrees: np.ndarray
    outputs: np.ndarray
    output_degree_noise: np.ndarray  # [n_outputs, 2]
    n_trivial_pbs: int

    @property
    def level_widths(self):
        w = np.diff(self.level_pbs_off)
        return [int(x) for x in w if x > 0]


class Program:
    def __init__(self, op: str, args=(), clear: str | bytes | None = None, params: dict | Params | None = None):
        self.lib = load_native()
        if params is None:
            params = PARAM_MESSAGE_2_CARRY_2_KS_PBS
        self.p = params if isinstance(params, Params) else Params(**params)
        a = np.ascontiguousarray(np.array(list(args), dtype=np.uint64))
        h = C.c_void_p()
        if isinstance(clear, str):
            clear = clear.encode("latin-1")
        if clear is not None and b"\0" in clear:   # the C ABI takes a NUL-terminated string: the pattern would be cut short
            raise ValueError(f"{op}: a clear operand cannot contain a NUL char")
        rc = self.lib.tfhe_b200_program_build(C.byref(self.p), op.encode(), a.ctypes.data if a.size else None, a.size, clear, C.byref(h))
        if rc != 0:
            raise NativeError(self.lib.tfhe_b200_last_error().decode())
        self.h = h
        self.op = op
        c = np.zeros(9, dtype=np.uint64)
        self._check(self.lib.tfhe_b200_program_counts(self.h, c.ctypes.data))
        (self.n_inputs, self.n_outputs, self.n_slots, self.n_levels, self.n_lin, self.n_terms, self.n_pbs, self.n_luts,
         self.n_trivial_pbs) = (int(x) for x in c)

    def _check(self, rc):
        if rc != 0:
            raise NativeError(self.lib.tfhe_b200_last_error().decode())

    def close(self):
        if getattr(self, "h", None):
            self.lib.tfhe_b200_program_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def ir(self) -> ProgramIR:
        tm = self.p.msg_mod * self.p.carry_mod
        llo = np.zeros(self.n_levels + 1, dtype=np.uint32)
        lpo = np.zeros(self.n_levels + 1, dtype=np.uint32)
        lin = np.zeros((self.n_lin, 3), dtype=np.uint32)
        lin_body = np.zeros(self.n_lin, dtype=np.uint64)
        ts = np.zeros(self.n_terms, dtype=np.uint32)
        tc = np.zeros(self.n_terms, dtype=np.int64)
        pbs = np.zeros((self.n_pbs, 3), dtype=np.uint32)
        lt = np.zeros((self.n_luts, tm), dtype=np.uint64)
        ld = np.zeros(self.n_luts, dtype=np.uint64)
        outs = np.zeros(self.n_outputs, dtype=np.uint32)
        odn = np.zeros((self.n_outputs, 2), dtype=np.uint64)
        ptr = lambda a: a.ctypes.data if a.size else None
        self._check(self.lib.tfhe_b200_program_copy(self.h, ptr(llo), ptr(lpo), ptr(lin), ptr(lin_body), ptr(ts), ptr(tc), ptr(pbs),
                                                    ptr(lt), ptr(ld), ptr(outs), ptr(odn)))
        return ProgramIR(self.n_inputs, self.n_slots, llo, lpo, lin, lin_body, ts, tc, pbs, lt, ld, outs, odn, self.n_trivial_pbs)

    @property
    def level_widths(self):
        return self.ir().level_widths

    def shard_plan(self, world: int, min_shard_width: int) -> tuple[int, int, int]:
        """(split levels, largest share in rows, rows each rank receives) of a run across `world` ranks (tfhe_b200_program_shard_plan)"""
        out = np.zeros(3, dtype=np.uint64)
        self._check(self.lib.tfhe_b200_program_shard_plan(self.h, world, min_shard_width, out.ctypes.data))
        return tuple(int(x) for x in out)

    def level_share(self, level: int, rank: int, world: int, min_shard_width: int) -> tuple[int, int, bool]:
        """(lo, hi, split): the PBS jobs of level `level` that `rank` runs, counted from the level's first job"""
        out = np.zeros(3, dtype=np.uint64)
        self._check(self.lib.tfhe_b200_program_level_share(self.h, level, rank, world, min_shard_width, out.ctypes.data))
        return int(out[0]), int(out[1]), bool(out[2])

    def accumulators(self) -> np.ndarray:
        acc = np.zeros((max(self.n_luts, 1), self.p.lut_len), dtype=np.uint64)
        if self.n_luts:
            self._check(self.lib.tfhe_b200_program_accumulators(self.h, acc.ctypes.data))
        return acc[: self.n_luts]

    def run(self, eng: Engine, inputs: np.ndarray, out: np.ndarray | None = None) -> np.ndarray:
        """Execute on the GPU of `eng`; inputs [n_inputs, k*N+1] u64 (host) -> outputs [n_outputs, k*N+1].  `out` lets the caller
        supply the result buffer (page-locked memory makes both copies DMA transfers instead of staged ones)."""
        inputs = np.ascontiguousarray(inputs, dtype=np.uint64).reshape(-1, self.p.big_len)
        if inputs.shape[0] != self.n_inputs:
            raise ValueError(f"{self.op}: expected {self.n_inputs} input blocks, got {inputs.shape[0]}")
        if out is None:
            out = np.empty((self.n_outputs, self.p.big_len), dtype=np.uint64)
        elif out.dtype != np.uint64 or not out.flags.c_contiguous or out.size != self.n_outputs * self.p.big_len:
            raise ValueError(f"{self.op}: out must be a C-contiguous uint64 array of {self.n_outputs} x {self.p.big_len} words")
        self._check(self.lib.tfhe_b200_program_run(eng.h, self.h, inputs.ctypes.data if inputs.size else None, out.ctypes.data if out.size else None))
        return out

    def pipe(self, execute, inputs):
        return execute(self, inputs)

    def last_ms(self) -> float:
        v = C.c_float()
        self._check(self.lib.tfhe_b200_program_last_ms(self.h, C.byref(v)))
        return v.value
