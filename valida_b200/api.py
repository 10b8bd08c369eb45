"""ctypes binding of libvalida_b200.so, shaped after the reference's Rust interfaces.

Reference interfaces mirrored (names and argument meaning kept):
  * p3_dft::TwoAdicSubgroupDft: dft_batch / idft_batch / coset_lde_batch        -> Radix2Dft
  * UnivariatePcsWithLde (machine/src/config.rs:17-22): commit_batches,
    commit_shifted_batches, get_ldes, coset_shift, log_blowup                    -> TwoAdicFriPcs
  * Machine::run / Chip::generate_trace (machine/src/machine.rs:13-30)          -> run_program / MachineTraces
Errors: the reference panics (derive/src/lib.rs:319,364,396); here every non-zero status raises
VgpuError carrying vgpu_last_error().
"""
import ctypes as C
import os
import weakref

import numpy as np

BABYBEAR_P = 2013265921
REPR_CANONICAL, REPR_MONTY_R32 = 0, 1
NUM_CHIPS = 14

_HERE = os.path.dirname(os.path.abspath(__file__))
lib_path = os.path.join(_HERE, "libvalida_b200.so")


class VgpuError(RuntimeError):
    pass


class _Matrix(C.Structure):
    _fields_ = [("data", C.POINTER(C.c_uint32)), ("height", C.c_uint64), ("width", C.c_uint64)]


def _load():
    if not os.path.exists(lib_path):
        raise VgpuError(
            "libvalida_b200.so is missing (%s): build it with `python -m valida_b200.build` — there is no CPU fallback" % lib_path
        )
    L = C.CDLL(lib_path)
    vp, u32p, u64 = C.c_void_p, C.POINTER(C.c_uint32), C.c_uint64
    sig = {
        "vgpu_ctx_create": (C.c_int32, [C.c_int32, vp, C.POINTER(vp)]),
        "vgpu_ctx_destroy": (None, [vp]),
        "vgpu_last_error": (C.c_char_p, [vp]),
        "vgpu_ctx_synchronize": (C.c_int32, [vp]),
        "vgpu_ctx_launch_count": (u64, [vp]),
        "vgpu_ctx_set_kernel_timing": (C.c_int32, [vp, C.c_int32]),
        "vgpu_ctx_kernel_stats": (C.c_uint32, [vp, C.POINTER(C.c_char_p), u32p, C.POINTER(C.c_float), C.POINTER(C.c_double), C.c_uint32]),
        "vgpu_host_register": (C.c_int32, [vp, vp, u64]),
        "vgpu_host_unregister": (C.c_int32, [vp, vp]),
        "vgpu_dmat_upload": (C.c_int32, [vp, C.POINTER(_Matrix), C.c_int32, C.POINTER(vp)]),
        "vgpu_dmat_upload_rows": (C.c_int32, [vp, C.POINTER(_Matrix), C.c_int32, C.POINTER(vp)]),
        "vgpu_dmat_local_rows": (C.c_int32, [vp, C.POINTER(u64), C.POINTER(u64)]),
        "vgpu_dmat_download": (C.c_int32, [vp, vp, C.c_int32, u32p]),
        "vgpu_dmat_dims": (C.c_int32, [vp, C.POINTER(u64), C.POINTER(u64)]),
        "vgpu_dmat_free": (None, [vp]),
        "vgpu_ntt_batch": (C.c_int32, [vp, vp, C.c_int32]),
        "vgpu_coset_lde_batch": (C.c_int32, [vp, vp, C.c_uint32, C.c_uint32, C.c_int32, C.POINTER(vp)]),
        "vgpu_ntt_batch_host": (C.c_int32, [vp, u32p, u64, u64, C.c_int32, C.c_int32]),
        "vgpu_commit_batches": (C.c_int32, [vp, C.POINTER(vp), C.c_uint32, u32p, u32p, C.POINTER(vp)]),
        "vgpu_commit_batches_host": (C.c_int32, [vp, C.POINTER(_Matrix), C.c_uint32, C.c_int32, u32p, u32p, C.POINTER(vp)]),
        "vgpu_prover_data_lde": (C.c_int32, [vp, C.c_uint32, C.POINTER(vp)]),
        "vgpu_prover_data_free": (None, [vp]),
        "vgpu_basic_machine_chip": (vp, [C.c_uint32]),
        "vgpu_perm_trace": (C.c_int32, [vp, vp, vp, vp, u32p, C.POINTER(vp), u32p]),
        "vgpu_quotient": (C.c_int32, [vp, vp, C.c_uint32, vp, vp, vp, u32p, u32p, u32p, C.POINTER(vp)]),
        "vgpu_set_challenger": (C.c_int32, [vp, u32p, u32p]),
        "vgpu_challenger_reset": (C.c_int32, [vp]),
        "vgpu_challenger_observe": (C.c_int32, [vp, u32p, C.c_uint32]),
        "vgpu_challenger_sample_ext": (C.c_int32, [vp, u32p]),
        "vgpu_comm_unique_id": (C.c_int32, [C.c_char_p]),
        "vgpu_comm_init": (C.c_int32, [vp, C.c_int32, C.c_int32, C.c_char_p]),
        "vgpu_comm_init_local": (C.c_int32, [C.POINTER(vp), C.c_int32]),
        "vgpu_comm_stats": (None, [vp, u32p, C.POINTER(C.c_double), C.c_int32]),
        "vgpu_comm_set_sharding": (C.c_int32, [vp, C.c_int32]),
        "vgpu_shard_range": (None, [u64, C.c_int32, C.c_int32, C.POINTER(u64), C.POINTER(u64)]),
        "vgpu_split_column_plan": (None, [C.c_int32, C.c_uint32, C.POINTER(u64), C.POINTER(u64), u32p]),
        "vgpu_tree_share": (None, [u64, C.c_int32, C.c_int32, C.POINTER(u64), C.POINTER(u64), C.POINTER(C.c_int32)]),
        "vgpu_open": (C.c_int32, [vp, C.POINTER(vp), C.c_uint32, u32p, u32p, C.POINTER(C.POINTER(C.c_uint8)), C.POINTER(u64)]),
        "vgpu_verify": (C.c_int32, [vp, C.c_char_p, u64, C.POINTER(_Matrix), C.c_int32, C.POINTER(C.c_int32)]),
        "vgpu_verify_batch": (C.c_int32, [vp, C.POINTER(C.c_char_p), C.POINTER(u64), C.c_uint32, C.POINTER(_Matrix), C.c_uint32, u32p, C.c_int32,
                                          C.POINTER(C.c_int32)]),
        "vgpu_last_verify_batch_phases": (C.c_uint32, [vp, C.POINTER(C.c_char_p), C.POINTER(C.c_float), C.c_uint32]),
        "vgpu_prove": (C.c_int32, [vp, C.POINTER(_Matrix), C.POINTER(_Matrix), C.c_int32, C.POINTER(C.POINTER(C.c_uint8)), C.POINTER(u64)]),
        "vgpu_prove_device": (C.c_int32, [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(C.POINTER(C.c_uint8)), C.POINTER(u64)]),
        "vgpu_free_bytes": (None, [C.POINTER(C.c_uint8)]),
        "vgpu_last_prove_phases": (C.c_uint32, [vp, C.POINTER(C.c_char_p), C.POINTER(C.c_float), C.c_uint32]),
        "vgpu_machine_run": (C.c_int32, [C.POINTER(C.c_int32), u64, C.c_uint32, C.c_uint32, u64, C.POINTER(vp), C.c_char_p, u64]),
        "vgpu_machine_run_static": (C.c_int32, [C.POINTER(C.c_int32), u64, C.c_uint32, C.c_uint32, u64, u32p, u32p, u64, C.POINTER(vp), C.c_char_p, u64]),
        "vgpu_traces_main": (C.POINTER(_Matrix), [vp, C.c_uint32]),
        "vgpu_traces_preprocessed": (C.POINTER(_Matrix), [vp, C.c_uint32]),
        "vgpu_traces_stats": (None, [vp, u32p, u32p, u32p]),
        "vgpu_traces_mem_cell": (C.c_int32, [vp, C.c_uint32, u32p]),
        "vgpu_traces_free": (None, [vp]),
        "vgpu_fib_program": (u64, [C.c_uint32, C.POINTER(C.c_int32)]),
        "vgpu_vm_run": (C.c_int32, [C.POINTER(C.c_int32), u64, C.c_uint32, C.c_uint32, u64, u32p, u32p, u64, C.POINTER(vp), C.c_char_p, u64]),
        "vgpu_vmlog_stats": (None, [vp, u32p, u32p, u32p]),
        "vgpu_vmlog_traces": (C.c_int32, [vp, C.POINTER(vp), C.c_char_p, u64]),
        "vgpu_witness_device": (C.c_int32, [vp, vp, C.POINTER(vp), C.POINTER(vp)]),
        "vgpu_vmlog_free": (None, [vp]),
    }
    for name, (res, args) in sig.items():
        f = getattr(L, name)
        f.restype, f.argtypes = res, args
    return L


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = _load()
    return _lib


def _as_u32(a):
    a = np.ascontiguousarray(a, dtype=np.uint32)
    return a


def _mat(a):
    return _Matrix(a.ctypes.data_as(C.POINTER(C.c_uint32)), a.shape[0], a.shape[1])


class Context:
    """One context per device/stream (single-threaded)."""

    def __init__(self, device=0, stream=None):
        self._children = weakref.WeakSet()      # handles that point into this context: released before the context goes
        self._h = C.c_void_p()
        rc = lib().vgpu_ctx_create(device, C.c_void_p(stream) if stream else None, C.byref(self._h))
        if rc != 0:
            msg = lib().vgpu_last_error(self._h).decode() if self._h else "context allocation failed"
            if self._h:
                lib().vgpu_ctx_destroy(self._h)
                self._h = None
            raise VgpuError(msg)

    def check(self, rc):
        if rc != 0:
            raise VgpuError(lib().vgpu_last_error(self._h).decode())

    def synchronize(self):
        self.check(lib().vgpu_ctx_synchronize(self._h))

    @property
    def launch_count(self):
        return int(lib().vgpu_ctx_launch_count(self._h))

    def set_kernel_timing(self, on):
        lib().vgpu_ctx_set_kernel_timing(self._h, 1 if on else 0)

    def kernel_stats(self):
        """[(kernel class, launches, total ms, algorithmic bytes)] since the last call (synchronises)."""
        names = (C.c_char_p * 16)(); ln = (C.c_uint32 * 16)(); ms = (C.c_float * 16)(); by = (C.c_double * 16)()
        n = lib().vgpu_ctx_kernel_stats(self._h, names, ln, ms, by, 16)
        return [(names[i].decode(), int(ln[i]), float(ms[i]), float(by[i])) for i in range(n)]

    # ---- multi-GPU: one rank per GPU (include/valida_b200.h, "multi-GPU") ----
    def comm_init(self, rank, world_size, unique_id):
        """Join the NCCL communicator named by unique_id (comm_unique_id() of rank 0, distributed by the caller)."""
        self.check(lib().vgpu_comm_init(self._h, world_size, rank, bytes(unique_id)))
        self.rank, self.world_size = rank, world_size

    def comm_init_from_torch(self):
        """Convenience for torchrun ranks: rank 0 creates the id, torch.distributed carries it to the others."""
        import torch.distributed as dist

        ids = [comm_unique_id() if dist.get_rank() == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        self.comm_init(dist.get_rank(), dist.get_world_size(), ids[0])

    def set_sharding(self, on):
        """False: this rank works alone (independent replicas); True: ONE proof is split across the ranks."""
        self.check(lib().vgpu_comm_set_sharding(self._h, 1 if on else 0))

    def comm_stats(self, reset=True):
        """Collectives since the last reset: {name: (calls, bytes sent to peers)} for barriers, all-gathers, peer-store exchanges."""
        calls = (C.c_uint32 * 3)(); by = (C.c_double * 3)()
        lib().vgpu_comm_stats(self._h, calls, by, 1 if reset else 0)
        return {n: (int(calls[i]), float(by[i])) for i, n in enumerate(("barrier", "allgather", "exchange"))}

    def upload_rows(self, row_major, repr=REPR_CANONICAL):
        """Split proof: of a trace tall enough to be split, keep this rank's run of rows only (otherwise like upload)."""
        a = _as_u32(row_major)
        m = _mat(a)
        out = C.c_void_p()
        self.check(lib().vgpu_dmat_upload_rows(self._h, C.byref(m), repr, C.byref(out)))
        return DeviceMatrix(self, out)

    def host_register(self, array):
        """Page-lock a numpy array the caller will prove from repeatedly (its uploads then overlap the commits)."""
        self.check(lib().vgpu_host_register(self._h, C.c_void_p(array.ctypes.data), array.nbytes))

    def host_unregister(self, array):
        self.check(lib().vgpu_host_unregister(self._h, C.c_void_p(array.ctypes.data)))

    def upload(self, row_major, repr=REPR_CANONICAL):
        """RowMajorMatrix<Val> (numpy h x w uint32) -> DeviceMatrix."""
        a = _as_u32(row_major)
        if a.ndim != 2:
            raise ValueError("expected a 2-D row-major matrix")
        m = _mat(a)
        out = C.c_void_p()
        self.check(lib().vgpu_dmat_upload(self._h, C.byref(m), repr, C.byref(out)))
        return DeviceMatrix(self, out)

    def close(self):
        """Destroys the context.  Device matrices / prover data created from it are released first (their handles would dangle)."""
        if getattr(self, "_h", None):
            for child in list(getattr(self, "_children", ())):
                try:
                    child.free()
                except Exception:
                    pass
            lib().vgpu_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DeviceMatrix:
    def __init__(self, ctx, handle, owned=True):
        self.ctx, self._h, self._owned = ctx, handle, owned
        ctx._children.add(self)

    @property
    def shape(self):
        h, w = C.c_uint64(), C.c_uint64()
        lib().vgpu_dmat_dims(self._h, C.byref(h), C.byref(w))
        return int(h.value), int(w.value)

    def local_rows(self):
        """(first row, rows) held on this rank — the whole matrix unless it is a row shard of a split proof."""
        r0, n = C.c_uint64(), C.c_uint64()
        lib().vgpu_dmat_local_rows(self._h, C.byref(r0), C.byref(n))
        return int(r0.value), int(n.value)

    def download(self, repr=REPR_CANONICAL):
        h, w = self.shape
        out = np.empty((h, w), dtype=np.uint32)
        self.ctx.check(lib().vgpu_dmat_download(self.ctx._h, self._h, repr, out.ctypes.data_as(C.POINTER(C.c_uint32))))
        return out

    def free(self):
        if self._h and self._owned and self.ctx._h:
            lib().vgpu_dmat_free(self._h)
        self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Radix2Dft:
    """p3_dft::TwoAdicSubgroupDft over device matrices (Radix2DitParallel / Radix2Bowers give the same values)."""

    def __init__(self, ctx):
        self.ctx = ctx

    def dft_batch(self, m):
        self.ctx.check(lib().vgpu_ntt_batch(self.ctx._h, m._h, 0))
        return m

    def idft_batch(self, m):
        self.ctx.check(lib().vgpu_ntt_batch(self.ctx._h, m._h, 1))
        return m

    def coset_lde_batch(self, m, added_bits, shift, bit_reversed=False):
        out = C.c_void_p()
        self.ctx.check(lib().vgpu_coset_lde_batch(self.ctx._h, m._h, added_bits, shift, 1 if bit_reversed else 0, C.byref(out)))
        return DeviceMatrix(self.ctx, out)


class ProverData:
    def __init__(self, ctx, handle, n):
        self.ctx, self._h, self.n = ctx, handle, n
        ctx._children.add(self)

    def free(self):
        if self._h and self.ctx._h:
            lib().vgpu_prover_data_free(self._h)
        self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class TwoAdicFriPcs:
    """UnivariatePcsWithLde surface used by Machine::prove (machine/src/config.rs:17-22)."""

    GENERATOR = 31

    def __init__(self, ctx, log_blowup=1, num_queries=40, proof_of_work_bits=8):
        if log_blowup != 1:
            raise VgpuError("the commit path is built for log_blowup = 1 (FriConfig of basic/src/bin/valida.rs:385-390); Radix2Dft.coset_lde_batch takes 1..4")
        self.ctx, self._log_blowup = ctx, log_blowup
        self.num_queries, self.proof_of_work_bits = num_queries, proof_of_work_bits

    def coset_shift(self):
        return self.GENERATOR

    def log_blowup(self):
        return self._log_blowup

    def commit_batches(self, polynomials):
        return self.commit_shifted_batches(polynomials, None)

    def commit_shifted_batches(self, polynomials, coset_shifts):
        n = len(polynomials)
        digest = (C.c_uint32 * 8)()
        out = C.c_void_p()
        shifts = None
        if coset_shifts is not None:
            shifts = (C.c_uint32 * n)(*[int(s) for s in coset_shifts])
        if n and isinstance(polynomials[0], DeviceMatrix):
            arr = (C.c_void_p * n)(*[m._h for m in polynomials])
            self.ctx.check(lib().vgpu_commit_batches(self.ctx._h, arr, n, shifts, digest, C.byref(out)))
        else:
            keep = [_as_u32(p) for p in polynomials]
            arr = (_Matrix * n)(*[_mat(a) for a in keep])
            self.ctx.check(lib().vgpu_commit_batches_host(self.ctx._h, arr, n, REPR_CANONICAL, shifts, digest, C.byref(out)))
        return np.array(list(digest), dtype=np.uint32), ProverData(self.ctx, out, n)

    def open_multi_batches(self, rounds, challenger=None):
        """rounds: [(ProverData, [[point, ...] per matrix])], points as 5 canonical words.  Uses the context's
        challenger (StarkConfig.challenger()).  Returns the CBOR bytes of (opened_values, proof)."""
        handles = (C.c_void_p * len(rounds))(*[pd._h for pd, _ in rounds])
        npts = np.array([len(p) for _, pts in rounds for p in pts], dtype=np.uint32)
        flat = np.array([w for _, pts in rounds for p in pts for z in p for w in z], dtype=np.uint32)
        out = C.POINTER(C.c_uint8)()
        n = C.c_uint64()
        self.ctx.check(lib().vgpu_open(self.ctx._h, handles, len(rounds), npts.ctypes.data_as(C.POINTER(C.c_uint32)),
                                       flat.ctypes.data_as(C.POINTER(C.c_uint32)), C.byref(out), C.byref(n)))
        data = C.string_at(out, n.value)
        lib().vgpu_free_bytes(out)
        return data

    def get_ldes(self, prover_data):
        """Committed LDEs (rows stored bit-reversed), borrowed views."""
        out = []
        for i in range(prover_data.n):
            v = C.c_void_p()
            self.ctx.check(lib().vgpu_prover_data_lde(prover_data._h, i, C.byref(v)))
            out.append(DeviceMatrix(self.ctx, v, owned=False))
        return out


def _u32arr(a, n):
    a = np.ascontiguousarray(a, dtype=np.uint32).reshape(-1)
    assert a.size == n
    return (C.c_uint32 * n)(*[int(x) for x in a])


def generate_permutation_trace(ctx, chip_id, main, prep, random_elements):
    """machine/src/chip.rs:121 — returns (flattened perm trace DeviceMatrix, cumulative_sum[5])."""
    chip = lib().vgpu_basic_machine_chip(chip_id)
    out = C.c_void_p()
    cs = (C.c_uint32 * 5)()
    ctx.check(lib().vgpu_perm_trace(ctx._h, chip, main._h, prep._h if prep is not None else None, _u32arr(random_elements, 15), C.byref(out), cs))
    return DeviceMatrix(ctx, out), np.array(list(cs), dtype=np.uint32)


def quotient(ctx, chip_id, log_degree, prep_lde, main_lde, perm_lde, cumulative_sum, perm_challenges, alpha):
    """machine/src/quotient.rs:18 — returns the h x 10 quotient-chunk DeviceMatrix."""
    chip = lib().vgpu_basic_machine_chip(chip_id)
    out = C.c_void_p()
    ctx.check(lib().vgpu_quotient(ctx._h, chip, log_degree, prep_lde._h if prep_lde is not None else None, main_lde._h, perm_lde._h,
                                  _u32arr(cumulative_sum, 5), _u32arr(perm_challenges, 15), _u32arr(alpha, 5), C.byref(out)))
    return DeviceMatrix(ctx, out)


class StarkConfig:
    """StarkConfigImpl (machine/src/config.rs:33-76): the PCS plus the initial challenger.

    round_constants: the 480 Poseidon round constants the caller's RNG produced
    (Poseidon::new_from_rng(4, 22, mds, rng), basic/src/bin/valida.rs:364-365), canonical words.
    """

    def __init__(self, ctx, round_constants, mds=None):
        self.ctx = ctx
        self.pcs_ = TwoAdicFriPcs(ctx)
        rc = _u32arr(round_constants, 480)
        m = _u32arr(mds, 256) if mds is not None else None
        ctx.check(lib().vgpu_set_challenger(ctx._h, rc, m))

    def pcs(self):
        return self.pcs_


def prove_machine(config, traces, device_resident=None):
    """Machine::prove (machine/src/machine.rs:22-24): returns the CBOR bytes of MachineProof.

    traces: MachineTraces (host, row-major canonical).  device_resident: optional pair
    ([14 DeviceMatrix], [2 DeviceMatrix]) already uploaded (bench's HBM-resident timing)."""
    ctx = config.ctx
    out = C.POINTER(C.c_uint8)()
    n = C.c_uint64()
    if device_resident is not None:
        dm, dp = device_resident
        a = (C.c_void_p * NUM_CHIPS)(*[m._h for m in dm])
        b = (C.c_void_p * 2)(*[m._h for m in dp])
        ctx.check(lib().vgpu_prove_device(ctx._h, a, b, C.byref(out), C.byref(n)))
    else:
        keep = [_as_u32(m) for m in traces.main] + [_as_u32(m) for m in traces.preprocessed]
        a = (_Matrix * NUM_CHIPS)(*[_mat(m) for m in keep[:NUM_CHIPS]])
        b = (_Matrix * 2)(*[_mat(m) for m in keep[NUM_CHIPS:]])
        ctx.check(lib().vgpu_prove(ctx._h, a, b, REPR_CANONICAL, C.byref(out), C.byref(n)))
    proof = C.string_at(out, n.value)
    lib().vgpu_free_bytes(out)
    return proof


COMM_ID_BYTES = 128


def comm_init_local(contexts):
    """One process, one worker THREAD per context (a Rust host with a thread per GPU): contexts[i] becomes rank i of a
    split proof.  Afterwards every rank's calls must come from its own thread — the collectives wait for all ranks.
    Several contexts may share a device (how the split-proof tests run on a one-GPU box)."""
    n = len(contexts)
    arr = (C.c_void_p * n)(*[c._h for c in contexts])
    rc = lib().vgpu_comm_init_local(arr, n)
    if rc != 0:
        raise VgpuError(lib().vgpu_last_error(contexts[0]._h).decode())
    for i, c in enumerate(contexts):
        c.rank, c.world_size = i, n


def run_ranks(fn, contexts):
    """Run fn(rank, ctx) on one thread per context and return the results in rank order (re-raises the first failure)."""
    import threading

    out, err = [None] * len(contexts), [None] * len(contexts)

    def work(i):
        try:
            out[i] = fn(i, contexts[i])
        except BaseException as e:   # noqa: BLE001
            err[i] = e

    th = [threading.Thread(target=work, args=(i,)) for i in range(len(contexts))]
    for t in th:
        t.start()
    for t in th:
        t.join()
    for e in err:
        if e is not None:
            raise e
    return out


def comm_unique_id():
    buf = C.create_string_buffer(COMM_ID_BYTES)
    if lib().vgpu_comm_unique_id(buf) != 0:
        raise VgpuError("NCCL is not available (libnccl.so.2 could not be loaded)")
    return buf.raw


def shard_range(total, world_size, rank):
    """Contiguous balanced split used for the column shares: (begin, end)."""
    b, e = C.c_uint64(), C.c_uint64()
    lib().vgpu_shard_range(total, world_size, rank, C.byref(b), C.byref(e))
    return int(b.value), int(e.value)


def split_column_plan(world_size, shapes):
    """Column ownership of one split commit: shapes = [(height, width), ...] -> per matrix the list of world_size + 1 first-column indices."""
    n = len(shapes)
    hs = (C.c_uint64 * n)(*[int(h) for h, _ in shapes])
    ws = (C.c_uint64 * n)(*[int(w) for _, w in shapes])
    out = (C.c_uint32 * (n * (world_size + 1)))()
    lib().vgpu_split_column_plan(world_size, n, hs, ws, out)
    return [[int(out[i * (world_size + 1) + r]) for r in range(world_size + 1)] for i in range(n)]


def tree_share(length, world_size, rank):
    """(begin, count, split) — the part of a tree layer a rank derives itself when commits are split."""
    b, c, sp = C.c_uint64(), C.c_uint64(), C.c_int32()
    lib().vgpu_tree_share(length, world_size, rank, C.byref(b), C.byref(c), C.byref(sp))
    return int(b.value), int(c.value), bool(sp.value)


class VerificationError(Exception):
    """Machine::verify rejected the proof; .verdict is the VGPU_REJECT_* code of include/valida_b200.h."""

    NAMES = {-1: "malformed proof", -2: "shape mismatch", -3: "invalid proof-of-work witness", -4: "input Merkle opening",
             -5: "FRI Merkle opening", -6: "FRI final polynomial mismatch", -7: "non-zero cumulative sum"}

    def __init__(self, verdict):
        self.verdict = verdict
        what = self.NAMES.get(verdict) or ("out-of-domain evaluation mismatch on chip %d" % (-100 - verdict))
        super().__init__("proof rejected: %s (verdict %d)" % (what, verdict))


def verify_machine(config, proof, preprocessed):
    """Machine::verify (machine/src/machine.rs:26-31): raises VerificationError unless the proof is accepted.

    proof: CBOR bytes of MachineProof; preprocessed: the two preprocessed traces (program, range), row-major canonical."""
    ctx = config.ctx
    keep = [_as_u32(m) for m in preprocessed]
    b = (_Matrix * 2)(*[_mat(m) for m in keep])
    verdict = C.c_int32(-1)
    ctx.check(lib().vgpu_verify(ctx._h, bytes(proof), len(proof), b, REPR_CANONICAL, C.byref(verdict)))
    if verdict.value != 0:
        raise VerificationError(verdict.value)


def verify_machines(config, proofs, preprocessed_list, program_of=None):
    """Machine::verify for many proofs in one call, checked on the device (vgpu_verify_batch).  Returns one verdict per proof:
    0 = accepted, otherwise the VGPU_REJECT_* code vgpu_verify gives that proof alone (no exception for a rejected proof).

    proofs: CBOR bytes; preprocessed_list: one (program, range) pair of row-major canonical traces per program;
    program_of[i]: the index in preprocessed_list of proof i's program (default: preprocessed_list[i])."""
    ctx = config.ctx
    n = len(proofs)
    if program_of is None:
        program_of = list(range(n))
    if len(program_of) != n:
        raise ValueError("program_of needs one entry per proof")
    keep = [_as_u32(m) for pair in preprocessed_list for m in pair]
    mats = (_Matrix * max(1, len(keep)))(*[_mat(m) for m in keep])
    blobs = [bytes(p) for p in proofs]
    ptrs = (C.c_char_p * max(1, n))(*blobs)
    lens = (C.c_uint64 * max(1, n))(*[len(p) for p in blobs])
    prog = (C.c_uint32 * max(1, n))(*[int(g) for g in program_of])
    verdicts = (C.c_int32 * max(1, n))()
    ctx.check(lib().vgpu_verify_batch(ctx._h, ptrs, lens, n, mats, len(preprocessed_list), prog, REPR_CANONICAL, verdicts))
    return [int(verdicts[i]) for i in range(n)]


def last_verify_batch_phases(ctx):
    """[(stretch, wall-clock ms)] of the last verify_machines call on ctx: decode, commitments, transcripts, packing, device."""
    names = (C.c_char_p * 16)()
    ms = (C.c_float * 16)()
    n = lib().vgpu_last_verify_batch_phases(ctx._h, names, ms, 16)
    return [(names[i].decode(), float(ms[i])) for i in range(min(n, 16))]


def last_prove_phases(ctx):
    names = (C.c_char_p * 32)()
    ms = (C.c_float * 32)()
    n = lib().vgpu_last_prove_phases(ctx._h, names, ms, 32)
    return [(names[i].decode(), float(ms[i])) for i in range(min(n, 32))]


class MachineTraces:
    """Host witness of one BasicMachine run: 14 main traces (chip order) + 2 preprocessed traces."""

    CHIPS = ["cpu", "program", "mem", "add", "sub", "mul", "div", "shift", "lt", "com", "bitwise", "output", "range", "static_data"]

    def __init__(self, handle):
        self._h = handle
        L = lib()
        self.main = []
        for i in range(NUM_CHIPS):
            m = L.vgpu_traces_main(handle, i).contents
            self.main.append(np.ctypeslib.as_array(m.data, shape=(m.height * m.width,)).reshape(m.height, m.width))
        self.preprocessed = []
        for i in range(2):
            m = L.vgpu_traces_preprocessed(handle, i).contents
            self.preprocessed.append(np.ctypeslib.as_array(m.data, shape=(m.height * m.width,)).reshape(m.height, m.width))
        c, mo, ao = C.c_uint32(), C.c_uint32(), C.c_uint32()
        L.vgpu_traces_stats(handle, C.byref(c), C.byref(mo), C.byref(ao))
        self.clock, self.mem_ops, self.add_ops = c.value, mo.value, ao.value

    def mem_cell(self, addr):
        v = C.c_uint32()
        if lib().vgpu_traces_mem_cell(self._h, addr, C.byref(v)) != 0:
            return None
        return v.value

    def free(self):
        if self._h:
            self.main, self.preprocessed = [], []
            lib().vgpu_traces_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class VmLog:
    """Machine::run without the row fill: the interpreter's logs (one record per cycle / memory operation / ALU operation)."""

    def __init__(self, handle):
        self._h = handle
        c, mo, ao = C.c_uint32(), C.c_uint32(), C.c_uint32()
        lib().vgpu_vmlog_stats(handle, C.byref(c), C.byref(mo), C.byref(ao))
        self.clock, self.mem_ops, self.add_ops = c.value, mo.value, ao.value

    def traces(self):
        """Chip::generate_trace x14 on the host from these logs."""
        h = C.c_void_p()
        err = C.create_string_buffer(512)
        if lib().vgpu_vmlog_traces(self._h, C.byref(h), err, 512) != 0:
            raise VgpuError(err.value.decode())
        return MachineTraces(h)

    def witness_device(self, ctx):
        """Chip::generate_trace x14 on the GPU: ([14 DeviceMatrix], [2 DeviceMatrix]) for prove_machine(device_resident=...)."""
        main = (C.c_void_p * NUM_CHIPS)()
        prep = (C.c_void_p * 2)()
        ctx.check(lib().vgpu_witness_device(ctx._h, self._h, main, prep))
        return [DeviceMatrix(ctx, C.c_void_p(main[i])) for i in range(NUM_CHIPS)], [DeviceMatrix(ctx, C.c_void_p(prep[i])) for i in range(2)]

    def free(self):
        if self._h:
            lib().vgpu_vmlog_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def run_program_log(program, initial_fp=0x1000, initial_pc=0, max_cycles=1 << 30, static_data=None):
    """Machine::run only (host interpreter): returns the VmLog the host or the device expands into traces."""
    p = np.ascontiguousarray(program, dtype=np.int32)
    h = C.c_void_p()
    err = C.create_string_buffer(512)
    sa = np.array(sorted((static_data or {}).keys()), dtype=np.uint32)
    sv = np.array([(static_data or {})[int(a)] for a in sa], dtype=np.uint32)
    u32ptr = C.POINTER(C.c_uint32)
    rc = lib().vgpu_vm_run(p.ctypes.data_as(C.POINTER(C.c_int32)), p.shape[0], initial_pc, initial_fp, max_cycles,
                           sa.ctypes.data_as(u32ptr), sv.ctypes.data_as(u32ptr), len(sa), C.byref(h), err, 512)
    if rc != 0:
        raise VgpuError(err.value.decode())
    return VmLog(h)


def fib_program(n):
    """fib_program() of basic/tests/test_prover.rs:35-188 with the `imm32 -8(fp)` operand set to n."""
    words = (C.c_int32 * (23 * 6))()
    cnt = lib().vgpu_fib_program(n, words)
    return np.array(list(words), dtype=np.int32).reshape(int(cnt), 6)


def run_program(program, initial_fp=0x1000, initial_pc=0, max_cycles=1 << 30, static_data=None):
    """Machine::run + generate_trace for every chip (host).  static_data: {address: 32-bit cell} preloaded through the
    static-data chip (machine.static_data_mut().write(addr, Word(..)), basic/tests/test_static_data.rs:59-60)."""
    p = np.ascontiguousarray(program, dtype=np.int32)
    h = C.c_void_p()
    err = C.create_string_buffer(512)
    sa = np.array(sorted((static_data or {}).keys()), dtype=np.uint32)
    sv = np.array([(static_data or {})[int(a)] for a in sa], dtype=np.uint32)
    u32ptr = C.POINTER(C.c_uint32)
    rc = lib().vgpu_machine_run_static(p.ctypes.data_as(C.POINTER(C.c_int32)), p.shape[0], initial_pc, initial_fp, max_cycles,
                                       sa.ctypes.data_as(u32ptr), sv.ctypes.data_as(u32ptr), len(sa), C.byref(h), err, 512)
    if rc != 0:
        raise VgpuError(err.value.decode())
    return MachineTraces(h)
