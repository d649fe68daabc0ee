"""ctypes binding of the ehmc C-ABI (include/ehmc.h) with DLPack tensor handoff.

PyTorch is used only to own device buffers; tensors (torch or NumPy) cross the
boundary as borrowed ``DLTensor`` views obtained from their ``__dlpack__``
capsules.  There is no CPU implementation behind this module: if the shared
library is missing, or no CUDA device is usable, every compute entry raises.
"""
from __future__ import annotations

import ctypes
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_ehmc.so")

EHMC_OK = 0
FAMILY_DIAG_GAUSSIAN = 1
FAMILY_DENSE_GAUSSIAN = 2
FAMILY_FUNNEL = 3
FAMILY_NBODY = 4
FAMILY_LOGISTIC = 5
FAMILY_COIN_TOSS = 6
FAMILY_HIERARCHICAL_NORMAL = 7
LEAPFROG = 0
STORMER_VERLET = 1
FLAG_BUGCOMPAT_MOMENTUM = 1
FLAG_REJECT_NONFINITE = 2
FLAG_REUSE_ENDPOINT = 4

# every symbol include/ehmc.h declares (tests/test_abi.py checks the export list)
SYMBOLS = (
    "ehmc_version", "ehmc_last_error", "ehmc_ctx_create", "ehmc_ctx_destroy", "ehmc_ctx_launch_count",
    "ehmc_ctx_overflow_count",
    "ehmc_ctx_device_info", "ehmc_ctx_set_option", "ehmc_measure_fp32_peak", "ehmc_potential_create", "ehmc_potential_destroy",
    "ehmc_potential_eval", "ehmc_set_position", "ehmc_set_momentum", "ehmc_philox_fill", "ehmc_leapfrog",
    "ehmc_stormer_verlet", "ehmc_integrate_nbody_mode", "ehmc_hmc_iter", "ehmc_hmc_run", "ehmc_adapt_step",
    "ehmc_comm_create", "ehmc_comm_handle", "ehmc_comm_connect", "ehmc_comm_destroy", "ehmc_hmc_run_ensemble",
)
COMM_HANDLE_BYTES = 64
COMM_MAX_RANKS = 16


class EhmcError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"ehmc error {code}: {message}")
        self.code = code


class HmcArgs(ctypes.Structure):
    """struct ehmc_hmc_args (include/ehmc.h)."""

    _fields_ = [
        ("struct_size", ctypes.c_uint32),
        ("flags", ctypes.c_uint32),
        ("integrator", ctypes.c_int32),
        ("numSteps", ctypes.c_int32),
        ("stepSize", ctypes.c_double),
        ("stepSizeSq", ctypes.c_double),
        ("boltzmann", ctypes.c_double),
        ("temperature", ctypes.c_double),
        ("seed", ctypes.c_uint64),
        ("iteration", ctypes.c_uint64),
        ("particleOffset", ctypes.c_uint64),
        ("dynamic", ctypes.c_void_p),
    ]


class Dynamic(ctypes.Structure):
    """struct ehmc_dynamic (include/ehmc.h): device-resident step size / iteration of an adaptive run."""

    _fields_ = [
        ("stepSize", ctypes.c_double),
        ("logStepSize", ctypes.c_double),
        ("iteration", ctypes.c_uint64),
        ("updates", ctypes.c_uint64),
        ("row", ctypes.c_uint64),
    ]


class AdaptArgs(ctypes.Structure):
    """struct ehmc_adapt_args (include/ehmc.h)."""

    _fields_ = [
        ("struct_size", ctypes.c_uint32),
        ("adaptIterations", ctypes.c_int32),
        ("targetAccept", ctypes.c_double),
        ("gain0", ctypes.c_double),
        ("kappa", ctypes.c_double),
        ("maxMove", ctypes.c_double),
        ("minStep", ctypes.c_double),
        ("maxStep", ctypes.c_double),
        ("numParticlesTotal", ctypes.c_double),
        ("lag", ctypes.c_int32),
        ("reserved", ctypes.c_int32),
    ]


_lib = None
_lib_lock = threading.Lock()


def load():
    """dlopen the in-tree library (built by ``build.build_library`` / __graft_entry__.build)."""
    global _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        if not os.path.isfile(LIB_PATH):
            raise EhmcError(
                -2, f"{LIB_PATH} is missing: build it with `python -m physicsbasedbayesianinference_b200.build` "
                "(needs nvcc); there is no CPU fallback")
        lib = ctypes.CDLL(LIB_PATH)
        vp, ci, cd, u64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_double, ctypes.c_uint64
        lib.ehmc_version.restype = ci
        lib.ehmc_last_error.restype = ctypes.c_char_p
        lib.ehmc_last_error.argtypes = [vp]
        sigs = {
            "ehmc_ctx_create": [ci, ctypes.POINTER(vp)],
            "ehmc_ctx_destroy": [vp],
            "ehmc_ctx_launch_count": [vp, ctypes.POINTER(u64)],
            "ehmc_ctx_overflow_count": [vp, ctypes.POINTER(u64), ci],
            "ehmc_ctx_device_info": [vp, ctypes.POINTER(cd)],
            "ehmc_ctx_set_option": [vp, ctypes.c_char_p, cd],
            "ehmc_measure_fp32_peak": [vp, cd, ctypes.POINTER(cd)],
            "ehmc_potential_create": [vp, ci, ctypes.POINTER(vp), ci, ctypes.POINTER(cd), ci, ci, ctypes.POINTER(vp)],
            "ehmc_potential_destroy": [vp],
            "ehmc_potential_eval": [vp, vp, vp, vp, vp, vp],
            "ehmc_set_position": [vp, vp, cd, u64, u64, vp],
            "ehmc_set_momentum": [vp, vp, vp, cd, cd, u64, u64, u64, vp],
            "ehmc_philox_fill": [vp, vp, vp, u64, u64, u64, vp],
            "ehmc_leapfrog": [vp, vp, vp, vp, vp, cd, cd, ci, vp],
            "ehmc_stormer_verlet": [vp, vp, vp, vp, vp, cd, cd, ci, vp],
            "ehmc_integrate_nbody_mode": [vp, ci, vp, vp, vp, cd, cd, cd, ci, vp],
            "ehmc_hmc_iter": [vp, vp, vp, vp, vp, ctypes.POINTER(HmcArgs), vp, vp, vp, vp, vp],
            "ehmc_hmc_run": [vp, vp, vp, vp, ctypes.POINTER(HmcArgs), ci, vp, vp, ctypes.c_int64, vp, vp],
            "ehmc_adapt_step": [vp, vp, cd, cd, cd, cd, cd, cd, cd, u64, vp, vp, u64, vp, vp, vp],
            "ehmc_comm_create": [vp, ci, ci, ctypes.POINTER(vp)],
            "ehmc_comm_handle": [vp, vp],
            "ehmc_comm_connect": [vp, vp],
            "ehmc_comm_destroy": [vp],
            "ehmc_hmc_run_ensemble": [vp, vp, vp, vp, ctypes.POINTER(HmcArgs), ci, ctypes.POINTER(AdaptArgs), vp, vp, vp,
                                      vp, vp, ctypes.c_int64, ctypes.c_int64, vp],
        }
        for name, args in sigs.items():
            fn = getattr(lib, name)
            fn.restype = ci
            fn.argtypes = args
        _lib = lib
        return lib


def check(rc):
    if rc != EHMC_OK:
        raise EhmcError(rc, load().ehmc_last_error(None).decode("utf-8", "replace"))


# ---------------------------------------------------------------------------
# DLPack handoff
# ---------------------------------------------------------------------------
_PyCapsule_GetPointer = ctypes.pythonapi.PyCapsule_GetPointer
_PyCapsule_GetPointer.restype = ctypes.c_void_p
_PyCapsule_GetPointer.argtypes = [ctypes.py_object, ctypes.c_char_p]


class DL:
    """Borrowed DLTensor view of a torch tensor or NumPy array.

    Holds the DLPack capsule (and therefore the producer's buffer) alive; ``ptr`` is
    the ``DLManagedTensor*`` whose first member is the ``DLTensor`` the C-ABI reads.
    """

    __slots__ = ("capsule", "ptr", "owner")

    def __init__(self, t):
        self.owner = t
        if isinstance(t, np.ndarray):
            if not t.flags.writeable:
                raise ValueError("read-only NumPy arrays cannot be exported through DLPack")
            self.capsule = t.__dlpack__()
        else:
            import torch

            if not isinstance(t, torch.Tensor):
                raise TypeError(f"expected a torch.Tensor or numpy.ndarray, got {type(t).__name__}")
            self.capsule = torch.utils.dlpack.to_dlpack(t.detach())
        self.ptr = _PyCapsule_GetPointer(self.capsule, b"dltensor")


def dl(t):
    """DL view or None (for optional arguments)."""
    if t is None:
        return None
    return t if isinstance(t, DL) else DL(t)


def _p(view):
    return None if view is None else view.ptr


def is_device_tensor(t):
    return not isinstance(t, np.ndarray) and getattr(t, "is_cuda", False)


def current_stream_ptr(t=None):
    """cudaStream_t of torch's current stream on t's device (None for host data)."""
    if t is None or isinstance(t, np.ndarray) or not getattr(t, "is_cuda", False):
        return None
    import torch

    return ctypes.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


# ---------------------------------------------------------------------------
# context
# ---------------------------------------------------------------------------
class Context:
    """One per CUDA device and process (ehmc_ctx)."""

    _by_device = {}

    def __init__(self, device=-1):
        lib = load()
        h = ctypes.c_void_p()
        check(lib.ehmc_ctx_create(int(device), ctypes.byref(h)))
        self.handle = h
        self.lib = lib

    @classmethod
    def get(cls, device=None):
        if device is None:
            device = -1
            try:
                import torch

                if torch.cuda.is_available():
                    device = torch.cuda.current_device()
            except ImportError:
                pass
        dev = int(device)
        ctx = cls._by_device.get(dev)
        if ctx is None:
            ctx = cls(dev)
            cls._by_device[dev] = ctx
        return ctx

    def launch_count(self):
        n = ctypes.c_uint64()
        check(self.lib.ehmc_ctx_launch_count(self.handle, ctypes.byref(n)))
        return n.value

    def overflow_count(self, reset=True):
        """Rows of integrate() calls on the tensor-core dense kernel that left the fp16 operand range (synchronises)."""
        n = ctypes.c_uint64()
        check(self.lib.ehmc_ctx_overflow_count(self.handle, ctypes.byref(n), 1 if reset else 0))
        return n.value

    def device_info(self):
        out = (ctypes.c_double * 4)()
        check(self.lib.ehmc_ctx_device_info(self.handle, out))
        return dict(sm_count=int(out[0]), sm_clock_mhz=out[1], hbm_bytes=out[2], l2_bytes=out[3])

    def set_option(self, name, value):
        check(self.lib.ehmc_ctx_set_option(self.handle, name.encode(), float(value)))

    def measure_fp32_peak(self, millis=200.0):
        out = ctypes.c_double()
        check(self.lib.ehmc_measure_fp32_peak(self.handle, float(millis), ctypes.byref(out)))
        return out.value


class PotentialHandle:
    """ehmc_potential: device-resident, kernel-ready parameters of one family."""

    def __init__(self, ctx, family, params, scalars, bits):
        self.ctx = ctx
        views = [dl(np.ascontiguousarray(p, dtype=np.float64) if isinstance(p, np.ndarray) else p) for p in params]
        arr = (ctypes.c_void_p * max(1, len(views)))(*[v.ptr for v in views])
        sc = (ctypes.c_double * max(1, len(scalars)))(*[float(s) for s in scalars])
        h = ctypes.c_void_p()
        check(ctx.lib.ehmc_potential_create(ctx.handle, int(family), arr, len(views), sc, len(scalars), int(bits),
                                            ctypes.byref(h)))
        self.handle = h

    def __del__(self):
        h = getattr(self, "handle", None)
        if h:
            try:
                self.ctx.lib.ehmc_potential_destroy(h)
            except Exception:
                pass
            self.handle = None


# ---------------------------------------------------------------------------
# thin call wrappers (arguments: torch tensors / NumPy arrays / DL views / None)
# ---------------------------------------------------------------------------
def potential_eval(ctx, pot, q, energy=None, grad=None, stream=None):
    vq, ve, vg = dl(q), dl(energy), dl(grad)
    check(ctx.lib.ehmc_potential_eval(ctx.handle, pot.handle, vq.ptr, _p(ve), _p(vg), stream))


def leapfrog(ctx, pot, q, p, mass, step_size, step_size_sq, num_steps, stream=None, stormer=False):
    vq, vp, vm = dl(q), dl(p), dl(mass)
    fn = ctx.lib.ehmc_stormer_verlet if stormer else ctx.lib.ehmc_leapfrog
    check(fn(ctx.handle, pot.handle, vq.ptr, vp.ptr, vm.ptr, float(step_size), float(step_size_sq), int(num_steps),
             stream))


def integrate_nbody_mode(ctx, integrator, q, p, mass, grav, step_size, step_size_sq, num_steps, stream=None):
    vq, vp, vm = dl(q), dl(p), dl(mass)
    check(ctx.lib.ehmc_integrate_nbody_mode(ctx.handle, int(integrator), vq.ptr, vp.ptr, vm.ptr, float(grav),
                                            float(step_size), float(step_size_sq), int(num_steps), stream))


def make_args(step_size, step_size_sq, num_steps, boltzmann, temperature, integrator=LEAPFROG, flags=0, seed=0,
              iteration=0, particle_offset=0, dynamic=None):
    a = HmcArgs()
    a.struct_size = ctypes.sizeof(HmcArgs)
    a.flags = int(flags)
    a.integrator = int(integrator)
    a.numSteps = int(num_steps)
    a.stepSize = float(step_size)
    a.stepSizeSq = float(step_size_sq)
    a.boltzmann = float(boltzmann)
    a.temperature = float(temperature)
    a.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    a.iteration = int(iteration) & 0xFFFFFFFFFFFFFFFF
    a.particleOffset = int(particle_offset)
    a.dynamic = None if dynamic is None else int(dynamic)
    return a


def dynamic_to_device(step_size, iteration, device, row=0):
    """A device copy of ehmc_dynamic (as a uint8 tensor; pass ``.data_ptr()`` as args.dynamic)."""
    import math

    import torch

    d = Dynamic(float(step_size), math.log(step_size), int(iteration), 0, int(row))
    return torch.frombuffer(bytearray(bytes(d)), dtype=torch.uint8).to(device)


def dynamic_from_device(t):
    return Dynamic.from_buffer_copy(t.cpu().numpy().tobytes())


def adapt_step(ctx, stats, num_particles_total, dynamic_ptr, target=0.8, gain0=1.5, kappa=0.5, max_move=0.7,
               min_step=1e-6, max_step=1e3, adapt_rows=1 << 62, state_ptr=None, stride=1, history=None, moments=None,
               stream=None):
    vs, vh, vm = dl(stats), dl(history), dl(moments)
    check(ctx.lib.ehmc_adapt_step(ctx.handle, vs.ptr, float(num_particles_total), float(target), float(gain0),
                                  float(kappa), float(max_move), float(min_step), float(max_step), int(adapt_rows),
                                  int(dynamic_ptr), None if state_ptr is None else int(state_ptr), int(stride),
                                  _p(vh), _p(vm), stream))


def hmc_iter(ctx, pot, q, mass, args, p_out=None, z=None, u=None, accept=None, stats=None, stream=None):
    vq, vm = dl(q), dl(mass)
    vp, vz, vu, va, vs = dl(p_out), dl(z), dl(u), dl(accept), dl(stats)
    check(ctx.lib.ehmc_hmc_iter(ctx.handle, pot.handle, vq.ptr, _p(vp), vm.ptr, ctypes.byref(args), _p(vz), _p(vu),
                                _p(va), _p(vs), stream))


def hmc_run(ctx, pot, q, mass, args, num_iterations, samples=None, momenta=None, sample_offset=0, accepted=None,
            stream=None):
    """numIterations iterations in one launch; samples / momenta are [D*P, S] views of (D, P, S) arrays."""
    vq, vm = dl(q), dl(mass)
    vs, vmo, va = dl(samples), dl(momenta), dl(accepted)
    check(ctx.lib.ehmc_hmc_run(ctx.handle, pot.handle, vq.ptr, vm.ptr, ctypes.byref(args), int(num_iterations), _p(vs),
                               _p(vmo), int(sample_offset), _p(va), stream))


class Comm:
    """ehmc_comm: this rank's mailbox plus the mapped mailboxes of its peers (CUDA IPC over NVLink)."""

    def __init__(self, ctx, rank, world):
        self.ctx, self.rank, self.world = ctx, int(rank), int(world)
        h = ctypes.c_void_p()
        check(ctx.lib.ehmc_comm_create(ctx.handle, self.rank, self.world, ctypes.byref(h)))
        self.handle = h

    def local_handle(self):
        buf = (ctypes.c_ubyte * COMM_HANDLE_BYTES)()
        check(self.ctx.lib.ehmc_comm_handle(self.handle, buf))
        return bytes(buf)

    def connect(self, handles):
        """handles: world x COMM_HANDLE_BYTES bytes, ordered by rank."""
        blob = b"".join(handles) if not isinstance(handles, (bytes, bytearray)) else bytes(handles)
        if len(blob) != self.world * COMM_HANDLE_BYTES:
            raise ValueError("need one handle per rank")
        buf = (ctypes.c_ubyte * len(blob)).from_buffer_copy(blob)
        check(self.ctx.lib.ehmc_comm_connect(self.handle, buf))

    def __del__(self):
        h = getattr(self, "handle", None)
        if h:
            try:
                self.ctx.lib.ehmc_comm_destroy(h)
            except Exception:
                pass
            self.handle = None


def make_adapt_args(num_particles_total, adapt_iterations, target=0.8, gain0=1.5, kappa=0.5, max_move=0.7,
                    min_step=1e-6, max_step=1e3, lag=1):
    a = AdaptArgs()
    a.lag = int(lag)
    a.struct_size = ctypes.sizeof(AdaptArgs)
    a.adaptIterations = int(adapt_iterations)
    a.targetAccept, a.gain0, a.kappa, a.maxMove = float(target), float(gain0), float(kappa), float(max_move)
    a.minStep, a.maxStep = float(min_step), float(max_step)
    a.numParticlesTotal = float(num_particles_total)
    return a


def hmc_run_ensemble(ctx, pot, q, mass, args, num_iterations, adapt, state, comm=None, history=None, moments=None,
                     trace=None, trace_particles=0, trace_offset=0, stream=None):
    vq, vm, vs = dl(q), dl(mass), dl(state)
    vh, vmo, vt = dl(history), dl(moments), dl(trace)
    check(ctx.lib.ehmc_hmc_run_ensemble(ctx.handle, pot.handle, vq.ptr, vm.ptr, ctypes.byref(args), int(num_iterations),
                                        ctypes.byref(adapt), None if comm is None else comm.handle, vs.ptr, _p(vh),
                                        _p(vmo), _p(vt), int(trace_particles), int(trace_offset), stream))


def philox_fill(ctx, z=None, u=None, seed=0, iteration=0, particle_offset=0, stream=None):
    vz, vu = dl(z), dl(u)
    check(ctx.lib.ehmc_philox_fill(ctx.handle, _p(vz), _p(vu), int(seed), int(iteration) & 0xFFFFFFFFFFFFFFFF,
                                   int(particle_offset), stream))


def set_position(ctx, q, q_std, seed, particle_offset=0, stream=None):
    vq = dl(q)
    check(ctx.lib.ehmc_set_position(ctx.handle, vq.ptr, float(q_std), int(seed), int(particle_offset), stream))


def set_momentum(ctx, p, mass, boltzmann, temperature, seed, iteration, particle_offset=0, stream=None):
    vp, vm = dl(p), dl(mass)
    check(ctx.lib.ehmc_set_momentum(ctx.handle, vp.ptr, vm.ptr, float(boltzmann), float(temperature), int(seed),
                                    int(iteration) & 0xFFFFFFFFFFFFFFFF, int(particle_offset), stream))
