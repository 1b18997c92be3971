"""ctypes binding of librokifd_b200.so - the host-side Python mirror of the reference's rkfd_sim
interface (reference include/roki_fd/rkfd_sim.h:58-102): same call names in snake_case, same argument
meaning, same life cycle Create -> (ContactInfo | ChainReg | SetDis/SetVel | SetSolver | PrpSet)* ->
UpdateInit -> Update* -> UpdateDestroy -> Destroy.

There is NO CPU fallback: loading fails loudly if the CUDA library has not been built, and
`update_init` raises if no device engine could be created.
"""
import ctypes as C
import os

import numpy as np

from .chains import NDOF, ChainModel, World

_HERE = os.path.dirname(os.path.abspath(__file__))
# ROKIFD_B200_LIB: a tuning aid (tools/build_exp.sh builds variants of the library); the default is the in-tree product library
LIB_PATH = os.environ.get("ROKIFD_B200_LIB") or os.path.join(_HERE, "librokifd_b200.so")

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)

JOINT = {"fixed": 0, "revolute": 1, "prismatic": 2, "spherical": 3, "float": 4, "cylindrical": 5, "hooke": 6, "breakablefloat": 7}
MOTOR = {None: 0, "none": 0, "dc": 1, "trq": 2}
CONTACT = {"rigid": 0, "elastic": 1}
SOLVER = {"Vert": 0, "MLCP": 1, "Volume": 2}


class LinkDesc(C.Structure):
    """rkB200LinkDesc of include/roki_fd/rkfd_b200.h"""
    _fields_ = [("name", C.c_char_p), ("stuff", C.c_char_p), ("parent", C.c_int), ("jointtype", C.c_int),
                ("frame_R", C.c_double * 9), ("frame_p", C.c_double * 3), ("mass", C.c_double),
                ("com", C.c_double * 3), ("inertia", C.c_double * 9),
                ("stiffness", C.c_double), ("viscosity", C.c_double), ("coulomb", C.c_double),
                ("staticfriction", C.c_double), ("motortype", C.c_int),
                ("motorconstant", C.c_double), ("admittance", C.c_double), ("gearratio", C.c_double),
                ("rotorinertia", C.c_double), ("gearinertia", C.c_double), ("minvoltage", C.c_double),
                ("maxvoltage", C.c_double), ("forcethreshold", C.c_double), ("torquethreshold", C.c_double)]


_LIB = None


def lib():
    """Loads the C-ABI library; raises if it was not built (no fallback path exists)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("rokifd_b200: %s not found - build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, ci, cd = C.c_void_p, C.c_int, C.c_double
    sig = {
        "rkFDB200Alloc": (vp, []), "rkFDB200Free": (None, [vp]), "rkChainB200Alloc": (vp, []), "rkChainB200Free": (None, [vp]),
        "rkFDCreate": (vp, [vp]), "rkFDDestroy": (None, [vp]),
        "rkChainInit": (vp, [vp]), "rkChainDestroy": (None, [vp]), "rkChainReadZTK": (vp, [vp, C.c_char_p]),
        "rkChainLinkNum": (ci, [vp]), "rkChainJointSize": (ci, [vp]), "rkChainLinkJoint": (vp, [vp, ci]),
        "rkCDPairChainUnreg": (None, [vp, vp]), "rkJointMotorSetInput": (None, [vp, _dp]), "rkJointGetDis": (None, [vp, _dp]), "rkJointGetVel": (None, [vp, _dp]),
        "rkJointDOF": (ci, [vp]),
        "rkB200LinkDescInit": (None, [C.POINTER(LinkDesc)]), "rkChainB200SetName": (ci, [vp, C.c_char_p]),
        "rkChainB200AddLink": (ci, [vp, C.POINTER(LinkDesc)]), "rkChainB200LinkAddVerts": (ci, [vp, ci, ci, _dp]),
        "rkChainB200LinkAddBox": (ci, [vp, ci, _dp, cd, cd, cd]),
        "rkFDChainReg": (vp, [vp, vp]), "rkFDChainRegFile": (vp, [vp, C.c_char_p]), "rkFDChainUnreg": (C.c_bool, [vp, vp]),
        "rkFDChainSetDis": (None, [vp, vp]), "rkFDChainSetVel": (None, [vp, vp]),
        "rkFDContactInfoScanFile": (C.c_bool, [vp, C.c_char_p]),
        "rkFDContactInfoAdd": (C.c_bool, [vp, C.c_char_p, C.c_char_p, ci, cd, cd, cd, cd, cd, cd]),
        "rkFDUpdateInit": (None, [vp]), "rkFDUpdate": (vp, [vp]), "rkFDUpdateN": (vp, [vp, ci]),
        "rkFDUpdateDestroy": (None, [vp]), "rkFDSolve": (vp, [vp]),
        "rkFDB200PrpSet": (None, [vp, cd, ci, cd, ci]), "rkFDB200SetSolver": (ci, [vp, ci]), "rkFDB200SetIntegrator": (ci, [vp, ci]), "rkFDB200Time": (cd, [vp]),
        "rkFDB200Size": (ci, [vp]), "rkFDB200CellChain": (vp, [vp]),
        "rkFDB200Dis": (_dp, [vp]), "rkFDB200Vel": (_dp, [vp]), "rkFDB200Acc": (_dp, [vp]),
        "zVecAlloc": (vp, [ci]), "zVecFree": (None, [vp]),
        "rkFDBatchSetEnvNum": (ci, [vp, ci]), "rkFDBatchSetDevices": (ci, [vp, _ip, ci]), "rkFDBatchSetStream": (ci, [vp, vp]),
        "rkFDBatchEnvNum": (ci, [vp]), "rkFDBatchReady": (ci, [vp]), "rkFDBatchLinkNum": (ci, [vp]), "rkFDBatchContactSlotNum": (ci, [vp]),
        "rkFDBatchSetState": (ci, [vp, vp, vp]), "rkFDBatchGetState": (ci, [vp, vp, vp, vp]),
        "rkFDBatchSetMotorInput": (ci, [vp, vp]), "rkFDBatchGetContactForce": (ci, [vp, vp]),
        "rkFDBatchGetContactState": (ci, [vp, vp, vp, vp]), "rkFDBatchSetContactState": (ci, [vp, vp, vp, vp]),
        "rkFDBatchGetPivot": (ci, [vp, vp, vp]), "rkFDBatchSetPivot": (ci, [vp, vp, vp]),
        "rkFDBatchSetStateAsync": (ci, [vp, vp, vp]), "rkFDBatchSetMotorInputAsync": (ci, [vp, vp]),
        "rkFDBatchGetStateAsync": (ci, [vp, vp, vp, vp]), "rkFDBatchJoin": (ci, [vp]),
        "rkFDBatchSetResortInterval": (ci, [vp, ci]), "rkFDBatchSlotMap": (ci, [vp, ci, _ip]), "rkFDBatchResortCount": (C.c_longlong, [vp]), "rkFDBatchResortKernelCount": (C.c_longlong, [vp]),
        "rkFDBatchGetStatus": (ci, [vp, vp]), "rkFDBatchStats": (ci, [vp, C.POINTER(cd)]), "rkFDBatchEval": (ci, [vp, ci]), "rkFDBatchSync": (ci, [vp]),
        "rkFDBatchDevicePtr": (vp, [vp, ci, ci, _ip, _ip]), "rkFDBatchLaunchCount": (C.c_longlong, [vp]),
        "rkFDBatchResetEnvs": (ci, [vp, ci, vp, vp, vp, vp]), "rkFDBatchResetEnvsDevice": (ci, [vp, ci, ci, vp, vp, vp, vp]),
        "rkFDBatchResetKernelCount": (C.c_longlong, [vp]),
        "rkFDBatchGetLinkFrames": (ci, [vp, ci, vp, vp, vp]), "rkFDBatchGetLinkFramesDevice": (ci, [vp, ci, ci, vp, vp, vp]),
        "rkFDBatchLinkFrameKernelCount": (C.c_longlong, [vp]), "rkFDBatchKernelVariant": (ci, [vp, ci, _ip]),
        "rkFDBatchSetExtWrenchLinks": (ci, [vp, ci, vp]), "rkFDBatchSetExtWrench": (ci, [vp, vp]), "rkFDBatchSetExtWrenchDevice": (ci, [vp, ci, vp]),
        "rkFDBatchSetMassPropLinks": (ci, [vp, ci, vp]), "rkFDBatchSetMassProp": (ci, [vp, vp]), "rkFDBatchSetMassPropDevice": (ci, [vp, ci, vp]),
        "rkFDB200DescribeModel": (ci, [vp, C.c_char_p, ci]), "rkFDBatchLastError": (C.c_char_p, []), "rkFDBatchDeviceCount": (ci, []), "rkFDB200MeasureFp64": (ci, [_dp]),
    }
    for name, (res, args) in sig.items():
        f = getattr(L, name)
        f.restype, f.argtypes = res, args
    _LIB = L
    return L


def _ptr(a):
    """address of a numpy array or a raw integer address (e.g. torch pinned tensor .data_ptr())"""
    if a is None:
        return None
    if isinstance(a, (int, np.integer)):
        return C.c_void_p(int(a))
    assert a.flags["C_CONTIGUOUS"]
    return C.c_void_p(a.ctypes.data)


class RkChain:
    """[EXT] rkChain stand-in: built programmatically or read from a ZTK file."""

    def __init__(self, model: ChainModel = None, ztk: str = None):
        L = lib()
        self.h = L.rkChainB200Alloc()
        if ztk is not None:
            if not L.rkChainReadZTK(self.h, ztk.encode()):
                L.rkChainB200Free(self.h)
                self.h = None
                raise RuntimeError("rkChainReadZTK(%s): %s" % (ztk, L.rkFDBatchLastError().decode()))
            return
        L.rkChainInit(self.h)
        if model is not None:
            L.rkChainB200SetName(self.h, model.name.encode())
            self._keep = []
            for k, l in enumerate(model.links):
                d = LinkDesc()
                L.rkB200LinkDescInit(C.byref(d))
                nm, st = l.name.encode(), l.stuff.encode()
                self._keep += [nm, st]
                d.name, d.stuff, d.parent, d.jointtype = nm, st, l.parent, JOINT[l.jtype]
                d.frame_R[:] = list(np.asarray(l.org_R, float).reshape(9))
                d.frame_p[:] = list(np.asarray(l.org_p, float))
                d.mass = l.mass
                d.com[:] = list(np.asarray(l.com, float))
                d.inertia[:] = list(np.asarray(l.inertia, float).reshape(9))
                d.stiffness, d.viscosity, d.coulomb, d.staticfriction = l.stiffness, l.viscosity, l.coulomb, l.sfriction
                d.forcethreshold, d.torquethreshold = getattr(l, "break_force", 0.0), getattr(l, "break_torque", 0.0)
                if l.motor is not None:
                    m = l.motor
                    d.motortype = MOTOR[m.type]
                    d.motorconstant, d.admittance, d.gearratio = m.k, m.admittance, m.gear
                    d.rotorinertia, d.gearinertia, d.minvoltage, d.maxvoltage = m.rotor_inertia, m.gear_inertia, m.min, m.max
                if L.rkChainB200AddLink(self.h, C.byref(d)) != k:
                    raise RuntimeError("rkChainB200AddLink: " + L.rkFDBatchLastError().decode())
                for v in l.shapes:
                    v = np.ascontiguousarray(v, np.float64)
                    L.rkChainB200LinkAddVerts(self.h, k, v.shape[0], v.ctypes.data_as(_dp))
                for (c, dd, w, hh) in l.boxes:
                    c = np.ascontiguousarray(c, np.float64)
                    L.rkChainB200LinkAddBox(self.h, k, c.ctypes.data_as(_dp), dd, w, hh)

    @property
    def link_num(self):
        return lib().rkChainLinkNum(self.h)

    @property
    def joint_size(self):
        return lib().rkChainJointSize(self.h)

    def destroy(self):
        if self.h:
            lib().rkChainDestroy(self.h)
            lib().rkChainB200Free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


class RkFDCell:
    def __init__(self, h):
        self.h = h

    @property
    def chain_handle(self):
        return lib().rkFDB200CellChain(self.h)

    def joint_motor_set_input(self, link, value):
        """rkJointMotorSetInput(rkChainLinkJoint(rkFDCellChain(cell), link), &value)"""
        L = lib()
        v = C.c_double(value)
        L.rkJointMotorSetInput(L.rkChainLinkJoint(self.chain_handle, link), C.byref(v))


class RkFD:
    """The forward-dynamics simulator object (reference `rkFD`, rkfd_sim.h:38-52)."""

    def __init__(self):
        L = lib()
        self.h = L.rkFDB200Alloc()
        if not L.rkFDCreate(self.h):
            raise RuntimeError("rkFDCreate failed")
        self._alive = True

    # ---- reference API ---------------------------------------------------------------------------
    def chain_reg(self, chain):
        c = chain if isinstance(chain, RkChain) else RkChain(chain)
        h = lib().rkFDChainReg(self.h, c.h)
        if not h:
            raise RuntimeError("rkFDChainReg: " + self.last_error())
        if c is not chain:
            c.destroy()          # the simulator holds a clone (reference rkfd_sim.c:217)
        return RkFDCell(h)

    def chain_reg_file(self, filename):
        h = lib().rkFDChainRegFile(self.h, filename.encode())
        return RkFDCell(h) if h else None

    def chain_unreg(self, cell):
        return bool(lib().rkFDChainUnreg(self.h, cell.h))

    def _zvec(self, a):
        L = lib()
        a = np.ascontiguousarray(a, np.float64)
        v = L.zVecAlloc(a.shape[0])
        buf = C.cast(C.cast(v, C.POINTER(C.c_void_p))[1], _dp)   # zVecStruct {int size; double *buf}
        for i in range(a.shape[0]):
            buf[i] = a[i]
        return v

    def chain_set_dis(self, cell, dis):
        v = self._zvec(dis)
        lib().rkFDChainSetDis(cell.h, v)
        lib().zVecFree(v)

    def chain_set_vel(self, cell, vel):
        v = self._zvec(vel)
        lib().rkFDChainSetVel(cell.h, v)
        lib().zVecFree(v)

    def contact_info_scan_file(self, filename):
        return bool(lib().rkFDContactInfoScanFile(self.h, filename.encode()))

    def contact_info_add(self, ci):
        return bool(lib().rkFDContactInfoAdd(self.h, ci.stuff_a.encode(), ci.stuff_b.encode(), CONTACT[ci.type],
                                             ci.K, ci.L, ci.E, ci.V, ci.SF, ci.KF))

    def prp_set(self, dt=0.001, pyramid=8, friction_weight=100.0, max_iter=10):
        lib().rkFDB200PrpSet(self.h, dt, pyramid, friction_weight, max_iter)

    def set_integrator(self, name):
        """rkFDODE2AssignRegular(fd, RKG | RK4 | Euler | Heun)."""
        if lib().rkFDB200SetIntegrator(self.h, {"RKG": 0, "RK4": 1, "Euler": 2, "Heun": 3}[name]) != 0:
            raise ValueError("integrator %r" % name)

    def set_solver(self, name):
        if lib().rkFDB200SetSolver(self.h, SOLVER[name]) != 0:
            raise RuntimeError(self.last_error())

    def update_init(self):
        lib().rkFDUpdateInit(self.h)
        if not lib().rkFDBatchReady(self.h):
            raise RuntimeError("rkFDUpdateInit: " + self.last_error())
        self._ck(lib().rkFDBatchSync(self.h))

    def update(self):
        if not lib().rkFDUpdate(self.h):          # NULL: no device engine (there is no CPU fallback)
            raise RuntimeError(self.last_error())

    def update_n(self, k):
        if not lib().rkFDUpdateN(self.h, k):
            raise RuntimeError(self.last_error())

    def update_destroy(self):
        lib().rkFDUpdateDestroy(self.h)

    def destroy(self):
        if getattr(self, "_alive", False):
            lib().rkFDDestroy(self.h)
            lib().rkFDB200Free(self.h)
            self._alive = False

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass

    @property
    def time(self):
        return lib().rkFDB200Time(self.h)

    @property
    def size(self):
        return lib().rkFDB200Size(self.h)

    def _vec(self, fn):
        n = self.size
        p = fn(self.h)
        return np.array([p[i] for i in range(n)], float)

    @property
    def dis(self):
        return self._vec(lib().rkFDB200Dis)

    @property
    def vel(self):
        return self._vec(lib().rkFDB200Vel)

    @property
    def acc(self):
        return self._vec(lib().rkFDB200Acc)

    # ---- batched extension -----------------------------------------------------------------------
    def last_error(self):
        return lib().rkFDBatchLastError().decode()

    def _ck(self, rc):
        if rc != 0:
            raise RuntimeError("rokifd_b200: " + self.last_error())

    def batch_set_env_num(self, B):
        self._ck(lib().rkFDBatchSetEnvNum(self.h, B))

    def batch_set_devices(self, ids):
        a = np.ascontiguousarray(ids, np.int32)
        self._ck(lib().rkFDBatchSetDevices(self.h, a.ctypes.data_as(_ip), a.shape[0]))

    def batch_set_stream(self, cuda_stream):
        self._ck(lib().rkFDBatchSetStream(self.h, C.c_void_p(int(cuda_stream))))

    @property
    def env_num(self):
        return lib().rkFDBatchEnvNum(self.h)

    @property
    def link_num(self):
        return lib().rkFDBatchLinkNum(self.h)

    @property
    def slot_num(self):
        return lib().rkFDBatchContactSlotNum(self.h)

    def batch_set_state(self, q, qd):
        if isinstance(q, np.ndarray):
            q, qd = np.ascontiguousarray(q, np.float64), np.ascontiguousarray(qd, np.float64)
        self._ck(lib().rkFDBatchSetState(self.h, _ptr(q), _ptr(qd)))

    def batch_get_state(self, q=None, qd=None, qdd=None):
        """Fills the given env-major arrays (or raw addresses); allocates numpy arrays when none is given."""
        if q is None and qd is None and qdd is None:
            shp = (self.env_num, max(self.size, 1))
            q, qd, qdd = np.zeros(shp), np.zeros(shp), np.zeros(shp)
            self._ck(lib().rkFDBatchGetState(self.h, _ptr(q), _ptr(qd), _ptr(qdd)))
            n = self.size
            return q[:, :n], qd[:, :n], qdd[:, :n]
        self._ck(lib().rkFDBatchGetState(self.h, _ptr(q), _ptr(qd), _ptr(qdd)))
        return q, qd, qdd

    def batch_set_state_async(self, q, qd):
        """pinned host buffers (numpy arrays or raw addresses); valid until batch_sync()"""
        self._ck(lib().rkFDBatchSetStateAsync(self.h, _ptr(q), _ptr(qd)))

    def batch_set_motor_input_async(self, u):
        self._ck(lib().rkFDBatchSetMotorInputAsync(self.h, _ptr(u)))

    def batch_get_state_async(self, q, qd, qdd):
        self._ck(lib().rkFDBatchGetStateAsync(self.h, _ptr(q), _ptr(qd), _ptr(qdd)))

    def batch_join(self):
        self._ck(lib().rkFDBatchJoin(self.h))

    def batch_set_motor_input(self, u):
        if isinstance(u, np.ndarray):
            u = np.ascontiguousarray(u, np.float64)
        self._ck(lib().rkFDBatchSetMotorInput(self.h, _ptr(u)))

    def batch_get_contact(self):
        B, ns = self.env_num, max(self.slot_num, 1)
        a, t = np.zeros((B, ns), np.int32), np.zeros((B, ns), np.int32)
        r, f = np.zeros((B, ns, 3)), np.zeros((B, ns, 3))
        self._ck(lib().rkFDBatchGetContactState(self.h, _ptr(a), _ptr(t), _ptr(r)))
        self._ck(lib().rkFDBatchGetContactForce(self.h, _ptr(f)))
        n = self.slot_num
        return a[:, :n], t[:, :n], r[:, :n], f[:, :n]

    def batch_set_contact(self, active, type_, ref):
        a = np.ascontiguousarray(active, np.int32)
        t = np.ascontiguousarray(type_, np.int32)
        r = np.ascontiguousarray(ref, np.float64)
        self._ck(lib().rkFDBatchSetContactState(self.h, _ptr(a), _ptr(t), _ptr(r)))

    def batch_get_pivot(self):
        B, n = self.env_num, max(self.size, 1)
        t, p = np.zeros((B, n), np.int32), np.zeros((B, n))
        self._ck(lib().rkFDBatchGetPivot(self.h, _ptr(t), _ptr(p)))
        return t[:, :self.size], p[:, :self.size]

    def batch_set_pivot(self, type_, prev):
        t = np.ascontiguousarray(type_, np.int32)
        p = np.ascontiguousarray(prev, np.float64)
        self._ck(lib().rkFDBatchSetPivot(self.h, _ptr(t), _ptr(p)))

    def batch_get_status(self):
        s = np.zeros(self.env_num, np.int32)
        self._ck(lib().rkFDBatchGetStatus(self.h, _ptr(s)))
        return s

    def describe_model(self):
        """The flattened device model of the last update_init as {name: [numbers]} (host side, no device needed)."""
        n = lib().rkFDB200DescribeModel(self.h, None, 0)
        buf = C.create_string_buffer(n + 1)
        lib().rkFDB200DescribeModel(self.h, buf, n + 1)
        out = {}
        for line in buf.value.decode().splitlines():
            k, _, v = line.partition(":")
            out[k] = [float(x) for x in v.split()]
        return out

    def batch_set_resort_interval(self, steps):
        self._ck(lib().rkFDBatchSetResortInterval(self.h, steps))

    @property
    def resort_count(self):
        return lib().rkFDBatchResortCount(self.h)

    @property
    def resort_kernel_count(self):
        return lib().rkFDBatchResortKernelCount(self.h)

    def batch_stats(self):
        """[envs, envs in contact, active contact vertices, flagged envs (sums), max|q''|, max|q'| (maxima)] of this process's batch."""
        out = (C.c_double * 8)()
        self._ck(lib().rkFDBatchStats(self.h, out))
        return [float(v) for v in out[:6]]

    def batch_eval(self, do_up_ref=False):
        self._ck(lib().rkFDBatchEval(self.h, int(do_up_ref)))

    def batch_sync(self):
        self._ck(lib().rkFDBatchSync(self.h))

    @property
    def launch_count(self):
        return lib().rkFDBatchLaunchCount(self.h)

    def batch_reset_envs(self, envs, q, qd=None, u=None):
        """rkFDBatchResetEnvs: environments envs[i] restart from (q[i], qd[i], u[i]) as after a new update_init; qd None: zero,
        u None: the current motor input.  The other environments go on unchanged."""
        e = np.ascontiguousarray(envs, np.int32).reshape(-1)
        n = e.shape[0]
        q = None if q is None else np.ascontiguousarray(q, np.float64)     # None: refused by the library (q is required)
        qd = None if qd is None else np.ascontiguousarray(qd, np.float64)
        u = None if u is None else np.ascontiguousarray(u, np.float64)
        for a, w in ((q, self.size), (qd, self.size), (u, self.link_num)):
            if a is not None and a.size != n * w:
                raise ValueError("batch_reset_envs: expected %d x %d values, got shape %s" % (n, w, a.shape))
        self._ck(lib().rkFDBatchResetEnvs(self.h, n, _ptr(e), _ptr(q), _ptr(qd), _ptr(u)))

    def batch_reset_envs_device(self, shard, n, envs_ptr, q_ptr, qd_ptr=None, u_ptr=None):
        """rkFDBatchResetEnvsDevice: raw device addresses (e.g. torch CUDA tensor .data_ptr()) of int32 envs[n] (indices local to
        the shard), q[n][size], qd[n][size], u[n][links]; stream-ordered on the engine's stream."""
        self._ck(lib().rkFDBatchResetEnvsDevice(self.h, shard, n, _ptr(envs_ptr), _ptr(q_ptr), _ptr(qd_ptr), _ptr(u_ptr)))

    @property
    def reset_kernel_count(self):
        return lib().rkFDBatchResetKernelCount(self.h)

    def batch_get_link_frames(self, links=None, frames=True, vel=True):
        """rkFDBatchGetLinkFrames: world frames (B, n, 12) - R row-major, then p - and velocities (B, n, 6) - linear, angular,
        world axes - of links (indices in flat_links() order; None: all links), from the committed state.  An output not
        requested is returned as None."""
        if links is None:
            n, pl = self.link_num, None
        else:
            pl = np.ascontiguousarray(links, np.int32).reshape(-1)
            n = pl.shape[0]
        B = self.env_num
        fr = np.zeros((B, n, 12)) if frames else None
        v = np.zeros((B, n, 6)) if vel else None
        self._ck(lib().rkFDBatchGetLinkFrames(self.h, n, _ptr(pl), _ptr(fr), _ptr(v)))
        return fr, v

    def batch_get_link_frames_device(self, shard, links, frame_ptr, vel_ptr):
        """rkFDBatchGetLinkFramesDevice: raw device addresses (e.g. torch CUDA tensor .data_ptr(), or None) of float64
        frame[Bs][n][12] and vel[Bs][n][6] of shard `shard`, indexed by the shard's local environment; stream-ordered on the
        engine's stream.  links: a host list of link indices (None: all links)."""
        if links is None:
            n, pl = self.link_num, None
        else:
            pl = np.ascontiguousarray(links, np.int32).reshape(-1)
            n = pl.shape[0]
        self._ck(lib().rkFDBatchGetLinkFramesDevice(self.h, shard, n, _ptr(pl), _ptr(frame_ptr), _ptr(vel_ptr)))

    @property
    def link_frame_kernel_count(self):
        return lib().rkFDBatchLinkFrameKernelCount(self.h)

    def batch_set_ext_wrench_links(self, links):
        """rkFDBatchSetExtWrenchLinks (before update_init): the links (indices in flat_links() order) that take an external
        wrench, in the order of its rows; an empty list clears the declaration."""
        pl = np.ascontiguousarray(links, np.int32).reshape(-1)
        self._ck(lib().rkFDBatchSetExtWrenchLinks(self.h, pl.shape[0], _ptr(pl)))

    def batch_set_ext_wrench(self, w):
        """rkFDBatchSetExtWrench: (B, n, 6) float64 host array, (force, torque about the centre of mass) in world axes per declared
        link; held as pending before update_init."""
        if isinstance(w, np.ndarray):
            w = np.ascontiguousarray(w, np.float64)
        self._ck(lib().rkFDBatchSetExtWrench(self.h, _ptr(w)))

    def batch_set_ext_wrench_device(self, shard, w_ptr):
        """rkFDBatchSetExtWrenchDevice: raw device address (e.g. torch CUDA tensor .data_ptr()) of float64 w[Bs][n][6] of shard
        `shard`, indexed by the shard's local environment; stream-ordered on the engine's stream."""
        self._ck(lib().rkFDBatchSetExtWrenchDevice(self.h, shard, _ptr(w_ptr)))

    def batch_set_mass_prop_links(self, links):
        """rkFDBatchSetMassPropLinks (before update_init): the links (indices in flat_links() order) that take per-environment
        mass properties, in the order of their rows; an empty list clears the declaration."""
        pl = np.ascontiguousarray(links, np.int32).reshape(-1)
        self._ck(lib().rkFDBatchSetMassPropLinks(self.h, pl.shape[0], _ptr(pl)))

    def batch_set_mass_prop(self, mp):
        """rkFDBatchSetMassProp: (B, n, 10) float64 host array, (mass, centre of mass, inertia about the centre of mass xx xy xz
        yy yz zz) in link axes per declared link; checked (finite, mass > 0, inertia positive definite); held as pending before
        update_init."""
        if isinstance(mp, np.ndarray):
            mp = np.ascontiguousarray(mp, np.float64)
        self._ck(lib().rkFDBatchSetMassProp(self.h, _ptr(mp)))

    def batch_set_mass_prop_device(self, shard, mp_ptr):
        """rkFDBatchSetMassPropDevice: raw device address (e.g. torch CUDA tensor .data_ptr()) of float64 mp[Bs][n][10] of shard
        `shard`, indexed by the shard's local environment; stream-ordered on the engine's stream, values unchecked."""
        self._ck(lib().rkFDBatchSetMassPropDevice(self.h, shard, _ptr(mp_ptr)))

    def kernel_variant(self, shard=0):
        """rkFDBatchKernelVariant: (block, gscr, rigid, spec, minb) of the step-kernel variant shard `shard` launches."""
        v = (C.c_int * 5)()
        self._ck(lib().rkFDBatchKernelVariant(self.h, shard, v))
        return tuple(v)


def create_world(world: World, B=None, devices=None):
    """Replays the reference's set-up call sequence (rkFDCreate, contact info, rkFDChainReg per chain,
    rkFDPrpSet*, rkFDSetSolver) for a World description.  Returns (fd, cells)."""
    fd = RkFD()
    for ci in world.contact_info:
        fd.contact_info_add(ci)
    cells = [fd.chain_reg(ch) for ch in world.chains]
    for chn, cell in zip(world.chains, cells):
        if not getattr(chn, "self_collide", False):        # as every example program of the reference does
            lib().rkCDPairChainUnreg(None, cell.chain_handle)
        # slide mode of collision cells (the reference's fake crawler): through the shapes of the REGISTERED chain
        L = lib()
        L.rkLinkShape.restype = C.c_void_p; L.rkLinkShape.argtypes = [C.c_void_p, C.c_int, C.c_int]
        for f in ("rkFDShape3DSetSlideMode", "rkFDShape3DSetSlideVel", "rkFDShape3DSetSlideAxis"):
            getattr(L, f).restype = C.c_void_p
        L.rkFDShape3DSetSlideMode.argtypes = [C.c_void_p, C.c_void_p, C.c_bool]
        L.rkFDShape3DSetSlideVel.argtypes = [C.c_void_p, C.c_void_p, C.c_double]
        L.rkFDShape3DSetSlideAxis.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_double)]
        for k, l in enumerate(chn.links):
            for ci_, (vel, axis) in getattr(l, "slides", {}).items():
                sh = L.rkLinkShape(cell.chain_handle, k, ci_)
                ax = (C.c_double * 3)(*[float(a) for a in axis])
                ok = sh and L.rkFDShape3DSetSlideMode(fd.h, sh, True) and L.rkFDShape3DSetSlideVel(fd.h, sh, float(vel)) and L.rkFDShape3DSetSlideAxis(fd.h, sh, ax)
                if not ok:
                    raise RuntimeError("rokifd_b200: slide mode: shape %d of link %d not found" % (ci_, k))
    fd.prp_set(world.dt, world.pyramid, world.friction_weight, world.max_iter)
    fd.set_solver(world.solver)
    fd.set_integrator(getattr(world, "integrator", "RKG"))
    if B is not None:
        fd.batch_set_env_num(B)
    if devices is not None:
        fd.batch_set_devices(devices)
    return fd, cells


def device_count():
    return lib().rkFDBatchDeviceCount()


def measure_fp64_tflops():
    """Measured fp64 FMA throughput of the current device (TFLOP/s)."""
    v = C.c_double(0.0)
    if lib().rkFDB200MeasureFp64(C.byref(v)) != 0:
        raise RuntimeError(lib().rkFDBatchLastError().decode())
    return v.value
