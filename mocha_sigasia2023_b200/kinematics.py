"""Torch-tensor level wrappers of the kinematics / inertialization kernels (C ABI rows a10-a18).

All inputs are CUDA tensors; outputs are new CUDA tensors. `quat.py` / `Inertialization.py` in this
package put the reference's NumPy signatures on top of these."""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib, skeleton


def _f32(t):
    _lib.require_cuda(t)
    if t.dtype != torch.float32:
        raise _lib.MochaError("expected float32 CUDA tensor")
    return t


def _f64(t):
    _lib.require_cuda(t)
    if t.dtype != torch.float64:
        raise _lib.MochaError("expected float64 CUDA tensor")
    return t


def parents_tensor(parents, device):
    return torch.as_tensor(list(parents), dtype=torch.int32, device=device)


def xy_to_quat(xy: torch.Tensor) -> torch.Tensor:
    """quat.from_xform_xy: [...,3,2] -> [...,4]."""
    xy = _f32(xy.contiguous())
    n = xy.numel() // 6
    out = torch.empty(xy.shape[:-2] + (4,), dtype=torch.float32, device=xy.device)
    _lib.check(_lib.load().mocha_xy_to_quat(_lib.ptr(xy), n, _lib.ptr(out), _lib.stream_ptr()), "mocha_xy_to_quat")
    return out


def quat_to_xy(q: torch.Tensor) -> torch.Tensor:
    """quat.to_xform_xy: [...,4] -> [...,3,2]."""
    q = _f32(q.contiguous())
    n = q.numel() // 4
    out = torch.empty(q.shape[:-1] + (3, 2), dtype=torch.float32, device=q.device)
    _lib.check(_lib.load().mocha_quat_to_xy(_lib.ptr(q), n, _lib.ptr(out), _lib.stream_ptr()), "mocha_quat_to_xy")
    return out


def _fp(ts):
    """All tensors float32 or all float64 (CUDA, contiguous); returns (tensors, suffix of the ABI entry)."""
    ts = [t.contiguous() for t in ts]
    for t in ts:
        _lib.require_cuda(t)
    dt = ts[0].dtype
    if dt not in (torch.float32, torch.float64) or any(t.dtype != dt for t in ts):
        raise _lib.MochaError("expected CUDA tensors of one floating type (float32 or float64)")
    return ts, ("_f64" if dt == torch.float64 else "")


def fk(lrot, lpos, parents):
    (lrot, lpos), sfx = _fp((lrot, lpos))
    J = lrot.shape[-2]
    F = lrot.numel() // (4 * J)
    grot, gpos = torch.empty_like(lrot), torch.empty_like(lpos)
    _lib.check(getattr(_lib.load(), "mocha_fk" + sfx)(_lib.ptr(lrot), _lib.ptr(lpos), _lib.ptr(parents), F, J,
                                                      _lib.ptr(grot), _lib.ptr(gpos), _lib.stream_ptr()), "mocha_fk")
    return grot, gpos


def fk_vel(lrot, lpos, lvel, lang, parents):
    (lrot, lpos, lvel, lang), sfx = _fp((lrot, lpos, lvel, lang))
    J = lrot.shape[-2]
    F = lrot.numel() // (4 * J)
    grot, gpos, gvel, gang = (torch.empty_like(t) for t in (lrot, lpos, lvel, lang))
    _lib.check(getattr(_lib.load(), "mocha_fk_vel" + sfx)(
        _lib.ptr(lrot), _lib.ptr(lpos), _lib.ptr(lvel), _lib.ptr(lang), _lib.ptr(parents), F, J, _lib.ptr(grot),
        _lib.ptr(gpos), _lib.ptr(gvel), _lib.ptr(gang), _lib.stream_ptr()), "mocha_fk_vel")
    return grot, gpos, gvel, gang


def ik(grot, gpos, parents):
    (grot, gpos), sfx = _fp((grot, gpos))
    J = grot.shape[-2]
    F = grot.numel() // (4 * J)
    lrot, lpos = torch.empty_like(grot), torch.empty_like(gpos)
    _lib.check(getattr(_lib.load(), "mocha_ik" + sfx)(_lib.ptr(grot), _lib.ptr(gpos), _lib.ptr(parents), F, J,
                                                      _lib.ptr(lrot), _lib.ptr(lpos), _lib.stream_ptr()), "mocha_ik")
    return lrot, lpos


QOPS = {"mul": 0, "inv_mul": 1, "mul_inv": 2, "mul_vec": 3, "inv_mul_vec": 4, "inv": 5, "abs": 6, "normalize4": 7,
        "normalize3": 8, "exp": 9, "log": 10, "between": 11, "from_angle_axis": 12, "to_xform": 13, "from_xform": 14,
        "to_euler_xyz": 15, "to_euler_yzx": 16, "cross": 17, "to_xform_xy": 18, "from_xform_xy": 19, "length3": 20,
        "length4": 21}
_QWIDTH = {0: (4, 4, 4), 1: (4, 4, 4), 2: (4, 4, 4), 3: (4, 3, 3), 4: (4, 3, 3), 5: (4, 0, 4), 6: (4, 0, 4), 7: (4, 0, 4),
           8: (3, 0, 3), 9: (3, 0, 4), 10: (4, 0, 3), 11: (3, 3, 4), 12: (1, 3, 4), 13: (4, 0, 9), 14: (9, 0, 4),
           15: (4, 0, 3), 16: (4, 0, 3), 17: (3, 3, 3), 18: (4, 0, 6), 19: (6, 0, 4), 20: (3, 0, 1), 21: (4, 0, 1)}


def quat_op(name: str, a: torch.Tensor, b: torch.Tensor | None = None, param: float = 0.0) -> torch.Tensor:
    """Element-wise quaternion algebra in the tensors' own precision (mocha_quat_op). a: [n, wa], b: [n, wb]
    dense CUDA tensors of one dtype (float32 / float64); returns [n, wo]."""
    op = QOPS[name]
    wa, wb, wo = _QWIDTH[op]
    ts, sfx = _fp((a,) if b is None else (a, b))
    a = ts[0]
    if a.dim() != 2 or a.shape[1] != wa or (wb and (ts[1].shape != (a.shape[0], wb))):
        raise _lib.MochaError(f"quat_op {name}: operand shapes {tuple(a.shape)} / "
                              f"{None if b is None else tuple(b.shape)} do not match widths {(wa, wb)}")
    n = a.shape[0]
    out = torch.empty((n, wo), dtype=a.dtype, device=a.device)
    if n:
        _lib.check(_lib.load().mocha_quat_op(op, int(sfx == "_f64"), _lib.ptr(a), None if b is None else _lib.ptr(ts[1]),
                                             n, float(param), _lib.ptr(out), _lib.stream_ptr()), "mocha_quat_op")
    return out


def fk_chain(lpos: torch.Tensor, lrot: torch.Tensor, start_pos=None, start_rot=None):
    """quat.fk_partial's chain walk: lpos [n,m,3], lrot [n,m,4]; bone c hangs off bone c-1, bone 0 off
    (start_pos [n,3], start_rot [n,4]) or is a root when they are None. Returns (gpos, grot)."""
    ts = (lpos, lrot) if start_pos is None else (lpos, lrot, start_pos, start_rot)
    ts, sfx = _fp(ts)
    n, m = ts[0].shape[0], ts[0].shape[1]
    gpos, grot = torch.empty_like(ts[0]), torch.empty_like(ts[1])
    _lib.check(_lib.load().mocha_fk_chain(int(sfx == "_f64"), None if start_pos is None else _lib.ptr(ts[2]),
                                          None if start_pos is None else _lib.ptr(ts[3]), _lib.ptr(ts[0]), _lib.ptr(ts[1]),
                                          n, m, _lib.ptr(gpos), _lib.ptr(grot), _lib.stream_ptr()), "mocha_fk_chain")
    return gpos, grot


def contact_update(state, lock, position, velocity, point, target, off_pos, off_vel, input_position, input_state,
                   unlock_radius, foot_height, halflife, dt):
    """In-place batched Inertialization.contact_update; state/lock/input_state int32 [n], vectors float64 [n,3]."""
    n = state.numel()
    for t in (position, velocity, point, target, off_pos, off_vel, input_position):
        _f64(t)
    _lib.check(_lib.load().mocha_contact_update(
        _lib.ptr(state), _lib.ptr(lock), _lib.ptr(position), _lib.ptr(velocity), _lib.ptr(point), _lib.ptr(target),
        _lib.ptr(off_pos), _lib.ptr(off_vel), _lib.ptr(input_position), _lib.ptr(input_state), n, unlock_radius,
        foot_height, halflife, dt, _lib.stream_ptr()), "mocha_contact_update")


def ik_two_bone(root, mid, end, target, fwd, root_gr, mid_gr, par_gr, max_length_buffer):
    ts = [_f64(t.contiguous()) for t in (root, mid, end, target, fwd, root_gr, mid_gr, par_gr)]
    n = ts[0].shape[0]
    a = torch.empty((n, 4), dtype=torch.float64, device=ts[0].device)
    b = torch.empty_like(a)
    _lib.check(_lib.load().mocha_ik_two_bone(
        _lib.ptr(ts[5]), _lib.ptr(ts[6]), *[_lib.ptr(t) for t in ts], max_length_buffer, n, _lib.ptr(a), _lib.ptr(b),
        _lib.stream_ptr()), "mocha_ik_two_bone")
    return a, b


def pose_transition(off, root, src, dst):
    """off/src/dst: 4-tuples (pos [n,J,3], vel, rot [n,J,4], ang) float64 (off updated in place);
    root: (pos [n,3], vel, rot [n,4], ang). Returns (tr_src_pos, tr_src_rot, tr_dst_pos, tr_dst_rot)."""
    n, J = off[0].shape[0], off[0].shape[1]
    dev = off[0].device
    tsp, tdp = torch.empty((n, 3), dtype=torch.float64, device=dev), torch.empty((n, 3), dtype=torch.float64, device=dev)
    tsr, tdr = torch.empty((n, 4), dtype=torch.float64, device=dev), torch.empty((n, 4), dtype=torch.float64, device=dev)
    args = [_lib.ptr(_f64(t)) for t in (*off, *root, *src, *dst)]
    _lib.check(_lib.load().mocha_pose_transition(*args, n, J, _lib.ptr(tsp), _lib.ptr(tsr), _lib.ptr(tdp),
                                                 _lib.ptr(tdr), _lib.stream_ptr()), "mocha_pose_transition")
    return tsp, tsr, tdp, tdr


def pose_update(off, inp, tr, halflife, dt):
    """Returns (pos, vel, rot, ang); off (4-tuple) is updated in place; tr = (src_pos, src_rot, dst_pos, dst_rot)."""
    n, J = off[0].shape[0], off[0].shape[1]
    out = tuple(torch.empty_like(t) for t in inp)
    args = [_lib.ptr(_f64(t)) for t in (*out, *off, *inp, *tr)]
    _lib.check(_lib.load().mocha_pose_update(*args, halflife, dt, n, J, _lib.stream_ptr()), "mocha_pose_update")
    return out


def make_post_params(parents=None, contact_bones=None, dt=1.0 / 60.0, ik_enabled=True, ik_max_length_buffer=0.015,
                     ik_foot_height=0.02, ik_unlock_radius=0.2, ik_blending_halflife=0.1) -> _lib.PostParams:
    parents = list(skeleton.BONE_PARENTS if parents is None else parents)
    contact_bones = list(skeleton.CONTACT_BONES if contact_bones is None else contact_bones)
    p = _lib.PostParams()
    p.J = len(parents)
    for i, v in enumerate(parents):
        p.parents[i] = int(v)
    p.contact_bones[0], p.contact_bones[1] = int(contact_bones[0]), int(contact_bones[1])
    p.dt = dt
    p.ik_max_length_buffer, p.ik_foot_height = ik_max_length_buffer, ik_foot_height
    p.ik_unlock_radius, p.ik_blending_halflife = ik_unlock_radius, ik_blending_halflife
    p.ik_enabled = int(ik_enabled)
    return p


class PostProcessor:
    """Device-resident per-clip post-process state + the fused per-frame kernel (mocha_post_frame)."""

    def __init__(self, B: int, device, params: _lib.PostParams | None = None):
        self.B = B
        self.params = params or make_post_params()
        self.state = torch.zeros(B * C.sizeof(_lib.ClipState), dtype=torch.uint8, device=device)
        self.out = torch.zeros(B * C.sizeof(_lib.FrameOut), dtype=torch.uint8, device=device)
        self.started = False

    def step(self, Y, src_hips_vel, src_rvel, src_rang, contacts):
        """Y [B,T,V,15] de-normalised; src_hips_vel [B,T,3]; src_rvel/src_rang [B,3]; contacts [B,2] uint8."""
        for t in (Y, src_hips_vel, src_rvel, src_rang):
            _f32(t)
        _lib.require_cuda(contacts)
        B, T, V, Cin = Y.shape
        init = 0 if self.started else 1
        _lib.check(_lib.load().mocha_post_frame(
            C.byref(self.params), _lib.ptr(Y), _lib.ptr(src_hips_vel), _lib.ptr(src_rvel), _lib.ptr(src_rang),
            _lib.ptr(contacts), B, T, V, Cin, init, _lib.ptr(self.state), _lib.ptr(self.out), _lib.stream_ptr()),
            "mocha_post_frame")
        self.started = True

    def step_packed(self, Y, side, contacts, lo: int = 0, init=None, start=None):
        """Same as step() with the source-motion inputs packed one row per clip:
        side [B', T*3+6] = [src_hips_vel | src_rvel | src_rang] (mocha_post_frame_packed). The B' clips are clips
        lo .. lo+B'-1 of this processor's state / output arrays (sub-batch lanes); init overrides `started`.
        start (uint8 [B'] CUDA tensor): clip b runs its frame 0 iff start[b] != 0, the others a steady-state step
        (mocha_post_frame_packed_masked); `init` and `started` are then ignored."""
        _f32(Y)
        _f32(side)
        _lib.require_cuda(contacts)
        B, T, V, Cin = Y.shape
        if side.dim() != 2 or side.shape[0] != B or side.shape[1] < T * 3 + 6 or side.stride(1) != 1:
            raise _lib.MochaError(f"side must be [B, >= T*3+6] with unit column stride, got {tuple(side.shape)}")
        if lo < 0 or lo + B > self.B:
            raise _lib.MochaError("step_packed: clip range outside this processor's state")
        state = C.c_void_p(self.state.data_ptr() + lo * C.sizeof(_lib.ClipState))
        out = C.c_void_p(self.out.data_ptr() + lo * C.sizeof(_lib.FrameOut))
        if start is not None:
            _lib.require_cuda(start)
            if start.dtype != torch.uint8 or start.shape != (B,):
                raise _lib.MochaError(f"start must be a uint8 [{B}] CUDA tensor, got {start.dtype} {tuple(start.shape)}")
            _lib.check(_lib.load().mocha_post_frame_packed_masked(
                C.byref(self.params), _lib.ptr(Y), _lib.ptr(side), side.stride(0), _lib.ptr(contacts), _lib.ptr(start),
                B, T, V, Cin, state, out, _lib.stream_ptr()), "mocha_post_frame_packed_masked")
            return
        init = (0 if self.started else 1) if init is None else int(bool(init))
        _lib.check(_lib.load().mocha_post_frame_packed(
            C.byref(self.params), _lib.ptr(Y), _lib.ptr(side), side.stride(0), _lib.ptr(contacts), B, T, V, Cin, init,
            state, out, _lib.stream_ptr()), "mocha_post_frame_packed")
        if lo == 0 and B == self.B:
            self.started = True

    def read(self):
        """Copy the frame outputs to the host as a dict of float64 numpy arrays [B, ...]."""
        import numpy as np
        raw = self.out.cpu().numpy()
        dt = np.dtype([("pos", "f8", (25, 3)), ("rot", "f8", (25, 4)), ("vel", "f8", (25, 3)), ("ang", "f8", (25, 3)),
                       ("blend_pos", "f8", (25, 3)), ("ik_pos", "f8", (25, 3)), ("ik_rot", "f8", (25, 4)),
                       ("src_root_pos", "f8", (3,)), ("src_root_rot", "f8", (4,)), ("src_root_vel", "f8", (3,)),
                       ("src_root_ang", "f8", (3,))])
        assert dt.itemsize == C.sizeof(_lib.FrameOut)
        rec = raw.view(dt)
        return {k: rec[k].copy() for k in dt.names}
