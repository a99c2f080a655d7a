"""DQN companion on the host side: load the reference's trained policy, pack
scene geometry, call the observe+act kernel.

Reference:
  weights     /root/reference/Model/ray/best_model.zip (SB3 1.6.2, policy.pth:
              q_net.q_net.{0,2,4}.{weight,bias}, net_arch [16,16], test_block_rl.py:52-56)
  observation SectorAndRayObservation (ext_obsv_sector_and_ray.py), 8 segments, memory
  action      model.predict(obsv, deterministic=True) -> argmax_a Q(s, a)  (main.py:148)
"""
from __future__ import annotations

import ctypes as C
import io
import zipfile
from typing import List, Sequence

import numpy as np

from . import _lib
from ._lib import TtdqnLayout, TtdqnMoving, TtdqnQnet


def default_layout(max_poly: int = 16, max_vert: int = 512) -> TtdqnLayout:
    lay = TtdqnLayout()
    _lib.load().ttdqn_default_layout(C.byref(lay))
    lay.max_poly, lay.max_vert = max_poly, max_vert
    return lay


class QNetWeights:
    """fp32 weights of the 3-layer Q-network, row-major [out][in]."""

    def __init__(self, w0, b0, w1, b1, w2, b2):
        self.arrays = [np.ascontiguousarray(a, dtype=np.float32) for a in (w0, b0, w1, b1, w2, b2)]
        w0, _, w1, _, w2, _ = self.arrays
        self.n_in, self.n_h1, self.n_h2, self.n_out = w0.shape[1], w0.shape[0], w1.shape[0], w2.shape[0]

    @classmethod
    def from_sb3_zip(cls, path: str) -> "QNetWeights":
        import torch
        with zipfile.ZipFile(path) as z:
            sd = torch.load(io.BytesIO(z.read("policy.pth")), map_location="cpu", weights_only=True)
        g = lambda k: sd[k].detach().cpu().numpy()
        return cls(g("q_net.q_net.0.weight"), g("q_net.q_net.0.bias"), g("q_net.q_net.2.weight"),
                   g("q_net.q_net.2.bias"), g("q_net.q_net.4.weight"), g("q_net.q_net.4.bias"))

    @classmethod
    def from_npz(cls, path: str) -> "QNetWeights":
        d = np.load(path)
        return cls(d["w0"], d["b0"], d["w1"], d["b1"], d["w2"], d["b2"])

    def save_npz(self, path: str) -> None:
        np.savez(path, **dict(zip(("w0", "b0", "w1", "b1", "w2", "b2"), self.arrays)))

    def host_struct(self) -> TtdqnQnet:
        a = self.arrays
        return TtdqnQnet(self.n_in, self.n_h1, self.n_h2, self.n_out,
                         *[x.ctypes.data for x in a])

    def device_struct(self, device="cuda"):
        import torch
        self._dev = [torch.from_numpy(a).to(device) for a in self.arrays]
        return TtdqnQnet(self.n_in, self.n_h1, self.n_h2, self.n_out,
                         *[t.data_ptr() for t in self._dev])


def pack_geometry(lay: TtdqnLayout, scenes: Sequence[Sequence[np.ndarray]],
                  solid: Sequence[Sequence[bool]]):
    """scenes[e] = list of rings ([nv,2] arrays); solid[e][i] marks filled polygons
    (obstacles) vs plain rings (the boundary LineString)."""
    n = len(scenes)
    xy = np.zeros((n, lay.max_vert, 2))
    off = np.zeros((n, lay.max_poly + 1), np.int32)
    sol = np.zeros((n, lay.max_poly), np.int32)
    cnt = np.zeros(n, np.int32)
    for e, rings in enumerate(scenes):
        if len(rings) > lay.max_poly:
            raise ValueError("too many rings for the layout")
        pos = 0
        for i, r in enumerate(rings):
            r = np.asarray(r, dtype=np.float64).reshape(-1, 2)
            if pos + len(r) > lay.max_vert:
                raise ValueError("too many vertices for the layout")
            xy[e, pos:pos + len(r)] = r
            off[e, i] = pos
            pos += len(r)
            off[e, i + 1] = pos
            sol[e, i] = int(bool(solid[e][i]))
        off[e, len(rings):] = pos
        cnt[e] = len(rings)
    return xy, off, sol, cnt


class DqnCompanion:
    """observe (sector + ray) -> Q-network -> argmax, batched over environments."""

    def __init__(self, lay: TtdqnLayout, weights: QNetWeights = None):
        self.lib = _lib.load()
        # the library's own layout checks (num_segments 3..16); with no environments nothing else runs
        rc = self.lib.ttdqn_observe_act_host(C.byref(lay), None, 0, *[None] * 12)
        if rc != 0:
            raise _lib.TtmpcError(f"DqnCompanion: bad layout (code {rc}): {self.lib.ttdqn_last_error().decode()}")
        self.lay = lay
        self.weights = weights
        self.ns = lay.num_segments
        self.n_ext = (4 if lay.use_memory else 2) * self.ns

    def observe_act(self, agent, xy, off, sol, cnt, internal=None, old_ext=None):
        n = len(agent)
        agent = np.ascontiguousarray(agent, np.float64)
        internal = None if internal is None else np.ascontiguousarray(internal, np.float32)
        if self.lay.use_memory and old_ext is None:
            old_ext = np.zeros((n, 2 * self.ns), np.float32)
        ext = np.zeros((n, self.n_ext), np.float32)
        seg = np.zeros((n, self.ns)); ray = np.zeros((n, self.ns))
        w = self.weights
        q = np.zeros((n, w.n_out if w else 1), np.float32)
        act = np.zeros(n, np.int32)
        qs = w.host_struct() if w else None
        P = lambda a: None if a is None else a.ctypes.data
        rc = self.lib.ttdqn_observe_act_host(
            C.byref(self.lay), C.byref(qs) if qs else None, n, P(agent), P(xy), P(off), P(sol), P(cnt),
            P(internal), P(old_ext), P(ext), P(q), P(act), P(seg), P(ray))
        if rc != 0:
            raise _lib.TtmpcError(f"ttdqn_observe_act_host failed (code {rc})")
        return dict(ext=ext, q=q, action=act, seg=seg, ray=ray, old_ext=old_ext)

    def observe_act_device(self, agent, xy, off, sol, cnt, internal, old_ext, out: dict, qstruct,
                           stream=None, moving=None):
        """All arguments are CUDA torch tensors; out holds ext/q/action/seg/ray tensors.
        moving=(centre [n][k][2] float64, shape_xy [n or 1][k][max_pv][2] float64, shape_nv [n or 1][k]
        int32): k moving solid rings per env, vertex offsets placed at the centres
        (ttdqn_observe_act_moving_device); None: the static rings alone."""
        import torch
        st = torch.cuda.current_stream().cuda_stream if stream is None else stream
        dp = lambda t: None if t is None else t.data_ptr()
        outs = (dp(out.get("ext")), dp(out.get("q")), dp(out.get("action")), dp(out.get("seg")), dp(out.get("ray")))
        qs = C.byref(qstruct) if qstruct else None
        if moving is None:
            rc = self.lib.ttdqn_observe_act_device(
                C.byref(self.lay), qs, agent.shape[0], dp(agent), dp(xy), dp(off), dp(sol), dp(cnt),
                dp(internal), dp(old_ext), *outs, C.c_void_p(st))
        else:
            mv = moving_struct(agent.shape[0], *moving)
            rc = self.lib.ttdqn_observe_act_moving_device(
                C.byref(self.lay), qs, agent.shape[0], dp(agent), dp(xy), dp(off), dp(sol), dp(cnt), C.byref(mv),
                dp(internal), dp(old_ext), *outs, C.c_void_p(st))
        if rc != 0:
            raise _lib.TtmpcError(f"ttdqn_observe_act_device failed (code {rc}): {self.lib.ttdqn_last_error().decode()}")
        return out


def rect_shape(radius: float) -> np.ndarray:
    """circle_to_rect of a moving obstacle as offsets from its centre, [4][2], in the vertex order the
    HintSwitcher's squares have (main.py:91-95): centre + rect_shape(r) is that square, bit for bit."""
    r = float(radius)
    return np.array([(-r, -r), (r, -r), (r, r), (-r, r)], dtype=np.float64)


def moving_struct(n: int, centre, shape_xy, shape_nv) -> TtdqnMoving:
    """ttdqn_moving of CUDA tensors centre [n][k][2] float64, shape_xy [n or 1][k][max_pv][2] float64
    and shape_nv [n or 1][k] int32 (shape_xy / shape_nv with one row: one template block for every
    env).  The tensors must outlive the call that uses the struct."""
    import torch
    if centre.dim() != 3 or centre.shape[0] != n or centre.shape[2] != 2 or centre.dtype != torch.float64:
        raise ValueError(f"moving centre must be float64 [{n}][k][2], got {tuple(centre.shape)} {centre.dtype}")
    k = centre.shape[1]
    if (shape_xy.dim() != 4 or shape_xy.shape[0] not in (1, n) or shape_xy.shape[1] != k or shape_xy.shape[3] != 2
            or shape_xy.dtype != torch.float64 or not 3 <= shape_xy.shape[2] <= 32):
        raise ValueError(f"moving shape_xy must be float64 [{n} or 1][{k}][3..32][2], got "
                         f"{tuple(shape_xy.shape)} {shape_xy.dtype}")
    if tuple(shape_nv.shape) != tuple(shape_xy.shape[:2]) or shape_nv.dtype != torch.int32:
        raise ValueError(f"moving shape_nv must be int32 {tuple(shape_xy.shape[:2])}, got "
                         f"{tuple(shape_nv.shape)} {shape_nv.dtype}")
    if not all(a.is_cuda and a.is_contiguous() for a in (centre, shape_xy, shape_nv)):
        raise ValueError("moving tensors must be contiguous CUDA tensors")
    return TtdqnMoving(k, shape_xy.shape[2], 1 if shape_xy.shape[0] == 1 else 0, 0,
                       centre.data_ptr(), shape_xy.data_ptr(), shape_nv.data_ptr())


def pack_paths(paths, max_nodes: int = None):
    """Reference-path polylines -> (xy [n][max_nodes][2] float64, count [n] int32)."""
    n = len(paths)
    m = max_nodes or max(len(p) for p in paths)
    xy = np.zeros((n, m, 2), np.float64)
    cnt = np.zeros(n, np.int32)
    for i, p in enumerate(paths):
        a = np.asarray(p, np.float64).reshape(-1, 2)
        xy[i, :len(a)] = a
        cnt[i] = len(a)
    return xy, cnt


def internal_obs_device(agent5, path_xy, path_n, corner_samples: int = 3, sample_offset: float = 0.0,
                        max_distance: float = 10.0, out=None, progress=None, stream=None):
    """``internal`` observation of the ray model (rays_reward1.py:27-31) for n environments.
    agent5 [n][5] (x y theta v w), path_xy [n][m][2], path_n [n]: CUDA torch tensors.
    Returns (internal [n][5 + 3*corner_samples] float32, path_progress [n] float64)."""
    import torch
    n = agent5.shape[0]
    if out is None:
        out = torch.empty(n, 5 + 3 * corner_samples, dtype=torch.float32, device=agent5.device)
    if progress is None:
        progress = torch.empty(n, dtype=torch.float64, device=agent5.device)
    st = torch.cuda.current_stream().cuda_stream if stream is None else stream
    rc = _lib.load().ttdqn_internal_obs_device(n, path_xy.shape[1], corner_samples, float(sample_offset),
                                               float(max_distance), agent5.data_ptr(), path_xy.data_ptr(),
                                               path_n.data_ptr(), out.data_ptr(), progress.data_ptr(), C.c_void_p(st))
    if rc != 0:
        raise _lib.TtmpcError(f"ttdqn_internal_obs_device failed (code {rc})")
    return out, progress


def rl_ref_device(agent5, action, steps: int = 20, ts: float = 0.2, ref_speed: float = 1.0, out=None, stream=None):
    """The DQN hint trajectory of main.py:184-193: positions [n][steps][2] (float64)."""
    import torch
    n = agent5.shape[0]
    if out is None:
        out = torch.empty(n, steps, 2, dtype=torch.float64, device=agent5.device)
    st = torch.cuda.current_stream().cuda_stream if stream is None else stream
    rc = _lib.load().ttdqn_rl_ref_device(n, steps, float(ts), float(ref_speed), agent5.data_ptr(), action.data_ptr(),
                                         out.data_ptr(), C.c_void_p(st))
    if rc != 0:
        raise _lib.TtmpcError(f"ttdqn_rl_ref_device failed (code {rc})")
    return out
