"""Drop-in replacement for `MPL/lib/models/multiview_mpl.py` of aghasemzadeh/OpenMPL — inference forward only.

Same factory (`get_multiview_mpl_net(cfg, is_train)`, multiview_mpl.py:649-654), same wrapper
(`MultiView_MPL_G(cfg)`, :528-585), same constructor keywords and defaults (`MultiView_MPL(...)`, :95-117), same
parameter / buffer names and shapes (so reference checkpoints load, `MPL/lib/utils/utils.py:148-153`), same
`forward(x, centers=None, rays=None)` list-of-views call convention (`MPL/lib/core/function_mpl.py:344-350`).
Behind that boundary nothing of the reference is left: the module owns the parameters and hands device pointers to
`libmpl_b200.so` (hand-written sm_100a CUDA, C ABI in `include/mpl_b200.h`).  PyTorch is used for device memory and
streams only.  There is no CPU or eager fallback: without the library or without a CUDA device the forward raises.

Selecting it from the reference's runner: `MODEL: multiview_mpl_b200` in the YAML (see INTEGRATION.md).
"""
from __future__ import annotations

import ctypes
import math
import os
import threading
from collections import OrderedDict

import torch
import torch.nn as nn

from .. import _lib
from ..spec import BUFFER_KINDS, CTOR_DEFAULTS, make_config, param_spec

# "fp32" is the bit-for-intent default (CUDA-core fp32, ~1e-6 of the output scale vs the reference); "tf32" is the
# fp32-grade TENSOR-CORE mode (split bf16 hi/lo operands, three tcgen05 MMAs per product; carries the north-star bound
# <= 1e-3 of scale / 0.1 mm); "bf16" is the throughput mode (tcgen05 bf16 projections + fused fp16-mma SPT).
DEFAULT_PRECISION = os.environ.get("MPL_B200_PRECISION", "fp32")


class _Node(nn.Module):
    """Anonymous container giving parameters the reference's dotted state_dict names."""


class _Handle:
    """Owns the `MplModel*` handles of a module, one per device (a handle is used by one thread at a time, and
    DataParallel runs one replica thread per GPU); shared by reference between replicas, never copied."""

    def __init__(self):
        self.ptrs = {}

    def __deepcopy__(self, memo):
        return _Handle()          # a deep-copied module lazily creates its own handles

    def __del__(self):
        try:
            for p in self.ptrs.values():
                _lib.lib().mpl_destroy(p)
        except Exception:
            pass


def _register(root: nn.Module, name: str, tensor: torch.Tensor, is_buffer: bool):
    parts = name.split(".")
    mod = root
    for p in parts[:-1]:
        if p not in mod._modules:
            mod.add_module(p, _Node())
        mod = mod._modules[p]
    if is_buffer:
        mod.register_buffer(parts[-1], tensor)
    else:
        mod.register_parameter(parts[-1], nn.Parameter(tensor, requires_grad=False))


def _default_init(shape, kind, fan_in):
    """PyTorch default initialisation of the layer kinds the reference builds (SURVEY.md §3.2-Q5)."""
    if kind in ("linear_w", "linear_b"):
        bound = 1.0 / math.sqrt(fan_in)
        return torch.empty(shape).uniform_(-bound, bound)
    if kind in ("norm_w", "bn_var"):
        return torch.ones(shape)
    if kind in ("norm_b", "pos", "bn_mean"):
        return torch.zeros(shape)
    if kind == "count":
        return torch.zeros(shape, dtype=torch.long)
    raise ValueError(kind)


def _invalidate_after_load(module, incompatible_keys):
    module.invalidate()


def pipeline_pieces(batch: int, chunk: int, first: int):
    """[b0, b1) pose ranges of the pipelined host staging: a short first piece (at most `first` poses, never more than a
    forward chunk), then whole chunks; every pose exactly once, in order."""
    first = min(chunk, max(1, first))
    bounds = [0] + list(range(first, batch, chunk)) + [batch]
    return [(b0, b1) for b0, b1 in zip(bounds[:-1], bounds[1:]) if b1 > b0]


class MultiView_MPL(nn.Module):
    """Same keyword arguments and defaults as the reference constructor (multiview_mpl.py:95-117)."""

    def __init__(self, num_joints=17, in_chans=2, embed_dim_ratio=32, depth=4,
                 num_heads=8, mlp_ratio=2., qkv_bias=True, qk_scale=None,
                 drop_rate=0., attn_drop_rate=0., drop_path_rate=0.2, norm_layer=None, num_views=5,
                 add_confidence_input=False,
                 mult_confidence_emb=False,
                 concat_confidence_emb=False,
                 confidence_input_as_third=False,
                 pose_3d_emb_learnable=False,
                 linear_weighted_mean=False,
                 pos_embedding_type="learnable",
                 add_3D_pos_encoding_in_Spatial=False,
                 input_rays_as_token=False,
                 add_3D_pos_encoding_to_rays=False,
                 confidence_as_attention_uncertainty_weight=False,
                 multiple_spatial_blocks=False,
                 no_transformer_spt=False,
                 no_transformer_fpt=False,
                 confidence_in_FPT=False,
                 deep_head=False,
                 head_kadkhod=False,
                 hidden_dim=1024,
                 FPT_blocks_view_keypoint_tokens=False, *, precision=None, ln_fusion=True, graph_batch=2048,
                 qkv_attn_fusion=True):
        super().__init__()
        kw = {k: v for k, v in locals().items() if k in CTOR_DEFAULTS}
        self.cfg = make_config(**kw)
        self.precision = precision or DEFAULT_PRECISION
        # implementation switch (MplDesc.ln_fusion): bf16 mode folds the FPT LayerNorms into the GEMMs unless
        # ln_fusion=False (checkpoints whose residual rows have |mean| >> std, see DESIGN.md section 5)
        self.ln_fusion = bool(ln_fusion)
        # batches of at most `graph_batch` poses (the reference runner's 256, valid_mpl.py:205-210) replay one captured CUDA
        # graph per batch size instead of ~130 kernel launches (mpl_set_graph_batch); 0 = always launch kernel by kernel
        self.graph_batch = int(graph_batch)
        # bf16 mode: QKV projection + cross-view attention as one kernel where the shape allows (MplDesc.qkv_attn_fusion)
        self.qkv_attn_fusion = bool(qkv_attn_fusion)
        # host inputs spanning more than one forward chunk are copied piece by piece on a side stream under the kernels of
        # the previous piece; the first piece (the only exposed copy) is this many poses
        self.pipeline_first_poses = int(os.environ.get("MPL_PIPE_FIRST", 4096))
        self.num_joints, self.num_views, self.embed_dim_ratio = num_joints, num_views, embed_dim_ratio
        self._spec = param_spec(self.cfg)
        for name, (shape, kind, fan_in) in self._spec.items():
            _register(self, name, _default_init(shape, kind, fan_in), kind in BUFFER_KINDS)
        self._names = list(self._spec.keys())
        self._h = _Handle()          # MplModel* per device, created at the first forward (the reference also fails there, Q6)
        self._dev = {}               # device index -> dict(packed, stamp, workspace)
        self._lock = threading.Lock()
        self._origin = [self]        # survives DataParallel's shallow replica copies: the module that owns the parameters
        self._chunk = None
        self._epoch = [0]            # bumped by invalidate(); part of the packed-weights stamp (shared with replicas)
        self.last_launches = 0
        # a loaded checkpoint always repacks, whatever path the copy took (utils.py:148-153 of the reference)
        self.register_load_state_dict_post_hook(_invalidate_after_load)

    # ---- handle / packing ------------------------------------------------------------------------------------------
    def _get_handle(self, index=None):
        if index is None:
            index = torch.cuda.current_device() if torch.cuda.is_available() else -1
        if index not in self._h.ptrs:
            L = _lib.lib()
            desc = _lib.make_desc(self.cfg.kw, self.precision, self.ln_fusion, self.qkv_attn_fusion)
            h = ctypes.c_void_p()
            _lib.check(L.mpl_create(ctypes.byref(desc), ctypes.byref(h)))
            n = L.mpl_num_params(h)
            name, numel, is_int = ctypes.c_char_p(), ctypes.c_int64(), ctypes.c_int32()
            lib_names = []
            for i in range(n):
                _lib.check(L.mpl_param_info(h, i, ctypes.byref(name), ctypes.byref(numel), ctypes.byref(is_int)))
                lib_names.append(name.value.decode())
                if numel.value != self._tensor(lib_names[-1]).numel():
                    raise RuntimeError(f"parameter table mismatch for {lib_names[-1]}")
            if lib_names != self._names:
                raise RuntimeError("parameter table of libmpl_b200.so differs from the module's state_dict")
            if self._chunk is not None:
                _lib.check(L.mpl_set_chunk_poses(h, int(self._chunk)))
            _lib.check(L.mpl_set_graph_batch(h, self.graph_batch))
            self._h.ptrs[index] = h
        return self._h.ptrs[index]

    def _tensor(self, name):
        mod = self
        parts = name.split(".")
        for p in parts[:-1]:
            mod = mod._modules[p]
        # getattr, not _parameters: in a DataParallel replica the parameters are plain tensor attributes
        return getattr(mod, parts[-1])

    def _stamp(self):
        """Cheap fingerprint of the ORIGINAL module's parameters (DataParallel re-broadcasts fresh copies to the replicas on
        every call, which must not trigger a repack while the master's weights are unchanged): the invalidate() epoch, every
        tensor's in-place version counter, and the storage addresses of a few sentinel tensors (a `.to()` / `.cuda()` moves
        them all).  ~0.1 ms for the 800 tensors of `hm_0` -- it runs on every forward, including the 256-pose ones."""
        origin = self._origin[0]
        slots = origin.__dict__.get("_slots")
        if slots is None:                                   # (container dict, key) of every tensor, resolved once
            slots = []
            for name in origin._names:
                mod = origin
                parts = name.split(".")
                for p in parts[:-1]:
                    mod = mod._modules[p]
                d = mod._parameters if parts[-1] in mod._parameters else mod._buffers
                slots.append((d, parts[-1]))
            origin.__dict__["_slots"] = slots
        ts = [d[k] for d, k in slots]
        n = len(ts)
        return (origin._epoch[0], tuple([t._version for t in ts]),
                tuple(ts[i].data_ptr() for i in (0, n // 3, (2 * n) // 3, n - 1)), tuple(ts[i].device for i in (0, n - 1)))

    def _state(self, device):
        """Per-device packed weights, repacked whenever the fingerprint of the parameters changes (see invalidate())."""
        L = _lib.lib()
        h = self._get_handle(device.index)
        stamp = self._stamp()
        with self._lock:
            st = self._dev.get(device.index)
            if st is None or st["stamp"] != stamp:
                tensors = [self._tensor(n) for n in self._names]
                srcs = [t if (t.device == device and t.dtype in (torch.float32, torch.long) and t.is_contiguous())
                        else t.to(device=device, dtype=torch.long if t.dtype == torch.long else torch.float32).contiguous()
                        for t in tensors]
                ptrs = (ctypes.c_void_p * len(srcs))(*[s.data_ptr() for s in srcs])
                nbytes = L.mpl_packed_bytes(h)
                packed = st["packed"] if st is not None else torch.empty(nbytes, dtype=torch.uint8, device=device)
                stream = torch.cuda.current_stream(device).cuda_stream
                _lib.check(L.mpl_pack_weights(h, ptrs, len(srcs), packed.data_ptr(), nbytes, stream))
                for s in srcs:                      # temporaries must outlive the enqueued copies
                    s.record_stream(torch.cuda.current_stream(device))
                new = {"packed": packed, "stamp": stamp, "workspace": st["workspace"] if st else None}
                if st is not None:
                    for k in ("static", "copy_stream"):
                        if k in st:
                            new[k] = st[k]
                st = new
                self._dev[device.index] = st
            return st

    def invalidate(self):
        """Force a repack of the device-side weight blob at the next forward.

        The packed blob is refreshed automatically when a parameter is replaced or modified through autograd-visible
        in-place operations (`p.copy_()`, `load_state_dict`, optimizer steps: they bump `Tensor._version`).  Writes that
        go through `p.data` (`p.data.copy_()`, `dist.broadcast(p.data)`, EMA updates on `.data`, `p.data = other`) bump
        nothing PyTorch exposes, and neither does re-assigning a parameter object -- call `invalidate()` after those.
        `dist.broadcast_state`, `load_state_dict` and moving the module (`.to()`, `.cuda()`) are detected."""
        self._origin[0]._epoch[0] += 1
        return self

    def set_chunk_poses(self, chunk: int):
        self._chunk = int(chunk)
        for h in self._h.ptrs.values():
            _lib.check(_lib.lib().mpl_set_chunk_poses(h, int(chunk)))

    def chunk_poses(self) -> int:
        """Poses per forward chunk (the workspace stops growing there)."""
        return int(_lib.lib().mpl_chunk_poses(self._get_handle()))

    def set_profile(self, enabled, serial: bool = False):
        """Bracket every kernel launch of the next forwards with CUDA events (see `profile()`).  The pose chunks always run
        one after the other, so the per-category times add up to the step; `serial` is accepted for old callers and changes
        nothing."""
        _lib.check(_lib.lib().mpl_set_profile(self._get_handle(), 1 if enabled else 0))

    def profile(self) -> dict:
        """{category: (milliseconds, launches)} of the last forward run with profiling enabled."""
        L = _lib.lib()
        n = L.mpl_profile_categories()
        ms = (ctypes.c_double * n)()
        cnt = (ctypes.c_int64 * n)()
        _lib.check(L.mpl_profile_collect(self._get_handle(), ms, cnt, n))
        return {L.mpl_profile_category_name(i).decode(): (ms[i], cnt[i]) for i in range(n) if cnt[i]}

    # ---- nn.Module plumbing ------------------------------------------------------------------------------------------
    def train(self, mode: bool = True):
        # construction leaves the module in training mode like any nn.Module; only the forward refuses it
        return super().train(mode)

    def __deepcopy__(self, memo):
        import copy
        cls = self.__class__
        new = cls.__new__(cls)
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            if k == "_dev":
                new.__dict__[k] = {}
            elif k == "_origin":
                new.__dict__[k] = [new]
            elif k == "_epoch":
                new.__dict__[k] = [0]
            elif k == "_slots":
                continue
            elif k == "_lock":
                new.__dict__[k] = threading.Lock()
            else:
                new.__dict__[k] = copy.deepcopy(v, memo)
        return new

    # ---- forward (multiview_mpl.py:450-525) --------------------------------------------------------------------------
    def forward(self, poses, rays=None, centers=None):
        if self.training:
            raise RuntimeError("multiview_mpl_b200 is an inference-only forward: call model.eval() "
                               "(training/backward is out of scope and there is no eager fallback)")
        if self.cfg.error is not None:
            raise {"IndexError": IndexError}.get(self.cfg.error[0], RuntimeError)(self.cfg.error[1])
        if not torch.cuda.is_available():
            raise RuntimeError("multiview_mpl_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        V, J = self.cfg.V, self.cfg.J
        device = self._tensor(self._names[0]).device
        if device.type != "cuda":
            first = poses[0] if isinstance(poses, (list, tuple)) else poses
            device = first.device if first.device.type == "cuda" else torch.device("cuda", torch.cuda.current_device())
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())

        def prep(x, last_shape, what):
            if x is None:
                return None, 0
            if isinstance(x, (list, tuple)):
                if len(x) != V:
                    raise RuntimeError(f"{what}: expected a list of {V} views, got {len(x)}")
                ts = [t.to(device=device, dtype=torch.float32, non_blocking=True).contiguous() for t in x]
                for t in ts:
                    if tuple(t.shape[1:]) != last_shape or t.shape[0] != ts[0].shape[0]:
                        raise RuntimeError(f"{what}: every view must be [B, {last_shape[0]}, {last_shape[1]}], got {tuple(t.shape)}")
                return ts, last_shape[0] * last_shape[1]
            t = x.to(device=device, dtype=torch.float32, non_blocking=True).contiguous()
            if t.dim() != 4 or t.shape[1] != V or tuple(t.shape[2:]) != last_shape:
                raise RuntimeError(f"{what}: packed input must be [B, {V}, {last_shape[0]}, {last_shape[1]}], got {tuple(t.shape)}")
            n = last_shape[0] * last_shape[1]
            return [t[:, v] for v in range(V)], V * n

        # Small batches: persistent staging buffers + one CUDA-graph launch
        small = self._graph_plan(poses, rays, centers)
        if small is not None:
            return self._forward_graph(small, device)

        # Host inputs larger than one forward chunk: the host->device copy of chunk i+1 runs on a side stream while
        # chunk i computes (same result, the copy disappears behind the kernels).
        pipelined = self._pipeline_plan(poses, rays, centers, device)
        if pipelined is not None:
            return self._forward_pipelined(pipelined, device)

        p_list, p_stride = prep(poses, (J, 3), "poses")
        r_list, r_stride = prep(rays, (J, 3), "rays")
        c_list, c_stride = prep(centers, (1, 3), "centers")
        if r_list is not None and r_stride != p_stride:
            raise RuntimeError("poses and rays must use the same layout (both lists of views or both packed)")
        B = p_list[0].shape[0]
        L = _lib.lib()
        with torch.cuda.device(device):
            st = self._state(device)
            h = self._get_handle(device.index)
            out = torch.empty((B, J, 3), dtype=torch.float32, device=device)
            aux = [torch.empty_like(out), torch.empty_like(out)] if self.cfg.kw["head_kadkhod"] else [None, None]
            need = L.mpl_workspace_bytes(h, B)
            ws = st["workspace"]
            if ws is None or ws.numel() < need:
                st["workspace"] = ws = torch.empty(need, dtype=torch.uint8, device=device)
            arr = lambda ts: (ctypes.c_void_p * V)(*[t.data_ptr() for t in ts]) if ts is not None else None
            stream = torch.cuda.current_stream(device).cuda_stream
            _lib.check(L.mpl_forward(h, st["packed"].data_ptr(), arr(p_list), arr(r_list), arr(c_list), p_stride, c_stride,
                                     out.data_ptr(), aux[0].data_ptr() if aux[0] is not None else None,
                                     aux[1].data_ptr() if aux[1] is not None else None, B, ws.data_ptr(), ws.numel(), stream))
            self.last_launches = int(L.mpl_last_launch_count(h))
        if self.cfg.kw["head_kadkhod"]:
            return out, [aux[0], aux[1]]
        return out


    # ---- small batches: persistent buffers + CUDA graph replay -------------------------------------------------------
    def _graph_plan(self, poses, rays, centers):
        """(inputs per kind, packed?, B) when the call qualifies for the graph path: well-formed fp32 inputs of at most
        `graph_batch` poses (anything else takes the plain path, which validates and reports errors)."""
        if self.graph_batch <= 0:
            return None
        V, J = self.cfg.V, self.cfg.J
        plan, B, packed_all = {}, None, None
        for kind, x, last in (("poses", poses, (J, 3)), ("rays", rays, (J, 3)), ("centers", centers, (1, 3))):
            if x is None:
                plan[kind] = None
                continue
            packed = not isinstance(x, (list, tuple))
            ts = [x] if packed else list(x)
            want = ((V,) + last) if packed else last
            if not packed and len(ts) != V:
                return None
            for t in ts:
                if not (isinstance(t, torch.Tensor) and t.dtype == torch.float32 and t.dim() == len(want) + 1
                        and tuple(t.shape[1:]) == want):
                    return None
                if B is None:
                    B = t.shape[0]
                if t.shape[0] != B:
                    return None
            if packed_all is None:
                packed_all = packed
            if kind == "rays" and packed != packed_all:
                return None
            plan[kind] = (ts, packed)
        if plan["poses"] is None or B is None or B == 0 or B > self.graph_batch:
            return None
        return plan, B

    def _forward_graph(self, planned, device):
        plan, B = planned
        V, J = self.cfg.V, self.cfg.J
        L = _lib.lib()
        kad = self.cfg.kw["head_kadkhod"]
        with torch.cuda.device(device):
            st = self._state(device)
            h = self._get_handle(device.index)
            key = (B,) + tuple(None if v is None else v[1] for v in plan.values())
            bufs = st.setdefault("static", {}).get(key)
            if bufs is None:
                bufs = {k: ([torch.empty(t.shape, dtype=torch.float32, device=device) for t in v[0]] if v is not None else None)
                        for k, v in plan.items()}
                bufs["out"] = torch.empty((B, J, 3), dtype=torch.float32, device=device)
                bufs["aux"] = [torch.empty_like(bufs["out"]), torch.empty_like(bufs["out"])] if kad else [None, None]
                if len(st["static"]) >= 16:
                    st["static"].pop(next(iter(st["static"])))
                st["static"][key] = bufs
            for k, v in plan.items():
                if v is not None:
                    for d, t in zip(bufs[k], v[0]):
                        d.copy_(t, non_blocking=True)           # host or device source; same stream as the graph launch
            need = L.mpl_workspace_bytes(h, max(B, self.graph_batch))
            ws = st["workspace"]
            if ws is None or ws.numel() < need:
                st["workspace"] = ws = torch.empty(need, dtype=torch.uint8, device=device)

            def views(k, row):
                if bufs[k] is None:
                    return None, 0
                if plan[k][1]:
                    return [bufs[k][0][:, v] for v in range(V)], V * row
                return bufs[k], row

            p_list, p_stride = views("poses", J * 3)
            r_list, _ = views("rays", J * 3)
            c_list, c_stride = views("centers", 3)
            arr = lambda ts: (ctypes.c_void_p * V)(*[t.data_ptr() for t in ts]) if ts is not None else None
            out, aux = bufs["out"], bufs["aux"]
            stream = torch.cuda.current_stream(device).cuda_stream
            _lib.check(L.mpl_forward(h, st["packed"].data_ptr(), arr(p_list), arr(r_list), arr(c_list), p_stride, c_stride,
                                     out.data_ptr(), aux[0].data_ptr() if kad else None, aux[1].data_ptr() if kad else None,
                                     B, ws.data_ptr(), ws.numel(), stream))
            self.last_launches = int(L.mpl_last_launch_count(h))
            # the persistent output buffer is overwritten by the next call of this batch size: hand out a copy
            if kad:
                return out.clone(), [aux[0].clone(), aux[1].clone()]
            return out.clone()

    def graph_stats(self):
        """(captures, replays) of the CUDA-graph path on the current device."""
        c, r = ctypes.c_int64(), ctypes.c_int64()
        _lib.check(_lib.lib().mpl_graph_stats(self._get_handle(), ctypes.byref(c), ctypes.byref(r)))
        return c.value, r.value

    # ---- pipelined host -> device staging ---------------------------------------------------------------------------
    def _pipeline_plan(self, poses, rays, centers, device):
        """(host tensors per kind, strides, B) when every input lives on the host, has the exact expected layout and
        spans more than one forward chunk; None otherwise (the plain path validates and reports errors)."""
        V, J = self.cfg.V, self.cfg.J
        plan, B = {}, None
        for kind, x, last in (("poses", poses, (J, 3)), ("rays", rays, (J, 3)), ("centers", centers, (1, 3))):
            if x is None:
                plan[kind] = None
                continue
            ts = list(x) if isinstance(x, (list, tuple)) else [x]
            packed = not isinstance(x, (list, tuple))
            want = ((V,) + last) if packed else last
            for t in ts:
                if not (isinstance(t, torch.Tensor) and t.device.type == "cpu" and t.dtype == torch.float32 and t.is_contiguous()
                        and t.dim() == len(want) + 1 and tuple(t.shape[1:]) == want):
                    return None
                if B is None:
                    B = t.shape[0]
                if t.shape[0] != B:
                    return None
            if not packed and len(ts) != V:
                return None
            plan[kind] = (ts, packed)
        if plan["poses"] is None or B is None:
            return None
        if plan["rays"] is not None and plan["rays"][1] != plan["poses"][1]:
            return None
        chunk = int(_lib.lib().mpl_chunk_poses(self._get_handle(device.index)))
        if B <= chunk:
            return None
        return plan, B, chunk

    def _forward_pipelined(self, planned, device):
        plan, B, chunk = planned
        V, J = self.cfg.V, self.cfg.J
        L = _lib.lib()
        with torch.cuda.device(device):
            st = self._state(device)
            h = self._get_handle(device.index)
            main = torch.cuda.current_stream(device)
            side = st.get("copy_stream")
            if side is None:
                side = st["copy_stream"] = torch.cuda.Stream(device)
            dev = {k: ([torch.empty(t.shape, dtype=torch.float32, device=device) for t in v[0]] if v is not None else None)
                   for k, v in plan.items()}
            side.wait_stream(main)                       # the fresh buffers may still be in use on the main stream
            # the first piece is small: its copy is the only one the forward has to wait for, every later piece arrives under
            # the kernels of the one before it
            pieces = pipeline_pieces(B, chunk, self.pipeline_first_poses)
            events = []
            with torch.cuda.stream(side):
                for b0, b1 in pieces:
                    for k, v in plan.items():
                        if v is not None:
                            for d, t in zip(dev[k], v[0]):
                                d[b0:b1].copy_(t[b0:b1], non_blocking=True)
                    ev = torch.cuda.Event()
                    ev.record(side)
                    events.append(ev)
            out = torch.empty((B, J, 3), dtype=torch.float32, device=device)
            kad = self.cfg.kw["head_kadkhod"]
            aux = [torch.empty_like(out), torch.empty_like(out)] if kad else [None, None]
            need = L.mpl_workspace_bytes(h, B)
            ws = st["workspace"]
            if ws is None or ws.numel() < need:
                st["workspace"] = ws = torch.empty(need, dtype=torch.uint8, device=device)

            def views(k, row):                             # per-view device tensors and the pose stride of kind k
                if dev[k] is None:
                    return None, 0
                if plan[k][1]:
                    return [dev[k][0][:, v] for v in range(V)], V * row
                return dev[k], row

            p_list, p_stride = views("poses", J * 3)
            r_list, _ = views("rays", J * 3)
            c_list, c_stride = views("centers", 3)
            launches = 0
            for ev, (b0, b1) in zip(events, pieces):
                main.wait_event(ev)
                arr = lambda ts: (ctypes.c_void_p * V)(*[t[b0:].data_ptr() for t in ts]) if ts is not None else None
                _lib.check(L.mpl_forward(h, st["packed"].data_ptr(), arr(p_list), arr(r_list), arr(c_list), p_stride, c_stride,
                                         out[b0:].data_ptr(), aux[0][b0:].data_ptr() if kad else None,
                                         aux[1][b0:].data_ptr() if kad else None, b1 - b0, ws.data_ptr(), ws.numel(),
                                         main.cuda_stream))
                launches += int(L.mpl_last_launch_count(h))
            for ts in dev.values():
                for t in ts or []:
                    t.record_stream(side)
            self.last_launches = launches
        return (out, [aux[0], aux[1]]) if kad else out


class MultiView_MPL_G(nn.Module):
    """cfg -> MultiView_MPL, with the reference's `num_views` rule (multiview_mpl.py:534-580)."""

    def __init__(self, cfg, **kwargs):
        super().__init__()
        ds, net = cfg.DATASET, cfg.NETWORK
        if ds.TEST_DATASET.startswith('multiview_cmu_panoptic') or ds.TEST_DATASET.startswith('multiview_amass_cmu_panoptic_mpl'):
            num_views = 5
        else:
            num_views = 4
        if ds.TRAIN_VIEWS is not None:
            num_views = len(ds.TRAIN_VIEWS)
            if ds.USE_HELPER_CAMERAS:
                assert ds.TRAIN_VIEWS_HELPER is not None
                num_views += len(ds.TRAIN_VIEWS_HELPER)
        if ds.TRAIN_ON_ALL_CAMERAS and ds.TEST_ON_ALL_CAMERAS:
            num_views = ds.N_VIEWS_TRAIN_TEST_ALL
        self.init_weights_from = net.INIT_WEIGHTS_FROM
        self.features = MultiView_MPL(
            num_joints=net.NUM_JOINTS,
            embed_dim_ratio=net.DIM,
            depth=net.TRANSFORMER_DEPTH,
            num_heads=net.TRANSFORMER_HEADS,
            drop_rate=net.TRANSFORMER_DROP_RATE,
            attn_drop_rate=net.TRANSFORMER_ATTN_DROP_RATE,
            drop_path_rate=net.TRANSFORMER_DROP_PATH_RATE,
            num_views=num_views,
            add_confidence_input=net.TRANSFORMER_ADD_CONFIDENCE_INPUT,
            mult_confidence_emb=net.TRANSFORMER_MULT_CONFIDENCE_EMB,
            concat_confidence_emb=net.TRANSFORMER_CONCAT_CONFIDENCE_EMB,
            confidence_input_as_third=net.TRANSFORMER_CONFIDENCE_INPUT_AS_THIRD,
            pose_3d_emb_learnable=net.POSE_3D_EMB_LEARNABLE,
            linear_weighted_mean=net.TRANSFORMER_LINEAR_WEIGHTED_MEAN,
            add_3D_pos_encoding_in_Spatial=net.TRANSFORMER_ADD_3D_POS_ENCODING_IN_SPATIAL,
            input_rays_as_token=net.TRANSFORMER_INPUT_RAYS_AS_TOKEN,
            add_3D_pos_encoding_to_rays=net.TRANSFORMER_ADD_3D_POS_ENCODING_TO_RAYS,
            confidence_as_attention_uncertainty_weight=net.TRANSFORMER_CONF_ATTENTION_UNCERTAINTY_WEIGHT,
            multiple_spatial_blocks=net.TRANSFORMER_MULTIPLE_SPATIAL_BLOCKS,
            no_transformer_spt=net.TRANSFORMER_NO_SPT,
            no_transformer_fpt=net.TRANSFORMER_NO_FPT,
            confidence_in_FPT=net.TRANSFORMER_CONFIDENCE_IN_FPT,
            deep_head=net.TRANSFORMER_OUTPUT_HEAD_DEEP,
            head_kadkhod=net.TRANSFORMER_OUTPUT_HEAD_KADKHOD,
            hidden_dim=net.TRANSFORMER_OUTPUT_HEAD_HIDDEN_DIM,
            FPT_blocks_view_keypoint_tokens=net.TRANSFORMER_FPT_BLOCKS_VIEW_KEYPOINT_TOKENS,
            precision=kwargs.get("precision"),
            ln_fusion=kwargs.get("ln_fusion", True),
            graph_batch=kwargs.get("graph_batch", 2048),
            qkv_attn_fusion=kwargs.get("qkv_attn_fusion", True),
        )

    def forward(self, x, centers=None, rays=None):
        return self.features(x, rays=rays, centers=centers)

    def init_weights(self, pretrained=''):
        """Reference behaviour for the branches that work there (multiview_mpl.py:587-646): a checkpoint file is
        loaded non-strictly; the default 'scratch' mode leaves the PyTorch default initialisation untouched."""
        if os.path.isfile(pretrained):
            sd = torch.load(pretrained, map_location='cpu')
            if isinstance(sd, dict) and 'state_dict' in sd:
                sd = sd['state_dict']
            self.load_state_dict(sd, strict=False)


def get_multiview_mpl_net(cfg, is_train, **kwargs):
    model = MultiView_MPL_G(cfg, **kwargs)
    if is_train and cfg.NETWORK.INIT_WEIGHTS:
        model.init_weights(cfg.NETWORK.PRETRAINED)
    return model
