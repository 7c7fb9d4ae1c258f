"""Batched, GPU-resident ``MComCore``.

Same constructor, config dictionary, plugin keys and attribute names as the reference
(mobile_env/core/base.py:28-296), but one object holds ``num_envs`` independent environments
as structure-of-arrays tensors on one B200 and ``step`` is a single fused CUDA launch through
the C ABI of ``libmbe.so`` (include/mbe.h).  There is no CPU fallback.

Two step semantics behind one kernel set (SURVEY.md section 0):

``mode="fork"``  the reference's real step: move -> nearest connectable BS -> ResourceFair split
                 -> utility (base.py:230-296).  ``step(epoch_number, curr_step)`` returns None
                 and results are read from attributes, like the reference.
``mode="gym"``   Gymnasium-shaped: ``step(actions) -> obs, reward, terminated, truncated, info``
                 with the central / multi-agent handlers (the fork dropped them; semantics are
                 this build's specification, see oracle/mbe_oracle.py).
"""
from __future__ import annotations

import ctypes as C
import math
import os
from dataclasses import dataclass, field
from typing import Dict, List, Optional

import numpy as np
import torch

from .. import _lib
from . import metrics as _metrics
from .arrival import NoDeparture
from .channels import Channel, OkumuraHata
from .entities import BaseStation, UserEquipment
from .logging import Monitor
from .movement import RandomWaypointMovement
from .schedules import ProportionalFair, RateFair, ResourceFair
from .util import deep_dict_merge
from .utilities import BoundedLogUtility

MAX_COORD = 32767


@dataclass
class LayoutMap:
    """What ``MComCore.layout_map`` computed, as device tensors (DESIGN.md section 10.2): ``stats`` int64
    ``[n, 6]`` = (points, covered, overlap, sum k, sum k^2, low) and ``area`` int32 ``[n, B]`` per requested
    env, and with ``maps`` the grids ``coverage`` uint8, ``serving`` int8 and ``qoe`` int8 ``[n, GY, GX]``,
    row j at y = j * stride, column i at x = i * stride."""

    stats: torch.Tensor
    area: torch.Tensor
    coverage: Optional[torch.Tensor]
    serving: Optional[torch.Tensor]
    qoe: Optional[torch.Tensor]

    def result(self, weights=(1.0, 0.1, 10.0)):
        """Per env dict of FP64 tensors: ``LayoutScorer.result()``'s keys over the map's QoE values
        k / 100 (``Score`` with ``weights``), plus ``Coverage`` and ``Overlap``, the shares of the points
        with at least one and at least two connectable BSs."""
        pts, cov, ovl, sk, sk2, low = self.stats.double().unbind(dim=1)
        mean = sk / (100 * pts)
        var = sk2 / (10000 * pts) - mean * mean
        p = low / pts
        w1, w2, w3 = weights
        return {"Average QoE": mean, "QoE Variance": var, "Low QoE Proportion": p,
                "Score": w1 * mean - w2 * var - w3 * p, "Coverage": cov / pts, "Overlap": ovl / pts}


@dataclass
class Plan:
    """Everything the C ABI needs, folded on the host (no GPU required to build it)."""

    num_envs: int
    num_ues: int
    num_bs: int
    mode: int
    handler: int
    bs_layout: int
    bs_random: tuple
    autoreset: bool
    reset_rng_episode: bool
    ep_time: int
    env_offset: int
    seed: int
    width: float
    height: float
    velocity: float
    move_d2max: int
    utility: tuple
    scheduler: int = 0
    shared_trajectory: bool = False
    num_trajectories: int = 1  # M: env of global id g follows shared trajectory g mod M
    classes: List[dict] = field(default_factory=list)  # link classes [bs class][ue class], ue class fastest
    bs_class: Optional[np.ndarray] = None
    bs_xy: Optional[np.ndarray] = None  # shared layout [B,2] int16
    num_bs_classes: int = 1
    ue_class: Optional[np.ndarray] = None  # [U] uint8, None = all UEs alike
    ue_classes: List[dict] = field(default_factory=list)  # per UE class: velocity, move_d2max

    @property
    def feature_size(self) -> int:
        if self.mode != _lib.MODE_GYM:
            return 0
        return (4 if self.handler == _lib.HANDLER_MA else 2) * self.num_bs + 1


class MComCore:
    NOOP_ACTION = 0
    metadata = {"render_modes": ["rgb_array", "human"]}

    # ------------------------------------------------------------------ configuration --
    @classmethod
    def default_config(cls) -> Dict:
        """Reference defaults (base.py:102-153) plus the batching keys of this build."""
        width, height, ep_time = 200, 200, 20
        return {
            "width": width,
            "height": height,
            "EP_MAX_TIME": ep_time,
            "seed": 2024,
            "reset_rng_episode": False,
            "arrival": NoDeparture,
            "channel": OkumuraHata,
            "scheduler": ResourceFair,
            "movement": RandomWaypointMovement,
            "utility": BoundedLogUtility,
            "bs": {"bw": 9e6, "freq": 2500, "tx": 40, "height": 50},
            "ue": {"velocity": 1.5, "snr_tr": 2e-8, "noise": 1e-9, "height": 1.6},
            "arrival_params": {"ep_time": ep_time, "reset_rng_episode": False},
            "channel_params": {},
            "scheduler_params": {},
            "movement_params": {"width": width, "height": height, "reset_rng_episode": True},
            "utility_params": {"lower": -20, "upper": 20, "coeffs": (10, 0, 10)},
            "metrics": {"scalar_metrics": {}, "ue_metrics": {}, "bs_metrics": {}},
            # ---- batching (new) ----
            "num_envs": 1,
            "env_offset": 0,  # global id of local env 0 when envs are sharded over GPUs
            "device": "cuda",
            "mode": "fork",  # "fork" | "gym"
            "handler": "central",  # "central" | "ma" (gym mode)
            "autoreset": False,
            "bs_random": None,  # (min, max): draw a BS layout per env and episode (custom.py:68-77)
            "max_bs": None,  # BS slots when bs_random is used
            "generic_kernel": False,  # True: never use the shape-specialised fused kernels
            # True: every env draws the same UE initial positions / waypoints (only BS layouts differ);
            # "follow_movement": True iff movement_params.reset_rng_episode -- the fork, where that flag
            # makes every epoch replay one UE trajectory (base.py:130-134) and env index = epoch number
            "shared_trajectory": False,
            # M > 1 (a power of two, with shared_trajectory): env g follows trajectory g mod M, so the M
            # env rows l*M .. l*M + M-1 score one BS layout over M UE trajectories (scoring.LayoutScorer)
            "num_trajectories": 1,
            # the fork's collect loop (collectData2.ipynb cell 4) as written: step() dumps the four JSON
            # files of base.py:298-349 and keeps the per-epoch lists for save_epoch_data().  MComCustom
            # (the class that loop drives) defaults to None = on when there is ONE env, like the
            # reference, and off for batches (use export.ReferenceDumpWriter / rollout there: same files
            # without a sync per step)
            "dumps": False,
            "dump_root": "..",  # the reference writes to ../collectData and ../collectData2
            # monitor.update(self) inside step() and info = monitor.info() (base.py:272): None = like the
            # reference when there is one env, off for batches (one clone per metric and step)
            "monitor_in_step": None,
        }

    @classmethod
    def seeding(cls, config: Dict) -> Dict:
        """Per-plugin seeds seed+1..seed+5 (base.py:155-170); movement gets seed+4."""
        for num, key in enumerate(
            ("arrival_params", "channel_params", "scheduler_params", "movement_params", "utility_params")
        ):
            config.setdefault(key, {})["seed"] = config["seed"] + num + 1
        return config

    # ------------------------------------------------------------------------- planning --
    @classmethod
    def build_plan(cls, stations: List[BaseStation], users: List[UserEquipment], config: Dict, plugins=None) -> Plan:
        """Maps plugin objects and entity parameters to the device description. Pure host code."""
        if plugins is None:
            plugins = cls._instantiate_plugins(config)
        arrival, channel, scheduler, movement, utility = plugins
        if not isinstance(arrival, NoDeparture):
            raise NotImplementedError(f"arrival {type(arrival).__name__}: only NoDeparture has a CUDA kernel")
        if not isinstance(scheduler, (ResourceFair, ProportionalFair, RateFair)):
            raise NotImplementedError(
                f"scheduler {type(scheduler).__name__}: only ResourceFair / ProportionalFair / RateFair have CUDA kernels")
        if not isinstance(utility, BoundedLogUtility):
            raise NotImplementedError(f"utility {type(utility).__name__}: only BoundedLogUtility has a CUDA kernel")
        if not isinstance(channel, Channel):
            raise TypeError("channel must derive from Channel")
        if not users:
            raise ValueError("at least one UE is required")
        # UE classes: UEs that share velocity / snr_threshold / noise / height (entities.py:32-57)
        users = sorted(users, key=lambda u: u.ue_id)
        ue_keys, ue_protos = [], []
        ue_class = np.zeros(len(users), dtype=np.uint8)
        for i, ue in enumerate(users):
            k = ue.radio_key()
            if k not in ue_keys:
                ue_keys.append(k)
                ue_protos.append(ue)
            ue_class[i] = ue_keys.index(k)
        if len(ue_keys) > _lib.MAX_UE_CLASSES:
            raise NotImplementedError(f"more than {_lib.MAX_UE_CLASSES} distinct UE parameter sets")
        ue0 = ue_protos[0]
        width, height = float(config["width"]), float(config["height"])
        if not (0 < width <= MAX_COORD and 0 < height <= MAX_COORD):
            raise ValueError("map does not fit int16 coordinates")
        mode = {"fork": _lib.MODE_FORK, "gym": _lib.MODE_GYM}[config["mode"]]
        handler = cls._handler_class(config).kernel_id
        bs_random = config.get("bs_random")
        max_d2 = int(width) ** 2 + int(height) ** 2 + 2
        if bs_random:
            nbs = int(config.get("max_bs") or bs_random[1])
            bs_protos = [BaseStation(0, (0, 0), **config["bs"])]
            bs_class, bs_xy, layout = None, None, _lib.BS_PER_ENV
            bs_random = (int(bs_random[0]), int(bs_random[1]))
        else:
            if not stations:
                raise ValueError("stations are required unless config['bs_random'] is set")
            stations = sorted(stations, key=lambda b: b.bs_id)
            nbs = len(stations)
            keys, bs_protos = [], []
            bs_class = np.zeros(nbs, dtype=np.uint8)
            for i, bs in enumerate(stations):
                k = bs.radio_key()
                if k not in keys:
                    keys.append(k)
                    bs_protos.append(bs)
                bs_class[i] = keys.index(k)
            bs_xy = np.array([[int(b.x), int(b.y)] for b in stations], dtype=np.int16)  # entities.py:24-26
            layout, bs_random = _lib.BS_SHARED, (0, 0)
        if len(bs_protos) * len(ue_protos) > _lib.MAX_CLASSES:
            raise NotImplementedError(
                f"{len(bs_protos)} BS parameter sets x {len(ue_protos)} UE parameter sets exceed {_lib.MAX_CLASSES} link classes")
        # one folded table set per (BS class, UE class) pair; UE classes that differ in velocity only
        # share the fold of their radio parameters
        folds = {}
        classes = []
        for bs in bs_protos:
            for ue in ue_protos:
                key = (bs.radio_key(), ue.radio_key()[1:])
                if key not in folds:
                    folds[key] = channel.fold(bs, ue, max_d2)
                classes.append(folds[key])
        ue_classes = [movement.device_params(ue.velocity) for ue in ue_protos]
        mv = ue_classes[0]
        w1, w2, w3 = utility.coeffs
        ep_time = int(min(config["EP_MAX_TIME"], arrival.ep_time))  # base.py:407-409 with NoDeparture
        shared = config.get("shared_trajectory", False)
        if shared == "follow_movement":
            shared = bool(movement.reset_rng_episode)
        num_envs, env_offset = int(config["num_envs"]), int(config.get("env_offset", 0))
        M = int(config.get("num_trajectories", 1))
        if M < 1:
            raise ValueError(f"num_trajectories={M} must be >= 1")
        if M > 1:  # the rules mbe_create enforces (include/mbe.h, mbe_config.num_trajectories)
            if not shared:
                raise ValueError(f"num_trajectories={M} needs shared_trajectory (M shared UE trajectories)")
            if M & (M - 1):
                raise ValueError(f"num_trajectories={M} must be a power of two")
            if M > num_envs or num_envs % M:
                raise ValueError(f"num_envs={num_envs} must be a multiple of num_trajectories={M}")
            if env_offset % M:
                raise ValueError(f"env_offset={env_offset} must be a multiple of num_trajectories={M}")
        return Plan(
            num_envs=num_envs, num_ues=len(users), num_bs=nbs, mode=mode, handler=handler,
            bs_layout=layout, bs_random=bs_random, autoreset=bool(config.get("autoreset")),
            reset_rng_episode=bool(movement.reset_rng_episode), ep_time=ep_time,
            env_offset=env_offset, seed=int(movement.seed),
            width=width, height=height, velocity=mv["velocity"], move_d2max=mv["move_d2max"],
            utility=(float(utility.lower), float(utility.upper), float(w1), float(w2), float(w3)),
            scheduler=int(scheduler.kernel_id), shared_trajectory=bool(shared), num_trajectories=M,
            classes=classes, bs_class=bs_class,
            bs_xy=bs_xy, num_bs_classes=len(bs_protos), ue_class=ue_class if len(ue_protos) > 1 else None,
            ue_classes=ue_classes,
        )

    @staticmethod
    def _handler_class(config):
        """config["handler"]: "central" | "ma" or a handler class (upstream passes the class)."""
        from ..handlers import HANDLERS

        h = config.get("handler") or "central"
        if isinstance(h, str):
            return HANDLERS[h]
        if getattr(h, "kernel_id", None) in (0, 1):
            return h
        raise NotImplementedError(f"handler {h!r} has no CUDA kernel (central / multi-agent only)")

    @staticmethod
    def _instantiate_plugins(config):
        return (
            config["arrival"](**config["arrival_params"]),
            config["channel"](**config["channel_params"]),
            config["scheduler"](**config["scheduler_params"]),
            config["movement"](**config["movement_params"]),
            config["utility"](**config["utility_params"]),
        )

    # ---------------------------------------------------------------------- construction --
    def __init__(self, stations: List[BaseStation], users: List[UserEquipment], config=None, render_mode=None):
        assert render_mode in self.metadata["render_modes"] + [None]
        self.render_mode = render_mode  # "rgb_array": render() returns env 0's map panel (render_frames)
        config = deep_dict_merge(self.default_config(), config or {})
        config = self.seeding(config)
        self.config = config
        self.width, self.height = config["width"], config["height"]
        self.seed = config["seed"]
        self.reset_rng_episode = config["reset_rng_episode"]
        self.EP_MAX_TIME = config["EP_MAX_TIME"]
        plugins = self._instantiate_plugins(config)
        (self.arrivalModel, self.channelModel, self.schedulerModel, self.movementModel, self.utilityModel) = plugins
        # upstream spellings
        self.arrival, self.channel, self.scheduler, self.movement, self.utility = plugins
        self.stationDict = {bs.bs_id: bs for bs in stations}
        self.userDict = {ue.ue_id: ue for ue in users}
        self.stations, self.users = self.stationDict, self.userDict
        self.NUM_USERS = len(self.userDict)
        self.closed = False

        self.plan = self.build_plan(list(stations), list(users), config, plugins)
        self.NUM_STATIONS = self.plan.num_bs
        self.num_envs = self.plan.num_envs
        self.mode = config["mode"]
        # Gymnasium-shaped surface (vector-env naming): spaces of ONE env; the batch adds axis 0
        self.handler = self._handler_class(config)
        if self.plan.mode == _lib.MODE_GYM:
            self.single_action_space = self.action_space = self.handler.action_space(self)
            self.single_observation_space = self.observation_space = self.handler.observation_space(self)

        config["metrics"]["scalar_metrics"].update(
            {
                "number connections": _metrics.number_connections,
                "number connected": _metrics.number_connected,
                "mean utility": _metrics.mean_utility,
                "mean datarate": _metrics.mean_datarate,
            }
        )
        self.monitor = Monitor(**config["metrics"])

        self._lib = _lib.load()  # raises if libmbe.so is not built: no CPU fallback
        if not torch.cuda.is_available():
            raise _lib.MbeError("MComCore needs a CUDA device (B200); there is no CPU fallback for step()")
        self.device = torch.device(config["device"])
        if self.device.type != "cuda":
            raise _lib.MbeError("config['device'] must be a CUDA device")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self._handle = C.c_void_p()
        self._keepalive = []
        self._create_handle()
        self._allocate()
        self._bind()
        self._needs_reset = True
        fork = self.plan.mode == _lib.MODE_FORK
        self.dumps = bool(config["dumps"]) if config["dumps"] is not None else (fork and self.num_envs == 1)
        if self.dumps and not fork:
            raise NotImplementedError("config['dumps']: the dump files are the fork's FORK-mode format")
        self.dump_root = config["dump_root"]
        self.monitor_in_step = (bool(config["monitor_in_step"]) if config["monitor_in_step"] is not None
                                else self.num_envs == 1)
        # the reference's per-epoch lists (base.py:99-100, 208-209; custom.py:60-62), env 0's view
        self.users_dataRateList = self.users_trajectoryList = self.userQoEList = None
        self._history = None

    def _create_handle(self):
        p = self.plan
        cfg = _lib.Config()
        cfg.abi_version = _lib.MBE_ABI_VERSION
        cfg.device = self.device.index
        cfg.num_envs, cfg.num_ues, cfg.num_bs = p.num_envs, p.num_ues, p.num_bs
        cfg.mode, cfg.handler, cfg.scheduler = p.mode, p.handler, p.scheduler
        cfg.bs_layout = p.bs_layout
        cfg.bs_random_min, cfg.bs_random_max = p.bs_random
        cfg.autoreset = int(p.autoreset)
        cfg.reset_rng_episode = int(p.reset_rng_episode)
        cfg.ep_time = p.ep_time
        cfg.move_d2max = p.move_d2max
        cfg.env_offset = p.env_offset
        cfg.seed = p.seed & 0xFFFFFFFFFFFFFFFF
        cfg.width, cfg.height, cfg.velocity = p.width, p.height, p.velocity
        cfg.util_lower, cfg.util_upper, cfg.util_w1, cfg.util_w2, cfg.util_w3 = p.utility
        cfg.num_classes = p.num_bs_classes
        cfg.flags = (_lib.FLAG_GENERIC_KERNEL if self.config.get("generic_kernel") else 0) | (
            _lib.FLAG_SHARED_TRAJECTORY if p.shared_trajectory else 0)
        cfg.num_trajectories = p.num_trajectories
        for i, c in enumerate(p.classes):
            lut = np.ascontiguousarray(c["rate_lut"], dtype=np.float64)
            self._keepalive.append(lut)
            cfg.classes[i].l0, cfg.classes[i].k, cfg.classes[i].l_zero = c["l0"], c["k"], c["l_zero"]
            cfg.classes[i].d2max = c["d2max"]
            cfg.classes[i].rate_lut = lut.ctypes.data_as(C.POINTER(C.c_double)) if len(lut) else None
            if c.get("log2snr_lut") is not None:
                ltab = np.ascontiguousarray(c["log2snr_lut"], dtype=np.float32)
                self._keepalive.append(ltab)
                cfg.classes[i].log2snr_lut = ltab.ctypes.data_as(C.POINTER(C.c_float))
                cfg.classes[i].log2snr_len = len(ltab)
        if p.ue_class is not None:
            self._keepalive.append(p.ue_class)
            cfg.num_ue_classes = len(p.ue_classes)
            cfg.ue_class = p.ue_class.ctypes.data_as(C.POINTER(C.c_uint8))
            for i, uc in enumerate(p.ue_classes):
                cfg.ue_classes[i].velocity, cfg.ue_classes[i].move_d2max = uc["velocity"], uc["move_d2max"]
        if p.bs_class is not None:
            self._keepalive.append(p.bs_class)
            cfg.bs_class = p.bs_class.ctypes.data_as(C.POINTER(C.c_uint8))
        _lib.check(self._lib.mbe_create(C.byref(cfg), C.byref(self._handle)))

    def _allocate(self):
        p, dev = self.plan, self.device
        E, U, B = p.num_envs, p.num_ues, p.num_bs
        z = lambda *s, dt: torch.zeros(*s, dtype=dt, device=dev)  # noqa: E731
        self.pos = z(E, U, 2, dt=torch.int16)
        self.wp = torch.full((E, U, 2), -1, dtype=torch.int16, device=dev)
        self.t = z(E, dt=torch.int32)
        self.episode = torch.full((E,), -1, dtype=torch.int32, device=dev)
        if p.bs_layout == _lib.BS_SHARED:
            self.bs_xy = torch.from_numpy(p.bs_xy).to(dev)
            self.nbs = None
        else:
            self.bs_xy = z(E, B, 2, dt=torch.int16)
            self.nbs = torch.full((E,), B, dtype=torch.int32, device=dev)
        self.rate = z(E, U, dt=torch.float64)
        self.utility_scaled = torch.full((E, U), -1.0, dtype=torch.float32, device=dev)
        self.done = z(E, dt=torch.uint8)
        self._terminated = z(E, dt=torch.bool)  # no natural termination, only truncation
        self.metrics = z(E, 4, dt=torch.float32)
        gym = p.mode == _lib.MODE_GYM
        mw = (B + 31) // 32  # connection bitmask words per UE
        self.conn = (z(E, U, dt=torch.int32) if mw == 1 else z(E, U, mw, dt=torch.int32)) if gym else None
        self.actions = z(E, U, dt=torch.int32) if gym else None
        self.obs = z(E, U, p.feature_size, dt=torch.float32) if gym else None
        self.reward = (z(E, U, dt=torch.float32) if p.handler == _lib.HANDLER_MA else z(E, dt=torch.float32)) if gym else None
        self.assoc = None if gym else torch.full((E, U), -1, dtype=torch.int32, device=dev)
        self.dbg_snr = None
        self.inj_wp = None
        self.wp_cnt = None

    def _bind(self):
        ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
        b = _lib.Buffers()
        b.pos, b.wp, b.t, b.episode, b.bs_xy, b.nbs = map(ptr, (self.pos, self.wp, self.t, self.episode, self.bs_xy, self.nbs))
        b.conn, b.assoc, b.actions = ptr(self.conn), ptr(self.assoc), ptr(self.actions)
        b.rate, b.utility, b.obs, b.reward = ptr(self.rate), ptr(self.utility_scaled), ptr(self.obs), ptr(self.reward)
        b.done, b.metrics, b.dbg_snr = ptr(self.done), ptr(self.metrics), ptr(self.dbg_snr)
        b.inj_wp, b.wp_cnt = ptr(self.inj_wp), ptr(self.wp_cnt)
        b.inj_k = 0 if self.inj_wp is None else self.inj_wp.shape[2]
        _lib.check(self._lib.mbe_bind(self._handle, C.byref(b)))

    # ------------------------------------------------------------------------ test hooks --
    def enable_debug_snr(self):
        """Allocates the optional [E,U,B] SNR output of the PRE phase."""
        p = self.plan
        self.dbg_snr = torch.zeros(p.num_envs, p.num_ues, p.num_bs, dtype=torch.float32, device=self.device)
        self._bind()
        return self.dbg_snr

    def inject_waypoints(self, waypoints):
        """Replays reference trajectories: ``waypoints`` int [E,U,K,2] are consumed in order per UE
        instead of Philox draws (movement.py:44-47)."""
        wp = torch.as_tensor(waypoints).to(device=self.device, dtype=torch.int16).contiguous()
        assert wp.dim() == 4 and wp.shape[:2] == self.pos.shape[:2] and wp.shape[3] == 2
        self.inj_wp = wp
        self.wp_cnt = torch.zeros(wp.shape[:2], dtype=torch.int32, device=self.device)
        self._bind()

    def set_positions(self, pos):
        self.pos.copy_(torch.as_tensor(pos).to(device=self.device, dtype=torch.int16))

    def set_station_positions(self, bs_xy, nbs=None):
        self.bs_xy.copy_(torch.as_tensor(bs_xy).to(device=self.device, dtype=torch.int16))
        if nbs is not None:
            self.nbs.copy_(torch.as_tensor(nbs).to(device=self.device, dtype=torch.int32))
        self._bind()  # a shared layout is folded into the kernel parameters at bind time

    # ----------------------------------------------------------------------------- run ----
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def reset(self, *, seed=None, options=None, env_mask=None):
        """MComCore.reset (base.py:172-209) for all envs, or those selected by ``env_mask``
        (uint8/bool tensor [E]).  GYM mode returns ``(obs, info)``."""
        if seed is not None:
            self.seed = seed  # like the reference: stored, plugins keep their seeds (base.py:178-180)
        for m in (self.arrivalModel, self.channelModel, self.schedulerModel, self.movementModel, self.utilityModel):
            m.reset()
        mask_ptr = None
        if env_mask is not None:
            env_mask = env_mask.to(device=self.device, dtype=torch.uint8).contiguous()
            mask_ptr = C.c_void_p(env_mask.data_ptr())
        _lib.check(self._lib.mbe_reset(self._handle, mask_ptr, self._stream()))
        self.monitor.reset()
        self._needs_reset = False
        if self.dumps:
            self._begin_epoch_history()
        if self.plan.mode == _lib.MODE_GYM:
            return self._obs_view(), {}
        return None

    def _obs_view(self):
        if self.plan.handler == _lib.HANDLER_CENTRAL:
            return self.obs.view(self.num_envs, -1)
        return self.obs

    def step(self, *args):
        """FORK: ``step(epoch_number, curr_step)`` -> None (base.py:230-296).
        GYM: ``step(actions)`` -> ``obs, reward, terminated, truncated, info``."""
        if self._needs_reset:
            raise RuntimeError("call reset() before step()")
        if self.plan.mode == _lib.MODE_FORK:
            _lib.check(self._lib.mbe_step(self._handle, self._stream()))
            if self.dumps:  # base.py:261-269: the four JSON files and the per-epoch lists
                epoch_number, curr_step = args if len(args) == 2 else (0, len(self._history["pos"]))
                self._record_step()
                self.save_layout_and_data_rates(epoch_number, curr_step)
            if self.monitor_in_step:
                self.monitor.update(self)  # base.py:272
            return None
        (actions,) = args
        if actions is not self.actions:
            self.actions.copy_(torch.as_tensor(actions).reshape(self.actions.shape), non_blocking=True)
        _lib.check(self._lib.mbe_step(self._handle, self._stream()))
        info = {"metrics": self.metrics}
        if self.monitor_in_step:
            self.monitor.update(self)
            info.update(self.monitor.info())
        # views only: no extra kernels on the step path (truncated aliases the done bytes)
        return self._obs_view(), self.reward, self._terminated, self.done.view(torch.bool), info

    # ---------------------------------------------- the fork's dump methods (env level) ----
    # Slow path by construction, like the reference: every step synchronises and copies the few
    # tensors a dump needs.  Env i of the batch plays epoch ``epoch_number + i``.  Batched collection
    # without the per-step sync: export.ReferenceDumpWriter (same files, byte for byte).
    def _util_params(self):
        up = self.config["utility_params"]
        return up["lower"], up["upper"], tuple(up["coeffs"])

    def _layouts(self):
        if self.nbs is None:
            bs = self.bs_xy.cpu().numpy()
            return [bs for _ in range(self.num_envs)]
        bs_all, nbs = self.bs_xy.cpu().numpy(), self.nbs.cpu().numpy()
        return [bs_all[i, : nbs[i]] for i in range(self.num_envs)]

    def _begin_epoch_history(self):
        ids = sorted(self.userDict)
        self.users_dataRateList = {u: [] for u in ids}
        self.users_trajectoryList = {u: [] for u in ids}
        self.userQoEList = {u: [] for u in ids}
        self._history = {"pos": [], "arrived": [], "assoc": [], "rate": [], "bs": None}

    def _record_step(self):
        from ..export import scaled_utility_fp64

        if self._history is None:
            self._begin_epoch_history()
        h = self._history
        if h["bs"] is None:
            h["bs"] = self._layouts()
        pos, wp = self.pos.cpu().numpy(), self.wp.cpu().numpy()
        assoc, rate = self.assoc.cpu().numpy(), self.rate.cpu().numpy()
        h["pos"].append(pos), h["arrived"].append(wp[:, :, 0] < 0), h["assoc"].append(assoc), h["rate"].append(rate)
        lower, upper, coeffs = self._util_params()
        for u in self.users_dataRateList:  # env 0 under the reference's attribute names (base.py:264-269)
            r = np.float64(rate[0][u]) if assoc[0][u] >= 0 else 0.0
            x, y = pos[0][u]
            self.users_dataRateList[u].append(round(r, 2))
            self.users_trajectoryList[u].append((int(x), int(y)) if wp[0][u][0] < 0 else (np.int64(x), np.int64(y)))
            self.userQoEList[u].append(round(scaled_utility_fp64(r, lower, upper, coeffs), 2))

    def _write_files(self, files):
        for rel, text in files.items():
            path = os.path.join(self.dump_root, rel)
            os.makedirs(os.path.dirname(path), exist_ok=True)
            with open(path, "w") as f:
                f.write(text)

    def save_layout_and_data_rates(self, epoch_number, curr_step):
        """base.py:298-349: stations_info / user_positions / data_rates / user_qoe JSON files of the
        current step under ``<dump_root>/collectData``, one set per env (epoch ``epoch_number + i``)."""
        from ..export import format_step_files

        if self.plan.mode != _lib.MODE_FORK:
            raise NotImplementedError("the dump files are the fork's FORK-mode format")
        if not self._history or not self._history["pos"]:
            self._record_step()
        h = self._history
        for i in range(self.num_envs):
            self._write_files(format_step_files(epoch_number + i, curr_step, h["bs"][i], h["pos"][-1][i],
                                                h["assoc"][-1][i], h["rate"][-1][i], self._util_params()))

    def save_base_station_positions(self, epoch_number):
        """custom.py:79-85: ``<dump_root>/collectData2/BaseStationPosition/stations_<epoch>.json``."""
        import json

        from ..export import EPOCH_DIRS

        for i, bs in enumerate(self._layouts()):
            positions = {b: (int(x), int(y)) for b, (x, y) in enumerate(bs)}
            self._write_files({os.path.join(*EPOCH_DIRS["stations"]).format(e=epoch_number + i): json.dumps(positions)})

    def save_epoch_data(self, epoch_number):
        """base.py:351-404: the per-epoch CSV files (data rates, trajectories, QoE) from the lists the
        dumping ``step`` kept since the last ``reset``."""
        from ..export import EPOCH_DIRS, format_epoch_files

        h = self._history
        if not h or not h["pos"]:
            print(f"warning: no user data rates in epoch {epoch_number}, nothing saved")  # cf. base.py:353-355
            return
        stations_key = os.path.join(*EPOCH_DIRS["stations"])
        for i in range(self.num_envs):
            files = format_epoch_files(epoch_number + i, h["bs"][i], [p[i] for p in h["pos"]],
                                       [a[i] for a in h["arrived"]], [a[i] for a in h["assoc"]],
                                       [r[i] for r in h["rate"]], self._util_params())
            files.pop(stations_key.format(e=epoch_number + i), None)  # written by save_base_station_positions
            self._write_files(files)

    def rollout(self, steps: int, qoe_acc=None, threshold: float = 0.0, record=()):
        """FORK mode: ``steps`` consecutive ``step`` calls (the fork's collect loop
        ``for s in range(20): env.step(e, s)``) through ``mbe_rollout`` -- one launch for the fork's
        own scenario.  ``qoe_acc``: f32 ``[E,4]`` tensor receiving the layout-score statistics
        (``scoring.LayoutScorer.acc``); ``record``: names out of ``("pos", "wp", "assoc", "rate",
        "utility")`` whose per-step series ``[T,E,U(,2)]`` are returned in a dict."""
        if self._needs_reset:
            raise RuntimeError("call reset() before rollout()")
        E, U, dev = self.num_envs, self.NUM_USERS, self.device
        shapes = {"pos": ((steps, E, U, 2), torch.int16), "wp": ((steps, E, U, 2), torch.int16),
                  "assoc": ((steps, E, U), torch.int32),
                  "rate": ((steps, E, U), torch.float64), "utility": ((steps, E, U), torch.float32)}
        series = {}
        out = _lib.RolloutOut()
        for name in record:
            shape, dt = shapes[name]
            series[name] = torch.empty(shape, dtype=dt, device=dev)
            setattr(out, name, series[name].data_ptr())
        acc = None if qoe_acc is None else C.c_void_p(qoe_acc.data_ptr())
        _lib.check(self._lib.mbe_rollout(self._handle, int(steps), acc, C.c_float(threshold),
                                         C.byref(out) if record else None, self._stream()))
        return series

    def step_window(self, first_env: int, num_envs: int, stream=None):
        """The fused step for envs ``[first_env, first_env + num_envs)`` only (``mbe_step_window``);
        actions are read from ``self.actions``, results land in the usual tensors.  ``stream``:
        a ``torch.cuda.Stream`` (default: the current one) -- windows on different streams overlap."""
        st = self._stream() if stream is None else C.c_void_p(stream.cuda_stream)
        _lib.check(self._lib.mbe_step_window(self._handle, int(first_env), int(num_envs), st))

    def stage(self, phase_mask: int):
        _lib.check(self._lib.mbe_stage(self._handle, int(phase_mask), self._stream()))

    def observe(self):
        _lib.check(self._lib.mbe_observe(self._handle, self._stream()))
        return self._obs_view()

    def channel_snr(self, want_elig=False):
        """Channel.calculateSNR for every UE x BS pair (channels.py:24-27) -> f32 [E,U,B]."""
        p = self.plan
        snr = torch.empty(p.num_envs, p.num_ues, p.num_bs, dtype=torch.float32, device=self.device)
        elig = torch.empty(p.num_envs, p.num_ues, dtype=torch.int32, device=self.device) if want_elig else None
        _lib.check(
            self._lib.mbe_channel(self._handle, C.c_void_p(snr.data_ptr()),
                                  None if elig is None else C.c_void_p(elig.data_ptr()), self._stream())
        )
        return (snr, elig) if want_elig else snr

    def step_host(self, actions_host, obs_host, reward_host, done_host):
        """Host-buffer step through ``mbe_step_host`` (pinned numpy/torch CPU tensors)."""
        ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())  # noqa: E731
        _lib.check(self._lib.mbe_step_host(self._handle, ptr(actions_host), ptr(obs_host), ptr(reward_host),
                                           ptr(done_host), self._stream()))

    def render(self):
        """Gymnasium ``render``: with ``render_mode="rgb_array"`` env 0's map panel as numpy uint8
        ``[H, W, 3]`` (slow path: synchronises and copies, like ``view``); ``None`` without a render mode.
        The reference's metric dashboard is not drawn (DESIGN.md section 9)."""
        if self.render_mode is None:
            return None
        if self.render_mode == "human":
            raise NotImplementedError('render_mode="human" needs a display backend, which this build does not have; '
                                      'use "rgb_array" and show the frames yourself')
        return self.render_frames([0])[0].cpu().numpy()

    def render_frames(self, envs=None, size=None, series=None):
        """Map-panel frames in one launch (``mbe_render``), as a device tensor uint8 ``[N, H, W, 3]`` of the
        current state of ``envs`` (index tensor or list, default all), or ``[T, N, H, W, 3]`` from ``series``,
        the dict of ``rollout(..., record=("pos", "assoc", "utility"))`` (FORK mode).  ``size`` = (height,
        width) pixels (default ``render.DEFAULT_SIZE``).  Series frames use the BS layouts bound now, so a
        series should stay within one episode (with ``autoreset`` the step that ends it draws new layouts)."""
        from .. import render as _render

        if envs is None:
            n, ids = self.num_envs, None
        else:
            ids = torch.as_tensor(envs).to(device=self.device, dtype=torch.int32).reshape(-1).contiguous()
            n = ids.numel()
            if n == 0:
                raise ValueError("render_frames: envs is empty")
            if bool(((ids < 0) | (ids >= self.num_envs)).any()):
                raise IndexError(f"render_frames: env ids must lie in 0..{self.num_envs - 1}")
        st = _render.style(size)
        steps, ro = 1, None
        if series is not None:
            ro = _lib.RolloutOut()
            for name in ("pos", "assoc", "utility"):
                if name in series:
                    setattr(ro, name, series[name].data_ptr())
            steps = int(next(iter(series.values())).shape[0]) if series else 0
        out = torch.empty((max(steps, 1), n, st.height, st.width, 3), dtype=torch.uint8, device=self.device)
        _lib.check(self._lib.mbe_render(self._handle, None if ids is None else C.c_void_p(ids.data_ptr()), int(n),
                                        None if ro is None else C.byref(ro), int(steps), C.byref(st),
                                        C.c_void_p(out.data_ptr()), self._stream()))
        return out if series is not None else out[0]

    def layout_map(self, envs=None, *, stride: int = 1, load: int = 1, ue_class: int = 0, threshold: float = 0.0,
                   maps: bool = True) -> LayoutMap:
        """Coverage, serving BS and QoE cent at every ``stride``-th integer map point of the BS layout of
        ``envs`` (index tensor or list, default all; an id outside 0..E-1 gives an empty map and zero
        statistics), and their map-wide statistics, in two launches (``mbe_layout_map``, DESIGN.md section
        10.2).  ``load``: UEs sharing the serving BS (1 = a UE alone); ``ue_class``: the map UE's class;
        ``threshold``: the low-QoE threshold of ``LayoutScorer``; ``maps=False``: statistics only."""
        if envs is None:
            n, ids = self.num_envs, None
        else:
            ids = torch.as_tensor(envs).to(device=self.device, dtype=torch.int32).reshape(-1).contiguous()
            n = ids.numel()
        gx = (math.ceil(self.plan.width) - 1) // max(int(stride), 1) + 1
        gy = (math.ceil(self.plan.height) - 1) // max(int(stride), 1) + 1
        dev = self.device
        out = LayoutMap(torch.empty(n, 6, dtype=torch.int64, device=dev),
                        torch.empty(n, self.plan.num_bs, dtype=torch.int32, device=dev),
                        *((torch.empty(n, gy, gx, dtype=dt, device=dev) if maps else None)
                          for dt in (torch.uint8, torch.int8, torch.int8)))
        ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())  # noqa: E731
        prm = _lib.MapParams(stride=int(stride), ue_class=int(ue_class), load=int(load), threshold=float(threshold))
        _lib.check(self._lib.mbe_layout_map(self._handle, ptr(ids), int(n), C.byref(prm), ptr(out.stats),
                                            ptr(out.area), ptr(out.coverage), ptr(out.serving), ptr(out.qoe),
                                            self._stream()))
        return out

    @property
    def launch_count(self) -> int:
        return int(self._lib.mbe_launch_count(self._handle))

    @property
    def step_kernel_name(self) -> str:
        """The kernel family ``step`` dispatches to for this shape (``mbe_step_kernel_name``)."""
        return self._lib.mbe_step_kernel_name(self._handle).decode()

    @property
    def time_is_up(self):
        """base.py:407-409, per env."""
        return self.done.view(torch.bool)

    @property
    def time(self):
        return self.t

    # ------------------------------------------------------------- reference-named views --
    def view(self, e: int = 0):
        """Host-side snapshot of env ``e`` with the reference's attribute names
        (stationDict, userDict, activeUsers, bs2ue_connections, bs2ue_dataRates,
        allUserDataRates, ue_utilities, time).  Slow path: synchronises and copies."""
        from .views import EnvView

        return EnvView(self, e)

    def bs_isolines(self, drate: float, env: int = 0) -> Dict:
        """Coverage outline of every base station (reference base.py:450-460, a rendering helper):
        ``{BaseStation: (xs, ys)}`` from ``Channel.isoline`` with the default UE parameters.  ``env``
        selects the layout when layouts are per env (``MComCustom``).  Host-side, off the step path."""
        ue_config = self.default_config()["ue"]
        per_env = self.plan.bs_layout == _lib.BS_PER_ENV
        stations = (self.view(env).stationDict if per_env else self.stationDict).values()
        return {bs: self.channelModel.isoline(bs, ue_config, (self.width, self.height), drate) for bs in stations}

    def state_dict(self):
        keys = ("pos", "wp", "t", "episode", "bs_xy", "nbs", "conn", "assoc", "rate", "utility_scaled", "done")
        return {k: getattr(self, k).clone() for k in keys if getattr(self, k) is not None}

    def load_state_dict(self, sd):
        for k, v in sd.items():
            getattr(self, k).copy_(v)
        if "bs_xy" in sd:
            self._bind()  # a shared layout is folded into the kernel parameters at bind time
        self._needs_reset = False
        if self.plan.mode == _lib.MODE_GYM:
            self.observe()  # obs is derived state: recompute it from the loaded positions / connections

    def close(self):
        if getattr(self, "_handle", None) and self._handle.value:
            self._lib.mbe_destroy(self._handle)
            self._handle = C.c_void_p()
        self.closed = True

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
