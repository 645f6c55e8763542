"""BatchedForestFire -- N independent forest-fire environments stepped by one CUDA launch.

Host-side mirror of the reference's ``ForestFire`` facade (Simulation/forest_fire.py:18-106):
same ``reset()`` / ``step(action)`` contract, same METADATA key names, same action set, reward and
done logic -- but every call acts on a whole batch and every array is a torch CUDA tensor.
PyTorch only provides device memory and the current stream; all arithmetic happens in
libwildfire_b200.so (hand-written sm_100a kernels) behind the C ABI of include/wildfire.h.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional

import numpy as np
import torch

from . import _lib
from .constants import ascii_of_type, make_metadata


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def config_from_metadata(m: dict) -> "_lib.WfConfig":
    """METADATA-style dict (constants.make_metadata) -> the C ABI's wf_config."""
    cfg = _lib.WfConfig()
    cfg.width, cfg.height = int(m["width"]), int(m["height"])
    cfg.n_actions, cfg.a_speed = int(m["n_actions"]), int(m["a_speed"])
    cfg.allow_dig_toggle = int(bool(m["allow_dig_toggle"]))
    cfg.make_rivers = int(bool(m["make_rivers"]))
    cfg.containment_wins = int(bool(m["containment_wins"]))
    if m["wind"] == "random":
        cfg.wind_random = 1
        cfg.wind_speed, cfg.wind_x, cfg.wind_y = 0.0, 0, 0
    else:
        cfg.wind_random = 0
        cfg.wind_speed = float(m["wind"][0])
        cfg.wind_x, cfg.wind_y = int(m["wind"][1][0]), int(m["wind"][1][1])
    cfg.fuel, cfg.radius = int(m["fuel"]), int(m["radius"])
    cfg.extra_ignitions = int(m["extra_ignitions"])
    cfg.auto_reset = int(bool(m["auto_reset"]))
    cfg.death_penalty = float(m["death_penalty"])
    cfg.contained_bonus = float(m["contained_bonus"])
    cfg.default_reward = float(m["default_reward"])
    cfg.heat, cfg.threshold = float(m["heat"]), float(m["threshold"])
    cfg.seed = int(m["seed"])
    cfg.env_id_base = int(m["env_id_base"])
    return cfg


_UNPACK_CODES = {torch.uint8: _lib.WF_OBS_U8, torch.float32: _lib.WF_OBS_F32, torch.bfloat16: _lib.WF_OBS_BF16}


def unpack_obs(bits: torch.Tensor, width: int, height: int, index=None, dtype: torch.dtype = torch.float32) -> torch.Tensor:
    """``"bits"`` observations -> ``[n, W, H, 3]`` of ``dtype`` (uint8, float32 or bfloat16) on the device, by
    ``wf_unpack_obs_bits`` on the current stream.

    ``bits``: ``[rows, words]`` int32 CUDA tensor (a ``[K, N, words]`` rollout: ``.view(-1, words)``).  ``index``: optional
    ``[n]`` row numbers (repeats and any order allowed; a row outside ``[0, rows)`` gives an all-zero observation), e.g. a
    minibatch drawn from a packed replay buffer; ``None`` = every row.  ``unpack_obs(...).flatten(1)`` feeds the reference's
    networks unchanged.
    """
    if dtype not in _UNPACK_CODES:
        raise ValueError("dtype must be torch.uint8, torch.float32 or torch.bfloat16")
    words = _lib.obs_bits_words(width, height)
    if not (isinstance(bits, torch.Tensor) and bits.is_cuda and bits.dtype == torch.int32 and bits.dim() == 2
            and bits.shape[1] == words):
        raise ValueError(f"bits must be an int32 CUDA tensor of shape [rows, {words}]")
    bits = bits.contiguous()
    idx = None
    if index is not None:
        idx = torch.as_tensor(index, device=bits.device).to(torch.int64).contiguous()
        if idx.dim() != 1:
            raise ValueError("index must be one-dimensional")
    n = bits.shape[0] if idx is None else idx.shape[0]
    with torch.cuda.device(bits.device):
        out = torch.empty((n, int(width), int(height), 3), dtype=dtype, device=bits.device)
        _lib.check(_lib.lib().wf_unpack_obs_bits(_ptr(bits), bits.shape[0], _ptr(idx), n, int(width), int(height), _ptr(out),
                                                 _UNPACK_CODES[dtype], C.c_void_p(torch.cuda.current_stream(bits.device).cuda_stream)))
    return out


def pack_obs(obs: torch.Tensor) -> torch.Tensor:
    """The inverse of ``unpack_obs``: ``[..., W, H, 3]`` 0/1 observations (any dtype, any device) -> ``[..., words]`` int32
    in the ``WF_OBS_BITS`` layout (include/wildfire.h: element k = (x*H + y)*3 + c is bit k % 32 of word k // 32, zero
    padding).  Plain torch, for packing stored uint8 memories once (e.g. demonstrations) into a packed replay buffer."""
    if obs.dim() < 3 or obs.shape[-1] != 3:
        raise ValueError("obs must have shape [..., W, H, 3]")
    lead, W, H = tuple(obs.shape[:-3]), int(obs.shape[-3]), int(obs.shape[-2])
    words = _lib.obs_bits_words(W, H)
    flat = (obs.reshape(*lead, W * H * 3) != 0).to(torch.int64)
    flat = torch.nn.functional.pad(flat, (0, words * 32 - W * H * 3)).reshape(*lead, words, 32)
    shifts = torch.arange(32, device=obs.device, dtype=torch.int64)
    packed = (flat << shifts).sum(-1)  # < 2**32: the uint32 pattern; as int32 with the same bits
    return torch.where(packed >= 2**31, packed - 2**32, packed).to(torch.int32)


class FinalStates:
    """The final states of the episodes that ended in one ``step`` / ``rollout`` call (``finals=True``), one entry per
    finished episode, sorted by ``(k, env)``: the state each env was in when it returned ``done`` at step ``k`` of the call,
    before the auto-reset replaced it (the ``final_observation`` of an auto-reset vector env).

    Written by the step kernels (``wf_set_final_capture``, include/wildfire.h) as one fixed-size record per episode.
    Tensors on the env's device: ``k``, ``env``, ``episode`` (the finished episode's number) and ``t`` (its length in
    steps) ``[F]`` int32; ``agent`` ``[F, 2]`` (final cell); ``alive``, ``visible``, ``dead``, ``digging`` ``[F]`` bool;
    ``next_start`` ``[F, 2]``, the next episode's start cell (-1, -1 without auto_reset); ``obs``, the terminal observation
    (``[F, words]`` bits rows for ``obs_dtype="bits"``, else ``[F, W, H, 3]`` of the env's dtype); ``records``, the raw
    ``[F, words]`` int32 records."""

    def __init__(self, records: torch.Tensor, width: int, height: int, obs_dtype=torch.uint8, n_envs: Optional[int] = None):
        W, H = int(width), int(height)
        self.width, self.height = W, H
        hdr = records[:, :_lib.FINAL_HEADER_WORDS]
        if records.shape[0] > 1:  # (k, env) order: the kernels' slot order is unspecified
            n = int(n_envs) if n_envs is not None else int(hdr[:, _lib.F_ENV].max()) + 1
            order = torch.argsort(hdr[:, _lib.F_K].long() * n + hdr[:, _lib.F_ENV].long())
            records, hdr = records[order], hdr[order]
        self.records = records
        self.k, self.env = hdr[:, _lib.F_K], hdr[:, _lib.F_ENV]
        self.episode, self.t = hdr[:, _lib.F_EPISODE], hdr[:, _lib.F_T]
        self.agent = hdr[:, _lib.F_AX:_lib.F_AY + 1]
        flags = hdr[:, _lib.F_FLAGS]
        self.alive = (flags & _lib.FINAL_ALIVE) != 0
        self.visible = (flags & _lib.FINAL_VISIBLE) != 0
        self.dead = (flags & _lib.FINAL_DEAD) != 0
        self.digging = (flags & _lib.FINAL_DIGGING) != 0
        self.next_start = hdr[:, _lib.F_NEXT_AX:_lib.F_NEXT_AY + 1]
        ow = _lib.obs_bits_words(W, H)
        bits = records[:, _lib.FINAL_OBS:_lib.FINAL_OBS + ow]
        if obs_dtype == "bits":
            self.obs = bits
        elif records.shape[0] == 0:
            self.obs = torch.empty((0, W, H, 3), dtype=obs_dtype, device=records.device)
        else:
            self.obs = unpack_obs(bits.contiguous(), W, H, dtype=obs_dtype)
        self._types = None
        self._host = None

    def __len__(self) -> int:
        return int(self.records.shape[0])

    def planes(self) -> torch.Tensor:
        """``[F, 4, W, H]`` bool: the fire, burnt, dirt and water planes of every record (grass is none of them)."""
        W, H = self.width, self.height
        pw, po = _lib.final_plane_words(W, H), _lib.final_plane_offset(W, H)
        words = self.records[:, po:po + 4 * pw].reshape(-1, 4, pw)
        shifts = torch.arange(32, device=words.device, dtype=torch.int32)
        bits = (words.unsqueeze(-1) >> shifts) & 1  # (an arithmetic shift of the sign bit is masked away)
        return bits.reshape(-1, 4, pw * 32)[:, :, :W * H].reshape(-1, 4, W, H).bool()

    def types(self) -> torch.Tensor:
        """``[F, W, H]`` uint8 cell types (``WF_GRASS`` 0, fire 1, burnt 2, dirt 3, water 4), computed on the device."""
        if self._types is None:
            p = self.planes().to(torch.uint8)
            code = torch.tensor([1, 2, 3, 4], dtype=torch.uint8, device=p.device).view(1, 4, 1, 1)
            self._types = (p * code).sum(1, dtype=torch.uint8)
        return self._types

    def render(self, i: int) -> str:
        """Record ``i`` as the string ``ForestFire.render(print_map=False)`` returns for that state (forest_fire.py:57-82):
        '+' grass, '@' fire, '#' burnt, '0' dirt, 'x' water, 'A' the agent while it is alive."""
        if self._host is None:  # one device-to-host copy for all the records
            self._host = (self.types().cpu().numpy(), self.agent.cpu().numpy(), self.alive.cpu().numpy())
        types, agent, alive = self._host
        t, (ax, ay), alive = types[i], (int(v) for v in agent[i]), bool(alive[i])
        rows = []
        for y in range(self.height):
            rows.append("".join("A" if alive and (x, y) == (ax, ay) else ascii_of_type[int(t[x, y])] for x in range(self.width)))
        return "\n" + "\n".join(rows) + "\n"


class BatchedForestFire:
    """``n_envs`` reference environments on one GPU.

    Parameters follow Simulation/constants.py:30-47 (``width``, ``height``, ``wind``, ``a_speed``,
    ``n_actions``, ``make_rivers``, ``allow_dig_toggle``, rewards) and Simulation/utility.py:94-102
    (``heat``, ``fuel``, ``threshold``), plus ``seed`` (key of the shared Philox stream),
    ``extra_ignitions``, ``auto_reset`` and ``env_id_base`` (global id of env 0 when a batch is
    sharded over several GPUs).

    Observations are ``[N, W, H, 3]`` (x is the slow axis, exactly ``World.get_state``'s layout,
    environment.py:399-402) so ``obs.flatten(1)`` feeds the reference's ``Flatten`` + ``Dense``
    networks unchanged (DQN.py:209-212).

    ``obs_dtype="bits"``: observations are packed one bit per element (``WF_OBS_BITS``, include/wildfire.h),
    ``[N, obs_bits_words(W, H)]`` ``torch.int32`` tensors holding the uint32 bit patterns, 8x smaller than uint8;
    ``unpack_obs`` turns rows of them back into ``[n, W, H, 3]`` on the device.
    """

    def __init__(self, n_envs: int, device=None, obs_dtype=torch.uint8, **metadata):
        if not torch.cuda.is_available():
            raise _lib.WildfireError("BatchedForestFire needs a CUDA device (no CPU fallback)")
        self.METADATA = make_metadata(**metadata)
        m = self.METADATA
        self.n_envs = int(n_envs)
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        self.device = dev
        self.width, self.height = int(m["width"]), int(m["height"])
        self.n_actions = int(m["n_actions"])
        codes = {torch.uint8: _lib.WF_OBS_U8, torch.float32: _lib.WF_OBS_F32, torch.bfloat16: _lib.WF_OBS_BF16, "bits": _lib.WF_OBS_BITS}
        if obs_dtype not in codes:
            raise ValueError('obs_dtype must be torch.uint8, torch.float32, torch.bfloat16 or "bits"')
        self.obs_dtype = obs_dtype
        self._obs_code = codes[obs_dtype]
        self.obs_bits = self._obs_code == _lib.WF_OBS_BITS

        L = _lib.lib()
        self._cfg = config_from_metadata(m)
        h = C.c_void_p()
        _lib.check(L.wf_create(C.byref(self._cfg), self.n_envs, self.device.index, C.byref(h)))
        self._h = h
        self.kernel_family = L.wf_kernel_family(h).decode()

        N, W, H = self.n_envs, self.width, self.height
        with torch.cuda.device(self.device):
            self._obs = torch.empty(self._obs_shape(N), dtype=self._obs_torch_dtype, device=self.device)
            self._reward = torch.empty((N,), dtype=torch.float64, device=self.device)
            self._done = torch.empty((N,), dtype=torch.uint8, device=self.device)
        self._done_bool = self._done.view(torch.bool)
        self._obs_ptr, self._reward_ptr, self._done_ptr = self._obs.data_ptr(), self._reward.data_ptr(), self._done.data_ptr()
        self._wf_step = L.wf_step
        nw = C.c_int32()
        coef = (C.c_double * (27 * 4))()
        speed = (C.c_double * 27)()
        vec = (C.c_int32 * 54)()
        _lib.check(L.wf_get_wind_table(h, coef, speed, vec, C.byref(nw)))
        self.wind_coef = np.array(coef[: nw.value * 4]).reshape(nw.value, 4)
        self.wind_speed_table = np.array(speed[: nw.value])
        self.wind_vector_table = np.array(vec[: nw.value * 2]).reshape(nw.value, 2)
        self._host = None

    # ------------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().wf_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    @property
    def obs_words(self) -> int:
        """int32 words per env of a ``"bits"`` observation (``obs_bits_words(width, height)``)."""
        return _lib.obs_bits_words(self.width, self.height)

    def _obs_shape(self, *lead):
        return (*lead, self.obs_words) if self.obs_bits else (*lead, self.width, self.height, 3)

    @property
    def _obs_torch_dtype(self):
        return torch.int32 if self.obs_bits else self.obs_dtype

    def _as_i32(self, t, shape):
        if not (isinstance(t, torch.Tensor) and t.dtype == torch.int32 and t.is_cuda and t.is_contiguous()):
            t = torch.as_tensor(t, device=self.device).to(torch.int32).contiguous()
        if tuple(t.shape) != tuple(shape):
            raise ValueError(f"expected shape {tuple(shape)}, got {tuple(t.shape)}")
        return t

    # ------------------------------------------------------------------------------------------
    def reset(self, mask=None, starts=None) -> torch.Tensor:
        """``ForestFire.reset()`` (forest_fire.py:52-54) for every env, or those with ``mask[n] != 0``.

        ``starts``: optional ``[N, 2]`` int agent start cells (negative x = draw from the stream).
        Returns the observation batch ``[N, W, H, 3]`` (``"bits"``: ``[N, words]``).
        """
        m = None
        if mask is not None:
            m = torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()
            if tuple(m.shape) != (self.n_envs,):
                raise ValueError("mask must have shape [n_envs]")
        s = None if starts is None else self._as_i32(starts, (self.n_envs, 2))
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().wf_reset(self._h, _ptr(m), _ptr(s), _ptr(self._obs), self._obs_code, self._stream()))
        return self._obs

    def step(self, actions, finals: bool = False, finals_capacity: Optional[int] = None):
        """``ForestFire.step(action)`` (forest_fire.py:30-49) for the whole batch.

        ``actions``: ``[N]`` ints, 0..3 = N,S,E,W; 4 = dig toggle iff ``allow_dig_toggle``; other = no-op.
        Returns ``(obs [N,W,H,3], reward float64 [N], done bool [N], {})``.  The returned tensors are
        the handle's persistent buffers (overwritten by the next call).
        ``finals=True``: the info dict holds ``"final"``, the ``FinalStates`` of the envs that returned done (as ``rollout``).
        """
        if finals:
            a = self._as_i32(actions, (self.n_envs,))
            with torch.cuda.device(self.device), self._capture(1, finals_capacity) as cap:
                _lib.check(self._wf_step(self._h, a.data_ptr(), self._obs_ptr, self._obs_code, self._reward_ptr, self._done_ptr,
                                         torch.cuda.current_stream(self.device).cuda_stream))
            return self._obs, self._reward, self._done_bool, {"final": cap.result}
        a = self._as_i32(actions, (self.n_envs,))
        rc = self._wf_step(self._h, a.data_ptr(), self._obs_ptr, self._obs_code, self._reward_ptr, self._done_ptr,
                           torch.cuda.current_stream(self.device).cuda_stream)
        if rc:
            _lib.check(rc)
        return self._obs, self._reward, self._done_bool, {}

    def rollout(self, k_steps: int, actions=None, obs: bool = True, out=None, policy: str = "stream",
                return_actions: bool = False, finals: bool = False, finals_capacity: Optional[int] = None):
        """``k_steps`` consecutive ``step`` calls in one launch (state stays on chip in between).

        ``actions``: ``[K, N]`` ints, or ``None`` = chosen on the device by ``policy``:
        ``"stream"`` (uniform random, ACTION stream), ``"walk"`` (the reference's heuristic
        demonstration / Baseline policy ``DQN.choose_randomwalk_action``, DQN.py:353-389) or ``"mlp"``
        (the Q-network given to ``set_policy_mlp``, eps-greedy, evaluated inside the step kernel of either family: on
        grids larger than 32x32 the tile kernel runs a policy pass after every step, with an exact fixed-point first layer).
        ``out``: optional ``(obs_or_None, reward, done_u8)`` buffers to write into.
        Returns ``(obs [K,N,W,H,3] or None, reward [K,N], done [K,N])`` (+ ``actions [K,N]`` if asked);
        with ``obs_dtype="bits"`` obs is ``[K, N, words]`` int32.
        ``finals=True``: a ``FinalStates`` of every episode that ended during the call is appended to the tuple.  The step
        kernels write one record per finished episode before the auto-reset; ``finals_capacity`` records fit (default
        ``N * K``, enough for every env ending at every step) and a call in which more episodes ended raises
        ``WildfireError``.  Without ``finals`` the same kernels as ever run.  Memory: the call allocates ``finals_capacity``
        records of ``final_record_words(W, H) * 4`` bytes (about W*H*2 bytes each: 256 B at 14x14, 57 KB at 256x256, so the
        default is 3.7 GB for 1024 envs of 256x256 and K = 64; pass a smaller ``finals_capacity`` where few episodes end),
        and reading the record count synchronises the stream.
        """
        if finals:
            with self._capture(k_steps, finals_capacity) as cap:
                res = self.rollout(k_steps, actions, obs, out, policy, return_actions)
            return (*res, cap.result)
        K, N = int(k_steps), self.n_envs
        a = None if actions is None else self._as_i32(actions, (K, N))
        pol = {"stream": _lib.WF_POLICY_STREAM, "walk": _lib.WF_POLICY_WALK, "mlp": _lib.WF_POLICY_MLP}[policy]
        with torch.cuda.device(self.device):
            if out is not None:
                o, r, d = out
                if self.obs_bits and o is not None and (tuple(o.shape) != self._obs_shape(K, N) or o.dtype != torch.int32
                                                        or not o.is_contiguous()):
                    raise ValueError(f"out obs must be a contiguous int32 tensor of shape {self._obs_shape(K, N)}")
            else:
                o = torch.empty(self._obs_shape(K, N), dtype=self._obs_torch_dtype, device=self.device) if obs else None
                r = torch.empty((K, N), dtype=torch.float64, device=self.device)
                d = torch.empty((K, N), dtype=torch.uint8, device=self.device)
            L = _lib.lib()
            if a is not None:
                _lib.check(L.wf_rollout(self._h, K, _ptr(a), _ptr(o), self._obs_code, _ptr(r), _ptr(d), self._stream()))
                chosen = a
            else:
                chosen = torch.empty((K, N), dtype=torch.int32, device=self.device) if return_actions else None
                _lib.check(L.wf_rollout_policy(self._h, K, pol, _ptr(chosen), _ptr(o), self._obs_code, _ptr(r), _ptr(d),
                                               self._stream()))
        if return_actions:
            return o, r, d.view(torch.bool), chosen
        return o, r, d.view(torch.bool)

    def _capture(self, k_steps: int, capacity: Optional[int]):
        """Context of one call with final-state capture on (``wf_set_final_capture``); ``.result`` afterwards."""
        env = self
        cap_n = env.n_envs * int(k_steps) if capacity is None else int(capacity)
        if cap_n < 0:
            raise ValueError("finals_capacity must be >= 0")

        class _Cap:
            def __enter__(self):
                words = _lib.final_record_words(env.width, env.height)
                with torch.cuda.device(env.device):
                    self.buf = torch.empty((max(cap_n, 1), words), dtype=torch.int32, device=env.device)
                    self.count = torch.zeros((1,), dtype=torch.int32, device=env.device)
                _lib.check(_lib.lib().wf_set_final_capture(env._h, _ptr(self.buf), cap_n, _ptr(self.count)))
                return self

            def __exit__(self, exc_type, exc, tb):
                _lib.check(_lib.lib().wf_set_final_capture(env._h, None, 0, None))
                if exc_type is not None:
                    return False
                n = int(self.count.item()) & 0xFFFFFFFF
                if n > cap_n:
                    raise _lib.WildfireError(f"{n} episodes ended in this call but finals_capacity is {cap_n}")
                self.result = FinalStates(self.buf[:n], env.width, env.height, env.obs_dtype, env.n_envs)
                return False

        return _Cap()

    def set_policy_mlp(self, kernel1, bias1, kernel2, bias2, eps: float = 0.0):
        """Weights of the in-kernel Q-network (``rollout(policy="mlp")``): Keras orientation, ``kernel1``
        ``[W*H*3, hidden]``, ``kernel2`` ``[hidden, n_actions]`` (DQN.make_network, DQN.py:209-233; for a
        dueling head pass the advantage stream).  ``eps``: exploration rate (DQN.choose_action :188-196).
        Both kernel families; on grids larger than 32x32 ``|kernel1|`` must stay below ``2**31 / (2*W*H + 1)``
        (the exact fixed-point sum, include/wildfire.h)."""
        arrs = [np.ascontiguousarray(torch.as_tensor(a).detach().cpu().numpy() if torch.is_tensor(a) else a, dtype=np.float32)
                for a in (kernel1, bias1, kernel2, bias2)]
        k1, b1, k2, b2 = arrs
        hidden = int(b1.shape[0])
        if k1.shape != (self.width * self.height * 3, hidden) or k2.shape != (hidden, self.n_actions) or b2.shape != (self.n_actions,):
            raise ValueError(f"weight shapes {[a.shape for a in arrs]} do not fit a {self.width}x{self.height}x3 -> {hidden} -> "
                             f"{self.n_actions} network")
        _lib.check(_lib.lib().wf_set_policy_mlp(self._h, k1.ctypes.data, b1.ctypes.data, k2.ctypes.data, b2.ctypes.data,
                                                hidden, float(eps)))

    def set_policy_mlp_dev(self, weight1, bias1, weight2, bias2, eps: float = 0.0):
        """``set_policy_mlp`` from float32 CUDA tensors in ``nn.Linear`` orientation (``weight1`` ``[hidden, W*H*3]``,
        ``weight2`` ``[n_actions, hidden]``), repacked by a kernel on the current stream: no host copy, no synchronisation
        (``wf_set_policy_mlp_dev``).  Rollouts queued after it on the same stream use the new weights, and they act
        exactly as after ``set_policy_mlp`` with the same weights.  For a dueling head pass the advantage stream.
        Both kernel families, as ``set_policy_mlp``."""
        ts = []
        for t in (weight1, bias1, weight2, bias2):
            if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float32 and t.device == self.device):
                raise ValueError(f"set_policy_mlp_dev takes float32 tensors on {self.device}")
            ts.append(t.detach().contiguous())
        w1, b1, w2, b2 = ts
        hidden = int(b1.shape[0]) if b1.dim() == 1 else -1
        if (b1.dim() != 1 or tuple(w1.shape) != (hidden, self.width * self.height * 3)
                or tuple(w2.shape) != (self.n_actions, hidden) or tuple(b2.shape) != (self.n_actions,)):
            raise ValueError(f"weight shapes {[tuple(t.shape) for t in ts]} do not fit a {self.width}x{self.height}x3 -> "
                             f"hidden -> {self.n_actions} network in nn.Linear orientation")
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().wf_set_policy_mlp_dev(self._h, _ptr(w1), _ptr(b1), _ptr(w2), _ptr(b2), hidden, float(eps),
                                                        self._stream()))

    def set_policy_mlp_flat_dev(self, params, hidden: int, dueling: bool, eps):
        """One in-kernel Q-network per group of envs (``wf_set_policy_mlp_nets_dev``): ``params`` is a float32 CUDA tensor
        ``[M, P]`` of M networks in the flat ``parameters_to_vector`` layout of ``wf_replay_fit`` (``mlp_param_count``;
        a dueling head acts with its advantage stream), ``eps`` M exploration rates.  Env n acts with network
        ``n // (n_envs // M)``; ``n_envs`` must be a multiple of M and ``n_envs // M`` a multiple of 8.  Repacked by a
        kernel on the current stream like ``set_policy_mlp_dev``, and network j acts exactly as ``set_policy_mlp_dev``
        with the same weights and ``eps[j]`` would."""
        if not (isinstance(params, torch.Tensor) and params.is_cuda and params.dtype == torch.float32
                and params.device == self.device and params.dim() == 2):
            raise ValueError(f"set_policy_mlp_flat_dev takes a float32 [M, P] tensor on {self.device}")
        M = int(params.shape[0])
        eps = [float(e) for e in eps]
        if len(eps) != M:
            raise ValueError(f"eps has {len(eps)} entries for {M} networks")
        P = _lib.mlp_param_count(self.width, self.height, int(hidden), self.n_actions, bool(dueling))
        if params.shape[1] != P:
            raise ValueError(f"params has {params.shape[1]} floats per network, a {self.width}x{self.height}x3 -> {hidden} -> "
                             f"{self.n_actions} network{' with a dueling head' if dueling else ''} has {P}")
        params = params.detach().contiguous()
        shape = _lib.WfMlpShape(width=self.width, height=self.height, hidden=int(hidden), n_actions=self.n_actions,
                                dueling=int(bool(dueling)), batch=1)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().wf_set_policy_mlp_nets_dev(self._h, C.byref(shape), M, _ptr(params),
                                                             (C.c_double * M)(*eps), self._stream()))

    def step_host(self, actions):
        """Host-buffer step through ``wf_step_host``: H2D actions, step, D2H obs/reward/done, sync.

        Uses page-locked staging arrays owned by this object; returns numpy views of them (numpy has no
        bfloat16: with ``obs_dtype=torch.bfloat16`` the observation is the pinned torch tensor itself;
        ``"bits"``: a ``uint32`` ``[N, words]`` array).
        """
        if self._host is None:
            N = self.n_envs
            t = dict(actions=torch.empty((N,), dtype=torch.int32).pin_memory(),
                     obs=torch.empty(self._obs_shape(N), dtype=self._obs_torch_dtype).pin_memory(),
                     reward=torch.empty((N,), dtype=torch.float64).pin_memory(),
                     done=torch.empty((N,), dtype=torch.uint8).pin_memory())
            np_obs = (t["obs"] if self.obs_dtype == torch.bfloat16 else
                      t["obs"].numpy().view(np.uint32) if self.obs_bits else t["obs"].numpy())
            self._host = dict(tensors=t, np_actions=t["actions"].numpy(), np_obs=np_obs,
                              np_reward=t["reward"].numpy(), np_done=t["done"].numpy().view(np.bool_),
                              ptrs=tuple(t[k].data_ptr() for k in ("actions", "obs", "reward", "done")),
                              fn=_lib.lib().wf_step_host)
        hb = self._host
        hb["np_actions"][:] = actions
        pa, po, pr, pd = hb["ptrs"]
        rc = hb["fn"](self._h, pa, po, self._obs_code, pr, pd)
        if rc:
            _lib.check(rc)
        return hb["np_obs"], hb["np_reward"], hb["np_done"], {}

    def host_session(self, on: bool = True, persistent_obs: bool = False) -> bool:
        """Turn the step-server session of ``step_host`` on / off (``wf_host_session``, include/wildfire.h): the step
        kernel stays resident and is driven through mapped host memory -- no launch, copy call or synchronise per
        step.  Returns whether a session is on afterwards (False for grids larger than 32x32: not supported there).

        ``persistent_obs=True``: ``step_host`` returns the same observation array every call anyway (like a vectorised
        Gym environment with ``copy=False``); with this flag the caller promises not to WRITE to it between steps, and
        only the elements that changed cross PCIe and are patched in place (mode 2 of ``wf_host_session``)."""
        L = _lib.lib()
        rc = L.wf_host_session(self._h, (2 if persistent_obs else 1) if on else 0)
        if rc == _lib.WF_ERR_INVALID and on:
            return False
        _lib.check(rc)
        return bool(L.wf_host_session_active(self._h))

    @property
    def host_session_state(self) -> int:
        """0: no session, 1: session on with the kernel parked, 2: step-server kernel resident."""
        return int(_lib.lib().wf_host_session_active(self._h))

    def observe(self) -> torch.Tensor:
        """``World.get_state()`` (environment.py:399-402) without stepping."""
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().wf_get_obs(self._h, _ptr(self._obs), self._obs_code, self._stream()))
        return self._obs

    # ------------------------------------------------------------------------------------------
    def get_state(self) -> dict:
        """Canonical planes of every env (``env[x, y, layer]`` order) as torch tensors.

        ``temp`` is rebuilt from the exact per-direction hit counters (``hits``) with the env's heat
        quanta: temp = sum_d hits[d] * coef[wind_id][d] (environment.py:286-290); it is only
        meaningful on grass cells (SURVEY.md section 7).
        """
        N, W, H = self.n_envs, self.width, self.height
        dev = self.device
        out = {k: torch.empty((N, W, H), dtype=torch.uint8, device=dev)
               for k in ("type", "burning", "fm_inf", "fuel", "apos")}
        out["hits"] = torch.empty((N, W, H, 4), dtype=torch.uint8, device=dev)
        out["scalars"] = torch.empty((N, _lib.WF_NSCALARS), dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().wf_get_state(self._h, _ptr(out["type"]), _ptr(out["burning"]), _ptr(out["fm_inf"]),
                                               _ptr(out["fuel"]), _ptr(out["hits"]), _ptr(out["apos"]),
                                               _ptr(out["scalars"]), self._stream()))
        coef = torch.as_tensor(self.wind_coef, device=dev)[out["scalars"][:, _lib.S_WIND_ID].long()]  # [N, 4]
        out["temp"] = (out["hits"].double() * coef[:, None, None, :]).sum(-1)
        # METADATA['a_speed_iter'] (Q8): ONE counter per handle, part of a checkpoint; kept as an [N] tensor (the same
        # value for every env) so that code that slices every entry of the dict per env keeps working
        out["a_iter"] = torch.full((N,), self.a_speed_iter, dtype=torch.int32, device=dev)
        return out

    @property
    def a_speed_iter(self) -> int:
        """``METADATA['a_speed_iter']`` (forest_fire.py:40-43): steps left until the next fire tick, 1..a_speed."""
        v = C.c_int32()
        _lib.check(_lib.lib().wf_get_a_iter(self._h, C.byref(v)))
        return int(v.value)

    @a_speed_iter.setter
    def a_speed_iter(self, value: int):
        _lib.check(_lib.lib().wf_set_a_iter(self._h, int(value)))

    def set_state(self, type=None, burning=None, fm_inf=None, fuel=None, hits=None, scalars=None, a_iter=None, **_ignored):
        """Overwrite planes / scalars / the tick phase counter (parity injection, checkpoint restore).  ``None`` = keep.
        ``set_state(**get_state())`` restores a checkpoint (derived entries such as ``temp`` / ``apos`` are ignored)."""
        N, W, H = self.n_envs, self.width, self.height
        if a_iter is not None:
            self.a_speed_iter = int(a_iter.flatten()[0]) if torch.is_tensor(a_iter) else int(a_iter)

        def u8(t, shape):
            if t is None:
                return None
            t = torch.as_tensor(t, device=self.device).to(torch.uint8).contiguous()
            if tuple(t.shape) != shape:
                raise ValueError(f"expected shape {shape}, got {tuple(t.shape)}")
            return t

        t_, b_, f_, fu_ = (u8(v, (N, W, H)) for v in (type, burning, fm_inf, fuel))
        h_ = u8(hits, (N, W, H, 4))
        s_ = None if scalars is None else self._as_i32(scalars, (N, _lib.WF_NSCALARS))
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().wf_set_state(self._h, _ptr(t_), _ptr(b_), _ptr(f_), _ptr(fu_), _ptr(h_), _ptr(s_),
                                               self._stream()))

    def set_fire_to(self, cells):
        """``World.set_fire_to(cell)`` (environment.py:233-246); ``cells``: ``[N, 2]`` ints, x < 0 = skip."""
        c = self._as_i32(cells, (self.n_envs, 2))
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().wf_set_fire_to(self._h, _ptr(c), self._stream()))

    def stats(self) -> dict:
        buf = (C.c_int64 * 8)()
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().wf_stats(self._h, buf, self._stream()))
        keys = ("env_steps", "episodes", "deaths", "contained", "burnouts", "ticks")
        return {k: int(buf[i]) for i, k in enumerate(keys)}

    def reset_stats(self):
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().wf_stats_reset(self._h, self._stream()))

    @property
    def tile_geometry(self):
        """Tile family: ``(threads per CTA, CTAs per cluster)`` of this handle's launches; warp family: ``(0, 0)``."""
        t, c = C.c_int32(), C.c_int32()
        _lib.check(_lib.lib().wf_tile_geometry(self._h, C.byref(t), C.byref(c)))
        return int(t.value), int(c.value)

    @property
    def launch_count(self) -> int:
        return int(_lib.lib().wf_launch_count(self._h))

    @property
    def host_threads(self) -> int:
        """Host threads ``step_host`` uses to expand packed observations (0 if that path is not in use)."""
        return int(_lib.lib().wf_host_threads(self._h))

    @property
    def state_bytes_per_env(self) -> int:
        return int(_lib.lib().wf_state_bytes_per_env(self._h))

    @staticmethod
    def heat_coefficients(wind_speed: float, wind_vector, heat: float = 0.3):
        """Heat quantum per direction (N, S, E, W as seen from the burning cell), the reference's
        own expression: ``wind_speed * heat * (angle + distance) ** -1`` (environment.py:260-290)."""
        wx, wy = wind_vector
        out = []
        for cx, cy in ((0, -1), (0, 1), (1, 0), (-1, 0)):
            angle = abs(math.atan2(wx * cy - wy * cx, wx * cx + wy * cy))
            out.append(wind_speed * heat * (angle + 1) ** (-1))
        return out
