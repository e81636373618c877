"""Scenario description: everything the reference derives from its ``params`` dict at construction.

Mirrors (without copying) the host-side set-up of
  PredatorPrey.__init__                envs/ma_gym/envs/predator_prey/predator_prey.py:51-108
  Coverage.__init__ / obstacles        envs/ma_gym/envs/coverage/coverage.py:39-109, 482-500
  init_communication                   custom_implement/env_communication.py:10-77
  runner sizing rules                  exp_runners/env_uitils.py:171-217
and turns it into the plain numbers ``cm_env_desc`` (include/commarl_b200.h) carries.
"""
import copy
from dataclasses import dataclass, field, fields
from typing import Optional

import numpy as np

from . import _native as N


def _neg_abs(x):
    # the reference stores costs as -abs(param) (predator_prey.py:67-69, coverage.py:87-91); an integer
    # zero stays +0.0, a float zero becomes -0.0 — kept, it is the same IEEE arithmetic afterwards.
    return float(-abs(x))


def coverage_wall_grid(map_size: int, obst: str = "Easy") -> np.ndarray:
    """(map+2)x(map+2) uint8 wall map: the border plus the fixed obstacles scaled by r = map/10
    (coverage.py:69-80 layouts; :162-168 border; :493-500 placement clipped to the grid)."""
    if map_size % 10:
        raise ValueError("Coverage needs a map size that is a multiple of 10 (coverage.py:67)")
    r, G = map_size // 10, map_size + 2
    wall = np.zeros((G, G), dtype=np.uint8)
    wall[0, :] = wall[-1, :] = 1
    wall[:, 0] = wall[:, -1] = 1
    blocks = {"Easy": [(2 * r + 1, 2 * r + 1, 6 * r, r), (3 * r + 1, 8 * r + 1, 4 * r, 2 * r)]}
    blocks["Hard"] = blocks["Easy"] + [(1, 2 * r + 1, r, 3 * r), (1, 7 * r + 1, 2 * r, r),
                                       (4 * r + 1, 4 * r + 1, 2 * r, 3 * r), (8 * r + 1, 5 * r + 1, 2 * r, 2 * r),
                                       (8 * r + 1, 8 * r + 1, r, r)]
    if obst not in blocks:
        raise ValueError(f"obstComplex must be Easy or Hard, got {obst!r}")
    for top, left, h, w in blocks[obst]:
        wall[top:min(top + h, G), left:min(left + w, G)] = 1
    return wall


@dataclass
class ScenarioSpec:
    scenario: str                      # 'pp' | 'co'
    map_size: int
    n_agents: int
    n_preys: int
    sensing: int
    max_steps: int
    n_layers: int = 2
    load: int = 2
    max_path_length: int = 0
    capture_reward: float = 10.0
    step_cost: float = -0.1
    moving_cost: float = 0.0
    penalty: float = 0.0
    lazy_penalty: float = 0.0
    revisit_penalty: float = 0.0
    final_reward: float = 0.0
    obst: str = "Easy"
    rcom: int = 9                      # 0 after the 'Rcom + 1 >= map' collapse = fully connected
    channel: int = N.CH_FC
    p_loss: float = 0.0
    pgb: float = 0.0196
    pbg: float = 0.282
    ge_init: int = 1
    loss_apply: int = 1
    seed: int = 1
    wall: Optional[np.ndarray] = field(default=None, repr=False)

    # ---- derived --------------------------------------------------------------------------------
    @property
    def grid(self) -> int:
        return self.map_size if self.scenario == "pp" else self.map_size + 2

    @property
    def window(self) -> int:
        return 2 * self.sensing + 1

    @property
    def obs_dim(self) -> int:
        """per-agent observation length (predator_prey.py:95-98, coverage.py:111-117 with add_clock=0)"""
        w2 = self.window ** 2
        return 2 * w2 + 3 if self.scenario == "pp" else 3 * w2 + 2

    @property
    def rcom2(self) -> int:
        return -1 if self.rcom == 0 else 2 * self.rcom * self.rcom

    @property
    def n_empty_cells(self) -> int:
        if self.scenario == "pp":
            return 0
        return int((self.wall == 0).sum()) - self.n_agents      # coverage.py:228-230 (counted after spawn)

    @property
    def bound_return(self) -> float:
        if self.scenario == "pp":                               # predator_prey.py:73
            return self.n_preys * self.capture_reward
        ne, n = self.n_empty_cells, self.n_agents               # coverage.py:214-219 (agg = mean)
        return self.capture_reward * ne / n - abs(self.step_cost) * ne / n + self.final_reward

    @property
    def ave_trput(self):
        return 0 if self.scenario == "pp" else self.n_empty_cells   # coverage.py:232

    def wall_rows(self) -> np.ndarray:
        """u64 [G] bit rows of the wall map (bit c of word r = cell (r, c) is a wall)."""
        G = self.grid
        rows = np.zeros(G, dtype=np.uint64)
        if self.wall is not None:
            for r in range(G):
                v = 0
                for c in range(G):
                    if self.wall[r, c]:
                        v |= 1 << c
                rows[r] = v
        return rows

    def lut(self) -> np.ndarray:
        """f32 [G + G + T + 1]: observation scalar features.
        PredatorPrey: row/m, col/(m-1) (asymmetric on purpose), t/T as float64 -> float32
        (predator_prey.py:195-196, then torch.Tensor(obs) at comm_categorical_mlp_policy.py:57);
        Coverage: Python round(pos/(G-1), 2) (coverage.py:206)."""
        G, T = self.grid, self.max_steps
        if self.scenario == "pp":
            m = self.map_size
            rows = [r / m for r in range(G)]
            cols = [c / (m - 1) for c in range(G)]
            tt = [t / T for t in range(T + 1)]
        else:
            rows = [round(r / (G - 1), 2) for r in range(G)]
            cols = list(rows)
            tt = [0.0] * (T + 1)
        return np.asarray(rows + cols + tt, dtype=np.float64).astype(np.float32)

    def validate(self):
        if not (1 <= self.n_agents <= N.MAX_AGENTS and 0 <= self.n_preys <= N.MAX_AGENTS):
            raise ValueError(f"n_agents/n_preys must be in 1..{N.MAX_AGENTS}")
        if not 2 <= self.grid <= N.MAX_GRID:
            raise ValueError(f"grid side {self.grid} exceeds {N.MAX_GRID}")
        if self.sensing not in (0, 1, 2):
            raise ValueError("Rsen must be 0, 1 or 2 (window bits are packed in 32-bit words)")
        if self.scenario == "pp" and self.load not in (2, 3, 4):
            raise ValueError("load must be 2, 3 or 4 (predator_prey.py:77-79 defines no capv otherwise)")
        if self.channel == N.CH_GE and self.ge_init == -1 and self.loss_apply == 0:
            raise ValueError("GE_INIT=-1 with loss_apply=0 is broken in the reference (env_communication.py:121)")

    # ---- construction ----------------------------------------------------------------------------
    @classmethod
    def from_params(cls, scenario: str, params: dict, seed: int = 1, max_path_length: Optional[int] = None,
                    channel_type: Optional[str] = None):
        """``params`` is the dict the reference runners pass as ``kwargs['params']`` (vars(args)).

        ``channel_type='GE'`` selects the Gilbert-Elliot branch, which the reference can only reach by
        setting ``env.channelType`` after construction (init_communication forces FC/IID/FL from the
        loss probability, env_communication.py:35-43)."""
        m = int(params["grid_size"])
        n = int(params["n_agents"])
        common = dict(scenario=scenario, map_size=m, n_agents=n, sensing=int(params["Rsen"]),
                      n_layers=int(params.get("n_gcn_layers", 2)), seed=int(seed),
                      max_path_length=int(max_path_length or 0), loss_apply=int(params.get("loss_apply", 1)))
        if scenario == "pp":
            spec = cls(n_preys=int(params["n_preys"]), max_steps=int(params["max_env_steps"]),
                       load=int(params["load"]), capture_reward=float(abs(params["capture_reward"])),
                       step_cost=_neg_abs(params["step_cost"]), moving_cost=_neg_abs(params["rm"]),
                       penalty=_neg_abs(params["penalty"]), **common)
        elif scenario == "co":
            obst = params.get("obstComplex", "Easy")
            spec = cls(n_preys=0, max_steps=int(params.get("max_env_steps", 400)), load=int(params.get("load", 2)),
                       capture_reward=float(abs(params["capture_reward"])), step_cost=_neg_abs(params["step_cost"]),
                       moving_cost=_neg_abs(params["rm"]), penalty=_neg_abs(params["penalty"]),
                       lazy_penalty=_neg_abs(params["lazy_penalty"]), revisit_penalty=_neg_abs(params["revisit_penalty"]),
                       final_reward=100.0,                      # hard-coded, coverage.py:92
                       obst=obst, wall=coverage_wall_grid(m, obst), **common)
            if n % int(params.get("n_groups", 3) or 1):
                raise ValueError("n_agents must be divisible by n_groups (coverage.py:53)")
        else:
            raise ValueError(f"unknown scenario {scenario!r}")
        pref = "tr" if params.get("mode", "train") in ("train", "restore") else "te"
        pl = params.get(f"{pref}pl")
        if pl is None:
            raise ValueError("Loss probability is not applied (env_communication.py:31-32)")
        return spec.with_channel(pl=pl, rcom=params.get(f"{pref}Rcom", 9), channel_type=channel_type,
                                 pgb=params.get("Pgb", 0.0196), pbg=params.get("Pbg", 0.282), ge_init=params.get("GE_INIT", 1))

    CHANNEL_FIELDS = ("channel", "p_loss", "rcom", "pgb", "pbg", "ge_init")

    def with_channel(self, pl=None, rcom=None, channel_type: Optional[str] = None, pgb=None, pbg=None, ge_init=None):
        """A copy under another channel condition, by the rules of the reference's init_communication
        (env_communication.py:26-75): ``pl`` 0 -> FC, 0 < pl < 1 -> IID, 1 -> FL; ``rcom`` collapses to fully connected when
        Rcom + 1 >= map; ``channel_type`` ('FC', 'FL', 'IID', 'GE') is applied last, as setting ``env.channelType`` after
        construction does.  Arguments left at None keep this spec's value."""
        spec = copy.copy(self)
        if pl is not None:
            if pl == 0:
                spec.channel = N.CH_FC
            elif 0 < pl < 1:
                spec.channel = N.CH_IID
            elif pl == 1:
                spec.channel = N.CH_FL
            else:
                raise ValueError(f"invalid Ploss value: pl={pl}")
            spec.p_loss = float(pl)
        if rcom is not None:
            rcom = int(rcom)
            spec.rcom = 0 if rcom + 1 >= spec.map_size else rcom     # :71-72
        if pgb is not None:
            spec.pgb = float(pgb)
        if pbg is not None:
            spec.pbg = float(pbg)
        if ge_init is not None:
            spec.ge_init = int(ge_init)
        if channel_type is not None:
            spec.channel = {"FC": N.CH_FC, "FL": N.CH_FL, "IID": N.CH_IID, "GE": N.CH_GE}[channel_type]
        spec.validate()
        return spec

    def same_except_channel(self, other: "ScenarioSpec") -> bool:
        """whether ``other`` differs from this spec in the channel fields (CHANNEL_FIELDS) at most"""
        for f in fields(self):
            if f.name in self.CHANNEL_FIELDS:
                continue
            a, b = getattr(self, f.name), getattr(other, f.name)
            if isinstance(a, np.ndarray) or isinstance(b, np.ndarray):
                if a is None or b is None or not np.array_equal(a, b):
                    return False
            elif a != b:
                return False
        return True

    def channel_cond(self) -> "N.ChannelCond":
        """this spec's channel as one entry of a cm_channel_cond table"""
        d = self.to_desc(None, None)
        return N.ChannelCond(d.channel, d.rcom2, d.p_loss, d.pgb, d.pbg, d.ge_bad_rate, d.ge_init)

    @classmethod
    def from_cli(cls, scenario: str, map_size: int, sen: int, den: float, cap: int = 2, loss: float = 0.0, **over):
        """The runners' sizing rule: n_agents = int(int(den*100) * (map/10)^2), n_preys = n_agents
        (exp_runners/env_uitils.py:194-201,35-43) with the default rewards of utils_pp.py:77-81 /
        utils_co.py:84-91."""
        n = int(int(den * 100) * (map_size / 10) ** 2)
        p = dict(grid_size=map_size, Rsen=sen, n_agents=n, n_gcn_layers=2, loss_apply=1, mode="train", trpl=loss,
                 trRcom=9, rm=0)
        if scenario == "pp":
            p.update(n_preys=n, load=cap, max_env_steps=200, capture_reward=10, step_cost=0.1, penalty=0)
        else:
            p.update(n_groups=3, obstComplex="Easy", load=2, capture_reward=2, step_cost=0, penalty=1,
                     revisit_penalty=0.5, lazy_penalty=1, max_env_steps=400)
        seed = over.pop("seed", 1)
        mpl = over.pop("max_path_length", None)
        ct = over.pop("channel_type", None)
        p.update(over)
        return cls.from_params(scenario, p, seed=seed, max_path_length=mpl, channel_type=ct)

    def to_desc(self, wall_rows_ptr, lut_ptr, env_id0=0) -> "N.EnvDesc":
        d = N.EnvDesc()
        d.scenario = N.PREDATOR_PREY if self.scenario == "pp" else N.COVERAGE
        d.n_agents, d.n_preys, d.grid, d.sensing = self.n_agents, self.n_preys, self.grid, self.sensing
        d.max_steps, d.max_path_length, d.load, d.n_layers = self.max_steps, self.max_path_length, self.load, self.n_layers
        d.n_empty_cells, d.rcom2, d.channel = self.n_empty_cells, self.rcom2, self.channel
        d.loss_apply, d.ge_init = self.loss_apply, self.ge_init
        # torch compares a float32 tensor with a Python scalar in float32 (SURVEY.md §8a a18/a19 [probed])
        d.p_loss = float(np.float32(self.p_loss))
        d.pgb, d.pbg = float(np.float32(self.pgb)), float(np.float32(self.pbg))
        d.ge_bad_rate = float(np.float32(self.pgb / (self.pgb + self.pbg))) if (self.pgb + self.pbg) > 0 else 0.0
        d.capture_reward, d.step_cost, d.moving_cost = self.capture_reward, self.step_cost, self.moving_cost
        d.penalty, d.lazy_penalty, d.revisit_penalty = self.penalty, self.lazy_penalty, self.revisit_penalty
        d.final_reward = self.final_reward
        d.seed, d.env_id0 = self.seed, env_id0
        d.wall_rows, d.lut = wall_rows_ptr, lut_ptr
        return d
