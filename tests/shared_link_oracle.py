"""Oracle of shared bottleneck links (SPEC §9) — TEST INFRASTRUCTURE.

Pure Python; IEEE doubles, operations in the order SPEC §9 writes them, so the results are the kernel's bit for bit.
Each link is a ``step_oracle.Session`` that stands for the trace position (its reset, ``_position`` and ``_advance``
are SPEC §2, §3.1 and §3.3); the players' decisions are the existing policy oracles' pure-Python rules
(``session_params_oracle.session_action`` on top of ``policy_oracle`` and ``dynamic_oracle``), used unchanged.
Small cases only: one Python-level event at a time.
"""
from __future__ import annotations

import math

import numpy as np

import dynamic_oracle as do
import policy_oracle as po
import session_params_oracle as spo
from oracle import step_oracle as so

FIXED, RANDOM, BBA, RATE, BOLA, DYNAMIC = 0, 1, po.POLICY_BBA, po.POLICY_RATE, po.POLICY_BOLA, do.POLICY_DYNAMIC
WAITING, ACTIVE, FINISHED = 0, 1, 2
_M32 = 0xffffffff


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """SPEC §4: Philox4x32-10 (the kernels' abr_common.cuh, oracle/abr_oracle.c)."""
    for _ in range(10):
        p0, p1 = 0xD2511F53 * c0, 0xCD9E8D57 * c2
        c0, c1, c2, c3 = ((p1 >> 32) ^ c1 ^ k0) & _M32, p1 & _M32, ((p0 >> 32) ^ c3 ^ k1) & _M32, p0 & _M32
        k0, k1 = (k0 + 0x9E3779B9) & _M32, (k1 + 0xBB67AE85) & _M32
    return c0, c1, c2, c3


def random_action(seed, g, k, A):
    """SPEC §4 RANDOM: draw k of global session g."""
    w = philox4x32_10(g & _M32, (g >> 32) & _M32, k >> 3, 0, seed & _M32, (seed >> 32) & _M32)[(k & 7) >> 1]
    return (((w >> (16 * (k & 1))) & 0xffff) * A) >> 16


class World:
    """Traces, video and parameters as the environment holds them: ``util`` must be the environment's own utility
    table (``env.state("utility")``), ``P`` a dict of the AbrParams fields the step reads, ``wide`` the seven
    environment-wide policy knobs of SPEC §4.7 (``session_params_oracle.env_wide``)."""

    def __init__(self, trace_bw, trace_len, trace_interval, sizes, util, P, wide):
        self.bw = [list(map(float, row)) for row in np.asarray(trace_bw, np.float64)]
        self.tl = [int(x) for x in trace_len]
        self.ti = [float(x) for x in np.broadcast_to(np.asarray(trace_interval, np.float64), (len(self.bw),))]
        self.sizes = [list(map(float, r)) for r in np.asarray(sizes, np.float64)]
        self.util = [list(map(float, r)) for r in np.asarray(util, np.float64)]
        self.V, self.A = len(self.sizes), len(self.sizes[0])
        self.P = dict(P)
        self.wide = list(wide)
        self.tables = {}
        positive = all(x > 0 for r in self.sizes for x in r)
        self.v, self.v_max = po.bola_table(self.sizes) if positive else (None, 0.0)

    def table(self, tr):
        if tr not in self.tables:
            self.tables[tr] = so.capacity_table(self.bw[tr][:self.tl[tr]], self.ti[tr], self.P["payload"])
        return self.tables[tr]


def run_shared(world, steps, G, link_trace_id, link_offset=None, join_delay=None, policy=BBA, player_policy=None,
               seed=0, session_base=0, actions=None, knobs=None, dyn_mode=None):
    """SPEC §9 for every link.  ``knobs``: the installed [7][N] per-session parameters (None: environment-wide);
    ``dyn_mode``: the [N] rules DYNAMIC players start from (zeros: a new environment).  Returns a dict of numpy arrays:
    the [steps][N] outputs, the [n_links] link outputs, acc [11][N], qoe_cost [N], ``state`` (the end state, a dict of [N] fields) and
    ``errors``."""
    P = world.P
    n_links = len(link_trace_id)
    N = n_links * G
    pols = list(player_policy) if player_policy is not None else [policy] * G
    res = {k: np.zeros((steps, N)) for k in ("delay", "sleep", "buffer", "rebuf", "reward", "request_time")}
    res["eov"] = np.zeros((steps, N), np.uint8)
    res["actions"] = np.zeros((steps, N), np.int32)
    for k in ("link_time", "link_capacity", "link_delivered"):
        res[k] = np.zeros(n_links)
    res["acc"] = np.zeros((11, N))
    res["qoe_cost"] = np.zeros(N)
    st = res["state"] = {}
    for k, dt in (("seg", np.int32), ("phase", np.float64), ("pos", np.float64), ("chunk", np.int32),
                  ("last_q", np.int32), ("buffer", np.float64), ("done", np.uint8), ("hist_len", np.int32),
                  ("trace_id", np.int32), ("dyn_mode", np.uint8)):
        st[k] = np.zeros(N, dt)
    if dyn_mode is not None:
        st["dyn_mode"][:] = dyn_mode
    res["errors"] = 0
    for l in range(n_links):
        _run_link(world, res, l, steps, G, int(link_trace_id[l]), 0.0 if link_offset is None else float(link_offset[l]),
                  join_delay, pols, seed, session_base, actions, knobs)
    return res


def _run_link(world, res, l, steps, G, tr, off, join_delay, pols, seed, session_base, actions, knobs):
    P, V, A = world.P, world.V, world.A
    K = max(1, P["hist_k"])
    n_bad = 0
    if not 0 <= tr < len(world.bw):
        n_bad, tr = 1, 0
    if not math.isfinite(off) or math.floor(off / world.ti[tr]) < 0:
        raise ValueError("the oracle takes finite start offsets >= 0")
    T = world.tl[tr]
    link = so.Session(world.bw[tr][:T], world.ti[tr], world.sizes, world.util, P, start_offset=off,
                      table=world.table(tr))
    C, I, Pc = link.C, link.I, link.C[T]
    pos_start = link.pos
    players = []
    for p in range(G):
        i = l * G + p
        w = 0.0 if join_delay is None else float(join_delay[i])
        bad = not (w >= 0.0 and w <= 1.7976931348623157e308)
        kn = world.wide if knobs is None else [float(x) for x in np.asarray(knobs)[:, i]]
        players.append(dict(i=i, pol=pols[p], state=WAITING if steps > 0 else FINISHED, wait=0.0 if bad else w,
                            flagged=bad, k=0, buffer=0.0, chunk=0, last_q=P["default_quality"], done=False, hist=[],
                            mode=int(res["state"]["dyn_mode"][i]), knobs=kn, sums=[0.0] * 6, n=0, eps=0, rem=0.0, q=0))
    clock, periods, delivered = 0.0, 0, 0.0

    def decide(pl):
        pol, k, i = pl["pol"], pl["k"], pl["i"]
        if pol == FIXED:
            a = int(actions[k][i])
            if a < 0 or a >= A:
                pl["flagged"] = True
                a = 0 if a < 0 else A - 1
            return a
        if pol == RANDOM:
            return random_action(seed, session_base + i, k, A)
        if pol == BBA:
            return spo.session_action(BBA, world.sizes[0], None, 0.0, None, pl["buffer"], pl["chunk"], 0,
                                      P["default_quality"], P["chunk_length"], pl["knobs"])[0]
        if pl["done"]:
            return 0
        c = pl["chunk"]
        hist = [np.float64(x) for x in pl["hist"][-K:]]   # IEEE division: a zero-size chunk's throughput is 0
        with np.errstate(divide="ignore"):
            q, m = spo.session_action(pol, world.sizes[c], world.v[c] if world.v else None, world.v_max, hist,
                                      pl["buffer"], c, pl["mode"], P["default_quality"], P["chunk_length"], pl["knobs"])
        q = int(q)
        if pol == DYNAMIC:
            pl["mode"] = m
        return q

    def put(pl, **vals):
        for key, x in vals.items():
            res[key][pl["k"]][pl["i"]] = x

    def requests():
        for pl in players:
            while pl["state"] == WAITING and pl["wait"] <= 0.0:
                if pl["k"] >= steps:          # the sleep after the last download is over
                    pl["state"] = FINISHED
                    break
                q = decide(pl)
                pl["req_time"] = clock
                if not P["auto_reset"] and pl["done"]:
                    put(pl, delay=0.0, sleep=0.0, buffer=pl["buffer"], rebuf=0.0, reward=0.0, eov=1, actions=q,
                        request_time=clock)
                    pl["k"] += 1
                    if pl["k"] >= steps:
                        pl["state"] = FINISHED
                    continue
                c = pl["chunk"]
                pl["q"], pl["size"], pl["rem"] = q, world.sizes[c][q], world.sizes[c][q]
                prow = c - 1 if (P.get("smooth_prev_ladder", 0) and pl["last_q"] >= 0 and c > 0) else c
                pl["u"] = world.util[c][q]
                pl["u_prev"] = world.util[prow][pl["last_q"]] if pl["last_q"] >= 0 else pl["u"]
                pl["req"] = (link.seg, link.phi, periods)
                pl["state"] = ACTIVE

    def complete(pl):
        seg_req, phi_req, per_req = pl["req"]
        kd = float(link.seg - seg_req) + float((periods - per_req) * T)
        x = (kd + (link.phi - phi_req)) * I
        delay = (x if x > 0 else 0.0) + P["rtt"]
        thr = pl["size"] / delay
        d = delay - pl["buffer"]
        rebuf = d if d > 0 else 0.0
        buffer = (pl["buffer"] - delay if pl["buffer"] - delay > 0 else 0.0) + P["chunk_length"]
        sleep = 0.0
        if buffer > P["max_buffer"]:
            sleep = math.ceil((buffer - P["max_buffer"]) / P["sleep_quantum"]) * P["sleep_quantum"]
            buffer = buffer - sleep
        u = pl["u"]
        smooth = abs(u - pl["u_prev"])
        reward = (u - P["rebuf_penalty"] * rebuf) - P["smooth_penalty"] * smooth
        pl["hist"].append(thr)
        pl["last_q"] = pl["q"]
        pl["chunk"] += 1
        pl["buffer"] = buffer
        eov = pl["chunk"] >= V
        if eov and P["auto_reset"]:
            pl["chunk"], pl["buffer"], pl["last_q"], pl["hist"] = 0, 0.0, P["default_quality"], []
        elif eov:
            pl["done"] = True
        s = pl["sums"]
        for j, val in enumerate((reward, rebuf, u, smooth, sleep, delay)):
            s[j] = s[j] + val
        pl["n"] += 1
        pl["eps"] += int(eov)
        put(pl, delay=delay, sleep=sleep, buffer=buffer, rebuf=rebuf, reward=reward, eov=int(eov), actions=pl["q"],
            request_time=pl["req_time"])
        pl["k"] += 1
        pl["wait"] = sleep
        pl["state"] = WAITING

    requests()
    while any(pl["state"] != FINISHED for pl in players):
        act = [pl for pl in players if pl["state"] == ACTIVE]
        n = len(act)
        m = min((pl["rem"] for pl in act), default=math.inf)
        tw = min((pl["wait"] for pl in players if pl["state"] == WAITING), default=math.inf)
        if n > 0:
            target = link.pos + float(n) * m
            w = 0
            while target >= Pc:
                target = target - Pc
                w += 1
            j = link.seg if w == 0 else 0
            while j + 1 < T and C[j + 1] <= target:
                j += 1
            phi_new = (target - C[j]) / (C[j + 1] - C[j])
            x = ((float(j - link.seg) + float(w * T)) + (phi_new - link.phi)) * I
            dc = x if x > 0 else 0.0
        if n > 0 and dc <= tw:
            dt = dc
            link.seg, link.phi, link.pos = j, phi_new, target
            periods += w
            for pl in act:
                pl["rem"] = pl["rem"] - m
        else:
            dt = tw
            seg0, pos0 = link.seg, link.pos
            nx = math.floor(link.phi + tw / I)
            link._advance(tw)
            crossed = (seg0 + nx) // T
            periods += crossed
            if n > 0:
                d = ((link.pos - pos0) + float(crossed) * Pc) / float(n)
                for pl in act:
                    pl["rem"] = pl["rem"] - d
        for pl in players:
            if pl["state"] == WAITING:
                pl["wait"] = pl["wait"] - dt
        clock = clock + dt
        for pl in players:
            if pl["state"] == ACTIVE and pl["rem"] <= 0.0:
                complete(pl)
                delivered = delivered + pl["size"]
        requests()
    res["link_time"][l] = clock
    res["link_capacity"][l] = (float(periods) * Pc + link.pos) - pos_start
    res["link_delivered"][l] = delivered
    for pl in players:
        i = pl["i"]
        res["errors"] += n_bad + int(pl["flagged"])
        res["acc"][:8, i] = pl["sums"] + [float(pl["n"]), float(pl["eps"])]
        res["qoe_cost"][i] = P["rebuf_penalty"] * pl["sums"][1] + P["smooth_penalty"] * pl["sums"][3]
        st = res["state"]
        st["seg"][i], st["phase"][i], st["pos"][i], st["trace_id"][i] = link.seg, link.phi, link.pos, tr
        st["chunk"][i], st["last_q"][i], st["buffer"][i] = pl["chunk"], pl["last_q"], pl["buffer"]
        st["done"][i] = int(pl["done"])
        st["hist_len"][i] = len(pl["hist"]) if P.get("track_history", 0) else 0
        if pl["pol"] == DYNAMIC:
            st["dyn_mode"][i] = pl["mode"]


def world_of_env(env, trace_bw, trace_len, trace_interval, sizes, policy_params=None, dynamic_params=None):
    """A World with the environment's own parameters and utility table (a GPU test's reference)."""
    p = env.params
    P = {f: getattr(p, f) for f, _ in type(p)._fields_}
    wide = spo.env_wide(p, policy_params, dynamic_params)
    return World(trace_bw, trace_len, trace_interval, sizes, env.state("utility").cpu().numpy(), P, wide)
