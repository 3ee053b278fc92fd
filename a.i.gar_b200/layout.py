"""Python view of the C ABI structs in include/agar_b200.h (AgarConfig, AgarLayout and
the per-env state record).  Used by the host API for agar_debug_dump/agar_debug_load and
by the tests to compare records coming from the GPU, the CPU oracle and the reference
harness field by field.
"""
import ctypes
import math

import numpy as np

ABI_VERSION = 1  # AGAR_ABI_VERSION
MAX_PLAYERS = 16
MAX_CELLS = 16
ACTION_DIM = 4

BOT_NN, BOT_GREEDY, BOT_RANDOM = 0, 1, 2
OBS_REFERENCE, OBS_CANONICAL = 0, 1
SIMPLE_STATE_LEN = 12  # Bot.getSimpleStateRepresentation, bot.py:511-548 (AGAR_SIMPLE_STATE_LEN)
CF_EJECT, CF_INHASH = 1, 2
REC_ERR_INDEX, REC_ERR_RECORD = 1, 2  # AGAR_REC_ERR_*

(GET_REWARD, GET_DONE, GET_VALID, GET_NEED_ACTION, GET_MASS, GET_FOV, GET_NCELLS, GET_ALIVE, GET_STATS,
 GET_OVERFLOW, GET_EVENT_HASH) = range(11)

EV_NAMES = {1: "EAT_PELLET", 2: "EAT_BLOB", 3: "EAT_VIRUS", 4: "VIRUS_EAT_BLOB", 5: "EAT_CELL", 6: "MERGE",
            7: "COLLIDE", 8: "SPAWN_PELLET", 9: "SPAWN_VIRUS", 10: "SPAWN_PLAYER", 11: "SPLIT", 12: "EJECT",
            13: "BLOB_TO_PELLET", 14: "PLAYER_DIED"}
(EV_EAT_PELLET, EV_EAT_BLOB, EV_EAT_VIRUS, EV_VIRUS_EAT_BLOB, EV_EAT_CELL, EV_MERGE, EV_COLLIDE, EV_SPAWN_PELLET,
 EV_SPAWN_VIRUS, EV_SPAWN_PLAYER, EV_SPLIT, EV_EJECT, EV_BLOB_TO_PELLET, EV_PLAYER_DIED) = range(1, 15)


class AgarConfig(ctypes.Structure):
    _fields_ = [
        ("n_players", ctypes.c_int32),
        ("bot_type", ctypes.c_int32 * MAX_PLAYERS),
        ("virus_enabled", ctypes.c_int32), ("enable_split", ctypes.c_int32), ("enable_eject", ctypes.c_int32),
        ("enable_greedy_split", ctypes.c_int32), ("pellet_spawn", ctypes.c_int32),
        ("grid_squares", ctypes.c_int32), ("frame_skip", ctypes.c_int32),
        ("pellet_grid", ctypes.c_int32), ("self_grid", ctypes.c_int32), ("wall_grid", ctypes.c_int32),
        ("enemy_grid", ctypes.c_int32), ("virus_grid", ctypes.c_int32),
        ("self_grid_lf", ctypes.c_int32), ("self_grid_slf", ctypes.c_int32),
        ("enemy_grid_lf", ctypes.c_int32), ("enemy_grid_slf", ctypes.c_int32),
        ("use_fovsize", ctypes.c_int32), ("use_last_fovsize", ctypes.c_int32), ("use_totalmass", ctypes.c_int32),
        ("use_last_action", ctypes.c_int32), ("use_second_last_action", ctypes.c_int32),
        ("mass_as_reward", ctypes.c_int32), ("obs_mode", ctypes.c_int32),
        ("fat_cap", ctypes.c_int32), ("virus_cap", ctypes.c_int32), ("blob_cap", ctypes.c_int32),
        ("event_cap", ctypes.c_int32),
        ("pellet_cap", ctypes.c_int32), ("all_player_grid", ctypes.c_int32), ("normalize_grid_by_max_mass", ctypes.c_int32),
        ("simple_state", ctypes.c_int32),
        ("reserved", ctypes.c_int32 * 3),
        ("reward_scale", ctypes.c_double), ("reward_term", ctypes.c_double),
        ("death_term", ctypes.c_double), ("death_factor", ctypes.c_double),
    ]


class AgarLayout(ctypes.Structure):
    _fields_ = [
        ("field_size", ctypes.c_int32), ("n_players", ctypes.c_int32), ("cell_cap", ctypes.c_int32),
        ("pellet_cap", ctypes.c_int32), ("fat_cap", ctypes.c_int32), ("virus_cap", ctypes.c_int32),
        ("blob_cap", ctypes.c_int32), ("event_cap", ctypes.c_int32), ("grid_squares", ctypes.c_int32),
        ("n_grids", ctypes.c_int32), ("n_extra", ctypes.c_int32), ("state_len", ctypes.c_int32),
        ("n_agents", ctypes.c_int32), ("action_len", ctypes.c_int32), ("n_hist", ctypes.c_int32),
        ("pad", ctypes.c_int32),
        ("max_pellets", ctypes.c_double), ("max_viruses", ctypes.c_double),
        ("off_header", ctypes.c_uint64), ("off_players", ctypes.c_uint64), ("off_cells", ctypes.c_uint64),
        ("off_viruses", ctypes.c_uint64), ("off_blobs", ctypes.c_uint64), ("off_fat", ctypes.c_uint64),
        ("off_pellets", ctypes.c_uint64), ("off_hist", ctypes.c_uint64), ("off_events", ctypes.c_uint64),
        ("record_bytes", ctypes.c_uint64),
    ]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


CELL_DT = np.dtype([("x", "f8"), ("y", "f8"), ("mass", "f8"), ("radius", "f8"), ("svx", "f8"), ("svy", "f8"),
                    ("merge_time", "f8"), ("counter", "i4"), ("uid", "u4"), ("flags", "u4"), ("pad", "u4")],
                   align=True)
MOTE_DT = np.dtype([("x", "f8"), ("y", "f8"), ("mass", "f8"), ("radius", "f8"), ("svx", "f8"), ("svy", "f8"),
                    ("counter", "i4"), ("aux", "u4")], align=True)
FAT_DT = np.dtype([("x", "f8"), ("y", "f8"), ("mass", "f8"), ("radius", "f8")], align=True)
BOT_DT = np.dtype([("type", "i4"), ("has_action", "i4"), ("has_last_action", "i4"), ("skip_frames", "i4"),
                   ("has_last_mass", "i4"), ("has_old_state", "i4"), ("time", "i4"), ("skipping", "i4"),
                   ("turn_begun", "i4"), ("need_action", "i4"), ("exp_valid", "i4"), ("exp_done", "i4"),
                   ("cur_action", "f8", (4,)), ("last_action", "f8", (4,)), ("cum_reward", "f8"),
                   ("last_reward", "f8"), ("last_mass", "f8"), ("fov_size_feat", "f8"),
                   ("last_fov_size_feat", "f8"), ("stat_mass_sum", "f8"), ("stat_mass_max", "f8"),
                   ("stat_frames", "f8"), ("stat_deaths", "f8")], align=True)
PLAYER_DT = np.dtype([("alive", "i4"), ("respawn_time", "i4"), ("n_cells", "i4"), ("do_split", "i4"),
                      ("do_eject", "i4"), ("fov_valid", "i4"), ("cmd_x", "f8"), ("cmd_y", "f8"), ("fov_x", "f8"),
                      ("fov_y", "f8"), ("fov_size", "f8"), ("bot", BOT_DT)], align=True)
HEADER_DT = np.dtype([("rng_field", "u4"), ("rng_bot", "u4"), ("next_uid", "u4"), ("frame", "u4"),
                      ("n_viruses", "i4"), ("n_blobs", "i4"), ("n_fat", "i4"), ("n_pellets", "i4"),
                      ("n_dead", "i4"), ("n_events", "i4"), ("overflow", "u4"), ("pad0", "u4"),
                      ("event_hash", "u8"), ("dead_order", "i4", (MAX_PLAYERS,))], align=True)
EVENT_DT = np.dtype([("type", "i4"), ("a", "i4"), ("b", "i4"), ("c", "i4"), ("d", "i4")], align=True)

assert CELL_DT.itemsize == 72 and MOTE_DT.itemsize == 56 and FAT_DT.itemsize == 32
assert BOT_DT.itemsize == 184 and PLAYER_DT.itemsize == 248 and HEADER_DT.itemsize == 120
assert EVENT_DT.itemsize == 20


def derive_config(num_nn=1, num_greedy=0, num_random=0, virus=False, split=False, eject=False, grid=11,
                  frame_skip=7, obs_mode=OBS_REFERENCE, event_cap=0, pellet_spawn=True, reward_scale=2.0,
                  reward_term=0.0, death_term=-40.0, death_factor=1.5, mass_as_reward=False, grid_view=True, overrides=None):
    """Build an AgarConfig the way src/model/networkParameters.py:75-102 derives its flags."""
    c = AgarConfig()
    k = num_nn + num_greedy + num_random
    c.n_players = k
    types = [BOT_NN] * num_nn + [BOT_GREEDY] * num_greedy + [BOT_RANDOM] * num_random
    for i, t in enumerate(types):
        c.bot_type[i] = t
    multiple = k > 1
    c.virus_enabled = int(virus)
    c.enable_split = int(split)
    c.enable_eject = int(eject)
    c.enable_greedy_split = 0
    c.pellet_spawn = int(pellet_spawn)
    c.grid_squares = grid
    c.frame_skip = frame_skip
    c.pellet_grid = 1
    c.self_grid = int(split or virus)
    c.self_grid_lf = int(split)
    c.self_grid_slf = 0
    c.wall_grid = int(multiple)
    c.virus_grid = int(virus)
    c.enemy_grid = int(multiple)
    c.enemy_grid_lf = int(split)
    c.enemy_grid_slf = 0
    c.use_fovsize = 1
    c.use_last_fovsize = int(split)
    c.use_totalmass = 1
    c.use_last_action = int(split)
    c.use_second_last_action = 0
    c.mass_as_reward = int(mass_as_reward)
    c.obs_mode = obs_mode
    c.simple_state = int(not grid_view)  # GRID_VIEW_ENABLED, networkParameters.py:119
    c.event_cap = event_cap
    c.reward_scale = reward_scale
    c.reward_term = reward_term
    c.death_term = death_term
    c.death_factor = death_factor
    for name, val in (overrides or {}).items():
        setattr(c, name, val)
    return c


def _align(v, a):
    return (v + a - 1) // a * a


def layout_for_config(c):
    """Pure-Python twin of agar_layout_compute() (include/agar_layout.h); tests check they agree."""
    L = AgarLayout()
    k = c.n_players
    if (c.enable_eject and not c.enable_split) or c.enable_greedy_split or (c.virus_grid and not c.virus_enabled) or \
            (c.all_player_grid and (c.self_grid or c.enemy_grid or c.self_grid_lf or c.self_grid_slf or c.enemy_grid_lf or
                                    c.enemy_grid_slf)):
        raise ValueError("config rejected (agar_layout_compute: eject without split, greedy split, a virus grid without viruses, "
                         "or the all-player grid together with self / enemy grids)")
    s = int(75.0 * math.sqrt(k))
    L.field_size, L.n_players = s, k
    L.n_agents = sum(1 for i in range(k) if c.bot_type[i] == BOT_NN)
    L.cell_cap = MAX_CELLS if (c.enable_split or c.virus_enabled) else 1
    L.max_pellets = (s * s) * 0.015 if c.pellet_spawn else 0.0
    L.max_viruses = (s * s) * 0.00005
    p = 0
    while p < L.max_pellets:
        p += 1
    v0 = 0
    while v0 < L.max_viruses:
        v0 += 1
    p = max(p, c.pellet_cap)
    L.pellet_cap = p
    L.virus_cap = (c.virus_cap if c.virus_cap > 0 else 2 * v0 + 6) if c.virus_enabled else 0
    L.blob_cap = (c.blob_cap if c.blob_cap > 0 else 8 * k + 8) if c.enable_eject else 0
    L.fat_cap = (c.fat_cap if c.fat_cap > 0 else 16 * k + 16) if c.enable_eject else 0
    L.event_cap = max(c.event_cap, 0)
    g = c.grid_squares
    L.grid_squares = g
    L.n_grids = sum(int(bool(x)) for x in (c.pellet_grid, c.self_grid, c.wall_grid, c.virus_grid, c.enemy_grid,
                                           c.self_grid_lf, c.self_grid_slf, c.enemy_grid_lf, c.enemy_grid_slf, c.all_player_grid))
    L.n_extra = (int(bool(c.use_fovsize)) + int(bool(c.use_totalmass)) + 4 * int(bool(c.use_last_action)) +
                 4 * int(bool(c.use_second_last_action)) + int(bool(c.use_last_fovsize)))
    L.state_len = g * g * L.n_grids + L.n_extra
    if c.simple_state:
        L.n_grids, L.n_extra, L.state_len = 0, 0, SIMPLE_STATE_LEN
    L.action_len = 2 + int(bool(c.enable_split)) + int(bool(c.enable_eject))
    L.n_hist = 4 if (not c.simple_state and (c.self_grid_lf or c.self_grid_slf or c.enemy_grid_lf or c.enemy_grid_slf)) else 0
    off = 0
    L.off_header = off
    off = _align(off + HEADER_DT.itemsize, 16)
    L.off_players = off
    off = _align(off + k * PLAYER_DT.itemsize, 16)
    L.off_cells = off
    off = _align(off + k * L.cell_cap * CELL_DT.itemsize, 16)
    L.off_viruses = off
    off = _align(off + L.virus_cap * MOTE_DT.itemsize, 16)
    L.off_blobs = off
    off = _align(off + L.blob_cap * MOTE_DT.itemsize, 16)
    L.off_fat = off
    off = _align(off + L.fat_cap * FAT_DT.itemsize, 16)
    L.off_pellets = off
    off = _align(off + p * 4, 16)
    L.off_hist = off
    off = _align(off + L.n_agents * L.n_hist * g * g * 4, 16)
    L.off_events = off
    off = off + L.event_cap * EVENT_DT.itemsize
    L.record_bytes = _align(off, 128)
    return L


class Record(object):
    """Numpy views over one env record (a writable buffer of layout.record_bytes bytes)."""

    def __init__(self, layout, buf=None):
        self.layout = layout
        n = int(layout.record_bytes)
        if buf is None:
            buf = np.zeros(n, dtype=np.uint8)
        else:
            buf = np.frombuffer(buf, dtype=np.uint8, count=n) if not isinstance(buf, np.ndarray) else buf
        assert buf.nbytes == n, (buf.nbytes, n)
        self.buf = buf
        L = layout
        k, g = L.n_players, L.grid_squares

        def view(off, dt, count):
            return buf[int(off):int(off) + dt.itemsize * count].view(dt)

        self.header = view(L.off_header, HEADER_DT, 1)
        self.players = view(L.off_players, PLAYER_DT, k)
        self.cells = view(L.off_cells, CELL_DT, k * L.cell_cap).reshape(k, L.cell_cap)
        self.viruses = view(L.off_viruses, MOTE_DT, L.virus_cap)
        self.blobs = view(L.off_blobs, MOTE_DT, L.blob_cap)
        self.fat = view(L.off_fat, FAT_DT, L.fat_cap)
        self.pellets = view(L.off_pellets, np.dtype("u4"), L.pellet_cap)
        self.hist = view(L.off_hist, np.dtype("f4"), L.n_agents * L.n_hist * g * g).reshape(L.n_agents, L.n_hist, g, g)
        self.events = view(L.off_events, EVENT_DT, L.event_cap)

    def event_list(self):
        n = int(self.header["n_events"][0])
        ev = self.events[:min(n, self.layout.event_cap)]
        return [(int(e["type"]), int(e["a"]), int(e["b"]), int(e["c"]), int(e["d"])) for e in ev]

    def pellet_list(self):
        """[(slot, x, y, mass)] of live integer pellets."""
        out = []
        for s, p in enumerate(self.pellets):
            p = int(p)
            if p:
                out.append((s, p & 1023, (p >> 10) & 1023, p >> 20))
        return out


def pack_pellet(x, y, m):
    return int(x) | (int(y) << 10) | (int(m) << 20)


_HASH_MUL = 0x100000001B3
_M64 = (1 << 64) - 1


def event_hash_step(h, ev):
    """Order-sensitive running hash of events (same arithmetic in oracle and kernels)."""
    for v in ev:
        h = ((h ^ (v & 0xFFFFFFFF)) * _HASH_MUL) & _M64
    return h


def compare_records(a, b, rtol=0.0, atol=0.0, what="", check_bots=True, check_events=False, check_hist=True):
    """Return a list of human-readable differences between two Records (empty = equal).

    Integer fields must match exactly; float fields within rtol/atol (0 = bit-exact)."""
    diffs = []

    def cmp_struct(name, xa, xb):
        for f in xa.dtype.names:
            if f in ("pad", "pad0"):
                continue
            va, vb = xa[f], xb[f]
            if xa.dtype[f].names:
                cmp_struct(name + "." + f, va, vb)
                continue
            if va.dtype.kind == "f":
                if rtol == 0.0 and atol == 0.0:
                    bad = ~((va == vb) | (np.isnan(va) & np.isnan(vb)))
                else:
                    bad = ~np.isclose(va, vb, rtol=rtol, atol=atol, equal_nan=True)
            else:
                bad = va != vb
            if np.any(bad):
                idx = np.argwhere(bad)[0]
                diffs.append("%s%s.%s%s: %r != %r (%d mismatches)" % (what, name, f, list(idx), va[tuple(idx)],
                                                                      vb[tuple(idx)], int(bad.sum())))

    ha, hb = a.header, b.header
    hdr_fields = ["rng_field", "rng_bot", "next_uid", "frame", "n_viruses", "n_blobs", "n_fat", "n_pellets",
                  "n_dead", "overflow"]
    if check_events:
        hdr_fields += ["n_events", "event_hash"]
    for f in hdr_fields:
        if ha[f][0] != hb[f][0]:
            diffs.append("%sheader.%s: %r != %r" % (what, f, ha[f][0], hb[f][0]))
    nd = int(ha["n_dead"][0])
    if list(ha["dead_order"][0][:nd]) != list(hb["dead_order"][0][:nd]):
        diffs.append("%sheader.dead_order differs" % what)
    pa, pb = a.players, b.players
    pfields = [f for f in PLAYER_DT.names if f != "bot"]
    cmp_struct("players", pa[pfields], pb[pfields])
    if check_bots:
        cmp_struct("players.bot", pa["bot"], pb["bot"])
    for k in range(a.layout.n_players):
        n = int(pa["n_cells"][k])
        if n == int(pb["n_cells"][k]) and n > 0:
            cmp_struct("cells[%d]" % k, a.cells[k, :n], b.cells[k, :n])
    nv = int(ha["n_viruses"][0])
    if nv == int(hb["n_viruses"][0]) and nv:
        cmp_struct("viruses", a.viruses[:nv], b.viruses[:nv])
    nb = int(ha["n_blobs"][0])
    if nb == int(hb["n_blobs"][0]) and nb:
        cmp_struct("blobs", a.blobs[:nb], b.blobs[:nb])
    if a.layout.fat_cap:
        live_a, live_b = a.fat["mass"] != 0, b.fat["mass"] != 0
        if np.any(live_a != live_b):
            diffs.append("%sfat pellet occupancy differs" % what)
        elif np.any(live_a):
            cmp_struct("fat", a.fat[live_a], b.fat[live_a])
    if np.any(a.pellets != b.pellets):
        idx = int(np.argwhere(a.pellets != b.pellets)[0][0])
        diffs.append("%spellets[%d]: %#x != %#x" % (what, idx, int(a.pellets[idx]), int(b.pellets[idx])))
    if a.hist.size and check_hist:
        if rtol == 0.0 and atol == 0.0:
            bad = a.hist != b.hist
        else:
            bad = ~np.isclose(a.hist, b.hist, rtol=max(rtol, 1e-6), atol=atol)
        if np.any(bad):
            diffs.append("%shistory grids differ (%d elements)" % (what, int(bad.sum())))
    if check_events:
        ea, eb = a.event_list(), b.event_list()
        if ea != eb:
            diffs.append("%sevents differ: %r vs %r" % (what, ea[:8], eb[:8]))
    return diffs
