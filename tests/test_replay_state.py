"""Replay-buffer state snapshots (agar_replay_save / agar_replay_load, GpuReplayBuffer.snapshot / restore / save_checkpoint /
load_checkpoint): a restored buffer continues bit for bit, banks are canonical, a load refuses any bank that could make a later
kernel index out of bounds and leaves the buffer unchanged, and checkpoint files are checked field by field."""
import copy
import ctypes

import numpy as np
import pytest

from aigar_b200 import replay as rpl
from oracle.replay_oracle import ReplayOracle

gpu = pytest.mark.gpu

# the header of include/agar_replay.h (AgarReplayStateHeader)
HEADER = np.dtype([("capacity", "<i8"), ("state_len", "<i8"), ("action_len", "<i8"), ("prioritized", "<i8"),
                   ("alpha_bits", "<u8"), ("beta_bits", "<u8"), ("next_idx", "<i8"), ("size", "<i8"), ("max_priority", "<f8")])
BAD_PRIORITIES = [0.0, -1.0, 1.75e308, float("nan")]   # skipped by update_priorities (flag 4)
EDGE_PRIORITIES = [5e-324, 1e-300, 1e300, 1.7e308]     # accepted; with alpha >= 1 their leaves are 0 or +inf


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("these tests need a GPU (the product has no CPU fallback; run with -m gpu on the B200 box)")
    return torch


def sections(cap, L, AL, prioritized):
    """{name: (offset, bytes per slot)} and the bank size, from the layout in include/agar_replay.h"""
    out, at = {}, 256
    for name, row in (("obs_t", 4 * L), ("obs_tp1", 4 * L), ("action", 4 * AL), ("reward", 4), ("done", 1),
                      ("leaf", 8 if prioritized else 0)):
        out[name] = (at, row)
        at = (at + cap * row + 255) // 256 * 256
    return out, at


def same(x, y):
    """bit for bit, NaN included (weights are NaN once a +inf leaf makes the tree's sum infinite)"""
    import torch
    return x.dtype == y.dtype and x.shape == y.shape and torch.equal(x.contiguous().view(torch.uint8),
                                                                     y.contiguous().view(torch.uint8))


def load_launches(cap, prioritized):
    """agar_replay_load: validate + install, and the tree rebuild at 11 levels per launch"""
    levels = (cap - 1).bit_length()
    return 2 + (-(-levels // 11) if prioritized else 0)


def header(bank_h):
    return bank_h[:HEADER.itemsize].view(HEADER)[0]


class Driver(object):
    """A seeded sequence of add / sample / update rounds, applied to a buffer and, where alpha keeps agar_pow in the domain
    where it equals libm, to the oracle: every output is recorded."""

    def __init__(self, torch, L, AL, seed, edge=False):
        self.torch, self.L, self.AL, self.edge = torch, L, AL, edge
        self.rng = np.random.default_rng(seed)

    def round(self, rp, n=None, ora=None):
        t, rng, dev = self.torch, self.rng, rp.device
        n = int(rng.integers(1, 80)) if n is None else n
        obs_t = rng.random((n, self.L)).astype(np.float32)
        obs_tp1 = rng.random((n, self.L)).astype(np.float32)
        act = rng.random((n, self.AL)).astype(np.float32)
        rew = rng.normal(size=n).astype(np.float32)
        done = (rng.random(n) < 0.2).astype(np.uint8)
        valid = rng.random(n) < 0.7
        rp.add_batch(*[t.tensor(x, device=dev) for x in (obs_t, act, rew, obs_tp1, done, valid)])
        if ora is not None:
            for i in np.flatnonzero(valid):
                ora.add(obs_t[i], act[i], float(rew[i]), obs_tp1[i], bool(done[i]))
        out = []
        size = len(rp)
        if size >= 2:
            u = rng.random(64)
            s = rp.sample(t.tensor(u, device=dev))
            out += [x.clone() for x in s]
            if ora is not None:
                so = ora.sample([float(x) for x in u])
                assert list(s[-1].cpu().numpy()) == list(so[-1])
                for a, b in zip(s[:5], so[:5]):
                    assert np.array_equal(a.cpu().numpy().astype(np.asarray(b).dtype), np.asarray(b))
                if rp.prioritized:
                    np.testing.assert_allclose(s[5].cpu().numpy(), so[5], rtol=1e-12)
            if rp.prioritized:
                idx = s[-1].cpu().numpy().astype(np.int64)[:16]
                idx = np.concatenate([idx, idx[:4], [-1, size, size + 7]])       # duplicates (the last wins), out of range
                pr = np.abs(rng.normal(size=idx.size)) + 1e-4
                k = int(rng.integers(0, 4))
                pr[16 + k] = BAD_PRIORITIES[k]                                    # a guarded priority on a valid index
                if self.edge:   # the last entries for their indices: with alpha >= 1, a 0 and a +inf leaf below size
                    pr[int(rng.integers(0, 16))] = EDGE_PRIORITIES[int(rng.integers(0, 4))]
                    idx = np.concatenate([idx, [int(rng.integers(0, size // 2)), size // 2 + int(rng.integers(0, size - size // 2))]])
                    pr = np.concatenate([pr, [1e-300, 1e300]])
                rp.update_priorities(t.tensor(idx, device=dev), t.tensor(pr, device=dev))
                if ora is not None:
                    # what the kernel applies: an entry whose index a later entry names is dropped before its checks
                    ok = [(int(i), float(p)) for j, (i, p) in enumerate(zip(idx, pr))
                          if i not in idx[j + 1:] and 0 <= i < size and 0 < p <= 1.7e308]
                    ora.update_priorities([i for i, _ in ok], [p for _, p in ok])
                    ora.max_priority = max([ora.max_priority] + [float(p) for p in pr if 0 < p <= 1.7e308])
        return out


def _fill(torch, rp, drv, ora=None):
    cap = rp.size_max
    for r in range(6):
        drv.round(rp, n=2 * cap + 3 if r == 2 else None, ora=ora)   # round 2 overflows the ring within one batch


ROUND_TRIP = [  # (prioritized, capacity, state_len, alpha, compare with the oracle)
    (False, 37, 123, 0.6, True), (True, 37, 123, 0.6, True), (False, 1000, 5, 0.6, True), (True, 1000, 5, 0.6, True),
    (False, 65536, 5, 0.6, True), (True, 65536, 5, 0.6, True), (True, 1000, 7, 1.0, False), (True, 65536, 3, 1.0, False)]


@gpu
@pytest.mark.parametrize("prioritized,cap,L,alpha,oracle", ROUND_TRIP,
                         ids=["%s-%d-L%d-a%g" % ("per" if c[0] else "uni", c[1], c[2], c[3]) for c in ROUND_TRIP])
def test_round_trip_continues_identically(torch_cuda, prioritized, cap, L, alpha, oracle):
    torch = torch_cuda
    from aigar_b200.replay import GpuReplayBuffer
    AL = 3
    mk = lambda: GpuReplayBuffer(cap, L, AL, prioritized, alpha, 0.4)   # noqa: E731
    a = mk()
    ora = ReplayOracle(cap, prioritized, alpha, 0.4) if oracle else None
    _fill(torch, a, Driver(torch, L, AL, 5, edge=alpha >= 1), ora)
    if prioritized:
        assert a.error_flags & 2                   # the out-of-range indices were refused
    bank = a.snapshot()
    assert bank.dtype == torch.uint8 and bank.dim() == 1 and bank.numel() == a.state_bytes == sections(cap, L, AL, prioritized)[1]
    ora0 = copy.deepcopy(ora)
    if alpha >= 1:   # the edge priorities put 0 and +inf leaves below size; they load
        leaf = bank.cpu().numpy()[sections(cap, L, AL, True)[0]["leaf"][0]:][:cap * 8].view(np.float64)[:len(a)]
        assert (leaf == 0).any() and np.isinf(leaf).any()

    def cont(rp, ora=None):
        d = Driver(torch, L, AL, 99, edge=alpha >= 1)
        out = []
        for _ in range(6):
            out += d.round(rp, ora=ora)
        return out + [rp.snapshot()]

    first = cont(a)
    b = mk()
    b.restore(bank)
    assert torch.equal(b.snapshot(), bank)
    second = cont(b, ora0)                         # a fresh buffer, checked against the oracle on the way
    a.restore(bank)                                # the original, after it diverged
    assert torch.equal(a.snapshot(), bank)
    third = cont(a)
    assert len(first) == len(second) == len(third)
    for i, (x, y, z) in enumerate(zip(first, second, third)):
        assert same(x, y) and same(x, z), "output %d differs after the restore" % i
    assert not (b.error_flags & rpl.ERR_STATE) and not (a.error_flags & rpl.ERR_STATE)


@gpu
@pytest.mark.parametrize("prioritized", [False, True])
def test_banks_are_canonical(torch_cuda, prioritized):
    torch = torch_cuda
    from aigar_b200.replay import GpuReplayBuffer
    cap, L, AL = 300, 5, 3
    rng = np.random.default_rng(3)
    n = 250
    data = [torch.tensor(x, device="cuda") for x in (rng.random((n, L), np.float32), rng.random((n, AL), np.float32),
                                                       rng.random(n, np.float32), rng.random((n, L), np.float32),
                                                       (rng.random(n) < 0.5).astype(np.uint8))]
    banks = []
    for cuts in ([0, n], [0, 1, 17, 100, 101, 250], [0, 200, 250]):
        rp = GpuReplayBuffer(cap, L, AL, prioritized, 0.6, 0.4)
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            rp.add_batch(*[x[lo:hi] for x in data])
        out = torch.full((rp.state_bytes,), 0xAB, dtype=torch.uint8, device=rp.device)   # every byte is written
        banks.append(rp.snapshot(out=out))
    for bk in banks[1:]:
        assert torch.equal(bk, banks[0])
    # a buffer whose allocations hold stale rows past size (it was full before the restore) saves the same bank
    full = GpuReplayBuffer(cap, L, AL, prioritized, 0.6, 0.4)
    for _ in range(2):
        full.add_batch(*data)
    full.restore(banks[0])
    assert torch.equal(full.snapshot(), banks[0])
    h = banks[0].cpu().numpy()
    hd = header(h)
    assert (hd["capacity"], hd["state_len"], hd["action_len"], hd["prioritized"], hd["next_idx"], hd["size"]) == \
        (cap, L, AL, int(prioritized), n, n)
    assert hd["alpha_bits"] == np.float64(0.6).view(np.uint64) and hd["max_priority"] == 1.0
    assert not h[HEADER.itemsize:256].any()
    secs, total = sections(cap, L, AL, prioritized)
    names = list(secs)
    for k, name in enumerate(names):
        off, row = secs[name]
        end = secs[names[k + 1]][0] if k + 1 < len(names) else total
        assert not h[off + n * row:end].any(), name                    # rows / leaves >= size and padding are zero
        if row:
            assert h[off:off + n * row].any(), name
    assert torch.equal(data[0], torch.from_numpy(h[secs["obs_t"][0]:][:n * L * 4].view(np.float32).reshape(n, L)).cuda())


def _corruptions(cap, L, AL, prioritized, size):
    """(name, function editing a host copy of a good bank) for every field a load checks"""
    secs = sections(cap, L, AL, prioritized)[0]

    def hdr(field, value):
        def f(h):
            hd = h[:HEADER.itemsize].view(HEADER)
            hd[field] = value
        return f

    def leaf(i, value):
        def f(h):
            h[secs["leaf"][0]:][:cap * 8].view(np.float64)[i] = value
        return f

    out = [("capacity", hdr("capacity", cap + 1)), ("state_len", hdr("state_len", L + 1)),
           ("action_len", hdr("action_len", AL - 1)), ("prioritized", hdr("prioritized", int(not prioritized))),
           ("prioritized=2", hdr("prioritized", 2)),
           ("alpha", hdr("alpha_bits", np.float64(0.6).view(np.uint64) + 1)),
           ("beta", hdr("beta_bits", np.float64(0.4).view(np.uint64) ^ (1 << 63))),
           ("next_idx<0", hdr("next_idx", -1)), ("next_idx=cap", hdr("next_idx", cap)), ("size<0", hdr("size", -1)),
           ("size>cap", hdr("size", cap + 1)), ("next_idx!=size", hdr("next_idx", size - 1)),
           ("max_priority nan", hdr("max_priority", np.nan)), ("max_priority<1", hdr("max_priority", 0.999)),
           ("max_priority>1.7e308", hdr("max_priority", 1.75e308)), ("max_priority inf", hdr("max_priority", np.inf))]
    if prioritized:
        out += [("leaf>=size nonzero", leaf(size + 3, 1.0)), ("leaf>=size -0.0", leaf(cap - 1, -0.0)),
                ("leaf<size nan", leaf(size // 2, np.nan)), ("leaf<size negative", leaf(0, -1e-300)),
                ("leaf<size -inf", leaf(size - 1, -np.inf))]
    return out


@gpu
@pytest.mark.parametrize("prioritized", [False, True])
def test_refused_banks_change_nothing(torch_cuda, prioritized):
    torch = torch_cuda
    from aigar_b200.replay import GpuReplayBuffer
    cap, L, AL = 1000, 5, 3
    mk = lambda: GpuReplayBuffer(cap, L, AL, prioritized, 0.6, 0.4)   # noqa: E731
    src, tgt = mk(), mk()
    d = Driver(torch, L, AL, 8)
    for _ in range(8):
        d.round(src)
    for _ in range(3):
        d.round(tgt)
    size = len(src)
    assert 10 < size < cap and len(tgt) != size
    good = src.snapshot()
    gh = good.cpu().numpy()
    before = tgt.snapshot()
    n0 = tgt.launch_count
    for name, edit in _corruptions(cap, L, AL, prioritized, size):
        h = gh.copy()
        edit(h)
        fresh = mk()
        fresh.restore(before)
        assert fresh.error_flags == 0, name
        fresh.restore(torch.from_numpy(h).cuda())
        assert torch.equal(fresh.snapshot(), before), name
        assert fresh.error_flags == rpl.ERR_STATE, name
        tgt.restore(torch.from_numpy(h).cuda())
        assert torch.equal(tgt.snapshot(), before), name
        assert len(tgt) == len(fresh) and tgt.next_idx == fresh.next_idx
    per_load = load_launches(cap, prioritized)
    n_cases = len(_corruptions(cap, L, AL, prioritized, size))
    assert tgt.launch_count - n0 == n_cases * (per_load + 1)   # each case: a load and a save
    tgt.restore(good)
    assert torch.equal(tgt.snapshot(), good) and len(tgt) == size
    u = torch.rand(64, dtype=torch.float64, device="cuda")
    for x, y in zip(tgt.sample(u), src.sample(u)):
        assert torch.equal(x, y)


@gpu
@pytest.mark.parametrize("alpha", [0.0, 0.6, 1.0, 2.5])
def test_reachable_states_load(torch_cuda, alpha):
    """Long random sequences with edge priorities: every state the live buffer reaches saves and loads without a flag."""
    torch = torch_cuda
    from aigar_b200.replay import GpuReplayBuffer
    for prioritized, cap, L in ((True, 700, 4), (True, 64, 2), (False, 300, 3)):
        a = GpuReplayBuffer(cap, L, 2, prioritized, alpha, 0.4)
        d = Driver(torch, L, 2, int(alpha * 10) + cap, edge=True)
        for r in range(60):
            d.round(a, n=3 * cap if r == 30 else None)
            if r % 10 == 9:
                b = GpuReplayBuffer(cap, L, 2, prioritized, alpha, 0.4)
                bank = a.snapshot()
                b.restore(bank)
                a.restore(bank.clone())
                assert b.error_flags == 0 and not (a.error_flags & rpl.ERR_STATE)
                assert torch.equal(b.snapshot(), bank)


@gpu
def test_host_refusals(torch_cuda):
    torch = torch_cuda
    from aigar_b200.replay import GpuReplayBuffer
    cap, L, AL = 100, 5, 3
    rp = GpuReplayBuffer(cap, L, AL, True, 0.6, 0.4)
    Driver(torch, L, AL, 1).round(rp, n=60)
    before = rp.snapshot()
    n0 = rp.launch_count
    vp = ctypes.c_void_p
    save = rp.lib.agar_replay_save
    load = rp.lib.agar_replay_load
    bank = torch.zeros(rp.state_bytes + 64, dtype=torch.uint8, device=rp.device)
    p, s = bank.data_ptr(), rp._stream()
    # the device pointers at the start of the handle (struct ReplayDev in csrc/agar_replay.cu): obs_t, obs_tp1, action,
    # reward, done, sum, mn, counters, max_priority, pos.  Every address named lies inside the buffer's own allocations, so
    # a regression of the check could not touch memory the test does not own.
    own = ctypes.cast(rp.h, ctypes.POINTER(ctypes.c_uint64))
    allocs = [int(own[i]) for i in range(10)]
    cases = [save(rp.h, None, s), load(rp.h, None, s), save(rp.h, vp(p + 8), s), load(rp.h, vp(p + 1), s)]
    for k, a in enumerate(allocs):
        cases += [save(rp.h, vp(a + (16 if k < 7 else 0)), s), load(rp.h, vp(a), s)]
    # a bank that starts before an allocation and runs into it
    cases.append(load(rp.h, vp(allocs[5] - (rp.state_bytes // 16 * 16 - 16)), s))
    assert cases == [-1] * len(cases)
    assert rp.lib.agar_replay_last_error(rp.h).decode().startswith("agar_replay_")
    assert rp.launch_count == n0
    assert torch.equal(rp.snapshot(), before) and rp.error_flags & rpl.ERR_STATE == 0
    strided = torch.zeros(2 * rp.state_bytes, dtype=torch.uint8, device=rp.device)[::2]
    for bad in (bank[:-64].to(torch.int8), bank[:-65], strided, bank[:-64].cpu(), bank[:-64].view(1, -1)):
        with pytest.raises(ValueError):
            rp.restore(bad)
        with pytest.raises(ValueError):
            rp.snapshot(out=bad)
    assert rp.launch_count == n0 + 1


@gpu
def test_restore_and_sample_in_a_cuda_graph(torch_cuda):
    torch = torch_cuda
    from aigar_b200.replay import GpuReplayBuffer
    cap, L, AL = 5000, 6, 2
    a, c = GpuReplayBuffer(cap, L, AL, True, 0.6, 0.4), GpuReplayBuffer(cap, L, AL, True, 0.6, 0.4)
    d = Driver(torch, L, AL, 4)
    for _ in range(10):
        d.round(a)
    bank = a.snapshot()
    u = torch.rand(512, dtype=torch.float64, device="cuda")
    want = a.sample(u)
    c.restore(bank)                            # warm-up: binds the calls before capture
    c.sample(u)
    for _ in range(5):
        d.round(c)
    graph = torch.cuda.CUDAGraph()
    n0 = c.launch_count
    with torch.cuda.graph(graph):
        c.restore(bank)
        got = c.sample(u)
    assert c.launch_count == n0 + load_launches(cap, True) + 2 == n0 + 6   # 13 tree levels: 2 rebuild launches; sample: 2
    for _ in range(2):
        d.round(c)
        graph.replay()
        torch.cuda.synchronize()
        for x, y in zip(got, want):
            assert torch.equal(x, y)
    # a graph that captured sample() sees a restore made between its replays
    g2 = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g2):
        got2 = c.sample(u)
    d.round(a)
    bank2 = a.snapshot()
    want2 = a.sample(u)
    c.restore(bank2)
    g2.replay()
    torch.cuda.synchronize()
    for x, y in zip(got2, want2):
        assert torch.equal(x, y)
    assert c.error_flags & rpl.ERR_STATE == 0


@gpu
def test_bank_larger_than_4_gib(torch_cuda):
    torch = torch_cuda
    from aigar_b200.replay import GpuReplayBuffer
    cap, L, AL = 1 << 20, 1024, 4
    a = GpuReplayBuffer(cap, L, AL, True, 0.6, 0.4)
    assert a.state_bytes > 8 << 30
    g = torch.Generator(device="cuda").manual_seed(0)
    chunk = 1 << 16
    obs = torch.rand((chunk, L), device="cuda", generator=g)
    act = torch.rand((chunk, AL), device="cuda", generator=g)
    done = torch.zeros(chunk, dtype=torch.uint8, device="cuda")
    n = 0
    for k in range(16):
        m = chunk - (1000 if k == 15 else 0)   # not full: the zeroed tail lies past 4 GiB in each ring section
        rew = torch.full((m,), float(k), device="cuda")
        a.add_batch(obs[:m] + k, act[:m], rew, obs[:m] - k, done[:m])
        n += m
    assert len(a) == n == cap - 1000
    a.update_priorities(torch.tensor([0, n - 1, n // 2], dtype=torch.int32, device="cuda"),
                        torch.tensor([3.0, 0.5, 7.0], dtype=torch.float64, device="cuda"))
    bank = a.snapshot()
    b = GpuReplayBuffer(cap, L, AL, True, 0.6, 0.4)
    b.restore(bank)
    assert torch.equal(b.snapshot(), bank)
    del bank
    idx = torch.tensor([0, 1, n // 2, n - 2, n - 1], dtype=torch.int32, device="cuda")
    for x, y in zip(a.gather(idx), b.gather(idx)):
        assert torch.equal(x, y)
    tail = b.gather(idx[-1:])
    assert torch.equal(tail[0][0], obs[m - 1] + 15) and torch.equal(tail[3][0], obs[m - 1] - 15)
    u = torch.rand(4096, dtype=torch.float64, device="cuda", generator=g)
    for x, y in zip(a.sample(u), b.sample(u)):
        assert torch.equal(x, y)
    assert a.error_flags == 0 and b.error_flags == 0


# ---- checkpoint files
FIELDS = dict(capacity=37, state_len=5, action_len=3, prioritized=True, alpha=0.6, beta=0.4)


def _rewrite(src, dst, **changes):
    with np.load(src, allow_pickle=False) as z:
        d = {k: z[k] for k in z.files}
    d.update(changes)
    for k in [k for k, v in changes.items() if v is None]:
        del d[k]
    with open(dst, "wb") as f:
        np.savez(f, **d)
    return dst


def _mismatched_files(tmp_path, good, bank, f=FIELDS):
    """(file, word its refusal must name) for each field a load checks"""
    out = []
    for name, value in (("capacity", f["capacity"] + 1), ("state_len", f["state_len"] - 1), ("action_len", 4),
                        ("prioritized", not f["prioritized"]), ("alpha", np.nextafter(f["alpha"], 1)), ("beta", 0.5)):
        p = str(tmp_path / ("bad_%s.npz" % name))
        rpl.write_replay_checkpoint(p, **dict(f, **{name: value}), bank=bank)
        out.append((p, name))
    p = str(tmp_path / "bad_bank.npz")
    rpl.write_replay_checkpoint(p, **f, bank=bank[:-256])
    out.append((p, "bank has"))
    out.append((_rewrite(good, str(tmp_path / "bad_format.npz"), format=np.array("agar_b200.records.v1")), "format"))
    tampered = bank.copy()
    tampered[300] ^= 1
    out.append((_rewrite(good, str(tmp_path / "bad_digest.npz"), bank=tampered), "sha256"))
    out.append((_rewrite(good, str(tmp_path / "no_beta.npz"), beta=None), "missing beta"))
    out.append((_rewrite(good, str(tmp_path / "bank_2d.npz"), bank=bank.reshape(-1, 16)), "1-D"))
    return out


def test_checkpoint_file_checks_without_a_device(tmp_path):
    """Parsing and matching a replay checkpoint needs no GPU: a stand-in writes the files."""
    bank = np.random.default_rng(0).integers(0, 256, 4096, dtype=np.uint8)
    good = str(tmp_path / "rp")                    # no .npz suffix: the file is written under exactly this name
    rpl.write_replay_checkpoint(good, **FIELDS, bank=bank)
    ck = rpl.read_replay_checkpoint(good)
    rpl.check_replay_checkpoint(ck, *FIELDS.values(), state_bytes=bank.size)
    assert str(ck["format"]) == rpl.REPLAY_CHECKPOINT_FORMAT == "agar_b200.replay.v1"
    assert np.array_equal(ck["bank"], bank)
    import hashlib
    assert str(ck["sha256"]) == hashlib.sha256(bank.tobytes()).hexdigest()
    for path, word in _mismatched_files(tmp_path, good, bank):
        with pytest.raises(rpl.CheckpointError, match=word):
            rpl.check_replay_checkpoint(rpl.read_replay_checkpoint(path), *FIELDS.values(), state_bytes=bank.size)
    from aigar_b200 import env as agar_env
    with pytest.raises(rpl.CheckpointError, match="not a records checkpoint"):   # the two kinds are not confused
        agar_env.read_checkpoint(good)


def test_error_bit_matches_the_header():
    import os
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = open(os.path.join(root, "include", "agar_replay.h")).read()
    assert int(re.search(r"AGAR_RP_ERR_STATE = (\d+)", src).group(1)) == rpl.ERR_STATE
    fields = re.search(r"typedef struct AgarReplayStateHeader \{(.*?)\}", src, re.S).group(1)
    names = re.findall(r"(\w+)[,;]", re.sub(r"/\*.*?\*/", "", fields))
    assert names == list(HEADER.names)


@gpu
def test_checkpoint_round_trip_and_refusals(torch_cuda, tmp_path):
    torch = torch_cuda
    from aigar_b200.replay import GpuReplayBuffer
    f = FIELDS
    a = GpuReplayBuffer(f["capacity"], f["state_len"], f["action_len"], f["prioritized"], f["alpha"], f["beta"])
    d = Driver(torch, f["state_len"], f["action_len"], 2)
    for _ in range(5):
        d.round(a)
    path = str(tmp_path / "replay.npz")
    a.save_checkpoint(path)
    b = GpuReplayBuffer.from_checkpoint(path)
    assert (b.size_max, b.state_len, b.action_len, b.prioritized, b.alpha, b.beta) == tuple(f.values())
    assert torch.equal(a.snapshot(), b.snapshot())
    u = torch.rand(64, dtype=torch.float64, device="cuda")
    for x, y in zip(a.sample(u), b.sample(u)):
        assert torch.equal(x, y)
    bank = a.snapshot().cpu().numpy()
    d.round(b)
    changed = b.snapshot()
    for p, word in _mismatched_files(tmp_path, path, bank):
        with pytest.raises(rpl.CheckpointError, match=word):
            b.load_checkpoint(p)
        assert torch.equal(b.snapshot(), changed), word
    # a file with a valid digest whose bank the device refuses: nothing is loaded, also once the sticky bit is set
    corrupt = bank.copy()
    corrupt[:HEADER.itemsize].view(HEADER)["size"] = f["capacity"] + 1
    bad = str(tmp_path / "bad_size.npz")
    rpl.write_replay_checkpoint(bad, **f, bank=corrupt)
    for _ in range(2):
        with pytest.raises(rpl.CheckpointError, match="device-side"):
            b.load_checkpoint(bad)
        assert torch.equal(b.snapshot(), changed)
    assert b.error_flags & rpl.ERR_STATE
    b.load_checkpoint(path)
    assert torch.equal(b.snapshot(), a.snapshot())


# ---- a training run resumes bit for bit
def _train(torch, env, drv, learner, rp, g, n_ticks, batch=256):
    """The un-graphed prioritized DQN tick of examples/train_dqn.py: decide -> step_observe -> add_batch -> sample with the
    generator's uniforms -> learn -> update_priorities."""
    import aigar_b200.layout as lay
    obs = env.obs.clone()
    for _ in range(n_ticks):
        acts = drv.decide()
        idx = drv.last_idx.float().unsqueeze(-1)
        nxt = env.step_observe(acts, env.cfg.frame_skip + 1)
        rp.add_batch(obs, idx, env.get(lay.GET_REWARD), nxt, env.get(lay.GET_DONE), env.get(lay.GET_VALID))
        obs = nxt.clone()
        s, a, r, s2, dn, w, ix = rp.sample(torch.rand(batch, dtype=torch.float64, device=env.device, generator=g))
        td, _ = learner.learn(s, a.squeeze(1), r, s2, dn, w.float())
        rp.update_priorities(ix, td.abs().double() + 1e-4)


def _setup(torch, cap):
    import aigar_b200.layout as lay
    from aigar_b200.dqn import DQNDriver, make_dqn
    from aigar_b200.env import AgarBatch
    from aigar_b200.learner import DQNLearner
    from aigar_b200.replay import GpuReplayBuffer
    env = AgarBatch(lay.derive_config(), 1024, seed=6)
    net = make_dqn(env.layout.state_len, device=env.device, seed=0)
    drv = DQNDriver(env, net=net, epsilon=0.3, seed=2)
    learner = DQNLearner(net, target_network_steps=7)
    rp = GpuReplayBuffer(cap, env.layout.state_len, 1, prioritized=True, alpha=0.6, beta=0.4)
    g = torch.Generator(device=env.device).manual_seed(1)
    return env, drv, learner, rp, g


@gpu
def test_training_run_resumes_bit_for_bit(torch_cuda, tmp_path):
    torch = torch_cuda
    N, cap = 12, 1 << 14                           # 1024 envs x 24 ticks wrap the ring
    env, drv, learner, rp, g = _setup(torch, cap)
    env.observe()
    _train(torch, env, drv, learner, rp, g, 2 * N)
    full = (env.state_tensor().clone(), rp.snapshot(), [p.detach().clone() for p in learner.net.parameters()],
            [p.detach().clone() for p in learner.target.parameters()])
    del env, drv, learner, rp, g

    env, drv, learner, rp, g = _setup(torch, cap)
    env.observe()
    _train(torch, env, drv, learner, rp, g, N)
    env.save_checkpoint(str(tmp_path / "env.npz"))
    rp.save_checkpoint(str(tmp_path / "replay.npz"))
    torch.save({"obs": env.obs.cpu(), "net": learner.net.state_dict(), "target": learner.target.state_dict(),
                "opt": learner.opt.state_dict(), "step": learner.step, "sample_gen": g.get_state(),
                "driver_gen": drv.gen.get_state()}, str(tmp_path / "learner.pt"))
    del env, drv, learner, rp, g
    torch.cuda.synchronize()

    from aigar_b200.dqn import DQNDriver, make_dqn
    from aigar_b200.env import AgarBatch
    from aigar_b200.learner import DQNLearner
    from aigar_b200.replay import GpuReplayBuffer
    env = AgarBatch.from_checkpoint(str(tmp_path / "env.npz"))
    rp = GpuReplayBuffer.from_checkpoint(str(tmp_path / "replay.npz"))
    st = torch.load(str(tmp_path / "learner.pt"))
    env.obs.copy_(st["obs"])
    net = make_dqn(env.layout.state_len, device=env.device, seed=123)   # another init: everything comes from the files
    net.load_state_dict(st["net"])
    drv = DQNDriver(env, net=net, epsilon=0.3, seed=77)
    drv.gen.set_state(st["driver_gen"])
    learner = DQNLearner(net, target_network_steps=7)
    learner.target.load_state_dict(st["target"])
    learner.opt.load_state_dict(st["opt"])
    learner.step = st["step"]
    g = torch.Generator(device=env.device)
    g.set_state(st["sample_gen"])
    _train(torch, env, drv, learner, rp, g, N)
    assert learner.step == 2 * N and learner.step // 7 > N // 7   # a target sync happens after the resume
    assert torch.equal(env.state_tensor(), full[0])
    assert torch.equal(rp.snapshot(), full[1])
    for x, y in zip(learner.net.parameters(), full[2]):
        assert torch.equal(x, y)
    for x, y in zip(learner.target.parameters(), full[3]):
        assert torch.equal(x, y)
    assert rp.error_flags & rpl.ERR_STATE == 0
