"""Terminal observations on the host-buffer step (``step_host()`` of a ``final_observation=True`` env,
``dexsim_step_host_final``).

Three twins take the same seed and actions: A steps with ``step()`` and final observations (the device-path yardstick,
``dexsim_step_final``), B with ``step_host()`` and final observations, C with plain ``step_host()``.  B must return what A
returns -- observation, reward, flags, contact counts, ``finished`` and, where finished, the final observation bit for
bit -- and what C returns; at the end all three hold the same state and counters.  The cases cover both host transports
(the copies and the zero-copy launch), one and several chunks, the fold rule, both tile widths, counts-only and full
tracking, both respawn modes, a loop bound, asynchronous calls on two slots and the primed static rows."""
import ctypes as C

import numpy as np
import pytest
import torch

import dexterous_rl_manipulation_b200 as dx
from dexterous_rl_manipulation_b200 import _lib

STATE = ("_obs", "_op64", "_thr", "_damp", "_step_count", "_cmask", "_size", "_mass", "_friction", "_episode",
         "_ep_return", "_ep_stats")
MAX_STEPS = 12


@pytest.fixture(scope="module")
def gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda")


def _kwargs(track, respawn, loop, seed=13):
    CC = dx.CurriculumConfig
    return dict(max_episode_steps=MAX_STEPS, reward_type="dense", respawn=respawn, loop_max_steps=loop,
                track_episodes=track, seed=seed, groups=[CC.easy(), CC.medium(), CC.hard()], auto_reset=True)


def _twins(n, track, respawn, loop, zero_copy="auto"):
    kw = _kwargs(track, respawn, loop)
    a = dx.BatchedManipulationEnv(n, "cuda", final_observation=True, **kw)
    b = dx.BatchedManipulationEnv(n, "cuda", final_observation=True, **kw)
    c = dx.BatchedManipulationEnv(n, "cuda", **kw)
    for e in (a, b, c):
        if loop:
            e._params.success_threshold = 6              # five fingers: the loop bound, not a success, ends episodes
        e.host_zero_copy = zero_copy
        e.reset(seed=13)
    return a, b, c


def _contact_mask(obs_dev):
    rows = obs_dev[:, 40:45].to(torch.uint8)
    return sum(rows[:, f] << f for f in range(5)).to(torch.uint8)


def _same_state(a, b, n):
    for k in STATE:
        x, y = getattr(a, k), getattr(b, k)
        assert (x is None and y is None) or torch.equal(x[..., :n], y[..., :n]), k
    assert torch.equal(a.counters, b.counters)
    torch.testing.assert_close(a.ret_sums, b.ret_sums, rtol=1e-9, atol=0.0)


# (n, chunks, full tracking, respawn, loop_max_steps, host_zero_copy, zero-copy steps expected)
CASES = [
    (100, None, False, True, 0, "auto", False),              # register kernel, one chunk
    (3122, 4, True, False, 0, "auto", True),                 # zero-copy: the 50-env last chunk folds into its neighbour
    (5000, 3, False, True, 5, "auto", True),                 # loop bound below the episode limit
    (70001, None, True, True, 0, "auto", True),              # zero-copy, narrow tile, ragged
    (131072, None, False, False, 0, "auto", True),           # zero-copy, wide tile
    (70001, None, False, True, 0, False, False),             # zero-copy forced off at a zero-copy size
    (300007, 8, False, True, 0, "auto", False),              # copy transport, eight chunks
]


@pytest.mark.gpu
@pytest.mark.parametrize("n,chunks,track,respawn,loop,zero_copy,zc_expected", CASES)
def test_step_host_final_matches_device_path(gpu, n, chunks, track, respawn, loop, zero_copy, zc_expected):
    a, b, c = _twins(n, track, respawn, loop, zero_copy)
    rng = np.random.default_rng(n)
    finished_total = 0
    for t in range(3 * MAX_STEPS + 2):
        act = rng.uniform(-1, 1, (n, 15)).astype(np.float32)
        oa, ra, ta, ua, ia = a.step(torch.from_numpy(act).cuda())
        zc0 = _lib.lib().dexsim_host_zero_copy_steps()
        ob, rb, tb, ub, ib = b.step_host(act, chunks=chunks)
        zc_used = _lib.lib().dexsim_host_zero_copy_steps() - zc0
        oc, rc, tc, uc, ic = c.step_host(act, chunks=chunks)
        # the first call primes the pinned observation; from then on sizes up to 160K take the zero-copy launch
        assert zc_used == (1 if zc_expected and t > 0 else 0), t
        fin = ia["finished"].cpu()
        assert torch.equal(ob, oa.cpu()) and torch.equal(rb, ra.cpu()), t
        assert torch.equal(tb, ta.cpu()) and torch.equal(ub, ua.cpu()), t
        assert torch.equal(ib["num_contacts"], ia["num_contacts"].cpu()), t
        assert torch.equal(ib["contact_mask"], _contact_mask(oa).cpu()), t
        assert torch.equal(ib["finished"], fin), t
        assert torch.equal(ib["final_observation"][fin], ia["final_observation"][fin.cuda()].cpu()), t
        for x, y in zip((ob, rb, tb, ub, ib["num_contacts"], ib["contact_mask"]),
                        (oc, rc, tc, uc, ic["num_contacts"], ic["contact_mask"])):
            assert torch.equal(x, y), t
        finished_total += int(fin.sum())
    assert finished_total > n                                    # several reset waves went through
    assert b._h_primed_slot == 0                                 # ... with the static rows carried, not re-downloaded
    _same_state(a, b, n)
    _same_state(b, c, n)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [5000, 70001])
def test_async_two_slots_packed_contacts(gpu, n):
    """sync=False on alternating slots with packed contacts: each slot's results (and its final observations) are
    valid after host_sync(), and the other slot's are not overwritten by it."""
    a, b, _ = _twins(n, False, True, 0)
    rng = np.random.default_rng(7)
    prev = None
    for t in range(3 * MAX_STEPS):
        act = rng.uniform(-1, 1, (n, 15)).astype(np.float32)
        oa, ra, ta, ua, ia = a.step(torch.from_numpy(act).cuda())
        fin = ia["finished"].cpu()
        want = (oa.cpu(), ra.cpu(), ta.cpu(), ua.cpu(), _contact_mask(oa).cpu(), fin,
                ia["final_observation"][fin.cuda()].cpu())
        slot = t % 2
        ob, rb, tb, ub, ib = b.step_host(act, chunks=3, sync=False, packed_contacts=True, slot=slot)
        b.host_sync()
        got = (ob[:, :40], rb, tb, ub, ib["contact_mask"], ib["finished"], ib["final_observation"][ib["finished"]])
        assert torch.equal(got[0], want[0][:, :40]), t
        for x, y in zip(got[1:], want[1:]):
            assert torch.equal(x, y), t
        if prev is not None:                                     # the other slot still holds the previous step
            pslot, pwant = prev
            pb = b._host_buffers(pslot)
            assert torch.equal(pb["fin"][:n].view(torch.bool), pwant[5]), t
            assert torch.equal(pb["final"][pwant[5]], pwant[6]), t
        prev = (slot, want)
    _same_state(a, b, n)


@pytest.mark.gpu
@pytest.mark.parametrize("n,zero_copy", [(4096 + 77, "auto"), (4096 + 77, False), (300007, "auto")])
def test_only_finished_rows_are_written(gpu, n, zero_copy):
    """The final buffer pre-filled with NaN before every step: exactly the rows of finished envs change."""
    _, b, _ = _twins(n, True, True, 0, zero_copy)
    rng = np.random.default_rng(3)
    final = b._host_buffers(0)["final"]
    seen = 0
    for t in range(2 * MAX_STEPS):
        final.fill_(float("nan"))
        _, _, _, _, ib = b.step_host(rng.uniform(-1, 1, (n, 15)).astype(np.float32), chunks=4)
        fin = ib["finished"]
        assert not bool(torch.isnan(final[fin]).any()), t
        assert bool(torch.isnan(final[~fin]).all()), t
        seen += int(fin.sum())
    assert 0 < seen


@pytest.mark.gpu
@pytest.mark.parametrize("n,chunks", [(1 << 20, 8), (131072, None)])
def test_truncation_wave(gpu, n, chunks):
    """Every episode truncates on the same step (no episode can succeed): every row of the final observation is written
    and equals the device path's."""
    T = 6
    CC = dx.CurriculumConfig
    kw = dict(max_episode_steps=T, reward_type="dense", respawn=True, track_episodes=False, seed=21,
              curriculum_config=CC.hard(), auto_reset=True, final_observation=True)
    a, b = dx.BatchedManipulationEnv(n, "cuda", **kw), dx.BatchedManipulationEnv(n, "cuda", **kw)
    for e in (a, b):
        e._params.success_threshold = 6
        e.reset(seed=21)
    final = b._host_buffers(0)["final"]
    final.fill_(float("nan"))
    gen = torch.Generator(device="cuda").manual_seed(1)
    waves = 0
    for t in range(2 * T + 3):
        act = torch.rand(n, 15, device="cuda", generator=gen) * 2 - 1
        oa, _, _, _, ia = a.step(act)
        ob, _, _, _, ib = b.step_host(act.cpu(), chunks=chunks)
        assert torch.equal(ib["finished"], ia["finished"].cpu()), t
        assert int(ib["finished"].sum()) in (0, n), t
        if bool(ib["finished"][0]):
            waves += 1
            assert torch.equal(final, ia["final_observation"].cpu()), t       # NaN-free and bit-equal
            final.fill_(float("nan"))
        assert torch.equal(ob, oa.cpu()), t
    assert waves == 2
    _same_state(a, b, n)


def test_host_final_argument_errors_without_gpu():
    """Each documented error of dexsim_step_host_final comes back before the device is touched (no GPU needed)."""
    L = _lib.lib()
    assert _lib.ABI_VERSION == 5 and L.dexsim_version() == 5
    assert "dexsim_step_host_final" in _lib.EXPORTS
    buf = (C.c_char * 256)()
    ptr = (C.addressof(buf) + 15) & ~15                     # non-NULL, 16-byte aligned, never dereferenced
    st = _lib.DexsimState()
    st.n, st.ld = 0, 32
    for name, _ in _lib.DexsimState._fields_[2:12]:
        setattr(st, name, ptr)
    p = _lib.DexsimParams()
    p.reward_type, p.success_threshold, p.num_groups, p.max_episode_steps, p.auto_reset = 1, 3, 1, 200, 1
    io = _lib.DexsimStepIO()
    io.action = io.reward = io.terminated = io.truncated = io.num_contacts = io.finished = ptr

    def call(fin=ptr, final=ptr):
        return L.dexsim_step_host_final(C.byref(st), C.byref(p), ptr, None, C.byref(io), ptr, ptr, ptr, ptr, ptr, ptr,
                                        ptr, fin, final, 1, 0, None)

    assert call() == -1004                                  # DEXSIM_E_PARAM: ordinary memory is not mapped page-locked
    p.auto_reset = 0
    assert call() == -1004                                  # DEXSIM_E_PARAM: no auto-reset
    p.auto_reset = 1
    io.sigma_obs = 0.05
    assert call() == -1004                                  # DEXSIM_E_PARAM: noise
    io.sigma_obs = 0.0
    assert call(fin=None) == -1001                          # DEXSIM_E_NULL: no finished buffer
    assert call(final=None) == -1001                        # DEXSIM_E_NULL: no final buffer
    io.finished = None
    assert call() == -1001                                  # DEXSIM_E_NULL: no device finished flags
