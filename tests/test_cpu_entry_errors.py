"""The error codes of the step entry points for bad arguments, alone and in pairs (no GPU needed).

Every call below is refused, or accepted with n == 0, before the library touches the device.  Where two bad arguments
coincide, the order of an entry point's checks decides which code it returns; the table pins that order.
"""
import ctypes as C
import itertools

from dexterous_rl_manipulation_b200 import _lib

ENTRIES = ("dexsim_step", "dexsim_step_single", "dexsim_step_final", "dexsim_step_next_reset", "dexsim_step_host",
           "dexsim_step_host_final", "dexsim_pack_env", "dexsim_pack_env_tagged")

# One bad argument each: a name and what it does to the call's arguments (a dict, see `call`).
BAD = {
    "st": lambda a: a.update(st=None),
    "p": lambda a: a.update(p=None),
    "io": lambda a: a.update(io=None),
    "n": lambda a: setattr(a["st_s"], "n", -1),
    "ld": lambda a: setattr(a["st_s"], "ld", 48),
    "auto": lambda a: setattr(a["p_s"], "auto_reset", 0),
    "fin": lambda a: setattr(a["io_s"], "finished", None),
    "final": lambda a: a.update(final=None),
    "hfin": lambda a: a.update(h_finished=None),
    "host": lambda a: a.update(host=None),                  # h_action of the host steps, out64 of the others
    "hsr": lambda a: setattr(a["io_s"], "host_static_rows", a["ptr"]),
    "layout": lambda a: setattr(a["io_s"], "action_layout", 2),
    "g0": lambda a: setattr(a["p_s"], "num_groups", 0),
    "g257": lambda a: setattr(a["p_s"], "num_groups", 257),
    "long": lambda a: (setattr(a["st_s"], "ep_return", a["ptr"]), setattr(a["st_s"], "ep_stats", a["ptr"]),
                       setattr(a["p_s"], "max_episode_steps", 5242)),   # tracked episodes of 5,243 steps
}

# `case: codes` with one letter per entry point in ENTRIES order: . ok, N NULL, S size, P param, G groups.
EXPECTED = """
none: .S...PSS
st: NNNNNNNN
p: NNNNNNSS
io: NNNNNNNN
n: SSSSSSSS
ld: SSSSSSSS
auto: .SPP.PSS
fin: .SNN.NSS
final: .SN..NSS
hfin: .S...NSS
host: .N..NNNN
hsr: .SPP.PSS
layout: PPPP.PSS
g0: GSGG.GSS
g257: GSGG.GSS
long: PSPP.PSS
st+p: NNNNNNNN
st+io: NNNNNNNN
st+n: NNNNNNNN
st+ld: NNNNNNNN
st+auto: NNPPNPNN
st+fin: NNNNNNNN
st+final: NNNNNNNN
st+hfin: NNNNNNNN
st+host: NNNNNNNN
st+hsr: NNPPNNNN
st+layout: NNNNNNNN
st+g0: NNNNNNNN
st+g257: NNNNNNNN
st+long: NNNNNNNN
p+io: NNNNNNNN
p+n: NNNNSNSS
p+ld: NNNNSNSS
p+auto: NNNNNNSS
p+fin: NNNNNNSS
p+final: NNNNNNSS
p+hfin: NNNNNNSS
p+host: NNNNNNNN
p+hsr: NNNNNNSS
p+layout: NNNNNNSS
p+g0: NNNNNNSS
p+g257: NNNNNNSS
p+long: NNNNNNSS
io+n: SSNNSNSS
io+ld: SSNNSNSS
io+auto: NNNNNNNN
io+fin: NNNNNNNN
io+final: NNNNNNNN
io+hfin: NNNNNNNN
io+host: NNNNNNNN
io+hsr: NNNNNNNN
io+layout: NNNNNNNN
io+g0: NNNNNNNN
io+g257: NNNNNNNN
io+long: NNNNNNNN
n+ld: SSSSSSSS
n+auto: SSPPSPSS
n+fin: SSNNSNSS
n+final: SSNSSNSS
n+hfin: SSSSSNSS
n+host: SNSSSSSS
n+hsr: SSPPSSSS
n+layout: SSSSSSSS
n+g0: SSSSSSSS
n+g257: SSSSSSSS
n+long: SSSSSSSS
ld+auto: SSPPSPSS
ld+fin: SSNNSNSS
ld+final: SSNSSNSS
ld+hfin: SSSSSNSS
ld+host: SNSSSSSS
ld+hsr: SSPPSSSS
ld+layout: SSSSSSSS
ld+g0: SSSSSSSS
ld+g257: SSSSSSSS
ld+long: SSSSSSSS
auto+fin: .SPP.PSS
auto+final: .SPP.PSS
auto+hfin: .SPP.PSS
auto+host: .NPPNPNN
auto+hsr: .SPP.PSS
auto+layout: PPPP.PSS
auto+g0: .SPP.PSS
auto+g257: .SPP.PSS
auto+long: .SPP.PSS
fin+final: .SNN.NSS
fin+hfin: .SNN.NSS
fin+host: .NNNNNNN
fin+hsr: .SPP.NSS
fin+layout: PPNN.NSS
fin+g0: GSNN.NSS
fin+g257: GSNN.NSS
fin+long: PSNN.NSS
final+hfin: .SN..NSS
final+host: .NN.NNNN
final+hsr: .SPP.NSS
final+layout: PPNP.NSS
final+g0: GSNG.NSS
final+g257: GSNG.NSS
final+long: PSNP.NSS
hfin+host: .N..NNNN
hfin+hsr: .SPP.NSS
hfin+layout: PPPP.NSS
hfin+g0: GSGG.NSS
hfin+g257: GSGG.NSS
hfin+long: PSPP.NSS
host+hsr: .NPPNNNN
host+layout: PNPPNNNN
host+g0: GNGGNGNN
host+g257: GNGGNGNN
host+long: PNPPNPNN
hsr+layout: PPPP.PSS
hsr+g0: GSPP.GSS
hsr+g257: GSPP.GSS
hsr+long: PSPP.PSS
layout+g0: PPGP.GSS
layout+g257: PPGP.GSS
layout+long: PPPP.PSS
g0+g257: GSGG.GSS
g0+long: PSPP.PSS
g257+long: PSPP.PSS
"""

LETTER = {0: ".", -1001: "N", -1002: "S", -1004: "P", -1005: "G"}


def call(L, name, bad):
    """`name` with valid arguments for n == 0, an auto-reset env and ordinary (not mapped) host memory, after `bad`."""
    buf = (C.c_char * 256)()
    ptr = (C.addressof(buf) + 15) & ~15                     # non-NULL, 16-byte aligned, never dereferenced
    st = _lib.DexsimState()
    st.n, st.ld = 0, 32
    for field, _ in _lib.DexsimState._fields_[2:12]:
        setattr(st, field, ptr)
    p = _lib.DexsimParams()
    p.reward_type, p.success_threshold, p.num_groups, p.max_episode_steps, p.auto_reset = 1, 3, 1, 200, 1
    io = _lib.DexsimStepIO()
    io.action = io.reward = io.terminated = io.truncated = io.num_contacts = io.finished = ptr
    io.action_layout = 1
    a = dict(st=C.byref(st), p=C.byref(p), io=C.byref(io), st_s=st, p_s=p, io_s=io, ptr=ptr, final=ptr, h_finished=ptr,
             host=ptr)
    for b in bad:
        BAD[b](a)
    head = (a["st"], a["p"], ptr, None, a["io"])
    host = (a["host"], ptr, ptr, ptr, ptr, ptr, ptr)          # h_action, h_obs, reward, flags, contacts, contact mask
    fn = getattr(L, name)
    if name == "dexsim_step":
        return fn(*head, None)
    if name == "dexsim_step_single":
        return fn(*head, a["host"], 1.0, None)
    if name == "dexsim_step_final":
        return fn(*head, a["final"], None)
    if name == "dexsim_step_next_reset":
        return fn(*head, None)
    if name == "dexsim_step_host":
        return fn(*head, *host, 1, 0, None)
    if name == "dexsim_step_host_final":
        return fn(*head, *host, a["h_finished"], a["final"], 1, 0, None)
    if name == "dexsim_pack_env":
        return fn(a["st"], a["io"], 0, 0, a["host"], None)
    return fn(a["st"], a["io"], 0, 0, a["host"], 1.0, None)


def cases():
    return [()] + [(b,) for b in BAD] + list(itertools.combinations(BAD, 2))


def table(L):
    return {"+".join(c) or "none": "".join(LETTER[call(L, e, c)] for e in ENTRIES) for c in cases()}


def test_step_entry_error_codes():
    expected = dict(line.split(": ") for line in EXPECTED.strip().splitlines())
    got = table(_lib.lib())
    assert list(got) == list(expected)
    wrong = {c: (got[c], expected[c]) for c in got if got[c] != expected[c]}
    assert not wrong, f"(got, expected) per case, entry points in the order {ENTRIES}: {wrong}"
