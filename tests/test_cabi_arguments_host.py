"""CPU test of the C ABI's argument rules: every env entry point, both host-buffer steps and the key derivation get
calls with exactly one faulty argument and must return that fault's MSAT_E* code before anything is enqueued.  The
"device" pointers are fake, suitably aligned addresses inside a host buffer; no kernel is launched."""
import ctypes as C
import functools

import pytest

import marl_sat_b200 as M
from marl_sat_b200 import _lib

EINVAL, EALIGN, EUNSUPPORTED, OK = _lib.MSAT_EINVAL, _lib.MSAT_EALIGN, _lib.MSAT_EUNSUPPORTED, _lib.MSAT_OK

_BUF = (C.c_char * 4096)()
A = (C.addressof(_BUF) + 127) // 128 * 128       # 128-byte aligned fake address; A + 64 holds a 40-byte chain
B = 4


@functools.lru_cache(maxsize=None)
def _env():
    return M.SATEnv(20, 91, 8, verbose=False, device="cpu")      # owns the plans: keep it alive


def plan(k):
    """uf20-91 plans: k = 3, and k = 16, one literal more than the clause-feature table covers."""
    return _env()._plan_for(k).handle


def _call(name, defaults, over):
    assert set(over) <= set(defaults), set(over) - set(defaults)
    args = {**defaults, **over}
    if isinstance(args.get("plan"), int) and args["plan"] < 100:     # a clause width: the plan for it
        args["plan"] = plan(args["plan"])
    return getattr(_lib.load(), name)(*args.values())


# Argument lists in the order of the C prototypes, each valid as given (so one override is one fault).
def reset(**o):
    return _call("msat_reset", dict(plan=3, bank=A, P=1, idx=A, keys=A, state=A, obs=A, B=B, stream=None), o)


def import_state(**o):
    return _call("msat_import_state", dict(plan=3, bank=A, P=1, idx=A, va=A, step=None, done=None, state=A, obs=A,
                                           B=B, stream=None), o)


def apply_start(**o):
    return _call("msat_apply_start_states", dict(plan=3, bank=A, P=1, state=A, rk=A, Bg=16, off=0, words=A, thr=A,
                                                 has=None, obs=A, ga=None, gc=None, B=B, stream=None), o)


def walksat(**o):
    return _call("msat_walksat", dict(plan=3, bank=A, P=1, state=A, keys=A, F=10, off=0, noise=0.5, solved=None,
                                      flips=None, B=B, stream=None), o)


_OUT = dict(reward=A, rcols=1, done=A, dcols=1, solved=None, nunsat=None, estep=None)


def step(**o):
    return _call("msat_step", dict(plan=3, bank=A, P=1, sin=A, sout=A, act=A, auto=1, idx=A, keys=A, obs=A, **_OUT,
                                   newly=None, B=B, stream=None), o)


def rollout_step(**o):
    return _call("msat_rollout_step", dict(plan=3, bank=A, P=1, sin=A, sout=A, act=A, rng=A, chain=A + 64, Bg=16,
                                           off=0, obs=A, **_OUT, B=B, stream=None), o)


def rollout_step_gnn(**o):
    return _call("msat_rollout_step_gnn", dict(plan=3, bank=A, P=1, sin=A, sout=A, act=A, rng=A, chain=A + 64, Bg=16,
                                               off=0, ga=A, gc=A, **_OUT, B=B, stream=None), o)


def rollout_steps(**o):
    return _call("msat_rollout_steps", dict(plan=3, bank=A, P=1, sin=A, sout=A, act=A, K=2, rng=A, chain=A + 64,
                                            Bg=16, off=0, obs=A, ga=None, gc=None, emit=0, **_OUT, newly=None, B=B,
                                            stream=None), o)


def get_obs(**o):
    return _call("msat_get_obs", dict(plan=3, bank=A, P=1, state=A, obs=A, B=B, stream=None), o)


def export_state(**o):
    outputs = {f"out{i}": None for i in range(10)}
    return _call("msat_export_state", dict(plan=3, bank=A, P=1, state=A, B=B, **outputs, stream=None), o)


def gnn_dynamic(**o):
    return _call("msat_gnn_dynamic", dict(plan=3, bank=A, P=1, state=A, B=B, ga=None, gc=None, stream=None), o)


def flip_gains(**o):
    return _call("msat_flip_gains", dict(plan=3, bank=A, P=1, state=A, B=B, tau=0.0, delta=None, labels=None,
                                         stream=None), o)


def env_keys(**o):
    return _call("msat_env_keys", dict(pk=A, rk=A, Bg=16, off=0, Bl=B, P=1, idx=A, keys=A, stream=None), o)


def env_keys_weighted(**o):
    return _call("msat_env_keys_weighted", dict(pk=A, rk=A, Bg=16, off=0, Bl=B, cum=A, P=1, idx=A, keys=A,
                                                stream=None), o)


_HOST = dict(plan=3, bank=A, P=1, state=A, ah=A, ad=A, rng=A, chain=A + 64, Bg=16, off=0, obs=A, **_OUT,
             rh=A, dh=A, sh=None, nh=None, eh=None, B=B, stream=None)


def step_host(**o):
    return _call("msat_rollout_step_host", _HOST, o)


def step_host_async(**o):
    return _call("msat_rollout_step_host_async", dict(pipe=None, slot=0, **_HOST), o)


def env_rule(fn, required, states, obs=True):
    """The rule every env entry point shares: plan, P > 0, B >= 0, the bank and the entry point's own required
    pointers (MSAT_EINVAL), then a 128-byte aligned bank and 16-byte aligned state and observations (MSAT_EALIGN)."""
    rows = [(fn, dict(plan=None), EINVAL), (fn, dict(P=0), EINVAL), (fn, dict(B=-1), EINVAL),
            (fn, dict(bank=None), EINVAL), (fn, dict(bank=A + 16), EALIGN)]
    rows += [(fn, {k: None}, EINVAL) for k in required]
    rows += [(fn, {k: A + 4}, EALIGN) for k in states + (["obs"] if obs else [])]
    return rows


def step_output_rule(fn):
    return [(fn, dict(rcols=0), EINVAL), (fn, dict(dcols=0), EINVAL)]


def shard_rule(fn):
    """[off, off + B) inside a global batch of Bg envs, Bg <= 2^30."""
    return [(fn, dict(off=14), EINVAL), (fn, dict(off=-1), EINVAL), (fn, dict(Bg=-1), EINVAL),
            (fn, dict(Bg=(1 << 30) + 1), EUNSUPPORTED)]


ROWS = (
    env_rule(reset, ["idx", "keys", "state"], ["state"])
    + env_rule(import_state, ["idx", "va", "state"], ["state"])
    + env_rule(get_obs, ["state", "obs"], ["state"])
    + env_rule(apply_start, ["state", "rk", "words", "thr"], ["state"]) + shard_rule(apply_start)
    + [(apply_start, dict(thr=A + 1), EALIGN), (apply_start, dict(gc=A + 2), EALIGN),
       (apply_start, dict(plan=16, gc=A), EUNSUPPORTED), (apply_start, dict(Bg=0, B=0), OK)]
    + env_rule(walksat, ["state", "keys"], ["state"], obs=False)
    + [(walksat, dict(noise=1.5), EINVAL), (walksat, dict(F=-1), EINVAL)]
    + env_rule(step, ["sin", "sout", "act", "idx", "keys"], ["sin", "sout"]) + step_output_rule(step)
    + [(step, dict(newly=A), EINVAL)]                      # newly_satisfied needs the shaped reward
    + [row for fn in (rollout_step, rollout_step_gnn, rollout_steps)
       for row in env_rule(fn, ["sin", "sout", "act", "rng", "chain"], ["sin", "sout"], obs=fn is not rollout_step_gnn)
       + step_output_rule(fn) + shard_rule(fn)
       + [(fn, dict(chain=A + 4), EINVAL), (fn, dict(Bg=0, B=0), EINVAL)]]
    + [(rollout_step_gnn, dict(plan=16), EUNSUPPORTED), (rollout_steps, dict(K=0), EINVAL),
       (rollout_steps, dict(K=65), EINVAL), (rollout_steps, dict(ga=A), EINVAL), (rollout_steps, dict(newly=A), EINVAL),
       (rollout_steps, dict(obs=None, gc=A, plan=16), EUNSUPPORTED)]
    + [row for fn in (export_state, gnn_dynamic, flip_gains)
       for row in [(fn, dict(plan=None), EINVAL), (fn, dict(P=0), EINVAL), (fn, dict(B=-1), EINVAL),
                   (fn, dict(bank=None), EINVAL), (fn, dict(state=None), EINVAL)]]
    + [row for fn in (env_keys, env_keys_weighted)
       for row in shard_rule(fn)
       + [(fn, dict(Bl=-1), EINVAL), (fn, dict(pk=None), EINVAL), (fn, dict(rk=None), EINVAL), (fn, dict(Bg=0, Bl=0), OK)]]
    + [(env_keys_weighted, dict(cum=None), EINVAL), (env_keys_weighted, dict(cum=A + 4), EALIGN)]
    # the host-buffer steps check the whole batch before they enqueue the action upload
    + [(step_host, dict(rng=None), EINVAL), (step_host, dict(off=14), EINVAL), (step_host, dict(rcols=0), EINVAL),
       (step_host, dict(chain=A + 4), EINVAL), (step_host, dict(ah=None), EINVAL), (step_host, dict(ad=None), EINVAL),
       (step_host, dict(plan=None), EINVAL), (step_host_async, dict(pipe=None), EINVAL)]
)


def _show(v):
    if v is None:
        return "NULL"
    return f"A+{v - A}" if isinstance(v, int) and A <= v < A + 4096 else str(v)


@pytest.mark.parametrize("fn,over,code", ROWS,
                         ids=[fn.__name__ + "-" + ",".join(f"{k}={_show(v)}" for k, v in o.items()) for fn, o, _ in ROWS])
def test_one_faulty_argument_gives_its_code(fn, over, code):
    assert fn(**over) == code
