"""Recorded calls of the unmodified RoBO reference into the robo_b200.compat shims, and their replay — TEST
INFRASTRUCTURE ONLY.

The reference's own classes reach the device path through two shims: ``george.GP`` (compat.GeorgeGP) and
``emcee.EnsembleSampler`` (robo_b200.util.ensemble_sampler).  ``Recorder`` logs every call the reference makes into
them while it runs (arguments, kernel parameters at the time of the call, answer); oracle/make_dropin_golden.py runs
the reference scenarios under it and stores the traces in tests/golden/dropin_*.npz.  ``replay`` issues the same calls
to the shims of the current tree and yields (recorded, replayed) answers, so the suite checks the shims against the
reference's call pattern without the reference tree.  Ensemble-sampler runs are replayed with the log-posterior values
the reference returned for each proposal: the sampler is deterministic given its random state, so it proposes the same
points and its chain must come out the same.

Size: a predict call on more than ``PREDICT_ROWS`` points is stored with a seeded subset of its rows (GP moments of a row
do not depend on the other rows, so the subset is a call of its own whose answers are the same rows of the answer), and
at most ``MAX_PREDICTS`` predict calls, evenly spaced, are kept per scenario; every other call is kept.

Storage: one ``.npz`` per scenario, no pickles: ``ops`` is a JSON list of the calls with scalars inline and each array
as [offset, shape] into ``data``, one float64 vector in which equal arrays are stored once."""
import json

import numpy as np

from robo_b200 import compat
from robo_b200.util import ensemble_sampler

GP_VERBS = ("compute", "log_likelihood", "predict")
PREDICT_ROWS = 16
MAX_PREDICTS = 120


class Recorder(object):
    """Context manager: patches the shim classes so that the reference's calls into them are logged into ``self.ops``."""

    def __init__(self, kernel_name):
        self.kernel_name = kernel_name
        self.ops = []
        self._depth = {}
        self._saved = []

    def _put(self, op, **arrays):
        op["arrays"] = {k: np.array(v, dtype=np.float64) for k, v in arrays.items() if v is not None}
        if op["op"] == "predict" and len(op["arrays"]["t"]) > PREDICT_ROWS:
            n = len(op["arrays"]["t"])
            rows = np.sort(np.random.RandomState(len(self.ops)).choice(n, PREDICT_ROWS, replace=False))
            for k, v in op["arrays"].items():
                if k == "t" or k.startswith("out"):
                    v = v[rows]
                    op["arrays"][k] = v[:, rows] if v.ndim == 2 and v.shape[1] == n else v
        self.ops.append(op)

    def log_calls(self, obj, *names):
        """Also log calls of ``obj``'s methods ``names`` (objects of the product that the reference drives directly):
        array arguments, keyword flags and the answer."""
        for name in names:
            def logged(*a, _name=name, _orig=getattr(obj, name), **kw):
                out = _orig(*a, **kw)
                arrays = {"arg%d" % j: v for j, v in enumerate(a) if isinstance(v, np.ndarray)}
                if isinstance(out, np.ndarray):
                    arrays["out"] = out
                self._put(dict(op=_name, kw=kw), **arrays)
                return out
            setattr(obj, name, logged)

    def _wrap(self, cls, name, log):
        orig = cls.__dict__[name]
        rec = self

        def wrapper(obj, *a, **kw):
            if rec._depth.get(cls):                # a shim calling itself: only the reference's calls are logged
                return orig(obj, *a, **kw)
            rec._depth[cls] = 1
            try:
                return log(orig, obj, *a, **kw)
            finally:
                rec._depth[cls] = 0
        self._saved.append((cls, name, orig))
        setattr(cls, name, wrapper)

    def __enter__(self):
        rec = self
        G, S = compat.GeorgeGP, ensemble_sampler.EnsembleSampler

        def gp_init(orig, gp, kernel, *a, **kw):
            orig(gp, kernel, *a, **kw)
            gp._trace_id = sum(op["op"] == "gp" for op in rec.ops)
            rec.ops.append(dict(op="gp", gp=gp._trace_id, kernel=rec.kernel_name, mean=float(gp.mean)))

        def call(verb):
            def log(orig, gp, *a, **kw):
                params = np.array(gp.kernel.get_parameter_vector(), dtype=np.float64)
                op = dict(op=verb, gp=gp._trace_id, kw={k: v for k, v in kw.items() if k != "yerr"})
                arrays = dict(params=params)
                if verb == "compute":
                    arrays.update(x=a[0], yerr=kw.get("yerr", a[1] if len(a) > 1 else 0.0))
                    flags = a[2:]
                else:
                    arrays.update(y=a[0], t=a[1] if verb == "predict" else None)
                    flags = a[2 if verb == "predict" else 1:]
                op["flags"] = list(flags)
                try:
                    out = orig(gp, *a, **kw)
                except np.linalg.LinAlgError:
                    op["raised"] = True
                    rec._put(op, **arrays)
                    raise
                op["raised"] = False
                op["n_out"] = len(out) if isinstance(out, tuple) else 0
                if isinstance(out, tuple):
                    arrays.update({"out%d" % j: o for j, o in enumerate(out)})
                else:
                    arrays["out"] = out
                rec._put(op, **arrays)
                return out
            return log

        def sampler_init(orig, s, nwalkers, dim, lnpostfn, *a, **kw):
            memo = []

            def lnp(theta):
                v = lnpostfn(theta)
                memo.append((np.array(theta, dtype=np.float64), float(v)))
                return v
            orig(s, nwalkers, dim, lnp, *a, **kw)
            s._trace_id = sum(op["op"] == "sampler" for op in rec.ops)
            s._trace_memo = memo
            rec.ops.append(dict(op="sampler", sampler=s._trace_id, nwalkers=int(nwalkers), dim=int(dim), a=s.a))

        def run_mcmc(orig, s, p0, N, rstate0=None, lnprob0=None):
            assert isinstance(rstate0, np.random.RandomState) and lnprob0 is None, "call pattern not recorded"
            state = rstate0.get_state()
            del s._trace_memo[:]
            pos, lnprob, st = orig(s, p0, N, rstate0=rstate0)
            thetas = np.array([m[0] for m in s._trace_memo])
            rec._put(dict(op="run_mcmc", sampler=s._trace_id, N=int(N), pos=int(state[2]),
                          has_gauss=int(state[3]), cached_gaussian=float(state[4])),
                     p0=p0, key=state[1], thetas=thetas, lnp=np.array([m[1] for m in s._trace_memo]),
                     out_pos=pos, out_lnprob=lnprob)
            return pos, lnprob, st

        self._wrap(G, "__init__", gp_init)
        for verb in GP_VERBS:
            self._wrap(G, verb, call(verb))
        self._wrap(S, "__init__", sampler_init)
        self._wrap(S, "run_mcmc", run_mcmc)
        return self

    def __exit__(self, *exc):
        for cls, name, orig in reversed(self._saved):
            setattr(cls, name, orig)
        self._saved = []
        return False

    def save(self, path, **extra):
        predicts = [i for i, op in enumerate(self.ops) if op["op"] == "predict"]
        keep = set(predicts[j] for j in np.linspace(0, len(predicts) - 1, min(len(predicts), MAX_PREDICTS)).astype(int)) \
            if predicts else set()
        data, where, ops = [], {}, []
        size = 0
        for i, op in enumerate(self.ops):
            if op["op"] == "predict" and i not in keep:
                continue
            op = dict(op)
            refs = {}
            for k, v in op.pop("arrays", {}).items():
                key = (v.shape, v.tobytes())
                if key not in where:
                    where[key] = size
                    data.append(v.ravel())
                    size += v.size
                refs[k] = [where[key], list(v.shape)]
            op["arrays"] = refs
            ops.append(op)
        np.savez_compressed(path, ops=np.array(json.dumps(ops)),
                            data=np.concatenate(data) if data else np.zeros(0),
                            **{"extra." + k: np.asarray(v) for k, v in extra.items()})


def load(path):
    """(ops with their arrays, extra) of a stored trace."""
    d = np.load(path, allow_pickle=False)
    data = d["data"]
    ops = json.loads(str(d["ops"]))
    for op in ops:
        op["arrays"] = {k: data[o:o + int(np.prod(shape, dtype=np.int64))].reshape(shape)
                        for k, (o, shape) in op["arrays"].items()}
    extra = {k[len("extra."):]: d[k] for k in d.files if k.startswith("extra.")}
    return ops, extra


def replay(path, kernels):
    """Issue the recorded calls to the shims of this tree.  ``kernels`` maps a recorded kernel name to a factory of a
    fresh robo_b200 kernel of the same structure (its parameters are set from the trace before every call).  Yields
    (call index, op, recorded answers, replayed answers) with answers as dicts of arrays."""
    ops, _ = load(path)
    gps, samplers = {}, {}
    for i, op in enumerate(ops):
        kind, arr = op["op"], op["arrays"]
        if kind == "gp":
            gps[op["gp"]] = compat.GeorgeGP(kernels[op["kernel"]](), mean=op["mean"])
        elif kind in GP_VERBS:
            gp = gps[op["gp"]]
            gp.kernel.set_parameter_vector(arr["params"])
            if kind == "compute":
                args = (arr["x"],)
                kw = dict(op["kw"], yerr=float(arr["yerr"]))
            else:
                args = (arr["y"], arr["t"]) if kind == "predict" else (arr["y"],)
                kw = dict(op["kw"])
            try:
                out = getattr(gp, kind)(*(args + tuple(op["flags"])), **kw)
                raised = False
            except np.linalg.LinAlgError:
                out, raised = None, True
            rec = {"raised": np.array(op["raised"])}
            got = {"raised": np.array(raised)}
            if not op["raised"] and not raised and kind != "compute":
                outs = out if op["n_out"] else (out,)
                names = ["out%d" % j for j in range(op["n_out"])] if op["n_out"] else ["out"]
                rec.update({k: arr[k] for k in names})
                got.update({k: np.asarray(o) for k, o in zip(names, outs)})
            yield i, op, rec, got
        elif kind == "sampler":
            samplers[op["sampler"]] = op
        elif kind == "run_mcmc":
            spec = samplers[op["sampler"]]
            table = {t.tobytes(): v for t, v in zip(arr["thetas"], arr["lnp"])}
            missing = []

            def lnp(theta):
                key = np.asarray(theta, dtype=np.float64).tobytes()
                if key not in table:
                    missing.append(key)
                    return -np.inf
                return table[key]
            s = ensemble_sampler.EnsembleSampler(spec["nwalkers"], spec["dim"], lnp, a=spec["a"])
            rng = np.random.RandomState()
            rng.set_state(("MT19937", arr["key"].astype(np.uint32), op["pos"], op["has_gauss"], op["cached_gaussian"]))
            pos, lnprob, _ = s.run_mcmc(arr["p0"], op["N"], rstate0=rng)
            rec = {"out_pos": arr["out_pos"], "out_lnprob": arr["out_lnprob"], "unrecorded_proposals": np.array(0)}
            got = {"out_pos": pos, "out_lnprob": lnprob, "unrecorded_proposals": np.array(len(missing))}
            yield i, op, rec, got
