"""Helpers shared by the oracle and GPU parity tests: golden reference trajectories -> packed problems."""
import numpy as np

from odam_b200.api import PackedTracks

TOL_PARAM = 1e-4   # BASELINE.json: relative error on parameters (denominator floored at 1e-3, SURVEY 8d)
TOL_LOSS = 1e-5    # BASELINE.json: relative error on the per-iteration loss
FLOOR = 1e-3


def rel_param(a, b):
    return np.abs(a - b) / np.maximum(np.abs(b), FLOOR)


def rel_loss(a, b):
    return np.abs(a - b) / np.maximum(np.abs(b), 1e-30)


class Case:
    def __init__(self, G, k):
        self.k = k
        self.obj = int(G["case_obj"][k])
        self.repr = str(G["case_repr"][k])
        self.use_prior = bool(G["case_prior"][k])
        self.iters = int(G["case_iters"][k])
        self.V = int(G["case_views"][k])
        i, V = self.obj, self.V
        self.Ms = np.ascontiguousarray(G["P_cws"][i][:V].reshape(V, 12), np.float32)
        self.box = np.ascontiguousarray(G["box"][i][:V], np.float32)
        self.mask = np.ascontiguousarray(G["mask"][i][:V], np.uint8)
        self.cls = int(G["cls"][i])
        self.prior33 = G["prior_by_class"][self.cls] if self.use_prior else None
        self.prior_table = np.stack([G["prior_by_class"][c].astype(np.float32).reshape(9) for c in range(8)]) \
            if self.use_prior else None
        self.init = G[f"c{k}_init"]
        for x in ("params", "grad", "m", "v", "loss", "final_points", "arg", "eta_idx", "resid_sign"):
            setattr(self, x, G[f"c{k}_{x}"])

    def states_before(self):
        """(params, m, v) BEFORE each step s = 0..iters-1 (teacher-forcing inputs)."""
        z = np.zeros((1, 9), np.float32)
        return (np.vstack([self.init[None], self.params[:-1]]), np.vstack([z, self.m[:-1]]),
                np.vstack([z, self.v[:-1]]))

    def tracks(self, inits):
        """n = len(inits) copies of this object's views, one per initial state."""
        n, V = len(inits), self.V
        return PackedTracks(init=np.ascontiguousarray(inits, np.float32), cls=np.full(n, self.cls, np.int32),
                            view_off=(np.arange(n + 1) * V).astype(np.int32), Ms=np.tile(self.Ms, (n, 1)),
                            box=np.tile(self.box, (n, 1)), mask=np.tile(self.mask, (n, 1)))


def all_cases(G):
    return [Case(G, k) for k in range(len(G["case_obj"]))]


class WideCase(Case):
    """A case of tests/golden/ref_runs_wide.npz (round 2: the BASELINE view counts and the loop's edge cases); every
    case carries its own views, so nothing is indexed through a shared scene."""

    def __init__(self, W, k):
        self.k = k
        self.name = str(W["names"][k])
        self.repr = str(W["case_repr"][k])
        self.use_prior = bool(W["case_prior"][k])
        self.iters = int(W["case_iters"][k])
        self.V = V = int(W["case_views"][k])
        self.Ms64, self.box64 = W[f"w{k}_Ms"], W[f"w{k}_box"]
        self.Ms = np.ascontiguousarray(self.Ms64.reshape(V, 12), np.float32)
        self.box = np.ascontiguousarray(self.box64, np.float32)
        self.mask = np.ascontiguousarray(W[f"w{k}_mask"], np.uint8)
        self.cls = int(W[f"w{k}_cls"])
        self.translate, self.angle, self.dims = W[f"w{k}_translate"], float(W[f"w{k}_angle"]), W[f"w{k}_dims"]
        self.prior33 = W["prior_by_class"][self.cls] if self.use_prior else None
        self.prior_table = np.stack([W["prior_by_class"][c].astype(np.float32).reshape(9) for c in range(8)]) \
            if self.use_prior else None
        self.init = W[f"w{k}_init"]
        for x in ("params", "grad", "m", "v", "loss", "final_points", "arg", "eta_idx", "resid_sign"):
            setattr(self, x, W[f"w{k}_{x}"])


def wide_cases(W):
    return [WideCase(W, k) for k in range(len(W["names"]))]


def teacher_forced(api, case, **kw):
    """From every recorded reference state of `case` run ONE kernel step (C ABI, host entry).  Returns the parameters
    after the step, the loss, and the step's discrete decisions: arg-extreme sample per (view, side), eta bucket per
    sample, sign of every residual."""
    P, M, V = case.states_before()
    s0 = np.tile(case.init[4:7], (len(P), 1))
    out_p = np.zeros_like(P)
    out_l = np.zeros(len(P), np.float32)
    args = np.zeros((len(P), case.V, 4), np.int32)
    sign = np.zeros((len(P), case.V, 4), np.int8)
    eta = np.zeros((len(P), 1000), np.uint8)
    for s in range(len(P)):   # Adam's bias correction depends on the step count: one launch per state
        o = api.optimize_host(case.tracks(P[s:s + 1]), prior=case.prior_table, n_iters=1, representation=case.repr,
                              m0=M[s:s + 1], v0=V[s:s + 1], step0=s, s0=s0[s:s + 1],
                              extras=("out_arg", "out_eta_idx", "out_pred"), **kw)
        out_p[s], out_l[s] = o["params"][0], o["loss"][0, 0]
        args[s], eta[s] = o["out_arg"].reshape(case.V, 4), o["out_eta_idx"][0]
        sign[s] = np.sign(o["out_pred"].reshape(case.V, 4) - case.box)
    return out_p, out_l, args, eta, sign


def teacher_forced_report(api, cases, label, **kw):
    """Teacher-forced parity of `cases` against the reference's recorded states.  Returns a dict of counts; prints one
    line per out-of-tolerance step and a summary (this is what profiles/r02_parity.txt records)."""
    total = viol_p = viol_l = disagree = viol_on_agree = 0
    worst_p = worst_l = 0.0
    for case in cases:
        out_p, out_l, args, eta, sign = teacher_forced(api, case, **kw)
        live = case.mask.astype(bool)
        for s in range(case.iters):
            rp = float(rel_param(out_p[s], case.params[s]).max())
            rl = 0.0 if (out_l[s] == 0 and case.loss[s] == 0) else float(rel_loss(out_l[s], case.loss[s]))
            bad = rp > TOL_PARAM or rl > TOL_LOSS
            same = (np.array_equal(case.arg[s][live], args[s][live]) and np.array_equal(case.eta_idx[s], eta[s])
                    and np.array_equal(case.resid_sign[s][live], sign[s][live]))
            total += 1
            viol_p += rp > TOL_PARAM
            viol_l += rl > TOL_LOSS
            disagree += not same
            if bad:
                print(f"  {label} case {getattr(case, 'name', case.k)} step {s}: rel err params {rp:.2e} loss {rl:.2e}; "
                      f"decisions {'AGREE' if same else 'differ'} (arg {int((case.arg[s][live] != args[s][live]).sum())}, "
                      f"eta {int((case.eta_idx[s] != eta[s]).sum())}, "
                      f"residual sign {int((case.resid_sign[s][live] != sign[s][live]).sum())})")
                viol_on_agree += same
            else:
                worst_p, worst_l = max(worst_p, rp), max(worst_l, rl)
    print(f"teacher-forced [{label}]: {total} steps; param violations {viol_p}, loss violations {viol_l}, steps with any "
          f"discrete decision differing from the reference {disagree}; violations on decision-agreeing steps "
          f"{viol_on_agree}; worst in-tolerance rel err params {worst_p:.2e}, loss {worst_l:.2e}")
    return dict(total=total, viol_p=viol_p, viol_l=viol_l, disagree=disagree, viol_on_agree=viol_on_agree)


def edge_object(kind, seed=31):
    """One synthetic object (views, init) with an edge of the backward pass forced: extreme shape exponents
    (h = +-6 puts e at 1.6 and 0.2, where samples sit in the 1e-6 clamp), yaws on the axes, a view behind the camera,
    an all-masked track, a single view."""
    from odam_b200 import synthetic
    from odam_b200.api import init_params
    V = 1 if kind == "V1" else 12
    sc = synthetic.make_scene(1, V, seed=seed)
    init = init_params(sc.translate[0], sc.angle[0], sc.dims[0])
    Ms = sc.P_cws[0].reshape(V, 12).astype(np.float32)
    box, mask = sc.box[0].astype(np.float32), sc.mask[0].copy()
    if kind.startswith("h"):
        init[7:9] = {"h+6": (6, 6), "h-6": (-6, -6), "h+-6": (6, -6)}[kind]
    if kind.startswith("yaw"):
        init[3] = {"yaw0": 0.0, "yaw+pi/2": np.pi / 2, "yaw-pi/2": -np.pi / 2, "yawpi": np.pi}[kind]
    if kind == "behind":
        Ms[0, 8:12] = -Ms[0, 8:12]
    if kind == "masked":
        mask[:] = 0
    return init, Ms, box, mask, int(sc.cls[0])


EDGE_KINDS = ["plain", "h+6", "h-6", "h+-6", "yaw0", "yaw+pi/2", "yaw-pi/2", "yawpi", "behind", "masked", "V1"]
