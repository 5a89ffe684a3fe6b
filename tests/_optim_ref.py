"""float64 references of the update rules (TF 1.x ApplyGradientDescent / ApplyMomentum / ApplyRMSProp) with a derived fp32
error bound, shared by the CPU and GPU optimizer tests.

Each fp32 operation of the rule may round once, by at most u * |result| (u = 2^-23: room for either rounding mode, as in
tests/_fp64_ref.py).  `RefState.step` carries the float64 value of every quantity AND a running bound on how far an fp32
implementation that starts from the same values and receives the same gradient sums may have drifted from it: the bound of
step k is propagated through the rule's formula (first-order, each input error times the formula's sensitivity to it) and
the fresh roundings of step k are added.  Nothing is tuned by hand: a test compares |fp32 - fp64| against `slack` x bound.
"""
import numpy as np

U = 2.0 ** -23
SLOT_INITS = {"sgd": (), "momentum": (0.0,), "rmsprop": (1.0, 0.0)}


class RefState:
    def __init__(self, rule: str, w0, momentum=0.9, decay=0.9, eps=1.0, slots0=None):
        self.rule, self.m, self.d, self.eps = rule, float(momentum), float(decay), float(eps)
        self.w = np.asarray(w0, dtype=np.float64).copy()
        n = self.w.shape
        if slots0 is None:
            self.s = [np.full(n, v, dtype=np.float64) for v in SLOT_INITS[rule]]
        else:
            self.s = [np.asarray(x, dtype=np.float64).copy() for x in slots0]
        self.ew = np.zeros(n)
        self.es = [np.zeros(n) for _ in self.s]

    def step(self, gsum, divisor, lr, e_gsum=0.0):
        """One committed step from the gradient SUM over the contributors (float64 values of what the fp32 code summed)
        and the bound `e_gsum` on the fp32 sum's own error."""
        gsum = np.asarray(gsum, dtype=np.float64)
        g = gsum / float(divisor)
        eg = np.asarray(e_gsum, dtype=np.float64) / float(divisor) + U * np.abs(g)
        lr = float(lr)
        if self.rule == "sgd":
            self.w = self.w - lr * g
            self.ew = self.ew + abs(lr) * eg + 3 * U * (np.abs(self.w) + np.abs(lr * g))
        elif self.rule == "momentum":
            a0 = self.s[0]
            a = self.m * a0 + g
            self.es[0] = self.m * self.es[0] + eg + 2 * U * (np.abs(self.m * a0) + np.abs(a))
            self.w = self.w - lr * a
            self.ew = self.ew + abs(lr) * self.es[0] + 3 * U * (np.abs(self.w) + np.abs(lr * a))
            self.s[0] = a
        else:
            ms0, mom0 = self.s
            ms = ms0 + (g * g - ms0) * (1.0 - self.d)
            self.es[0] = (self.d * self.es[0] + (1.0 - self.d) * 2 * np.abs(g) * eg
                          + 4 * U * (g * g + np.abs(ms0) + np.abs(ms)))
            den = np.sqrt(ms + self.eps)
            t = lr * g / den
            et = abs(lr) * eg / den + np.abs(t) * (0.5 * self.es[0] / (ms + self.eps) + 4 * U)
            mom = self.m * mom0 + t
            self.es[1] = self.m * self.es[1] + et + 2 * U * (np.abs(self.m * mom0) + np.abs(mom))
            self.w = self.w - mom
            self.ew = self.ew + self.es[1] + 2 * U * (np.abs(self.w) + np.abs(mom))
            self.s = [ms, mom]

    def check(self, w32, slots32=(), slack=2.0, what=""):
        """Assert the fp32 values lie within slack x bound of the float64 ones; returns the worst err / bound."""
        worst = 0.0
        for name, got, ref, bound in [("w", w32, self.w, self.ew)] + [
                ("slot%d" % i, s, r, b) for i, (s, r, b) in enumerate(zip(slots32, self.s, self.es))]:
            err = np.abs(np.asarray(got, dtype=np.float64) - ref)
            lim = slack * bound + 1e-30
            ratio = float(np.max(err / lim))
            worst = max(worst, ratio)
            assert ratio <= 1.0, "%s %s: max err/bound %.3f (err %.3g at %d)" % (what, name, ratio, float(err.max()),
                                                                                 int(err.argmax()))
        return worst
