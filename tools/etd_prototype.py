"""CPU prototype (numpy + the C oracle's right-hand side): classical RK4 against ETD-RK4 (Cox-Matthews) with the cover pair's
conduction mode -- the constant 0.653 1/s eigenvalue that caps the nominal RK4 step at 3.58 s -- treated exactly.  The conduction
operator on (tCovIn, tCovE) is -lambda M with M a projector, so every phi-function of it is phi(0) (I - M) + phi(-lambda h) M: scalar
work.  Error against the Radau(1e-12) truth fixtures, WITHOUT the transient-stiffness rule (intervals of the rule-based set whose
top-compartment mode exceeds the step's stability limit therefore diverge at the coarse grids).  Result recorded in DESIGN.md
"Known limits": 215 steps (n_sub 180) stay within 3.5e-7 on the random-action set, 192 steps within 6.8e-7 -- 1.4-1.5x fewer steps
than the shipped 300 at a 2-3x margin to the 1e-6 gate instead of 19x.      python tools/etd_prototype.py"""
import os, sys, numpy as np, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests")); sys.path.insert(0, os.path.join(ROOT, "greenlight-gym2_b200"))
import oracle_binding as ob
def phis(z):
    # phi1..phi3 at z (z <= 0), series for small |z|
    if abs(z) < 1e-3:
        p1 = 1 + z/2 + z*z/6 + z**3/24; p2 = 0.5 + z/6 + z*z/24 + z**3/120; p3 = 1/6 + z/24 + z*z/120 + z**3/720
    else:
        e = np.exp(z); p1 = (e-1)/z; p2 = (e-1-z)/z**2; p3 = (e-1-z-z*z/2)/z**3
    return np.exp(z), p1, p2, p3
def make(p, x, u, d):
    a = ob.aux_rhs(x, u, d, p)[0]
    K = p[71]/p[73]; ia, ib = 1.0/a[33], 1.0/a[34]
    lam = K*(ia+ib)
    M = np.array([[ia, -ia], [-ib, ib]])/(ia+ib)     # projector: L = -lam M on states (5, 6)
    return lam, M
def step_etd(x, h, f, lam, M):
    I2 = np.eye(2)
    def op(g0, gz):  # g(hL) restricted to the cover pair
        return g0*(I2-M) + gz*M
    def N(y):
        r = f(y); r[5:7] += lam*(M @ y[5:7]); return r
    eh, p1h, _, _ = phis(-lam*h/2); e1, p1, p2, p3 = phis(-lam*h)
    Eh, P1h = op(1.0, eh), op(1.0, p1h)
    def apply(A, v, g0=1.0):  # matrix on the pair, scalar g0 on every other state
        w = g0*v; w[5:7] = A @ v[5:7]; return w
    Nx = N(x)
    a_ = apply(Eh, x) + (h/2)*apply(P1h, Nx)
    Na = N(a_)
    b_ = apply(Eh, x) + (h/2)*apply(P1h, Na)
    Nb = N(b_)
    c_ = apply(Eh, a_) + (h/2)*apply(P1h, 2*Nb - Nx)
    Nc = N(c_)
    A1 = op(1 - 3*0.5 + 4/6, p1 - 3*p2 + 4*p3); A2 = op(2*0.5 - 4/6, 2*p2 - 4*p3); A3 = op(-0.5 + 4/6, -p2 + 4*p3)
    E1 = op(1.0, e1)
    out = apply(E1, x) + h*(apply(A1, Nx, 1/6) + apply(A2, Na + Nb, 1/3) + apply(A3, Nc, 1/6))
    return out
def integrate(x, u, d, p, n_sub, sched, etd=True):
    f = lambda y: ob.rhs(y, u, d, p)
    lam, M = make(p, x, u, d)
    h0 = 900.0/n_sub; steps = 0
    for s in range(n_sub):
        m = sched[s] if s < len(sched) else 1
        h = h0/m
        for q in range(m):
            if etd: x = step_etd(x, h, f, lam, M)
            else:
                k1=f(x); k2=f(x+h/2*k1); k3=f(x+h/2*k2); k4=f(x+h*k3); x = x + h/6*(k1+2*k2+2*k3+k4)
            steps += 1
    return x, steps
if __name__ == "__main__":
    rel=lambda a,b: float(np.max(np.abs(a-b)/np.maximum(np.abs(b),1e-3)))
    gold = os.path.join(ROOT, "tests", "golden")
    zr=np.load(os.path.join(gold, "truth_random_actions.npz")); zb=np.load(os.path.join(gold, "truth_rule_based.npz"))
    sets={"random":(zr, range(0,120,4)), "rule-based":(zb, range(0,249,6))}
    for n_sub, sched in ((260,[16,8,4,4,4,4,2,2,2,2,2,2]), (180,[16,8,4,4,4,2,2,2,2]), (150,[16,8,8,4,4,4,2,2,2,2]), (120,[32,16,8,4,4,4,2,2,2,2]), (100,[32,16,8,4,4,4,2,2,2,2])):
        for name,(z,idx) in sets.items():
            t0=time.time(); errs=[]; st=0
            for i in idx:
                y,st=integrate(z["x"][i].copy(), z["u"][i], z["d"][i], z["p"], n_sub, sched, True)
                errs.append(rel(y,z["y"][i]) if np.all(np.isfinite(y)) else np.inf)
            errs=np.array(errs)
            print(f"ETD n_sub={n_sub} steps={st} {name}: worst {errs.max():.2e} p90 {np.percentile(errs,90):.2e} med {np.median(errs):.2e} ({time.time()-t0:.0f}s)",flush=True)
