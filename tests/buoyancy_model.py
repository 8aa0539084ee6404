"""TEST INFRASTRUCTURE ONLY. Coupled (Boussinesq) SIMPLE iterations (DESIGN.md §1, "Buoyancy"), composed from pinned parts: the
loop of fast_simple.simple_iterations, unchanged, with the body force added to the momentum right-hand sides in the device's operator
order (every numpy elementwise operation rounds once, like the -fmad=false kernel), and after each iteration the scalar sweeps built by
scalar_oracle.build and solved with the given solve. The source enters through the solve the loop is given: the momentum solves are
the only calls on the loop's own momentum matrices, and there b + b_di is exactly the right-hand side they receive. With
fast_simple.oracle_solve this is the reference-order model, with fast_simple.model_solve the fast-mode model."""
import numpy as np

import fast_simple as fs
import scalar_oracle as so


def coupled_iterations(om, bcs, settings, rho, mu, fields, phi, iterations, solve, gamma, beta, phi_ref, gravity, sweeps=1, state=None,
                       pos=None, first=1, on_iteration=None):
    """`iterations` coupled iterations from `fields` (u, v, w, p) and the scalar `phi`; `bcs` is a scalar_oracle.ScalarBcs of `om`.
    Returns fast_simple.simple_iterations's records, each with the iteration's `phi` (after its sweeps) added."""
    state = state or fs.State(om, mu)
    vol = np.asarray(om.export()["cell_volume"], dtype=np.float64)
    g = [float(x) for x in gravity]
    rho_beta = rho * beta
    cur = [np.array(phi, dtype=np.float64)]

    def source(a, B):   # b_k <- (b_k + b_di,k) - (s_P * g_k), s_P = ((rho * beta) * (phi_P - phi_ref)) * V_P, phi as the iteration started
        s = (rho_beta * (cur[0] - phi_ref)) * vol
        if len(B) == 3:   # the lockstep solve of u, v, w on a_u
            return np.stack([B[k] - s * g[k] for k in range(3)])
        k = next(q for q, m in enumerate(state.a) if m is a)
        return (B[0] - s * g[k])[None]

    def loop_solve(a, B, X, pos=None):
        if any(a is m for m in state.a):
            B = source(a, B)
        return solve(a, B, X, pos)

    def sweep(rec):
        x = cur[0]
        for _ in range(sweeps):
            a, b = so.build(om, bcs, rec["u"], rec["v"], rec["w"], rec["p"], x, *state.a, gamma, rho, settings.momentum, settings.limiter,
                            settings.velocity_interpolation, settings.gradient)
            x = solve(a, b[None], x[None], pos)[0]
        cur[0] = x
        rec["phi"] = x
        if on_iteration:
            on_iteration(rec)

    return fs.simple_iterations(om, settings, rho, mu, fields, iterations, loop_solve, state=state, pos=pos, first=first, on_iteration=sweep)


def zone_terms(om, bcs, rec, state, settings, gamma, rho, name):
    """The (diffusive, convective) outward flux terms of rec['phi'] through each face of zone `name`, in ascending face order, on
    rec's flow (u, v, w, p) and the state's diagonals (DESIGN.md §1)."""
    g = om.export()
    zones = om.zones()
    k = zones["names"].index(name)
    zid = int(zones["ids"][k])
    F = so.face_flux(om, rec["u"], rec["v"], rec["w"], rec["p"], *state.a, settings.velocity_interpolation, settings.gradient)
    phi = rec["phi"]
    terms = []
    for f in np.nonzero(g["face_zone"] == zid)[0]:
        c = int(g["face_c0"][f])
        fl = (rho * g["face_area"][f]) * F[f]
        if bcs.kind[k] == so.FIXED:
            pb = float(bcs.value[k])
            d_b = gamma * g["face_area"][f] / np.linalg.norm(g["face_centroid"][f] - g["cell_centroid"][c])
            terms.append((d_b * (phi[c] - pb), max(fl, 0.0) * phi[c] + min(fl, 0.0) * pb))
        else:
            terms.append((0.0, fl * phi[c]))
    return np.array(terms).reshape(-1, 2)


def zone_flux(om, bcs, rec, state, settings, gamma, rho, name):
    """(diffusive, convective) sums of zone_terms in ascending face order."""
    diff = conv = 0.0
    for d, c in zone_terms(om, bcs, rec, state, settings, gamma, rho, name):
        diff += d
        conv += c
    return float(diff), float(conv)
