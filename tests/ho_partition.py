"""Test support for higher-order elements on a partitioned network: the oracle of one rank's part (global node
degrees, so that a cut bifurcation keeps its multiplier), the map of its dofs into the whole network's numbering,
and the sizes of the exchanged sections."""

import numpy as np

from oracle import reference_port as rp


def oracle_ho(pos, edges, colors, N, fd, pd, degree=None):
    """``OracleNetworkHO``; ``degree``: global node degrees when (pos, edges) is one part of a partitioned network."""
    net = rp.OracleNetworkHO(pos, edges, colors, N, fd, pd)
    if degree is not None:
        base = rp.OracleNetwork(pos, edges, colors, N, degree=degree)
        for key in ("degree", "bifurcation_values", "boundary_values", "lm_index", "n_bif"):
            setattr(net, key, getattr(base, key))
        net.n_dofs = net.loff + net.n_bif
        net.block_sizes[-1] = net.n_bif
    return net


def local_to_global(part, lnet, gnet):
    """Global dof of every local dof: flux and interior pressures follow their edge, vertex pressures their node
    (shared nodes included), multipliers their bifurcation."""
    N, fd, pd = lnet.N, lnet.fd, lnet.pd
    ge = part.global_edges
    idx = np.full(lnet.n_dofs, -1, dtype=np.int64)
    per = fd * N + 1
    idx[lnet.fb[:, None] + np.arange(per)[None, :]] = gnet.fb[ge][:, None] + np.arange(per)[None, :]
    k = np.arange(ge.size)[:, None]
    if pd == 0:
        idx[lnet.poff + k * N + np.arange(N)[None, :]] = gnet.poff + ge[:, None] * N + np.arange(N)[None, :]
    else:
        nl, ng = lnet.n_nodes, gnet.n_nodes
        idx[lnet.poff + np.arange(nl)] = gnet.poff + part.global_nodes
        j = np.arange(N - 1)[None, :]
        idx[lnet.poff + nl + k * (N - 1) + j] = gnet.poff + ng + ge[:, None] * (N - 1) + j
        nvl, nvg = lnet.x.shape[0], gnet.x.shape[0]
        i = np.arange(N * (pd - 1))[None, :]
        idx[lnet.poff + nvl + k * N * (pd - 1) + i] = gnet.poff + nvg + ge[:, None] * N * (pd - 1) + i
    idx[lnet.loff:] = gnet.loff + part.global_bif
    assert (idx >= 0).all() and np.unique(idx).size == idx.size
    return idx


def expected_exchange_sizes(n_shared, continuous_pressure):
    """(setup, apply, residual) doubles of the host-driven exchange of the table-driven path
    (include/nxfx_b200.h, nxfx_exchange_sizes)."""
    nt = max(n_shared, 1)
    return 12 * nt, 2 * nt, (3 if continuous_pressure else 1) * n_shared + 2


def place(gnet, vals):
    """Rank 0: the gathered ``DistributedSolver.dof_values()`` of every rank -> one vector in ``gnet``'s numbering."""
    N, fd, pd = gnet.N, gnet.fd, gnet.pd
    x = np.full(gnet.n_dofs, np.nan)
    per = fd * N + 1
    for v in vals:
        ge = np.asarray(v["edges"], dtype=np.int64)
        x[gnet.fb[ge][:, None] + np.arange(per)[None, :]] = v["flux"]
        if pd == 0:
            x[gnet.poff + ge[:, None] * N + np.arange(N)[None, :]] = v["pressure"]
        else:
            inner = gnet.poff + gnet.n_nodes + ge[:, None] * (N - 1) + np.arange(N - 1)[None, :]
            cell = gnet.poff + gnet.x.shape[0] + ge[:, None] * N * (pd - 1) + np.arange(N * (pd - 1))[None, :]
            x[np.concatenate([inner, cell], axis=1)] = v["pressure"]
            x[gnet.poff + np.asarray(v["nodes"], dtype=np.int64)] = v["node_pressure"]
        x[gnet.loff + np.asarray(v["multipliers"], dtype=np.int64)] = v["lam"]
    return x
