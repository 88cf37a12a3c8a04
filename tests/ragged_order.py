"""A numpy restatement of the plan's elimination-order rule (tb_plan_create, csrc/tb_plan.cu): reverse Cuthill-McKee over
the joints, kept when it shrinks sum (i - first_i + 1)^2 below 0.85x that of the natural order, and the envelope
statistics of K_ff in the chosen order.  The envelope kernel of ragged batches (tb_ragged_env_order) must reproduce it
joint for joint."""
import numpy as np

from oracle import truss_oracle as orc


def adjacency(nJ, conn):
    """Joint adjacency from the members in ascending order: sorted, de-duplicated, self-loops dropped."""
    adj = [set() for _ in range(nJ)]
    for a, b in np.asarray(conn).reshape(-1, 2):
        if a != b:
            adj[a].add(int(b))
            adj[b].add(int(a))
    return [sorted(s) for s in adj]


def rcm(nJ, adj):
    """Reverse Cuthill-McKee: each component from its lowest unseen joint, three bfs_far passes to a pseudo-peripheral
    start, newly seen neighbours stable-sorted by degree, the whole order reversed."""
    deg = [len(a) for a in adj]

    def bfs_far(start):
        q, level, mark = [start], {start: 0}, {start}
        h = 0
        while h < len(q):
            for v in adj[q[h]]:
                if v not in mark:
                    mark.add(v)
                    level[v] = level[q[h]] + 1
                    q.append(v)
            h += 1
        best = q[-1]
        for v in q:
            if level[v] == level[q[-1]] and deg[v] < deg[best]:
                best = v
        return best

    order, seen = [], [False] * nJ
    for s0 in range(nJ):
        if seen[s0]:
            continue
        start = s0
        for _ in range(3):
            start = bfs_far(start)
        q = [start]
        seen[start] = True
        h = 0
        while h < len(q):
            nb = [v for v in adj[q[h]] if not seen[v]]
            for v in nb:
                seen[v] = True
            q += sorted(nb, key=lambda v: deg[v])        # (sorted() is stable)
            h += 1
        order += q
    return order[::-1]


def _first(dim, nJ, conn, free, rows):
    """first[i] of every free DOF row under the map rows[dof] (row index, -1 at supports)."""
    n = int(free.sum())
    first = np.arange(n)
    has_member = np.zeros(nJ, bool)
    for a, b in np.asarray(conn).reshape(-1, 2):
        has_member[a] = has_member[b] = True
        for ja, jb in ((a, b), (b, a)):
            ra, rb = rows[ja * dim:(ja + 1) * dim], rows[jb * dim:(jb + 1) * dim]
            ra, rb = ra[ra >= 0], rb[rb >= 0]
            if len(ra) and len(rb):
                first[ra] = np.minimum(first[ra], rb.min())
    for j in np.flatnonzero(has_member):
        r = rows[j * dim:(j + 1) * dim]
        r = r[r >= 0]
        if len(r):
            first[r] = np.minimum(first[r], r.min())
    return first


def plan_order(dim, support, conn):
    """The elimination order of tb_plan_create for this topology: dict(order=joints in elimination order, reordered,
    envelope_size, envelope_flops, half_bandwidth)."""
    support = np.asarray(support)
    nJ = len(support)
    free = orc.free_mask(dim, support).reshape(-1)
    nat_rows = np.where(free, np.cumsum(free) - 1, -1)
    order = rcm(nJ, adjacency(nJ, conn))
    rank = np.empty(nJ, int)
    rank[order] = np.arange(nJ)
    # free DOFs by (RCM rank of the joint, reference free index)
    dofs = np.flatnonzero(free)
    cand = sorted(range(len(dofs)), key=lambda x: (rank[dofs[x] // dim], x))
    rcm_rows = np.full(free.shape, -1)
    rcm_rows[dofs[cand]] = np.arange(len(dofs))

    def score(rows):
        first = _first(dim, nJ, conn, free, rows)
        i = np.arange(len(first))
        return float(np.sum((i - first + 1).astype(np.float64) ** 2)), first

    s_nat, f_nat = score(nat_rows)
    s_rcm, f_rcm = score(rcm_rows)
    use = len(dofs) > 0 and s_rcm < 0.85 * s_nat
    first = f_rcm if use else f_nat
    n = len(first)
    env = int(np.sum(np.arange(n) - first + 1))
    fl = 0.0
    for i in range(n):
        j = np.arange(first[i], i + 1)
        fl += float(np.sum(2.0 * (j - np.maximum(first[i], first[j])) + 1.0))
        fl += 4.0 * (i - first[i]) + 2.0
    return {"order": list(order) if use else list(range(nJ)), "reordered": int(use), "envelope_size": env,
            "envelope_flops": fl, "half_bandwidth": int(np.max(np.arange(n) - first)) if n else 0}


def host_cubes(num_cube, count, seed):
    """``count`` cube trusses of ``num_cube`` cells on a 6^3 grid from the host generator."""
    from python_stable_3d_truss_analysis_b200.generate import GenerateRandomCubeTrusses

    return GenerateRandomCubeTrusses(gridRange=(6, 6, 6), numCubeRange=(num_cube, num_cube), numEachRange=(1, count),
                                     lengthRange=(100, 200), forceRange=[(-1000, 1000)] * 3, seed=seed,
                                     isPrintMessage=False)
