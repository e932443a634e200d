"""CPU reference of C0 assembly (b200fe_assembly_*), bit-exact to the contract in include/b200fe.h, and the maps the
tests feed it:
  structured_map  the C0 map and signs of the modified basis on a box of nex^d elements, with optional element mirror
                  flips and homogeneous Dirichlet boundaries;
  random_map      dofs with multiplicities from 0 to ~1000, NO_DOF entries and optional random signs;
  box_points      the physical coordinates of every element's quadrature points on the same mesh (flips included)."""
import numpy as np

NO_DOF = 0xFFFFFFFF


def _map_1d(nex, nm):
    """direction-wise map and sign: g[ex, flip, p], s[flip, p]"""
    ex = np.arange(nex)[:, None]
    p = np.arange(nm)[None, :]
    g = np.where(p == 0, ex * (nm - 1), np.where(p == 1, (ex + 1) * (nm - 1), ex * (nm - 1) + p - 1))
    gf = g.copy()
    gf[:, [0, 1]] = g[:, [1, 0]]  # a mirrored element swaps its two vertex modes ...
    s = np.ones((2, nm), dtype=np.int64)
    s[1, 2:] = (-1) ** np.arange(2, nm)  # ... and bubble p changes sign with the parity of p
    return np.stack([g, gf], axis=1), s


def structured_map(dim, nex, nm, flips=None, dirichlet=False):
    """(map uint32, sign int8, ndof) of the modified basis (mode 0 = (1 - x)/2, mode 1 = (1 + x)/2, bubbles p >= 2) on
    nex^d box elements, element e = (ez*nex + ey)*nex + ex, local entry l = e*nm^d + (r*nm + q)*nm + p, global dof
    (gz*N + gy)*N + gx with N = nex*(nm - 1) + 1.  flips: (nelmt, dim) booleans, True = the element is mirrored in that
    direction.  dirichlet: every dof with a 1-D index 0 or N - 1 becomes NO_DOF and the rest are renumbered in order."""
    assert nm >= 2
    nelmt = nex ** dim
    n1 = nex * (nm - 1) + 1
    g1, s1 = _map_1d(nex, nm)
    flips = np.zeros((nelmt, dim), dtype=bool) if flips is None else np.asarray(flips, dtype=bool)
    e = np.arange(nelmt)
    eidx = [(e // nex ** a) % nex for a in range(dim)]  # element index per direction, direction 0 fastest
    # per element and direction: the 1-D dof and sign of each mode
    gd = [g1[eidx[a], flips[:, a].astype(int)] for a in range(dim)]  # (nelmt, nm)
    sd = [s1[flips[:, a].astype(int)] for a in range(dim)]
    if dim == 2:
        gx, gy = gd[0][:, None, :], gd[1][:, :, None]
        glob = gy * n1 + gx
        sign = sd[1][:, :, None] * sd[0][:, None, :]
        inner = (gx > 0) & (gx < n1 - 1) & (gy > 0) & (gy < n1 - 1)
    else:
        gx, gy, gz = gd[0][:, None, None, :], gd[1][:, None, :, None], gd[2][:, :, None, None]
        glob = (gz * n1 + gy) * n1 + gx
        sign = sd[2][:, :, None, None] * sd[1][:, None, :, None] * sd[0][:, None, None, :]
        inner = (gx > 0) & (gx < n1 - 1) & (gy > 0) & (gy < n1 - 1) & (gz > 0) & (gz < n1 - 1)
    glob = glob.reshape(-1).astype(np.int64)
    sign = np.broadcast_to(sign, (nelmt,) + (nm,) * dim).reshape(-1).astype(np.int8)
    ndof = n1 ** dim
    if dirichlet:
        inner = np.broadcast_to(inner, (nelmt,) + (nm,) * dim).reshape(-1)
        keep = np.zeros(ndof, dtype=bool)
        keep[glob[inner]] = True
        renum = np.cumsum(keep) - 1
        glob = np.where(inner, renum[glob], NO_DOF)
        ndof = int(keep.sum())
    return glob.astype(np.uint32), sign, ndof


def random_map(nloc, ndof, seed, no_dof=0.05, signed=True, hubs=3, hub_size=1000):
    """(map uint32, sign int8 or None): `hubs` dofs with hub_size entries each, the other entries uniform over the dofs
    (so some dofs have none), a fraction no_dof of NO_DOF entries, random signs"""
    rng = np.random.default_rng(seed)
    m = rng.integers(0, ndof, nloc, dtype=np.int64)
    pos = rng.permutation(nloc)
    hubs = min(hubs, ndof)
    nh = min(hubs * hub_size, nloc)
    m[pos[:nh]] = rng.choice(ndof, hubs, replace=False)[np.arange(nh) % hubs]
    nd = int(no_dof * nloc)
    m[pos[nh:nh + nd]] = NO_DOF
    sign = rng.choice(np.array([-1, 1], dtype=np.int8), nloc) if signed else None
    return m.astype(np.uint32), sign


def gather_ref(map_, sign, glob):
    """local[l] = sign[l] * glob[map[l]], +0 for NO_DOF"""
    glob = np.asarray(glob)
    valid = map_ != NO_DOF
    x = glob[np.where(valid, map_, 0).astype(np.int64)] if glob.size else np.zeros(map_.size, glob.dtype)
    if sign is not None:
        x = np.where(sign < 0, -x, x)
    return np.where(valid, x, glob.dtype.type(0))


def assemble_ref(map_, sign, loc, ndof):
    """glob[g] = ((+0 + v_l0) + v_l1) + ... over map[l] = g in ascending l, v_l = sign[l] * loc[l], rounded to the dtype
    of loc: one vectorised pass per position k inside the segments, k ascending"""
    loc = np.asarray(loc)
    order = np.argsort(map_, kind="stable")
    keys = map_[order]
    nvalid = int(np.searchsorted(keys, NO_DOF))  # NO_DOF sorts last
    order, keys = order[:nvalid], keys[:nvalid].astype(np.int64)
    v = loc[order]
    if sign is not None:
        v = np.where(sign[order] < 0, -v, v)
    start = np.searchsorted(keys, np.arange(ndof))
    count = np.searchsorted(keys, np.arange(ndof), side="right") - start
    out = np.zeros(ndof, dtype=loc.dtype)
    for k in range(int(count.max()) if ndof else 0):
        d = np.nonzero(count > k)[0]
        out[d] = out[d] + v[start[d] + k]
    return out


def box_points(dim, nex, x1, flips=None):
    """(nelmt, dim, nq^d) physical coordinates of the quadrature points x1 (on [-1, 1]) of the nex^d elements of the unit
    box, point (k*nq + j)*nq + i; a mirrored direction runs from the element's right edge to its left"""
    nelmt, nq, h = nex ** dim, len(x1), 1.0 / nex
    flips = np.zeros((nelmt, dim), dtype=bool) if flips is None else np.asarray(flips, dtype=bool)
    e = np.arange(nelmt)
    out = np.empty((nelmt, dim, nq ** dim))
    for a in range(dim):
        xi = np.where(flips[:, a:a + 1], -x1[None, :], x1[None, :])  # (nelmt, nq)
        xa = ((e // nex ** a) % nex)[:, None] * h + (xi + 1) / 2 * h
        shape = [nelmt] + [1] * dim
        shape[dim - a] = nq  # direction 0 is the last (fastest) axis
        out[:, a] = np.broadcast_to(xa.reshape(shape), (nelmt,) + (nq,) * dim).reshape(nelmt, -1)
    return out
