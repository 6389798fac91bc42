"""CWBVH bytes written by hand: one node encoder, and a seeded generator of valid trees in the layouts that neither of the
project's builders writes.

`encode_node` writes one 80-byte CwBvhNode.  By default it writes the way host/cwbvh_build.cpp's Collapser does (p = box min,
tight exponents, leaf triangles packed in child order from offset 0, zeroed empty slots); its keyword arguments take each of
those choices away.

`random_cwbvh` / `random_tlas` build trees that `tray_host_cwbvh_validate` accepts but that use the freedoms of the format:
overlapping boxes, 1-8 children in any slots, single-child chains, inner blocks anywhere in the node array, leaf ranges in any
order with gaps, loose exponents and q bytes, any bytes in empty slots, and, in two-level scenes, permuted `blas_offsets` and a
BLAS shared by two instances.  Whatever a correct traversal never reads holds POISON: record slots in leaf-offset gaps hold a
huge triangle across the scene, unreferenced node slots hold a node whose leaves cover all space and lead to poison records, and
unreferenced `blas_offsets` entries lead to a poison BLAS.  A traversal that reads one of them returns a poison id.

Every index the generator writes, poison included, lies inside its array (`check_indices`).  Leaf ranges of one node never
overlap: the kernel's fused node test adds child bits instead of OR-ing them, which is only right when they are disjoint."""
import math

import numpy as np

import oracle_binding as ob
from tray_racing_b200 import cuda, host

EXACT_EXP_BYTE = 167                  # build_gpu.h: an exponent byte >= 167 sends the scene to the unfused node test
POISON_SPAN = 100.0                   # half-size of a poison triangle (scenes live in [-1, 1]^3; f16 edges stay finite)
POISON_BOX = float(2 ** 12)           # poison nodes cover [-POISON_BOX, POISON_BOX]^3


# ---- one node --------------------------------------------------------------------------------------------------------------
def quant_exponent(extent):
    extent = max(extent, 1e-20)
    k = math.ceil(math.log2(extent / 255.0))
    while math.ldexp(255.0, k) < extent:
        k += 1
    while math.ldexp(255.0, k - 1) >= extent:
        k -= 1
    return k


def _vec3(x):
    return np.broadcast_to(np.asarray(x, np.float32), (3,)).astype(np.float32)


def encode_node(lo, hi, children, child_base=0, prim_base=0, exp=None, slack=0, p=None, leaf_offsets=None, empty_fill=None):
    """One 80-byte CwBvhNode over the box [lo, hi] (scalars: a cube).  children: (slot, child_lo, child_hi, kind), kind "inner"
    or the triangle count of a leaf; inner children are the nodes child_base, child_base + 1, .. in slot order.
      exp           exponent per axis (scale 2^exp), at least the tight one; default: the tight exponent of hi - p
      slack         q bytes widened by this many steps on each side (clamped to 0 .. 255): an int, or one per child
      p             the node origin, <= lo on every axis; default lo
      leaf_offsets  the triangle offset of each child (None for inner ones); default: packed in child order from 0
      empty_fill    (6, 8) bytes: the q bytes (lo x, lo y, lo z, hi x, hi y, hi z) of the slots no child uses; default zero"""
    n = np.zeros(80, np.uint8)
    lo, hi = _vec3(lo), _vec3(hi)
    p = lo if p is None else _vec3(p)
    assert (p <= lo).all()
    n[0:12] = p.view(np.uint8)
    k = [quant_exponent(float(hi[a]) - float(p[a])) for a in range(3)]
    if exp is not None:
        e = np.broadcast_to(np.asarray(exp), (3,))
        assert all(int(e[a]) >= k[a] for a in range(3)), (e, k)
        k = [int(e[a]) for a in range(3)]
    assert all(1 <= ka + 127 <= 254 for ka in k)
    n[12:15] = [ka + 127 for ka in k]
    n[16:24] = np.array([child_base, prim_base], np.uint32).view(np.uint8)
    if empty_fill is not None:
        used = {c[0] for c in children}
        for s in set(range(8)) - used:
            for a in range(3):
                n[32 + 16 * a + s], n[40 + 16 * a + s] = empty_fill[a][s], empty_fill[3 + a][s]
    tri_offset = 0
    for i, (slot, clo, chi, kind) in enumerate(children):
        clo, chi = _vec3(clo), _vec3(chi)
        sl = slack if np.isscalar(slack) else slack[i]
        for a in range(3):
            scale = math.ldexp(1.0, k[a])
            n[32 + 16 * a + slot] = min(255, max(0, math.floor((float(clo[a]) - float(p[a])) / scale) - sl))
            n[40 + 16 * a + slot] = min(255, max(0, math.ceil((float(chi[a]) - float(p[a])) / scale) + sl))
        if kind == "inner":
            n[15] |= 1 << slot
            n[24 + slot] = 0x20 | (24 + slot)
        else:
            off = tri_offset if leaf_offsets is None else leaf_offsets[i]
            assert 0 <= off and off + kind <= 24
            n[24 + slot] = (0x20, 0x60, 0xE0)[kind - 1] | off
            tri_offset = off + kind
    return n


class Scene:
    """nodes + triangle soup (+ blas_offsets, tlas_start of a two-level scene), as the oracle and the CUDA scene take them;
    `rec` overrides the records made from `tris` (records that are not triangles of the soup: poison)"""

    def __init__(self, nodes, tris, blas=None, tlas_start=0, stride=48, rec=None):
        self.nodes, self.tris, self.blas, self.tlas_start, self.stride = nodes, tris, blas, tlas_start, stride
        self.rec = host.tri_records(tris, stride) if rec is None else rec

    def oracle(self):
        return ob.Oracle(self.nodes, self.rec, self.stride, self.blas, self.tlas_start, self.blas is not None)

    def cuda(self):
        return cuda.TrayCudaScene(self.nodes, self.rec, self.stride, self.blas, self.tlas_start)


# ---- geometry --------------------------------------------------------------------------------------------------------------
def random_tris(n, seed, flat_fraction=0.2, size=(0.005, 0.25)):
    """n triangles in [-1, 1]^3 of log-uniform size; `flat_fraction` of them lie in the planes z = 0.25 and x = -0.4 (flat
    sheets: zero-extent boxes on one axis)"""
    rng = np.random.default_rng(seed)
    c = rng.uniform(-0.9, 0.9, (n, 1, 3))
    s = 10 ** rng.uniform(np.log10(size[0]), np.log10(size[1]), (n, 1, 1))
    t = (c + s * rng.uniform(-1, 1, (n, 3, 3))).astype(np.float32)
    k = int(n * flat_fraction)
    t[: k // 2, :, 2] = np.float32(0.25)
    t[k // 2:k, :, 0] = np.float32(-0.4)
    return t.reshape(n, 9)


def poison_tris(n, seed):
    """huge triangles through the middle of the scene, cycling through the three axis planes"""
    rng = np.random.default_rng(seed)
    out = np.zeros((n, 3, 3), np.float32)
    S = POISON_SPAN
    for i in range(n):
        a, b, c = i % 3, (i + 1) % 3, (i + 2) % 3
        out[i, :, a] = rng.uniform(-0.5, 0.5)
        out[i, :, b] = (-S, 2 * S, -S)
        out[i, :, c] = (-S, -S, 2 * S)
    return out.reshape(n, 9)


def random_objects(tris, n_objects, seed):
    """(tris reordered, object_offsets): the soup cut into `n_objects` slabs along x of random widths (each >= 1 triangle)"""
    rng = np.random.default_rng(seed)
    t = np.asarray(tris, np.float32).reshape(-1, 9)
    t = t[np.argsort(t.reshape(-1, 3, 3)[:, :, 0].mean(axis=1), kind="stable")]
    cuts = np.sort(rng.choice(np.arange(1, len(t)), n_objects - 1, replace=False))
    return t, np.concatenate([[0], cuts, [len(t)]]).astype(np.uint64)


def tri_bounds(tris):
    t3 = np.asarray(tris, np.float32).reshape(-1, 3, 3)
    return t3.min(axis=1), t3.max(axis=1)


# ---- the generator ---------------------------------------------------------------------------------------------------------
KNOBS = dict(
    split="random",          # "random": random partitions (boxes overlap), "median": spatial median splits, "mix"
    slots="random",          # "random", "octant" (builder-like), "low", "high", "mix": one of the four per node
    order="random",          # node order: "bfs", "dfs", "random" (child blocks shuffled)
    node_gaps=0.1,           # chance of 1-2 poison nodes before a child block
    leaf_order="random",     # leaf ranges "slot" ordered or in a "random" order of the node's leaves
    leaf_gaps=0.3,           # chance of a poison record before a leaf range (or of pushing the ranges to end at 24)
    record_gaps=0.2,         # chance of poison records between two nodes' record blocks
    chain=0.1,               # chance that a node has one inner child (single-child chains)
    full=0.3,                # chance that a node over >= 24 primitives carves 8 leaves of 3 (tri_y = 0xFFFFFF)
    loose_p=0.3,             # chance of p below the box minimum
    exp_raise=0.3,           # chance, per axis, of an exponent 1-8 above the tight one
    slack=0.3,               # chance, per child, of q bytes widened by 1-6 steps
    empty_fill=True,         # random q bytes in empty slots
    exact_node=False,        # one node with an exponent byte >= EXACT_EXP_BYTE
    root_leaf=False,         # a root over <= 3 primitives holds them as one leaf
)


class _Node:
    __slots__ = ("ids", "lo", "hi", "kids", "slots", "index", "full")

    def __init__(self, ids, lo, hi):
        self.ids, self.lo, self.hi, self.kids, self.slots, self.index, self.full = ids, lo, hi, [], [], -1, False


class _Gen:
    """one tree (a flat scene, one BLAS or the TLAS) over primitive boxes, written into its own region of nodes and appending
    its leaf ranges to a shared record list (primitive id, or -1 for a poison record)"""

    def __init__(self, rng, knobs, plo, phi):
        self.rng, self.k, self.plo, self.phi = rng, knobs, plo, phi
        self.cen = (plo.astype(np.float64) + phi) / 2

    def box(self, ids):
        return self.plo[ids].min(axis=0), self.phi[ids].max(axis=0)

    def pick(self, name, choices):
        v = self.k[name]
        return choices[self.rng.integers(len(choices))] if v == "mix" else v

    def partition(self, ids, k):
        rng = self.rng
        if self.pick("split", ("random", "median")) == "median":
            ax = int(np.argmax(self.cen[ids].max(axis=0) - self.cen[ids].min(axis=0)))
            ids = ids[np.argsort(self.cen[ids, ax], kind="stable")]
            cuts = np.linspace(0, len(ids), k + 1).astype(int)
        else:
            ids = rng.permutation(ids)
            cuts = np.concatenate([[0], np.sort(rng.choice(np.arange(1, len(ids)), k - 1, replace=False)), [len(ids)]])
        return [ids[cuts[i]:cuts[i + 1]] for i in range(k)]

    def build(self, ids, depth=0, full=False):
        rng, k = self.rng, self.k
        node = _Node(ids, *self.box(ids))
        n = len(ids)
        if full or n == 24 and rng.random() < k["full"]:                     # 8 leaves of 3: tri_y = 0xFFFFFF
            assert n == 24
            node.full = True
            ax = int(rng.integers(3))
            node.kids = np.array_split(ids[np.argsort(self.cen[ids, ax], kind="stable")], 8)
        elif n <= 3 and (depth == 0 and k["root_leaf"] or depth > 0 and rng.random() < 0.5):
            node.kids = [ids]                                                    # one leaf
        elif depth > 40:
            node.kids = np.array_split(ids, (n + 2) // 3) if n <= 24 else [self.build(g, depth + 1) for g in self.partition(ids, 8)]
        elif n > 3 and rng.random() < k["chain"]:
            node.kids = [self.build(ids, depth + 1)]                             # a single-child chain
        else:
            carved = None
            if n >= 48 and rng.random() < k["full"]:                             # carve 24 neighbours: 8 leaves of 3 below
                ax = int(rng.integers(3))
                srt = ids[np.argsort(self.cen[ids, ax], kind="stable")]
                at = int(rng.integers(0, n - 23))
                carved = srt[at:at + 24]
                ids = np.concatenate([srt[:at], srt[at + 24:]])
                node.kids.append(self.build(carved, depth + 1, full=True))
            m = min(int(rng.integers(1, 9 - len(node.kids))), len(ids))
            if m == 1 and len(ids) > 3 and carved is None:
                m = 2
            for g in self.partition(ids, m):
                if len(g) <= 3 and (rng.random() < 0.75 or len(g) == len(node.ids)):
                    node.kids.append(g)
                else:
                    node.kids.append(self.build(g, depth + 1))
        node.slots = self.assign_slots(node)
        return node

    def kid_box(self, kid):
        return (kid.lo, kid.hi) if isinstance(kid, _Node) else self.box(kid)

    def assign_slots(self, node):
        m = len(node.kids)
        how = self.pick("slots", ("random", "octant", "low", "high"))
        if how == "random":
            return [int(s) for s in self.rng.permutation(8)[:m]]
        if how == "low":
            return [int(s) for s in self.rng.permutation(m)]
        if how == "high":
            return [int(s) + 8 - m for s in self.rng.permutation(m)]
        # octant: each child to the octant of its centre around the node centre (x -> bit 2, y -> bit 1, z -> bit 0), the
        # nearest free slot when taken
        c = (node.lo.astype(np.float64) + node.hi) / 2
        free, out = set(range(8)), []
        for kid in node.kids:
            klo, khi = self.kid_box(kid)
            kc = (klo.astype(np.float64) + khi) / 2
            want = (4 if kc[0] > c[0] else 0) | (2 if kc[1] > c[1] else 0) | (1 if kc[2] > c[2] else 0)
            s = min(free, key=lambda s: (bin(s ^ want).count("1"), s))
            free.discard(s)
            out.append(s)
        return out

    # -- layout ----------------------------------------------------------------------------------------------------------
    def layout(self, root):
        """node indices inside the region: the root at 0, each node's inner children one block in slot order; returns the
        region's slot list (a _Node, or None for a poison node)"""
        rng, order = self.rng, self.k["order"]
        region = [root]
        root.index = 0

        def inner(node):
            return [kid for _, kid in sorted(zip(node.slots, node.kids), key=lambda x: x[0]) if isinstance(kid, _Node)]

        def place(block):
            if rng.random() < self.k["node_gaps"]:
                region.extend([None] * int(rng.integers(1, 3)))
            for kid in block:
                kid.index = len(region)
                region.append(kid)

        if order == "bfs":
            queue = [root]
            while queue:
                node = queue.pop(0)
                place(inner(node))
                queue += inner(node)
        elif order == "dfs":
            def visit(node):
                place(inner(node))
                for kid in inner(node):
                    visit(kid)
            visit(root)
        else:
            blocks, todo = [], [root]
            while todo:
                node = todo.pop()
                if inner(node):
                    blocks.append(inner(node))
                    todo += inner(node)
            for i in rng.permutation(len(blocks)):
                place(blocks[i])
        if rng.random() < self.k["node_gaps"]:
            region.append(None)
        return region

    def leaf_ranges(self, node, records):
        """offsets of the node's leaves, and their records appended to `records` (poison in the gaps); returns prim_base"""
        rng = self.rng
        leaves = [i for i, kid in enumerate(node.kids) if not isinstance(kid, _Node)]
        if not leaves:
            return 0, {}
        if self.k["leaf_order"] == "random":
            leaves = [leaves[i] for i in rng.permutation(len(leaves))]
        else:
            leaves.sort(key=lambda i: node.slots[i])
        spare = 24 - sum(len(node.kids[i]) for i in leaves)
        gaps = [0] * len(leaves)                                                 # poison records in front of each range
        for j in range(len(leaves)):
            if spare and rng.random() < self.k["leaf_gaps"]:
                gaps[j] += 1
                spare -= 1
        if spare and rng.random() < self.k["leaf_gaps"] / 3:
            gaps[-1] += spare                                                    # the last range ends exactly at 24
        if rng.random() < self.k["record_gaps"]:
            records.extend([-1] * int(rng.integers(1, 4)))
        base, off, offsets = len(records), 0, {}
        for j, i in enumerate(leaves):
            records.extend([-1] * gaps[j])
            off += gaps[j]
            offsets[i] = off
            records.extend(int(p) for p in node.kids[i])
            off += len(node.kids[i])
        assert off <= 24
        return base, offsets

    def encode(self, node, region_nodes, records, exact):
        rng, k = self.rng, self.k
        kids = node.kids
        prim_base, offsets = self.leaf_ranges(node, records)
        inner_kids = [kid for kid in kids if isinstance(kid, _Node)]
        child_base = min(kid.index for kid in inner_kids) if inner_kids else 0
        children, leaf_off, slack = [], [], []
        for i, kid in enumerate(kids):
            klo, khi = self.kid_box(kid)
            children.append((node.slots[i], klo, khi, "inner" if isinstance(kid, _Node) else len(kid)))
            leaf_off.append(offsets.get(i))
            slack.append(int(rng.integers(1, 7)) if rng.random() < k["slack"] else 0)
        lo, hi = node.lo, node.hi
        p = lo
        if rng.random() < k["loose_p"]:
            p = (lo - (hi - lo + np.float32(0.01)) * rng.uniform(0, 2, 3).astype(np.float32)).astype(np.float32)
            p = np.minimum(p, lo)
        tight = [quant_exponent(float(hi[a]) - float(p[a])) for a in range(3)]
        exp = [t + (int(rng.integers(1, 9)) if rng.random() < k["exp_raise"] else 0) for t in tight]
        if exact:
            exp[int(rng.integers(3))] = EXACT_EXP_BYTE - 127 + int(rng.integers(0, 4))
        fill = rng.integers(0, 256, (6, 8)) if k["empty_fill"] else None
        return encode_node(lo, hi, children, child_base, prim_base, exp=exp, slack=slack, p=p, leaf_offsets=leaf_off,
                           empty_fill=fill)

    def emit(self, ids, records, poison_base):
        """the region's node bytes (poison nodes included) and the number of poison nodes in it"""
        root = self.build(np.asarray(ids))
        region = self.layout(root)
        nodes = [n for n in region if n is not None]
        exact_at = int(self.rng.integers(len(nodes))) if self.k["exact_node"] else -1
        out = np.zeros((len(region), 80), np.uint8)
        for j, node in enumerate(region):
            if node is None:
                out[j] = poison_node(poison_base)
        for i, node in enumerate(nodes):
            out[node.index] = self.encode(node, out, records, i == exact_at)
        return out, sum(n is None for n in region)


def poison_node(poison_base):
    """8 leaves of 3 poison records each (records poison_base .. + 23), every one over all of space"""
    B = POISON_BOX
    kids = [(s, -B, B, 3) for s in range(8)]
    return encode_node(-B, B, kids, prim_base=poison_base)


class Generated:
    """nodes, records (`rec_tri`: the triangle of each record slot, -1 = poison), and for two-level scenes blas_offsets and
    tlas_start; `regions`: (first node, node count, nodes unreached, records missing) of each tree the validator checks"""

    def __init__(self, **kw):
        self.__dict__.update(kw)

    def scene(self, tris, stride, seed=0):
        """a Scene over the records (poison records: huge triangles)"""
        rec_tris = np.zeros((len(self.rec_tri), 9), np.float32)
        real = self.rec_tri >= 0
        rec_tris[real] = np.asarray(tris, np.float32).reshape(-1, 9)[self.rec_tri[real]]
        rec_tris[~real] = poison_tris(int((~real).sum()), seed)
        return Scene(self.nodes, rec_tris, self.blas, self.tlas_start, stride)

    def poison_ids(self):
        return np.flatnonzero(self.rec_tri < 0).astype(np.uint32)


def _knobs(overrides):
    unknown = set(overrides) - set(KNOBS)
    assert not unknown, unknown
    return {**KNOBS, **overrides}


def random_cwbvh(tris, seed, **knobs):
    """a flat CWBVH over `tris` (n x 9), root at node 0: Generated(nodes, rec_tri, blas=None, tlas_start=0, regions)"""
    k = _knobs(knobs)
    rng = np.random.default_rng(seed)
    n = len(tris)
    records = []
    if n == 0:
        return Generated(nodes=np.zeros((0, 80), np.uint8), rec_tri=np.zeros(0, np.int64), blas=None, tlas_start=0, regions=[])
    plo, phi = tri_bounds(tris)
    g = _Gen(rng, k, plo, phi)
    records.extend([-1] * 24)                                               # the poison block the poison nodes point at
    nodes, n_poison_nodes = g.emit(np.arange(n), records, 0)
    rec_tri = np.array(records, np.int64)
    out = Generated(nodes=nodes, rec_tri=rec_tri, blas=None, tlas_start=0,
                    regions=[(0, len(nodes), n_poison_nodes, int((rec_tri < 0).sum()))])
    check_indices(out)
    return out


def random_tlas(tris, object_offsets, seed, shared=True, **knobs):
    """a two-level scene: one BLAS per object (records hold global primitive indices), a TLAS over the instance boxes with
    permuted blas_offsets, one BLAS referenced by two instances when `shared`, BLAS regions before and after the TLAS, and a
    poison BLAS behind every unreferenced blas_offsets entry.  Generated(nodes, rec_tri, blas, tlas_start, regions); the TLAS
    region's 'records' are instance slots"""
    k = _knobs(knobs)
    rng = np.random.default_rng(seed)
    plo, phi = tri_bounds(tris)
    records = [-1] * 24                                                     # the poison block of the triangle records
    n_obj = len(object_offsets) - 1
    blas_regions = []
    for o in range(n_obj):
        ids = np.arange(int(object_offsets[o]), int(object_offsets[o + 1]))
        region, n_poison = _Gen(rng, {**k, "exact_node": k["exact_node"] and o == 0}, plo, phi).emit(ids, records, 0)
        blas_regions.append((region, n_poison, len(ids)))
    poison_blas = poison_node(0)[None]
    # instances: one per object, plus a second instance of object 0
    inst_obj = list(range(n_obj)) + ([0] if shared and n_obj else [])
    off = [int(x) for x in object_offsets]
    ilo = np.stack([plo[off[o]:off[o + 1]].min(axis=0) for o in inst_obj])
    ihi = np.stack([phi[off[o]:off[o + 1]].max(axis=0) for o in inst_obj])
    slots_rec = [-1] * 24                                                   # instance slots; -1: a poison entry
    tk = {**k, "exact_node": False}
    tlas, tlas_poison = _Gen(rng, tk, ilo, ihi).emit(np.arange(len(inst_obj)), slots_rec, 0)
    # node array: a random split of the BLAS regions before / after the TLAS, the poison BLAS somewhere among them
    parts = [("blas", i) for i in range(n_obj)] + [("poison", 0)]
    parts = [parts[i] for i in rng.permutation(len(parts))]
    cut = int(rng.integers(1, len(parts)))                                  # BLAS nodes before and after the TLAS
    parts = parts[:cut] + [("tlas", 0)] + parts[cut:]
    chunks, base = [], 0
    where = {}
    for kind, i in parts:
        arr = {"blas": lambda: blas_regions[i][0], "poison": lambda: poison_blas, "tlas": lambda: tlas}[kind]()
        where[(kind, i)] = base
        chunks.append(arr)
        base += len(arr)
    nodes = np.concatenate(chunks)
    tlas_start = where[("tlas", 0)]
    blas = np.array([where[("blas", inst_obj[s])] if s >= 0 else where[("poison", 0)] for s in slots_rec], np.uint32)
    rec_tri = np.array(records, np.int64)
    n_rec = len(rec_tri)
    regions = [(where[("blas", o)], len(blas_regions[o][0]), blas_regions[o][1], n_rec - blas_regions[o][2]) for o in range(n_obj)]
    regions.append((tlas_start, len(tlas), tlas_poison, int(sum(s < 0 for s in slots_rec))))
    out = Generated(nodes=nodes, rec_tri=rec_tri, blas=blas, tlas_start=tlas_start, regions=regions,
                    inst_lo=np.array([ilo[s] if s >= 0 else (0, 0, 0) for s in slots_rec], np.float32).reshape(-1, 3),
                    inst_hi=np.array([ihi[s] if s >= 0 else (0, 0, 0) for s in slots_rec], np.float32).reshape(-1, 3))
    check_indices(out)
    return out


def decode(node):
    """(imask, child_base, prim_base, [(slot, meta)] of the used slots) of an 80-byte node"""
    cb, pb = node[16:24].view(np.uint32)
    return int(node[15]), int(cb), int(pb), [(s, int(node[24 + s])) for s in range(8) if node[24 + s]]


def check_indices(g):
    """every node, record and blas_offsets index the tree holds, poison included, lies inside its array; leaf ranges of a
    node are disjoint"""
    N, R = len(g.nodes), len(g.rec_tri)
    if g.blas is not None:
        assert (g.blas < N).all()
        spans = sorted((b, n) for b, n, _, _ in g.regions) + [(int(b), 1) for b in set(g.blas.tolist()) - {r[0] for r in g.regions}]
    else:
        spans = [(0, N)] if N else []
    spans.sort()
    covered = sum(n for _, n in spans)
    assert covered == N, (covered, N)
    for base, size in spans:
        tlas = g.blas is not None and base == g.tlas_start
        for j in range(base, base + size):
            imask, cb, pb, used = decode(g.nodes[j])
            assert imask == 0 or cb + bin(imask).count("1") <= size, (j, cb, imask, size)
            bits = 0
            for s, meta in used:
                if meta == 0x20 | (24 + s):
                    assert imask >> s & 1
                    continue
                cnt = {1: 1, 3: 2, 7: 3}[meta >> 5]
                off = meta & 31
                assert off + cnt <= 24
                r = ((1 << cnt) - 1) << off
                assert not bits & r, f"node {j}: leaf ranges overlap"
                bits |= r
                limit = len(g.blas) if tlas else R
                assert pb + off + cnt <= limit, (j, pb, off, cnt, limit)
