"""oracle/pyref.py — second, independently written restatement (object style, pure Python).

TEST INFRASTRUCTURE ONLY (never imported by the product path).  PARITY UNPINNED: see the
header of oracle/nnet_oracle.cpp.  This file exists so that two restatements written in
different styles (C++ handle arrays vs Python objects that mirror the Java classes) can be
required to agree bit-for-bit; it is used for small n only.

Citations are file:line into /root/reference.
"""
import math

DBL_MAX = 1.7976931348623157e308
M64 = (1 << 64) - 1


def splitmix64(z):
    """splitmix64's output function (Steele, Lea, Flood 2014), mod 2**64: restated here independently of csrc/fnn_record.h."""
    z = (z + 0x9E3779B97F4A7C15) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def draw_digest_term(k, i, j):
    """The strategy record's term for draw k of an iteration going from position i to position j."""
    return splitmix64(splitmix64(k) ^ (((i & 0xFFFFFFFF) << 32) | (j & 0xFFFFFFFF)))


class JavaRandom:
    """java.util.Random(seed): 48-bit LCG, nextInt(bound) with the documented rejection loop."""

    def __init__(self, seed):
        self.s = (seed ^ 0x5DEECE66D) & ((1 << 48) - 1)
        self.calls = 0  # LCG steps taken

    def _next(self, bits):
        self.calls += 1
        self.s = (self.s * 0x5DEECE66D + 0xB) & ((1 << 48) - 1)
        v = self.s >> (48 - bits)
        if v >= 1 << 31:
            v -= 1 << 32
        return v

    def next_int(self, bound):
        r = self._next(31)
        m = bound - 1
        if bound & m == 0:
            return (bound * r) >> 31
        u = r
        while True:
            r = u % bound
            t = (u - r + m) & 0xFFFFFFFF
            if t < 0x80000000:
                return r
            u = self._next(31)


class NetNode:  # NetNode.java:5-15
    __slots__ = ("id", "distID", "positionID", "nbr", "ch1", "ch2", "next", "prev", "Sx")

    def __init__(self):
        self.id = 0
        self.distID = 0
        self.positionID = 0
        self.nbr = None
        self.ch1 = None
        self.ch2 = None
        self.next = None
        self.prev = None
        self.Sx = 0.0


class NeighborNet:
    def __init__(self, D, ntax, mode="canonical", seed=0, mult=5, additive=False, fallback=1024):
        self.D = D  # list of lists, mutated
        self.ntax = ntax
        self.mode = mode
        self.rng = JavaRandom(seed)
        self.mult = mult
        self.additive = additive
        self.fallback = fallback
        self.Cx = None
        self.Cy = None
        self.best = 0.0
        self.trace = []
        self.first_time = True
        self.top = 0
        self.row_perm = []
        self.record = []  # Random modes: per iteration [draws, rejected, remapped, digest] (fnn_ctx_strategy_record)

    # the cluster-distance ladder, e.g. NetMakerOriginal.java:218-225
    def dpq(self, p, q):
        D = self.D
        if p.nbr is None and q.nbr is None:
            return D[p.distID][q.distID]
        if p.nbr is not None and q.nbr is None:
            return (D[p.distID][q.distID] + D[p.nbr.distID][q.distID]) / 2.0
        if p.nbr is None and q.nbr is not None:
            return (D[p.distID][q.distID] + D[p.distID][q.nbr.distID]) / 2.0
        return (D[p.distID][q.distID] + D[p.distID][q.nbr.distID] + D[p.nbr.distID][q.distID]
                + D[p.nbr.distID][q.nbr.distID]) / 4.0

    def run(self):  # NetMakerOriginal.java:129-162
        n = self.ntax
        if n <= 3:
            return list(range(n + 1))
        nodes = [None] * n
        for i in range(n, 0, -1):
            t = NetNode()
            t.id = i
            t.positionID = i - 1
            t.distID = i - 1
            nodes[i - 1] = t
        self.nodes = nodes
        self.amalgs = []
        # initialize :164-191 (all singletons at this point)
        for p in nodes:
            for j in range(p.positionID + 1, n):
                q = nodes[j]
                v = self.D[p.distID][q.distID]
                p.Sx += v
                q.Sx += v
        num_nodes = self.agglom(n)
        return self.expand(num_nodes)

    def find_default(self, num_active, num_clusters):  # :197-236
        nodes = self.nodes
        self.Cx = self.Cy = None
        self.best = DBL_MAX
        for i in range(num_active):
            p = nodes[i]
            if p.nbr is not None and p.nbr.id < p.id:
                continue
            for j in range(i):
                q = nodes[j]
                if q.nbr is not None and q.nbr.id < q.id:
                    continue
                if q.nbr is p:
                    continue
                Q = (float(num_clusters) - 2.0) * self.dpq(p, q) - p.Sx - q.Sx
                if (self.Cx is None or Q < self.best) and p.nbr is not q:
                    self.Cx, self.Cy, self.best = p, q, Q

    def find_row_min(self, p, found, num_active, num_clusters):  # NeighborNetLocal.java:88-157
        if id(p) in found:
            return found[id(p)]
        if p.nbr is not None and id(p.nbr) in found:
            return found[id(p.nbr)]
        mins = []
        my_min = DBL_MAX
        for row in range(num_active):
            q = self.nodes[row]
            if p is q or (p.nbr is not None and p.nbr is q):
                continue
            Q = (float(num_clusters) - 2.0) * self.dpq(p, q) - p.Sx - q.Sx
            if Q < my_min:
                my_min = Q
                mins = [(p, q, Q)]
            elif Q == my_min:
                mins.append((p, q, Q))
        found[id(p)] = mins
        return mins

    def find_relaxed(self, num_active, num_clusters):  # NeighborNetLocal.java:170-264
        if self.additive:
            raise NotImplementedError("pyref covers relaxed without -additive")
        found = {}
        my_minimums = []
        rp = self.row_perm
        if self.first_time:
            rp[:] = list(range(self.ntax))
            self.first_time = False
            self.top = self.ntax - 1
        i = self.top + 1
        while i > 0:
            swap_cell = self.rng.next_int(i)
            if rp[swap_cell] >= num_active:
                rp[swap_cell], rp[self.top] = rp[self.top], rp[swap_cell]
                if i == self.top + 1:
                    i -= 1
                else:
                    i += 1
                self.top -= 1
                i -= 1
                continue
            rp[i - 1], rp[swap_cell] = rp[swap_cell], rp[i - 1]
            p = self.nodes[rp[i - 1]]
            if p.nbr is not None and p.nbr.id < p.id:
                i -= 1
                continue
            for (_, row, _) in self.find_row_min(p, found, num_active, num_clusters):
                for t in self.find_row_min(row, found, num_active, num_clusters):
                    tr = t[1]
                    if (tr is p or (tr.nbr is not None and tr.nbr is p)
                            or (tr.nbr is not None and p.nbr is not None and tr.nbr is p.nbr)
                            or (p.nbr is not None and tr is p.nbr)):
                        my_minimums.append(t)
                        break
            if my_minimums:
                c = my_minimums[self.rng.next_int(len(my_minimums))]
                self.Cx, self.Cy = c[0], c[1]
                return
            i -= 1

    def find_random(self, num_active, num_clusters):  # NeighborNetRandom.java:130-178
        nodes = self.nodes
        self.best = DBL_MAX
        lg = int(math.ceil(math.log10(num_active)))
        amount = {"random_logn": lg, "random_n": num_active, "random_nlogn": lg * num_active}[self.mode] * self.mult
        i = self.rng.next_int(num_active)
        self.Cx = self.Cy = None
        row = self.record[-1]
        row[0] = amount
        for k in range(amount):
            calls_before = self.rng.calls
            if nodes[i].nbr is not None:
                inbr = nodes[i].nbr.positionID
                j = j0 = self.rng.next_int(num_active - 2)
                if i == j and num_active - 1 == inbr:
                    j = num_active - 2
                elif i == j and num_active - 1 != inbr:
                    j = num_active - 1
                elif inbr == j and num_active - 2 == i:
                    j = num_active - 1
                elif inbr == j and num_active - 2 != i:
                    j = num_active - 2
            else:
                j = j0 = self.rng.next_int(num_active - 1)
                if i == j:
                    j = num_active - 1
            row[1] += self.rng.calls - calls_before > 1
            row[2] += j != j0
            row[3] = (row[3] + draw_digest_term(k, i, j)) & M64
            p, q = nodes[i], nodes[j]
            Q = (float(num_clusters) - 2.0) * self.dpq(p, q) - p.Sx - q.Sx
            if (self.Cx is None or Q < self.best) and p.nbr is not q:
                self.Cx, self.Cy, self.best = p, q, Q
            i = j

    def compute_rx(self, z, Cx, Cy, num_active):  # NetMakerOriginal.java:549-561
        rx = 0.0
        for i in range(num_active):
            p = self.nodes[i]
            if p is Cx or p is Cx.nbr or p is Cy or p is Cy.nbr or p.nbr is None:
                rx += self.D[z.distID][p.distID]
            else:
                rx += self.D[z.distID][p.distID] / 2.0
        return rx

    def subtract(self, p, x):  # :681-696
        if p is not x and p is not x.nbr and (p.nbr is None or p.nbr.id > p.id):
            v = self.dpq(p, x)
            p.Sx -= v
            if p.nbr is not None:
                p.nbr.Sx -= v

    def agg3way(self, x, y, z, num_nodes, num_active):  # :589-674
        D, nodes = self.D, self.nodes
        u = NetNode()
        u.id = num_nodes + 1
        u.ch1, u.ch2 = x, y
        v = NetNode()
        v.id = num_nodes + 2
        v.ch1, v.ch2 = y, z
        nodes[x.positionID] = u
        u.positionID, u.distID = x.positionID, x.distID
        nodes[z.positionID] = v
        v.positionID, v.distID = z.positionID, z.distID
        nodes[y.positionID] = nodes[num_active - 1]
        nodes[y.positionID].positionID = y.positionID
        nodes[num_active - 1] = None
        u.nbr, v.nbr = v, u
        for i in range(num_active - 1):
            p = nodes[i]
            D[u.distID][p.distID] = D[p.distID][u.distID] = (2.0 / 3.0) * D[x.distID][p.distID] + D[y.distID][p.distID] / 3.0
            D[v.distID][p.distID] = D[p.distID][v.distID] = (2.0 / 3.0) * D[z.distID][p.distID] + D[y.distID][p.distID] / 3.0
        D[u.distID][u.distID] = D[v.distID][v.distID] = 0.0
        self.amalgs.append(u)
        return u

    def handle(self, Cx, Cy, num_nodes, num_active, num_clusters):  # :397-515
        D = self.D
        x, y = Cx, Cy
        rcx = rcxn = rcy = rcyn = 0.0
        if Cx.nbr is not None or Cy.nbr is not None:
            rcx = self.compute_rx(Cx, Cx, Cy, num_active)
            if Cx.nbr is not None:
                rcxn = self.compute_rx(Cx.nbr, Cx, Cy, num_active)
            rcy = self.compute_rx(Cy, Cx, Cy, num_active)
            if Cy.nbr is not None:
                rcyn = self.compute_rx(Cy.nbr, Cx, Cy, num_active)
        m = num_clusters + (Cx.nbr is not None) + (Cy.nbr is not None)
        best = (float(m) - 2.0) * D[Cx.distID][Cy.distID] - rcx - rcy
        if Cx.nbr is not None:
            Q = (float(m) - 2.0) * D[Cx.nbr.distID][Cy.distID] - rcxn - rcy
            if Q < best:
                x, y, best = Cx.nbr, Cy, Q
        if Cy.nbr is not None:
            Q = (float(m) - 2.0) * D[Cx.distID][Cy.nbr.distID] - rcx - rcyn
            if Q < best:
                x, y, best = Cx, Cy.nbr, Q
        if Cx.nbr is not None and Cy.nbr is not None:
            Q = (float(m) - 2.0) * D[Cx.nbr.distID][Cy.nbr.distID] - rcxn - rcyn
            if Q < best:
                x, y, best = Cx.nbr, Cy.nbr, Q
        self.best = best
        rec = [x.id, y.id]
        for i in range(num_active):
            p = self.nodes[i]
            if i != x.positionID and i != y.positionID:
                self.subtract(p, x)
                self.subtract(p, y)
        if x.nbr is None and y.nbr is None:
            x.nbr, y.nbr = y, x
            u = x
            num_clusters -= 1
            kind = 2
        elif x.nbr is None:
            u = self.agg3way(x, y, y.nbr, num_nodes, num_active)
            num_nodes += 2
            num_active -= 1
            num_clusters -= 1
            kind = 3
        elif y.nbr is None or num_active == 4:
            u = self.agg3way(y, x, x.nbr, num_nodes, num_active)
            num_nodes += 2
            num_active -= 1
            num_clusters -= 1
            kind = 3
        else:
            x2, y2 = x.nbr, y.nbr
            u1 = self.agg3way(x2, x, y, num_nodes, num_active)
            u = self.agg3way(u1, u1.nbr, y2, num_nodes + 2, num_active - 1)
            num_nodes += 4
            num_active -= 2
            num_clusters -= 1
            kind = 4
        # updateClusterDistances :517-536
        u.Sx = 0.0
        u.nbr.Sx = 0.0
        for i in range(num_active):
            p = self.nodes[i]
            if (p.nbr is None or p.nbr.id > p.id) and u.nbr is not p and u is not p:
                if p.nbr is None:
                    v = (D[p.distID][u.distID] + D[p.distID][u.nbr.distID]) / 2.0
                else:
                    v = (D[p.distID][u.distID] + D[p.distID][u.nbr.distID] + D[p.nbr.distID][u.distID]
                         + D[p.nbr.distID][u.nbr.distID]) / 4.0
                p.Sx += v
                if p.nbr is not None:
                    p.nbr.Sx += v
                u.Sx += v
        u.nbr.Sx = u.Sx
        return num_nodes, num_active, num_clusters, rec, kind

    def agglom(self, num_nodes):  # :331-395
        D, nodes = self.D, self.nodes
        num_active = num_clusters = num_nodes
        while num_active > 3:
            self.record.append([0, 0, 0, 0])
            if num_active == 4 and num_clusters == 2:
                p = nodes[0]
                q = nodes[1] if p.nbr is not nodes[1] else nodes[2]
                if D[p.distID][q.distID] + D[p.nbr.distID][q.nbr.distID] < D[p.distID][q.nbr.distID] + D[p.nbr.distID][q.distID]:
                    xid = q.id
                    self.agg3way(p, q, q.nbr, num_nodes, num_active)
                else:
                    xid = q.nbr.id
                    self.agg3way(p, q.nbr, q, num_nodes, num_active)
                self.trace.append((num_active, num_clusters, p.id, q.id, xid, 0, 5, 0.0))
                num_nodes += 2
                break
            if num_active <= self.fallback or self.mode == "canonical":
                self.find_default(num_active, num_clusters)
            elif self.mode == "relaxed":
                self.find_relaxed(num_active, num_clusters)
            else:
                self.find_random(num_active, num_clusters)
            if self.Cx.id > self.Cy.id:
                self.Cx, self.Cy = self.Cy, self.Cx
            m0, c0, cx, cy = num_active, num_clusters, self.Cx.id, self.Cy.id
            num_nodes, num_active, num_clusters, rec, kind = self.handle(self.Cx, self.Cy, num_nodes, num_active, num_clusters)
            self.trace.append((m0, c0, cx, cy, rec[0], rec[1], kind, self.best))
        return num_nodes

    def expand(self, num_nodes):  # :246-325
        nodes = self.nodes
        x, y, z = nodes[0], nodes[1], nodes[2]
        x.next, y.next, z.next = y, z, x
        x.prev, y.prev, z.prev = z, x, y
        while self.amalgs:
            u = self.amalgs.pop()
            v = u.nbr
            x, y, z = u.ch1, u.ch2, v.ch2
            if v is not u.next:
                u, v = v, u
                x, z = z, x
            x.prev = u.prev
            x.prev.next = x
            x.next = y
            y.prev = x
            y.next = z
            z.prev = y
            z.next = v.next
            z.next.prev = z
        while x.id != 1:
            x = x.next
        ordering = [0] * (self.ntax + 1)
        a, t = x, 0
        while True:
            t += 1
            ordering[t] = a.id
            a = a.next
            if a is x:
                break
        return ordering


def live_design_matrix(n, ordering):
    """The dense system of FastNN.java:401-441: row = taxon pair (file order), column = split
    (i,j) = {ordering[i+1..j]}.  Returned as a list of rows of 0/1 (for scipy NNLS, small n)."""
    splits = []
    for i in range(n):
        s = set()
        for j in range(i + 1, n):
            s.add(ordering[j])
            splits.append(frozenset(s))
    pairs = [(i + 1, j + 1) for i in range(n) for j in range(i + 1, n)]
    return [[0.0 if ((a in sp) == (b in sp)) else 1.0 for sp in splits] for (a, b) in pairs]
