"""Seeded programs over ONE 2-D shape that mix statement forms inside long pending stretches: integer, float and bool arrays,
arithmetic / comparisons / logical ops / where / minimum / maximum / abs / astype, floor division and modulo on integers,
in-place updates, strided and reversed slice views as operands, sliced assignments, transposed and broadcast (row / column)
operands, global and axis reductions.  Integer-valued data: every result is exact in NumPy and here.  Aimed at the lowering
(forwarding, dead stores, register allocation, SINCOS-free) and at the fuser's alias rules under the DAG's statement orders."""
import numpy as onp

R, C = 13, 22


def _h(x):
    return onp.array(x.asarray() if hasattr(x, "asarray") else x)


def expr_program(np, seed, n_actions=40):
    rng = onp.random.RandomState(9000 + seed)
    fa = (lambda x: x.copy()) if np is onp else np.fromarray
    F = [fa(rng.randint(-6, 7, size=(R, C)).astype(onp.float64)) for _ in range(3)]   # float pool
    I = [fa(rng.randint(-6, 7, size=(R, C)).astype(onp.int64)) for _ in range(2)]     # int pool
    row = fa(rng.randint(-3, 4, size=(C,)).astype(onp.float64))
    col = fa(rng.randint(-3, 4, size=(R, 1)).astype(onp.float64))
    sq = fa(rng.randint(-3, 4, size=(C, R)).astype(onp.float64))                     # read through .T
    out = []

    def f():
        return F[int(rng.randint(len(F)))]

    def i():
        return I[int(rng.randint(len(I)))]

    def put(pool, v):
        if len(pool) >= 6:
            del pool[int(rng.randint(len(pool)))]
        pool.append(v)

    def sl():
        a = int(rng.randint(0, R - 4)); b = int(rng.randint(0, C - 6))
        return (slice(a, a + 4), slice(b, b + 6))

    held = []   # temporaries built by one statement, consumed by a LATER one and dropped before anything flushes them
    for _ in range(n_actions):
        k = int(rng.randint(0, 27))
        if k == 0:
            put(F, f() + f() * 2.0)
        elif k == 1:
            put(F, np.where(f() > f(), f(), f() - 1.0))
        elif k == 2:
            put(F, np.minimum(f(), 3.0) - np.maximum(f(), -2.0))
        elif k == 3:
            put(F, abs(f()) + row)                      # row-broadcast operand
        elif k == 4:
            put(F, f() * col)                           # column-broadcast operand
        elif k == 5:
            put(F, f() + sq.T)                          # transposed operand
        elif k == 6:
            put(I, i() * 3 - i())
        elif k == 7:
            put(I, i() // 4 + i() % 5)
        elif k == 8:
            put(F, i().astype(onp.float64) * 0.5 + f())
        elif k == 9:
            put(I, (f() * 2.0).astype(onp.int64) + i())
        elif k == 10:
            m = np.logical_and(f() > 0.0, i() < 2)
            put(F, np.where(m, f(), -f()))
        elif k == 11:
            x = f(); x += f()
        elif k == 12:
            x = f(); x *= 2.0; x -= 1.0
        elif k == 13:
            x = i(); x += i()
        elif k == 14:
            x = f(); x[sl()] = 0.0
        elif k == 15:
            x, y = f(), f(); s1, s2 = sl(), sl(); x[s1] = y[s2] + 1.0          # maybe the same array, maybe overlapping
        elif k == 16:
            x = f(); put(F, x[::-1, :] - x[:, ::-1])                            # reversed views
        elif k == 17:
            x = f(); v = x[1:R:2, 0:C:3]; put(F, f() * 1.0); out.append(_h(v * 2.0))   # strided view read
        elif k == 18:
            out.append(onp.asarray(float(f().sum())))
        elif k == 19:
            out.append(_h((f() + 1.0).sum(axis=int(rng.randint(0, 2)))))
        elif k == 20:
            out.append(onp.asarray(float((f() * 2.0 - f()).max())))
        elif k in (21, 22):
            if len(held) < 2:
                held.append(f() * 2.0 - f() if k == 21 else abs(f()) + 1.0)      # built now ...
        elif k == 23:
            if held:
                x = f(); x[:, :] = held.pop(0)                                    # ... stored whole, statements later
        elif k == 24:
            if held:
                x = f(); w = sl(); x[w] = held.pop()[w]                           # ... or a window of it
        elif k == 25:
            if held:
                put(F, held.pop(0) + f())                                         # ... or consumed as an operand
        elif k == 26:
            if held:
                held.pop()                                                        # ... or dropped unused
        else:
            out.append(_h(F[int(rng.randint(len(F)))] if rng.rand() < 0.5 else I[int(rng.randint(len(I)))]))
    for x in F + I:
        out.append(_h(x))
    return out


def _case(seed):
    def f(np):
        return expr_program(np, seed)

    f.__name__ = "expr_program_%d" % seed
    return f


CASES = [_case(s) for s in range(200)]


def trig_mask_program(np, seed, n_actions=36):
    """sin / cos of shared operands (the SINCOS pairing and the store it moves), sqrt / exp, boolean-mask assignment and
    masked sums, float32 arrays next to float64 ones - around in-place updates and held temporaries.  Compared with a
    tolerance (transcendentals) by the caller."""
    rng = onp.random.RandomState(12000 + seed)
    fa = (lambda x: x.copy()) if np is onp else np.fromarray
    F = [fa(rng.randint(-6, 7, size=(R, C)).astype(onp.float64) * 0.25) for _ in range(3)]
    G = [fa(rng.randint(-6, 7, size=(R, C)).astype(onp.float32)) for _ in range(2)]      # float32 pool (array-with-array ops only)
    out = []
    held = []

    def f():
        return F[int(rng.randint(len(F)))]

    def g():
        return G[int(rng.randint(len(G)))]

    def put(pool, v):
        if len(pool) >= 5:
            del pool[int(rng.randint(len(pool)))]
        pool.append(v)

    for _ in range(n_actions):
        k = int(rng.randint(0, 18))
        if k == 0:
            x = f(); put(F, np.sin(x) * np.sin(x) + np.cos(x) * np.cos(x))
        elif k == 1:
            x = f(); s = np.sin(x); y = f(); y += 1.0; c = np.cos(x); put(F, s - c)       # an in-place update between the pair
        elif k == 2:
            x = f(); s = np.sin(x); y = f(); u = y * 2.0; y[:, :] = np.cos(x); put(F, u + s)   # the pair's second half overwrites y
        elif k == 3:
            # (+ 0.25 keeps sqrt's slope at most 1: an operand such as sin(x)**2 + cos(x)**2 - 1.0 is rounding noise, and
            # sqrt(abs(.)) of it would turn one ulp of another sin / cos implementation into 1e-8)
            put(F, np.sqrt(abs(f()) + 0.25) + np.exp(np.minimum(f(), 2.0)))
        elif k == 4:
            x = f(); m = g() > 0.0; x[m] = 0.5                 # boolean-mask assignment (mask from exact data: no comparison
                                                               # can fall differently on another sin / cos implementation)
        elif k == 5:
            x = f(); m = g() > g(); out.append(onp.asarray(float(x[m].sum())))            # masked sum
        elif k == 6:
            put(G, np.minimum(np.maximum(g() + g(), -8.0), 8.0))      # (kept small: float32 results stay exact, so NumPy's
        elif k == 7:                                                   # rounding of every temporary cannot differ)
            put(G, np.minimum(np.maximum(g() * g() - g(), -8.0), 8.0))
        elif k == 8:
            put(F, g().astype(onp.float64) * 0.5 + f())
        elif k == 9:
            put(G, np.minimum(np.maximum((g().astype(onp.float64) * 2.0).astype(onp.float32) - g(), -8.0), 8.0))
        elif k == 10:
            x = g(); x += g()
        elif k in (11, 12):
            if len(held) < 2:
                x = f(); held.append(np.cos(x) if k == 11 else np.sin(x) + 1.0)
        elif k == 13:
            if held:
                x = f(); x[:, :] = held.pop(0)
        elif k == 14:
            if held:
                put(F, held.pop() * 2.0)
        elif k == 15:
            out.append(_h(f()))
        elif k == 16:
            out.append(onp.asarray(float((np.sin(f()) + np.cos(f())).sum())))
        else:
            x = f(); x -= f()
    for x in F + G:
        out.append(_h(x))
    return out


def _tcase(seed):
    def f(np):
        return trig_mask_program(np, seed)

    f.__name__ = "trig_mask_program_%d" % seed
    return f


TRIG_CASES = [_tcase(s) for s in range(120)]


def view_program(np, seed, n_actions=34):
    """Writes THROUGH views: strided, reversed and transposed targets, row / column broadcast assignment, windows of one array
    combined with shifted windows of the same or another array (the stencil form, also in place), slices of slices,
    axis sums fed back as broadcast operands.  Integer-valued float64 / int64 data (weights 2, 0.5, -1): exact."""
    rng = onp.random.RandomState(15000 + seed)
    fa = (lambda x: x.copy()) if np is onp else np.fromarray
    A = [fa(rng.randint(-4, 5, size=(R, C)).astype(onp.float64) * 2.0) for _ in range(3)]
    T = [fa(rng.randint(-4, 5, size=(C, R)).astype(onp.float64) * 2.0)]                    # transposed shape
    out = []

    def a():
        return A[int(rng.randint(len(A)))]

    def put(v):
        if len(A) >= 5:
            del A[int(rng.randint(len(A)))]
        A.append(v)

    def win(h, w):
        i = int(rng.randint(0, R - h + 1)); j = int(rng.randint(0, C - w + 1))
        return (slice(i, i + h), slice(j, j + w))

    for _ in range(n_actions):
        k = int(rng.randint(0, 16))
        if k == 0:
            x = a(); x[::2, :] = a()[1::2, :][:x[::2, :].shape[0], :] if R % 2 == 0 else a()[::2, :] * 0.5     # strided target
        elif k == 1:
            x = a(); x[:, ::-1] = a() - 1.0                                          # reversed target
        elif k == 2:
            x = a(); x[::-1, ::3] = a()[:, ::3] * 2.0                                # reversed + strided target
        elif k == 3:
            t = T[0]; t.T[:, :] = a() + 1.0                                          # transposed target
        elif k == 4:
            put(T[0].T * 0.5 + a())                                                  # transposed operand
        elif k == 5:
            x = a(); x[2:5, :] = a()[0, :]                                           # row broadcast into a window
        elif k == 6:
            x = a(); x[:, 3:7] = a()[:, 5:6]                                         # column broadcast into a window
        elif k == 7:
            x = a(); h, w = 6, 9; w1, w2, w3 = win(h, w), win(h, w), win(h, w)
            x[w1] = x[w2] * 0.5 + a()[w3]                                            # shifted windows, possibly of the same array
        elif k == 8:
            x, y = a(), a()
            y[1:-1, 1:-1] = x[:-2, 1:-1] + x[2:, 1:-1] + x[1:-1, :-2] + x[1:-1, 2:] - 4.0 * x[1:-1, 1:-1]   # 5-point stencil, maybe in place
        elif k == 9:
            x = a(); v = x[2:11, 4:20]; v[1:4, ::2] = 7.0; out.append(_h(v[::2, 1:5] * 2.0))   # slices of slices
        elif k == 10:
            x = a(); put(x - x.sum(axis=0) * 0.5)                                    # axis sum fed back as a row operand
        elif k == 11:
            x = a(); s = x.sum(axis=1); out.append(_h(s)); put(x * 2.0 - a())
        elif k == 12:
            x = a(); x += a()[::-1, ::-1]                                            # in place from a reversed view
        elif k == 13:
            x = a(); x[win(4, 5)] *= 2.0                                             # in place on a window
        elif k == 14:
            out.append(_h(a()))
        else:
            out.append(onp.asarray(float((a()[1:, :] - a()[:-1, :]).sum())))
    for x in A + T:
        out.append(_h(x))
    return out


def _vcase(seed):
    def f(np):
        return view_program(np, seed)

    f.__name__ = "view_program_%d" % seed
    return f


VIEW_CASES = [_vcase(s) for s in range(120)]


def api_program(np, seed, n_actions=30):
    """Library-level calls inside pending stretches, with the sources updated in place AFTER the call and before anything is
    read: cumsum (a direct scan at call time), concatenate / stack / pad (slice assignments into a new array), reshape_copy
    (a direct redistribution at call time), clip, where, axis sums, transposes, unit-dim reshapes, broadcast_to, astype."""
    rng = onp.random.RandomState(18000 + seed)
    fa = (lambda x: x.copy()) if np is onp else np.fromarray
    A = [fa(rng.randint(-4, 5, size=(R, C)).astype(onp.float64)) for _ in range(3)]
    V = [fa(rng.randint(-4, 5, size=(150,)).astype(onp.float64)) for _ in range(2)]
    out = []

    def a():
        return A[int(rng.randint(len(A)))]

    def v():
        return V[int(rng.randint(len(V)))]

    def bump(x):
        if rng.rand() < 0.6:
            x += 1.0            # the source changes right after the call: the result must not see it

    for _ in range(n_actions):
        k = int(rng.randint(0, 16))
        if k == 0:
            x = v(); c = np.cumsum(x); bump(x); out.append(_h(c))
        elif k == 1:
            x = a(); ax = int(rng.randint(0, 2)); c = np.cumsum(x * 2.0, axis=ax); bump(x); out.append(_h(c))
        elif k == 2:
            x, y = a(), a(); c = np.concatenate([x, y * 2.0], axis=int(rng.randint(0, 2))); bump(x); bump(y); out.append(_h(c + 1.0))
        elif k == 3:
            x, y = v(), v(); c = np.stack([x, y - 1.0]); bump(y); out.append(_h(c))
        elif k == 4:
            x = a(); c = np.pad(x, ((1, 2), (0, 3)), mode="constant", constant_values=7); bump(x); out.append(_h(c))
        elif k == 5:
            x = a(); c = (x.reshape_copy((C, R)) if np is not onp else onp.reshape(x, (C, R)).copy()); bump(x); out.append(_h(c * 2.0))
        elif k == 6:
            x = a(); c = np.clip(x, -2.0, 3.0); bump(x); A.append(c); del A[0]
        elif k == 7:
            x = a(); c = np.where(x > 0.0, x, -x); bump(x); out.append(_h(c))
        elif k == 8:
            x = a(); m = x.sum(axis=0) * 0.5; bump(x); out.append(_h(m))   # (mean is sum * (1/n) here, like the reference: not bit-equal to NumPy's)
        elif k == 9:
            x = a(); t = x.T; y = t * 2.0; bump(x); out.append(_h(y))
        elif k == 10:
            x = v(); e = np.expand_dims(x, 0); y = e + 1.0; bump(x); out.append(_h(y))
        elif k == 11:
            x = v(); b = np.broadcast_to(x, (4, 150)); y = b * 2.0; bump(x); out.append(_h(y))
        elif k == 12:
            x = a(); i = (x * 2.0).astype(onp.int64); bump(x); out.append(_h(i // 3))
        elif k == 13:
            x = a(); x[2:9, 3:12] = x[3:10, 4:13] + 1.0
        elif k == 14:
            x = a(); s = float(x.sum()); x -= 1.0; out.append(onp.asarray(s + float(x.sum())))
        else:
            x = v(); V.append(x[::-1] * 1.0 + v()); del V[0]
    for x in A + V:
        out.append(_h(x))
    return out


def _acase(seed):
    def f(np):
        return api_program(np, seed)

    f.__name__ = "api_program_%d" % seed
    return f


API_CASES = [_acase(s) for s in range(100)]


SHAPES = [(7,), (3, 5), (1,), (0,), (4, 0), (200,), (101,), (6, 7, 8), (2, 3, 4, 5), (1, 150), (150, 1), (99,), (100,)]


def shape_program(np, seed, n_actions=26):
    """Shapes around the distribution threshold (arrays under 100 elements live on one rank), single elements, empty arrays,
    3-D and 4-D arrays, unit dims - int64 / float64 / bool / int32 data, elementwise ops, comparisons, where, reductions
    over all axes and over one, in-place updates, slices, transposes, scalar reads."""
    rng = onp.random.RandomState(21000 + seed)
    fa = (lambda x: x.copy()) if np is onp else np.fromarray
    out = []
    for _round in range(3):
        shp = SHAPES[int(rng.randint(len(SHAPES)))]
        P = [fa(rng.randint(-5, 6, size=shp).astype(onp.float64)) for _ in range(2)]
        Q = [fa(rng.randint(-5, 6, size=shp).astype(onp.int64)), fa(rng.randint(0, 5, size=shp).astype(onp.int32))]
        nd = len(shp)
        for _ in range(n_actions // 3):
            k = int(rng.randint(0, 14))
            p, q = P[int(rng.randint(2))], Q[0]
            if k == 0:
                P[int(rng.randint(2))] = p * 2.0 - P[int(rng.randint(2))]
            elif k == 1:
                P[int(rng.randint(2))] = np.where(p > 0.0, p, p * -1.0) + q.astype(onp.float64)
            elif k == 2:
                Q[0] = q * 2 - Q[0] // 3
            elif k == 3:
                Q[1] = Q[1] + Q[1] % 3              # int32 with int32
            elif k == 4:
                p += 1.0
            elif k == 5:
                q -= 2
            elif k == 6:
                out.append(onp.asarray(float(p.sum())))
            elif k == 7:
                out.append(onp.asarray(int(q.sum())))
            elif k == 8 and nd >= 2 and 0 not in shp:
                out.append(_h(p.sum(axis=int(rng.randint(nd)))))
            elif k == 9 and nd >= 2:
                out.append(_h(np.transpose(p) * 2.0))
            elif k == 10 and shp[0] >= 3:
                s = (slice(1, shp[0] - 1),) + (slice(None),) * (nd - 1)
                p[s] = p[s] * 0.5
            elif k == 11 and 0 not in shp:
                idx = tuple(int(rng.randint(n)) for n in shp)
                out.append(onp.asarray(float(p[idx])))          # a single element, read back as a scalar
            elif k == 12:
                out.append(_h((p > 0.0) & (q < 2) if np is onp else np.logical_and(p > 0.0, q < 2)))
            else:
                out.append(_h(Q[1] * 2))
        out += [_h(x) for x in P + Q]
    return out


def _scase(seed):
    def f(np):
        return shape_program(np, seed)

    f.__name__ = "shape_program_%d" % seed
    return f


SHAPE_CASES = [_scase(s) for s in range(100)]


def _st_cross(a):
    return a[-1, 0] + a[1, 0] + a[0, -1] + a[0, 1] - 4.0 * a[0, 0]


def _st_row(a, b):
    return a[0, -2] + a[0, 2] - 2.0 * b[0, 0]


def skeleton_program(np, seed, n_actions=24):
    """The skeletons (functions traced into the op list) inside pending stretches, their sources updated right after the
    call: smap / smap_index with Python and string lambdas, sreduce with +, max, sstencil / stencil with relative indices,
    scumulative with + and max, fromfunction, triu."""
    rng = onp.random.RandomState(24000 + seed)
    fa = (lambda x: x.copy()) if np is onp else np.fromarray
    A = [fa(rng.randint(-4, 5, size=(R, C)).astype(onp.float64)) for _ in range(3)]
    V = [fa(rng.randint(-4, 5, size=(160,)).astype(onp.int64)) for _ in range(2)]
    # two arrays with padded shards (local_border: the neighbours' edges are received into the ring of the block)
    fb = (lambda x: x.copy()) if np is onp else (lambda x: np.fromarray(x, local_border=2))
    B = [fb(rng.randint(-4, 5, size=(R, C)).astype(onp.float64)) for _ in range(2)]
    out = []
    is_np = np is onp

    def a():
        return A[int(rng.randint(len(A)))]

    def v():
        return V[int(rng.randint(len(V)))]

    def bump(x, by):
        if rng.rand() < 0.6:
            x += by

    for _ in range(n_actions):
        k = int(rng.randint(0, 16))
        if k == 12:
            x = B[int(rng.randint(2))]
            if is_np:
                r = onp.zeros((R, C)); r[1:-1, 1:-1] = x[:-2, 1:-1] + x[2:, 1:-1] + x[1:-1, :-2] + x[1:-1, 2:] - 4.0 * x[1:-1, 1:-1]
            else:
                r = np.sstencil(np.stencil(_st_cross), x)
            bump(x, 1.0); out.append(_h(r))
        elif k == 13:
            x, y = B[0], B[1]
            if is_np:
                r = onp.zeros((R, C)); r[:, 2:-2] = x[:, :-4] + x[:, 4:] - 2.0 * y[:, 2:-2]
            else:
                r = np.stencil(_st_row)(x, y)
            bump(x, 2.0); out.append(_h(r))
        elif k == 14:
            x = B[int(rng.randint(2))]; x += a() * 0.5                     # padded and plain arrays in one statement
        elif k == 15:
            x = B[int(rng.randint(2))]; x[1:-1, 1:-1] = x[:-2, 1:-1] * 0.5 + x[1:-1, 2:]   # in place through shifted views of a padded array
        elif k == 0:
            x, y = v(), v()
            r = 3 * x - 7 * y if is_np else np.smap(lambda p, q: 3 * p - 7 * q, x, y)
            bump(x, 1); out.append(_h(r))
        elif k == 1:
            x = v()
            r = 3 * x - 7 if is_np else np.smap("lambda x: 3*x-7", x)
            bump(x, 2); out.append(_h(r))
        elif k == 2:
            x = v()
            r = 7 * onp.arange(160) + x if is_np else np.smap_index(lambda i, p: 7 * i + p, x)
            bump(x, 1); out.append(_h(r))
        elif k == 3:
            x = v()
            r = (x * x).sum() if is_np else np.sreduce(lambda p: p * p, lambda s, t: s + t, 0, x)
            x -= 1; out.append(onp.asarray(int(r)))
        elif k == 4:
            x = v()
            r = onp.max(2 * x + 1) if is_np else np.sreduce(lambda p: 2 * p + 1, lambda s, t: max(s, t), -10**9, x)
            x += 1; out.append(onp.asarray(int(r)))
        elif k == 5:
            x = a()
            if is_np:
                r = onp.zeros((R, C)); r[1:-1, 1:-1] = x[:-2, 1:-1] + x[2:, 1:-1] + x[1:-1, :-2] + x[1:-1, 2:] - 4.0 * x[1:-1, 1:-1]
            else:
                r = np.sstencil(np.stencil(_st_cross), x)
            bump(x, 1.0); out.append(_h(r))
        elif k == 6:
            x, y = a(), a()
            if is_np:
                r = onp.zeros((R, C)); r[:, 2:-2] = x[:, :-4] + x[:, 4:] - 2.0 * y[:, 2:-2]
            else:
                r = np.stencil(_st_row)(x, y)
            bump(y, 1.0); out.append(_h(r))
        elif k == 7:
            x = v()
            r = onp.cumsum(x) if is_np else np.scumulative(lambda p, q: p + q, lambda p, q: p + q, x)
            bump(x, 1); out.append(_h(r))
        elif k == 8:
            x = v()
            r = onp.maximum.accumulate(x) if is_np else np.scumulative(lambda p, q: np.maximum(p, q), lambda p, q: np.maximum(p, q), x)
            bump(x, 3); out.append(_h(r))
        elif k == 9:
            r = np.fromfunction(lambda i, j: (i * 3 + j) % 7, (R, C)) + a()
            A.append(r); del A[0]
        elif k == 10:
            x = a(); r = np.triu(x, 1) * 2.0; bump(x, 1.0); out.append(_h(r))
        else:
            x = a(); x[1:-1, :] = x[:-2, :] + x[2:, :]
    for x in A + V + B:
        out.append(_h(x))
    return out


def _kcase(seed):
    def f(np):
        return skeleton_program(np, seed)

    f.__name__ = "skeleton_program_%d" % seed
    return f


SKELETON_CASES = [_kcase(s) for s in range(80)]


def partition_program(np, seed, n_actions=26):
    """Operands with DIFFERENT partitions in one statement (multi-rank: pieces exchanged, operands all-gathered, boxes cut
    into ranges): arrays split by rows, by columns and by the default rule; misaligned windows; transposes (a row-split
    array read as a column-split one); vectors with their own 1-D partition broadcast along either axis; axis sums over the
    split and the unsplit axis; in-place updates whose operand lives elsewhere."""
    rng = onp.random.RandomState(27000 + seed)
    H, W_ = 24, 36
    is_np = np is onp

    def mk(kw):
        x = rng.randint(-4, 5, size=(H, W_)).astype(onp.float64)
        return x.copy() if is_np else np.fromarray(x, **kw)

    layouts = [{}, {"dist_dims": 0}, {"dist_dims": 1}]
    A = [mk(layouts[i % 3]) for i in range(4)]
    S = [(lambda x: x.copy() if is_np else np.fromarray(x, dist_dims=d))(rng.randint(-4, 5, size=(W_, H)).astype(onp.float64)) for d in (0, 1)]
    row = (lambda x: x.copy() if is_np else np.fromarray(x))(rng.randint(-3, 4, size=(W_,)).astype(onp.float64))
    col = (lambda x: x.copy() if is_np else np.fromarray(x))(rng.randint(-3, 4, size=(H,)).astype(onp.float64))
    out = []

    def a():
        return A[int(rng.randint(len(A)))]

    def put(v):
        del A[int(rng.randint(len(A)))]
        A.append(v)

    for _ in range(n_actions):
        k = int(rng.randint(0, 14))
        if k == 0:
            put(a() + a() * 2.0 - a())                                    # three partitions in one statement
        elif k == 1:
            put(a() + S[int(rng.randint(2))].T)                           # transposed operand with its own split
        elif k == 2:
            put(a() * row + col.reshape(H, 1) if is_np else a() * row + np.expand_dims(col, 1))
        elif k == 3:
            x = a(); x += a()                                             # in place, operand elsewhere
        elif k == 4:
            x = a(); out.append(_h(x.sum(axis=0))); out.append(_h(x.sum(axis=1)))
        elif k == 5:
            x, y = a(), a(); i, j = int(rng.randint(0, 6)), int(rng.randint(0, 9))
            put(np.concatenate([x[i:i + 12, :], y[i + 3:i + 15, :]], axis=0) if rng.rand() < 0.5 else x * 1.0)
        elif k == 6:
            x, y = a(), a(); i, j = int(rng.randint(0, 8)), int(rng.randint(0, 12))
            x[2:18, 3:27] = y[i:i + 16, j:j + 24] * 0.5                   # misaligned window of another layout
        elif k == 7:
            x = a(); y = a()
            x[1:-1, 1:-1] = y[:-2, 1:-1] + y[2:, 1:-1] + y[1:-1, :-2] + y[1:-1, 2:]
        elif k == 8:
            out.append(onp.asarray(float((a() * S[0].T).sum())))
        elif k == 9:
            s = S[int(rng.randint(2))]; s += a().T
        elif k == 10:
            put(np.where(a() > a(), a(), S[1].T))
        elif k == 11:
            out.append(_h(a()[::2, ::3] - a()[1::2, 1::3]))
        elif k == 12:
            out.append(_h(a()))
        else:
            x = a(); x[:, :] = x.sum(axis=0) * 0.25 + x                  # a reduction over the (maybe split) axis fed back
    for x in A + S:
        out.append(_h(x))
    return out


def _pcase(seed):
    def f(np):
        return partition_program(np, seed)

    f.__name__ = "partition_program_%d" % seed
    return f


PARTITION_CASES = [_pcase(s) for s in range(80)]


def reduction_program(np, seed, n_actions=22):
    """Reductions in every form: sum / min / max / prod / all / any, over all axes, one axis and several, keepdims, of
    views (strided, reversed, transposed, windows), of expressions whose temporary dies, chained (a reduction of a
    reduction), next to in-place updates of the source.  2-D and 3-D integer-valued arrays."""
    rng = onp.random.RandomState(30000 + seed)
    fa = (lambda x: x.copy()) if np is onp else np.fromarray
    A2 = [fa(rng.randint(-4, 5, size=(R, C)).astype(onp.float64)) for _ in range(2)]
    A3 = [fa(rng.randint(-3, 4, size=(6, 9, 11)).astype(onp.int64)) for _ in range(2)]
    out = []

    def red(x, name, **kw):
        return getattr(x, name)(**kw)

    for _ in range(n_actions):
        k = int(rng.randint(0, 14))
        x2, x3 = A2[int(rng.randint(2))], A3[int(rng.randint(2))]
        name = ["sum", "min", "max"][int(rng.randint(3))]
        if k == 0:
            out.append(_h(red(x2, name, axis=int(rng.randint(2)))))
        elif k == 1:
            out.append(_h(red(x3, name, axis=int(rng.randint(3)))))
        elif k == 2:
            ax = [(0, 1), (0, 2), (1, 2)][int(rng.randint(3))]
            out.append(_h(x3.sum(axis=ax)))
        elif k == 3:
            out.append(_h(x2.sum(axis=int(rng.randint(2)), keepdims=True)))
        elif k == 4:
            out.append(onp.asarray(float(red(x2 * 2.0 + 1.0, name))))                    # temporary dies in the reduction
        elif k == 5:
            out.append(_h(red(x2[1::2, ::-1], name, axis=int(rng.randint(2)))))          # strided + reversed view
        elif k == 6:
            out.append(_h(red(x2.T, name, axis=int(rng.randint(2)))))                    # transposed view
        elif k == 7:
            out.append(_h(x3[1:5, :, 2:9].sum(axis=1)))                                  # window of a 3-D array
        elif k == 8:
            out.append(onp.asarray(float(x2.sum(axis=0).sum())))                         # a reduction of a reduction
            out.append(onp.asarray(float(x2.sum(axis=1).max())))
        elif k == 9:
            s = x2.sum(axis=1); x2 += 1.0; out.append(_h(s))                             # source updated after the call
        elif k == 10:
            out.append(onp.asarray(bool((x3 > -4).all()))); out.append(onp.asarray(bool((x3 > 2).any())))
        elif k == 11:
            out.append(onp.asarray(int((abs(x3) % 2 + 1)[0:2, 0:3, 0:4].prod())))
        elif k == 12:
            x3 -= A3[int(rng.randint(2))] // 2
        else:
            A2[int(rng.randint(2))] = x2 - x2.sum(axis=0) * 0.125
    for x in A2 + A3:
        out.append(_h(x))
    return out


def _rcase(seed):
    def f(np):
        return reduction_program(np, seed)

    f.__name__ = "reduction_program_%d" % seed
    return f


REDUCTION_CASES = [_rcase(s) for s in range(80)]


def mixed_program(np, seed, n_actions=40):
    """Everything on ONE pool: arrays with three partitions (default, row-split, column-split) and one with padded shards;
    arithmetic / where / in-place / overlapping windows / strided, reversed and transposed targets / boolean masks (from
    exact data) / sin-cos pairs / temporaries held across statements / cumsum, concatenate, pad, reshape_copy, smap,
    sstencil / reductions fed back / rebinding, del, sync, partial reads.  Compared with a tolerance (transcendentals)."""
    rng = onp.random.RandomState(33000 + seed)
    is_np = np is onp
    kws = [{}, {"dist_dims": 0}, {"dist_dims": 1}]

    def mk(i):
        x = rng.randint(-4, 5, size=(R, C)).astype(onp.float64)
        return x.copy() if is_np else np.fromarray(x, **kws[i % 3])

    P = [mk(i) for i in range(4)]
    K = (lambda x: x.copy() if is_np else np.fromarray(x))(rng.randint(-4, 5, size=(R, C)).astype(onp.int64))     # exact data for masks
    B = (lambda x: x.copy() if is_np else np.fromarray(x, local_border=2))(rng.randint(-4, 5, size=(R, C)).astype(onp.float64))
    held = []
    out = []

    def p():
        return P[int(rng.randint(len(P)))]

    def put(v):
        if len(P) >= 6:
            del P[int(rng.randint(len(P)))]
        P.append(v)

    def win(h, w):
        i = int(rng.randint(0, R - h + 1)); j = int(rng.randint(0, C - w + 1))
        return (slice(i, i + h), slice(j, j + w))

    for _ in range(n_actions):
        k = int(rng.randint(0, 30))
        if k == 0:
            put(p() * 2.0 - p() + np.where(p() > 0.0, p(), 1.0 - p()))
        elif k == 1:
            x = p(); x += p() * 0.5
        elif k == 2:
            x = p(); w1, w2 = win(5, 8), win(5, 8); x[w1] = x[w2] - p()[w1]
        elif k == 3:
            x = p(); x[::2, ::-1] = p()[::2, :] + 1.0
        elif k == 4:
            x = p(); x.T[:, :] = p().T * 2.0
        elif k == 5:
            x = p(); m = K > int(rng.randint(-3, 3)); x[m] = -1.0
        elif k == 6:
            x = p(); m = K < 0; out.append(onp.asarray(float(x[m].sum())))
        elif k == 7:
            x = p(); put(np.sin(x) * np.cos(x))
        elif k == 8:
            x = p(); s = np.sin(x); y = p(); y -= 1.0; put(s + np.cos(x))
        elif k in (9, 10):
            if len(held) < 2:
                held.append(p() * 2.0 + 1.0 if k == 9 else np.cos(p()))
        elif k == 11:
            if held:
                x = p(); x[:, :] = held.pop(0)
        elif k == 12:
            if held:
                put(held.pop() - p())
        elif k == 13:
            x = p(); c = np.cumsum(x, axis=int(rng.randint(2))); x += 1.0; put(c * 0.125)
        elif k == 14:
            x, y = p(), p(); c = np.concatenate([x[:6, :], y[6:, :]], axis=0); y -= 1.0; put(c)
        elif k == 15:
            x = p(); c = np.pad(x[1:-1, 2:-2], ((1, 1), (2, 2)), mode="edge"); x += 1.0; put(c)
        elif k == 16:
            x = p(); c = x.reshape_copy((C, R)) if not is_np else onp.reshape(x, (C, R)).copy(); x -= 1.0; out.append(_h(c))
        elif k == 17:
            x = p(); r = 3 * x - 7 if is_np else np.smap("lambda x: 3*x-7", x); x += 1.0; put(np.minimum(np.maximum(r, -50.0), 50.0))
        elif k == 18:
            if is_np:
                r = onp.zeros((R, C)); r[1:-1, 1:-1] = B[:-2, 1:-1] + B[2:, 1:-1] + B[1:-1, :-2] + B[1:-1, 2:] - 4.0 * B[1:-1, 1:-1]
            else:
                r = np.sstencil(np.stencil(_st_cross), B)
            B += p() * 0.5; put(r * 0.25)
        elif k == 19:
            x = p(); put(x - x.sum(axis=0) * 0.0625)
        elif k == 20:
            x = p(); out.append(_h(x.max(axis=1))); out.append(onp.asarray(float((x * 0.5 + p()).sum())))
        elif k == 21:
            x = p(); y = p(); y[1:-1, 1:-1] = x[:-2, 1:-1] + x[2:, 1:-1] - 2.0 * x[1:-1, 1:-1]
        elif k == 22:
            i = int(rng.randint(len(P))); P[i] = np.minimum(np.maximum(P[i], -30.0), 30.0)      # rebinding keeps values small
        elif k == 23:
            if len(P) > 3:
                del P[int(rng.randint(len(P)))]
        elif k == 24:
            if not is_np:
                np.sync()
        elif k == 25:
            out.append(_h(p()))
        elif k == 26:
            x = p(); _ = np.cos(x) * 3.0; del _                                          # never observed
        elif k == 27:
            K += 1; K[K > 4] = -4                                                        # the mask source itself changes
        elif k == 28:
            x = p(); v = x[2:11, 3:19]; v *= 0.5; out.append(_h(v[::2, ::3]))
        else:
            x = p(); put((x > p()).astype(onp.float64) + (K % 3).astype(onp.float64))
    for x in P + [K, B]:
        out.append(_h(x))
    return out


def _mcase(seed):
    def f(np):
        return mixed_program(np, seed)

    f.__name__ = "mixed_program_%d" % seed
    return f


MIXED_CASES = [_mcase(s) for s in range(120)]


def typing_program(np, seed, n_actions=16):
    """float32 / float64 / int64 arrays with Python and NumPy scalars, values that are NOT exactly representable: the result
    depends on the class every operation is computed in and on where roundings happen (the reference's rules: Numba's
    scalar typing inside the fused loop, division as multiplication by the reciprocal, float32 arrays with Python floats
    computed in float64 and rounded once when STORED).  Not comparable with NumPy - pinned by the outputs of the real
    reference (tests/golden/fuzz_golden.npz)."""
    rng = onp.random.RandomState(36000 + seed)
    fa = (lambda x: x.copy()) if np is onp else np.fromarray
    A = fa((rng.randint(-40, 41, size=(120,)) * 0.1).astype(onp.float32))
    B = fa((rng.randint(1, 41, size=(120,)) * 0.3).astype(onp.float32))
    D = fa(rng.randint(-40, 41, size=(120,)) * 0.1)
    I = fa(rng.randint(1, 9, size=(120,)).astype(onp.int64))
    out = []
    for _ in range(n_actions):
        k = int(rng.randint(0, 14))
        if k == 0:
            r = A * 2.5 + B
        elif k == 1:
            r = A * B - 0.1
        elif k == 2:
            r = A + D
        elif k == 3:
            r = A * I
        elif k == 4:
            r = A / 3.0
        elif k == 5:
            r = 1.0 / B
        elif k == 6:
            r = B ** 2 + B ** 0.5
        elif k == 7:
            r = np.sqrt(B) * A
        elif k == 8:
            r = A.astype(onp.float64) * 0.1
        elif k == 9:
            r = (D * 0.1).astype(onp.float32) + A
        elif k == 10:
            r = np.where(A > 0.5, A, B * 0.3)
        elif k == 11:
            A += 0.1; r = A
        elif k == 12:
            r = D / I + A
        else:
            t = A * 0.1; r = t + B; del t
        out.append(_h(r))
    out.append(_h(A)); out.append(_h(D))
    return out


def typing2_program(np, seed, n_actions=14):
    """More statement forms for the typing rules (see typing_program): integer arrays with float scalars, floor division and
    modulo on inexact floats, abs / negation, minimum / maximum with scalars, comparisons stored as float32, truncating
    casts, exp.  Pinned by the real reference where it can run them."""
    rng = onp.random.RandomState(39000 + seed)
    fa = (lambda x: x.copy()) if np is onp else np.fromarray
    A = fa((rng.randint(-40, 41, size=(120,)) * 0.1).astype(onp.float32))
    B = fa((rng.randint(1, 41, size=(120,)) * 0.3).astype(onp.float32))
    D = fa(rng.randint(-40, 41, size=(120,)) * 0.1)
    I = fa(rng.randint(-9, 10, size=(120,)).astype(onp.int64))
    out = []
    for _ in range(n_actions):
        k = int(rng.randint(0, 16))
        if k == 0:
            r = I * 0.5 + A
        elif k == 1:
            r = I / 3
        elif k == 2:
            r = I // 2 + I % 3
        elif k == 3:
            r = A // 0.3
        elif k == 4:
            r = D % 0.7
        elif k == 5:
            r = abs(A) - (-B)
        elif k == 6:
            r = np.minimum(A, 0.5) + np.maximum(B, 2.25)
        elif k == 7:
            r = np.maximum(A, B) * D
        elif k == 8:
            r = (A > 0.3).astype(onp.float32) * B
        elif k == 9:
            r = (A * 10.0).astype(onp.int64) + I
        elif k == 10:
            r = (D * 7.0).astype(onp.int32)
        elif k == 11:
            r = I.astype(onp.float32) * 0.1
        elif k == 12:
            r = np.exp(A * 0.1) * B
        elif k == 13:
            r = A * A * A - B * 0.5
        elif k == 14:
            r = (A + B) * (A - B)
        else:
            B *= 1.1; r = B
        out.append(_h(r))
    out.append(_h(B))
    return out
