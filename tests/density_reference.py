"""Noisy density-matrix semantics in plain numpy: the reference the noisy simulator is tested against.

Restates, independently of the package's lowering and kernels, what ``B200Backend(noise_model=nm)`` computes for
one circuit (the semantics are listed in the package's ``noise.py`` docstring):

* ``ρ`` starts as ``|0><0|``; every instruction applies ``U ρ U†`` and then the error registered for its name on
  its qubits (specific qubits first, else all qubits), as a superoperator on the vectorised ``ρ``, index
  ``r | c << n``;
* a measurement whose qubit is used again splits every branch into its two projected, un-normalised density
  matrices and records the outcome in its clbit; terminal measurements are read off the diagonal at the end;
* ``p(key)`` = trace of everything that ends with classical value ``key`` (bit i = clbit i; unwritten clbits 0);
* then every written clbit's recorded value passes through the readout error of the qubit that wrote it last.

Runs on any circuit object ``oracle.statevector`` takes, so ``oracle.instantiate`` instances knit with
``oracle.sparse_knit.knit`` into the noisy reference of a cut circuit.  The noise model is read from its
registries (``_all``, ``_local``, ``_readout``, ``_readout_all``) and the errors' ``superop`` matrices.
"""
import numpy as np

from oracle import gates


def _apply(v, n2, bits, m):
    """``m`` (2^k x 2^k, little-endian in ``bits``) on the bits ``bits`` of the 2^n2 vector ``v``."""
    k = len(bits)
    t = v.reshape((2,) * n2)                                # axis a <-> bit n2 - 1 - a
    axes = [n2 - 1 - b for b in reversed(bits)]             # most significant of m first
    mt = m.reshape((2,) * (2 * k))
    t = np.tensordot(mt, t, axes=(list(range(k, 2 * k)), axes))
    t = np.moveaxis(t, list(range(k)), axes)
    return np.ascontiguousarray(t).reshape(-1)


def _error(model, name, qubits):
    err = model._local.get((name, tuple(qubits)))
    if err is None:
        err = model._all.get(name)
    return None if err is None else np.asarray(err.superop)


def _readout(model, q):
    err = model._readout.get(q)
    if err is None:
        err = model._readout_all
    return None if err is None else np.asarray(err.probabilities)


def noisy_distribution(circuit, model):
    """dict[int, float]: the exact noisy probability of every classical outcome (zeros omitted)."""
    n = len(circuit.qubits)
    n2 = 2 * n
    qidx = {q: i for i, q in enumerate(circuit.qubits)}
    cidx = {c: i for i, c in enumerate(circuit.clbits)}
    ops = []
    for ins in circuit.data:
        op = ins.operation
        if op.name in ("barrier", "wire_cut") or type(op).__name__ in ("Barrier", "WireCut"):
            continue
        qs = tuple(qidx[q] for q in ins.qubits)
        if op.name == "measure":
            ops.append(("m", qs, cidx[ins.clbits[0]]))
            continue
        u = getattr(op, "_matrix", None)
        if u is None:
            u = gates.matrix(op.name, op.params)
        ops.append((op.name, qs, np.asarray(u, dtype=complex)))
    last_use = {}
    for i, (_name, qs, _x) in enumerate(ops):
        for q in qs:
            last_use[q] = i
    rho = np.zeros(1 << n2, dtype=complex)
    rho[0] = 1.0
    branches = [(rho, 0)]
    deferred, writer = [], {}
    for i, (name, qs, x) in enumerate(ops):
        bits = list(qs) + [q + n for q in qs]
        if name == "m":
            q, cb = qs[0], x
            writer[cb] = q
            if last_use[q] == i:
                deferred.append((q, cb))
                continue
            new = []
            idx = np.arange(1 << n2)
            for b in (0, 1):
                keep = (((idx >> q) & 1) == b) & (((idx >> (q + n)) & 1) == b)
                for r, c in branches:
                    p = np.where(keep, r, 0)
                    if np.any(p):
                        new.append((p, (c & ~(1 << cb)) | (b << cb)))
            branches = new
            continue
        s = np.kron(np.conj(x), x)
        e = _error(model, name, qs)
        if e is not None:
            s = e @ s
        branches = [(_apply(r, n2, bits, s), c) for r, c in branches]
    idx = np.arange(1 << n, dtype=np.int64)
    dkey = np.zeros(1 << n, dtype=np.int64)
    dmask = 0
    for q, cb in deferred:
        dkey = (dkey & ~(1 << cb)) | (((idx >> q) & 1) << cb)
        dmask |= 1 << cb
    out = {}
    for r, c in branches:
        prob = r[idx * ((1 << n) + 1)].real
        keys = dkey | (c & ~dmask)
        uniq, inv = np.unique(keys, return_inverse=True)
        sums = np.bincount(inv, weights=prob)
        for k, v in zip(uniq.tolist(), sums.tolist()):
            out[k] = out.get(k, 0.0) + v
    for cb, q in sorted(writer.items()):
        ro = _readout(model, q)
        if ro is None:
            continue
        new = {}
        for k, v in out.items():
            m = (k >> cb) & 1
            k0 = k & ~(1 << cb)
            new[k0] = new.get(k0, 0.0) + ro[m, 0] * v
            new[k0 | (1 << cb)] = new.get(k0 | (1 << cb), 0.0) + ro[m, 1] * v
        out = new
    return {k: v for k, v in out.items() if v != 0.0}
