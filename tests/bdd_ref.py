"""Reference BDD evaluation for the tests: the semantics of pgb_glwe_bdd_eval_batched (include/poulpy_b200.h) for one item, node by node
over cmux_ref.glwe_cmux,

    state[j] = leaf j;  state[n_leaves + k] = cmux(t = state[t_k], f = state[f_k], s_{bit of k's level});
    output o = state[outputs[o]]: a node as is, a leaf's first min(a.size, res.size) limbs with the rest zeroed,

and the same circuit evaluated in plain integers.  GLWEs are int64 arrays (size, cols, n); sels[i] is the oracle VmpPMat of input bit i
of this one item."""
import numpy as np

import cmux_ref as CR


def eval_plain(circuit, bits):
    """The leaf values the outputs of `circuit` (poulpy_b200.circuit.BddCircuit) select for the input bits `bits` (a sequence of 0/1)."""
    state = list(circuit.leaves)
    for bit, nodes in circuit.levels:
        state += [state[t] if bits[bit] else state[f] for t, f in nodes]
    return [state[o] for o in circuit.outputs]


def glwe_bdd_eval(o, res_size, leaves, circuit, base2k, sels, ggsw_base2k, dsize=1):
    """-> the n_out GLWEs (n_out, res_size, cols, n) of one item whose leaves are `leaves` (n_leaves, a_size, cols, n)."""
    _, a_size, cols, n = leaves.shape
    state = [np.ascontiguousarray(x, dtype=np.int64) for x in leaves]
    for bit, nodes in circuit.levels:
        for t, f in nodes:
            out = np.zeros((res_size, cols, n), dtype=np.int64)
            CR.glwe_cmux(o, out, state[t], state[f], base2k, sels[bit], ggsw_base2k, dsize)
            state.append(out)
    res = np.zeros((len(circuit.outputs), res_size, cols, n), dtype=np.int64)
    for i, s in enumerate(circuit.outputs):
        m = min(state[s].shape[0], res_size)
        res[i, :m] = state[s][:m]
    return res


def complete_tree(n_bits):
    """The CMux tree of pgb_glwe_cmux_tree_batched as a circuit: 2^n_bits leaves, level i (bit i) holds g_{i+1,j} = cmux(g_{i,2j+1},
    g_{i,2j}), one output."""
    from poulpy_b200.circuit import BddCircuit
    L = 1 << n_bits
    levels, prev, nxt = [], list(range(L)), L
    for i in range(n_bits):
        nodes = [(prev[2 * j + 1], prev[2 * j]) for j in range(len(prev) // 2)]
        levels.append((i, nodes))
        prev = list(range(nxt, nxt + len(nodes)))
        nxt += len(nodes)
    return BddCircuit(list(range(L)), levels, [prev[0]])
