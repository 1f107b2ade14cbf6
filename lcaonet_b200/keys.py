"""Names of the entries a graph batch carries (the input/side-effect contract of `forward`).

Same strings as the reference contract (lcaonet/data/keys.py:4-27) so that batches built for the
reference model work unchanged.
"""


class GraphKeys:
    Lattice = "lattice"  # (B, 3, 3)
    PBC = "pbc"  # (B, 3)
    Neighbors = "neighbors"  # (B)

    Batch_idx = "batch"  # (N)
    Z = "z"  # (N)
    Pos = "pos"  # (N, 3)

    Edge_idx = "edge_index"  # (2, E), row 0 = centre/source s, row 1 = neighbour/target t
    Edge_shift = "edge_shift"  # (E, 3)
    Edge_dist = "edge_dist"  # (E)
    Edge_vec_st = "edge_vec"  # (E, 3) unit vectors

    Idx_s_3b = "idx_s_3b"
    Idx_t_3b = "idx_t_3b"
    Idx_k_3b = "idx_k_3b"  # (T)
    Edge_idx_ks_3b = "edge_idx_ks_3b"  # (T)
    Edge_idx_st_3b = "edge_idx_st_3b"  # (T)
    Angles_3b = "angles_3b"  # (T) cos(theta)

    # written by LCAONet.forward when regress_atom_energy / regress_atom_virial is set (no reference counterpart)
    Atom_energy = "atom_energy"  # (N, out_size)
    Atom_virial = "atom_virial"  # (N, 3, 3), or (N, out_size, 3, 3)


KEYS = [v for k, v in vars(GraphKeys).items() if not k.startswith("__")]
