"""Debug: tensor-core walk (int8 residual form) vs oracle / sweep_pipe walk (fp64 residual form) on the lowrank test cases."""
import os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
from conftest import glorot, hidden_pair
from oracle import c_oracle, gpfq_oracle as O
from quantized_neural_networks_b200 import get_engine

eng = get_engine(0)
for (N0, N1, m, first) in ((520, 2048, 48, True), (600, 2200, 64, False)):
    rng = np.random.default_rng(N0 + N1 + m)
    if first:
        X = (rng.uniform(0, 1, (N0, m)) * (rng.uniform(0, 1, (N0, m)) < 0.5)).astype(np.float32)
        X[:10] = 0
        Xq = X
    else:
        X, Xq = hidden_pair(rng, N0, m)
    W = glorot(rng, N0, N1)
    for bits in (np.log2(3), 2, 4):
        A = O.layer_alphabet(W, 3 if bits != np.log2(3) else 2, O.unit_alphabet(bits))
        Qref = c_oracle.quantize_layer(W, X, Xq, A)
        eng.set_option("sweep_outer", 2)
        Q = eng.dense_layer(X, None if first else Xq, W, A, method="gram")
        eng.set_option("sweep_i8", 2)
        Qo = eng.dense_layer(X, None if first else Xq, W, A, method="gram")
        eng.set_option("sweep_i8", 0)
        eng.set_option("sweep_outer", 0)
        bad = np.argwhere(Q != Qref)
        print((N0, N1, m, first), "bits", bits, "K", len(A), "agree tc/oracle", O.agreement(Q, Qref), "old/oracle", O.agreement(Qo, Qref),
              "tc/old", O.agreement(Q, Qo), "n_bad", len(bad))
        if len(bad):
            ts = np.unique(bad[:, 0]); js = np.unique(bad[:, 1])
            print("  first bad t:", ts[:20], "n neurons:", len(js), "first bad j:", js[:10])
            t, j = bad[0]
            print("  at", t, j, "Q", Q[t, j], "ref", Qref[t, j], "levels", A)
