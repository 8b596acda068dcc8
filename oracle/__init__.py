"""CPU oracle for the nn-active-learning query-scoring hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``oracle/`` is imported by the product
package (``nn-active-learning_b200`` / ``nnal_b200``).  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl
reference`` legs may import it, and there only as the checker / CPU baseline.

Parity status
-------------
``oracle/check_against_reference.py`` (run with $NNAL_REFERENCE set to the
original sources) imports the UNMODIFIED reference in place, missing
third-party modules stubbed, compares on seeded inputs and writes the golden
vectors in ``tests/golden/``:

* PINNED, NumPy helpers executed as they are: patch gather, multi-image gather +
  normalise, global2local_inds, compute_entropy, uncertainty_filtering,
  binary_uncertainty_filter, shrink_gradient, sample_query_dstr, append_zero,
  get_self_sims, get_cross_sims.
* PINNED, the query dispatch executed as it is over a fake TF session / fake
  cvxopt (everything AROUND the TF graph and the SDP solve is the reference's own
  code): PW_NN.batch_eval, PW_NNAL.CNN_query 'entropy' and 'fi',
  bin_uncertainty_filter_multimg, every method of PW_NNAL.query_multimg
  (entropy, fi, rep-entropy, core-set, MC-entropy, BALD, ensemble, QBC-JS),
  NNAL.CNN_query 'entropy' / 'rep-entropy' / 'fi' (image loader replaced by an
  in-memory pool), gen_A_matrices, FC_gradnorms_batch, LLFC_grads, LLFC_hess, and the SDP programme (c, G, h, A, b) that
  SDP_query_distribution / inequality_cvx_matrix hand to cvxopt.
* "Parity unpinned": the arithmetic INSIDE TensorFlow 1.x (conv/pool/fc/softmax
  forward, tf.gradients, dropout masks) and inside cvxopt -- TF 1.x is not
  installable here and the reference ships no golden vectors for it (SURVEY.md
  §8c).  The float64 restatement encodes the documented TF semantics and is
  cross-checked against torch-CPU float64 (forward and autograd) in
  ``tests/test_oracle.py``; SDP solutions are certified by their duality gap.
"""
from .nnal_oracle import *   # noqa: F401,F403
from .fi_oracle import *     # noqa: F401,F403
from .rep_oracle import *    # noqa: F401,F403
from .mc_oracle import *     # noqa: F401,F403
