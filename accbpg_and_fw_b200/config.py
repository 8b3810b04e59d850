"""Run-time switches of the package (plain module attributes; set them before calling a driver).

linear_images
    D-opt's Gram matrix M(x) = H diag(x) H^T and the linear-inverse objectives' A x are *linear* in x.  The
    accelerated drivers only ever evaluate f at x0, at fresh prox points z+ and at convex combinations
    (1-theta) a + theta b of points whose image they already hold, so with this switch on they carry the images
    along and form the image of a combination with one axpby instead of another pass over H / A
    (SURVEY.md section 8d: "linearity shortcuts are allowed as optimisations").  Values agree with the
    direct evaluation to rounding (the tests run both ways); the image of x is re-formed from scratch every
    `reanchor_every` iterations so rounding cannot accumulate.  Set to False to evaluate every point from scratch.

pipeline
    ABPG, ABDA and BPG without line search take no data-dependent decision inside an iteration except the stopping
    test, so the drivers enqueue iteration k+1 before the scalars of iteration k have been read back (deferred read,
    accbpg_ctx_read_async): the GPU never idles between iterations.  Recorded values and the returned iterate are
    those of the synchronous loop; when the stopping test fires, the one iteration enqueued beyond it is discarded.
    Switched off automatically with verbose=True or restart=True.

peer_allreduce
    Column-sharded runs exchange through NVLink peer memory inside this library's kernels instead of NCCL calls between
    them (buffers from torch.distributed._symmetric_memory): the ranks' Gram matrices are summed behind the SYRK
    (accbpg_dopt_gram_allreduce), and D_opt_FW(_away) exchanges its selection records and the chosen column
    (accbpg_fw_run_peer).  Falls back to NCCL when symmetric memory cannot be set up.

fused_small
    BPG on a D-optimal design objective with the Burg kernel on the simplex whose H fits in the shared memory of one SM
    (configs[0], 80 x 200, does): the whole solve is ONE kernel launch (accbpg_dopt_bpg_small) instead of a dozen launches
    and a host decision per line-search trip.  Same control flow and histories; T is stamped evenly over the solve's
    wall time (the host does not see individual iterations).
    The same holds for BPG on PoissonRegression / KLdivRegression with BurgEntropy, BurgEntropyL1, BurgEntropyL2,
    ShannonEntropy, ShannonEntropyL1 or ShannonEntropySimplex when A fits the shared memory of a cluster of at most 8 SMs
    (accbpg_linreg_bpg_small; the notebook instances, Poisson 200 x 100 and KL 1000 x 100, do).  There T[k] is the
    device clock at the top of iteration k.
    ABPG and ABPG_gain on the same objectives and kernels run as one launch too (accbpg_linreg_abpg_small, a plan of
    its own that holds more vectors) when linear_images is also on: the kernel follows that scheme - carried A x and
    A z, A x re-formed every `reanchor_every` iterations - so results differ from the operator loop only in the order
    of sums.  With linear_images off the operator loop evaluates every point from scratch, as that switch says.
    ABPG and ABPG_gain on the D-optimal design objective with BurgEntropySimplex run as one launch as well
    (accbpg_dopt_abpg_small, on the machinery of the BPG kernel with three more vectors) when H fits.  That kernel
    evaluates every point from scratch, which is what linear_images = False asks for, and the carried Gram images agree
    with it to rounding, so it is taken under both settings of linear_images.  SparseDOptimalObj stays on the operator
    loop.
"""
linear_images = True
reanchor_every = 64
pipeline = True
peer_allreduce = __import__('os').environ.get('ACCBPG_PEER_ALLREDUCE', '1') != '0'
fused_small = __import__('os').environ.get('ACCBPG_FUSED_SMALL', '1') != '0'
