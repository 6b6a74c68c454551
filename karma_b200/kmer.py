"""Drop-in mirror of ``karma/kmer.py`` (reference: /root/reference/karma/kmer.py).

Same class, constructor, ``run`` signature, attributes, files and messages as the
reference's ``KmerClustering`` (kmer.py:14-325); the k-mer profile matrix
(``__calc_kmer_profile``, kmer.py:199-264) and the neighbour search that
``umap.UMAP(...).fit_transform`` performs first (kmer.py:285-290) run on a B200
through libkarma_b200.so.  There is no CPU path: without the GPU library the
profile step raises ``KarmaB200Error``.

karma.py keeps doing (karma.py:197-213)::

    k = KmerClustering(sequences=sequences, output_dir=kmer_dir,
                       kmer_size=args.KMER_SIZE, threads=args.THREADS)
    k.run(neighbors=..., components=..., dist=..., r_state=..., min_cluster_size=...)
    labeled_contigs = k.clusters; unlabeled_contigs = k.unlabeled_cluster[0]
"""
import logging
import os
import sys
import time

import numpy as np

try:                                    # inside karma: the shared logger (kmer.py:11)
    from karma.logs import logger
except Exception:                       # stand-alone: same format as karma/logs.py:9-11
    logger = logging.getLogger("karma_b200.kmer")
    if not logger.handlers:
        _h = logging.StreamHandler()
        _h.setFormatter(logging.Formatter("{asctime} [{levelname}]: {message}",
                                          datefmt="%Y-%m-%d %H:%M:%S", style="{"))
        logger.addHandler(_h)
    logger.setLevel(logging.INFO)


def _accepts(fn, *names):
    import inspect
    try:
        params = inspect.signature(fn).parameters
    except (TypeError, ValueError):
        return False
    if any(p.kind is inspect.Parameter.VAR_KEYWORD for p in params.values()):
        return True
    return all(n in params for n in names)


def umap_embedding(profile, knn_indices, knn_dists, umap_args, umap_module=None):
    """The call of kmer.py:285-290, ``umap.UMAP(**umap_args).fit_transform(profile)``, fed with the exact
    kNN graph from the GPU so that UMAP does not search for neighbours again.  Three hand-off routes, chosen
    by FEATURE (signatures), never by catching errors out of ``fit_transform``:

    1. umap-learn >= 0.5: ``UMAP(precomputed_knn=(idx, dist[, None]))``.  0.5.0-0.5.3 insist on an NNDescent
       object as third element; the parameters are validated up front (``_validate_parameters``) and a
       rejection falls through to the next route.
    2. umap-learn 0.3.x / 0.4.x -- the reference pins 0.3.9 (conda/meta.yaml:15): the stages ``UMAP.fit``
       itself runs, ``umap.umap_.fuzzy_simplicial_set(..., knn_indices=, knn_dists=)`` followed by
       ``simplicial_set_embedding`` with UMAP's defaults (spread 1, learning rate 1, repulsion 1, 5 negative
       samples, spectral init, default epochs), on the float32 copy of the profile as ``fit`` makes it.
    3. neither available (or no graph: fewer contigs than neighbours): the stock call.

    Returns (embedding, route) with route in {"precomputed_knn", "fuzzy_simplicial_set", "stock"}."""
    if umap_module is None:
        import umap as umap_module
    n = profile.shape[0]
    k = umap_args["n_neighbors"]
    have_graph = knn_indices is not None and knn_dists is not None and knn_indices.shape == (n, k) and k < n
    if have_graph and _accepts(umap_module.UMAP.__init__, "precomputed_knn"):
        idx = np.ascontiguousarray(knn_indices, dtype=np.int64)
        dst = np.ascontiguousarray(knn_dists, dtype=np.float32)
        for graph in ((idx, dst), (idx, dst, None)):
            try:
                reducer = umap_module.UMAP(precomputed_knn=graph, **umap_args)
                if hasattr(reducer, "_validate_parameters"):
                    reducer._validate_parameters()
            except (TypeError, ValueError):
                continue
            return reducer.fit_transform(profile), "precomputed_knn"
    um = getattr(umap_module, "umap_", None)
    fss = getattr(um, "fuzzy_simplicial_set", None)
    sse = getattr(um, "simplicial_set_embedding", None)
    fab = getattr(um, "find_ab_params", None)
    if (have_graph and fss is not None and sse is not None and fab is not None and
            _accepts(fss, "X", "n_neighbors", "random_state", "metric", "knn_indices", "knn_dists") and
            _accepts(sse, "data", "graph", "n_components", "initial_alpha", "a", "b", "gamma", "negative_sample_rate",
                     "n_epochs", "init", "random_state", "metric", "metric_kwds") and
            not _accepts(sse, "densmap")):
        from sklearn.utils import check_array, check_random_state
        x = check_array(profile, dtype=np.float32, accept_sparse="csr")          # UMAP.fit's own cast
        rs = check_random_state(umap_args.get("random_state"))
        a, b = fab(1.0, umap_args["min_dist"])
        fss_kw = dict(X=x, n_neighbors=k, random_state=rs, metric="euclidean", metric_kwds={},
                      knn_indices=np.ascontiguousarray(knn_indices, dtype=np.int64),
                      knn_dists=np.ascontiguousarray(knn_dists, dtype=np.float32),
                      angular=False, set_op_mix_ratio=1.0, local_connectivity=1.0, verbose=False)
        import inspect
        fss_kw = {kk: v for kk, v in fss_kw.items() if kk in inspect.signature(fss).parameters}
        graph = fss(**fss_kw)
        if isinstance(graph, tuple):                                              # 0.4.x returns (graph, sigmas, rhos)
            graph = graph[0]
        sse_kw = dict(data=x, graph=graph, n_components=umap_args["n_components"], initial_alpha=1.0, a=a, b=b, gamma=1.0,
                      negative_sample_rate=5, n_epochs=0, init="spectral", random_state=rs, metric="euclidean",
                      metric_kwds={}, verbose=False)
        sse_kw = {kk: v for kk, v in sse_kw.items() if kk in inspect.signature(sse).parameters}
        emb = sse(**sse_kw)
        if isinstance(emb, tuple):
            emb = emb[0]
        return emb, "fuzzy_simplicial_set"
    return umap_module.UMAP(**umap_args).fit_transform(profile), "stock"


CLUSTER_ROUTES = ("host", "device")


class KmerClustering:
    """Mirror of kmer.py's class.  ``kmer_size``: "5p6" (kmer.py's default), an integer k (kmer.py:83-85): k <= 7
    counts into dense shared-memory histograms, 8 <= k <= 16 through sorted 128-bit k-mer keys, k > 16 raises
    KarmaB200Error (the sort key holds 16 characters); or the fixed-column throughput shapes "5+6" / "4+5" of this
    library (A/C/G/T only: other bytes are rejected there).  Sequences must be single-byte characters (latin-1;
    FASTA is ASCII): one byte per character keeps byte order == the code-point order sorted() uses (kmer.py:172).

    ``cluster_on`` selects where UMAP and HDBSCAN run: "host" (umap-learn and hdbscan, through ``umap_embedding``)
    or "device" (``cluster.cluster_from_lists``: the same stages as umap 0.3.9's route, on the GPU, with the profile
    and the k-lists never downloaded for them).  None reads the environment variable KARMA_B200_CLUSTER, so that an
    unmodified karma.py can choose; unset or empty means "host"."""

    def __init__(self, sequences, output_dir, kmer_size, threads, cluster_on=None):
        # kmer.py:15-27
        self.sequences = sequences
        self.output_dir = output_dir
        self.output_eval = f"{self.output_dir}/eval.txt"
        self.output_file = f"{self.output_dir}/cluster.txt"

        self.threads = threads          # kept for interface parity; the GPU path does not fork
        self.kmer_size = kmer_size

        self.clusters = []
        self.unlabeled_cluster = []
        self.kmers = None
        self.sorted_kmer_set = set()

        # GPU-side products of the last profile computation
        self.knn_indices = None
        self.knn_dists = None
        self._engine = None
        self._d_knn = None

        if cluster_on is None:
            cluster_on = os.environ.get("KARMA_B200_CLUSTER") or "host"
        if cluster_on not in CLUSTER_ROUTES:
            raise ValueError("cluster_on (or KARMA_B200_CLUSTER) must be one of %s, got %r" % (CLUSTER_ROUTES, cluster_on))
        self.cluster_on = cluster_on

    # ------------------------------------------------------------------ helpers
    @staticmethod
    def __mask_list(list_to_mask, mask):
        """kmer.py:30-44 -- same grouping and ordering (labels in ``set(mask)``
        iteration order, members in input order) without rebuilding
        ``list(keys())`` per element (the reference is O(N^2) there)."""
        names = [k.lstrip(">") for k in list_to_mask.keys()]
        groups = {}
        for j, lab in enumerate(mask):
            groups.setdefault(lab, []).append(names[j])
        labeled, unlabeled = [], []
        for i in set(mask):
            (unlabeled if i == -1 else labeled).append(groups[i])
        return (labeled, unlabeled)

    @staticmethod
    def is_palindrome(sequence):
        """kmer.py:46-54 -- plain string palindrome (not reverse complement)."""
        return sequence == sequence[::-1]

    def fill_array_for_contig(self, *args):
        """kmer.py:108-122 -- (row, col, count/length) triples of one contig's Counter.
        Kept because it is public in the reference; the GPU path does not call it."""
        row, contig, length = args[0], args[1], args[2]
        return [(row, self.kmers[kmer], count / length) for kmer, count in contig.items()]

    @staticmethod
    def _first_token(names):
        return [n.split(" ")[0] for n in names]

    def __fix_fasta_headers(self):
        """Keep only the first space-delimited token of every contig name (kmer.py:94-106)."""
        self.unlabeled_cluster = [self._first_token(self.unlabeled_cluster[0])]
        self.clusters = [self._first_token(members) for members in self.clusters]

    def __save_groups_to_file(self):
        """cluster.txt (kmer.py:124-133): tab-separated names, one group per line, the unlabeled
        group first."""
        rows = [self.unlabeled_cluster[0]] + list(self.clusters)
        with open(self.output_file, "w") as out:
            out.writelines("\t".join(members) + "\n" for members in rows)

    def __read_clusters(self):
        """Resume from a previous cluster.txt (kmer.py:135-144)."""
        with open(self.output_file, "r") as src:
            rows = [line.rstrip("\n").split("\t") for line in src]
        if not rows:                                   # readline() on an empty file gives "" -> [""]
            rows = [[""]]
        self.unlabeled_cluster = [rows[0]]
        self.clusters.extend(rows[1:])

    def __write_eval_information(self, **fields):
        """eval.txt (kmer.py:266-272): a header line and a value line, tab separated."""
        with open(self.output_eval, "w") as out:
            out.write("\t".join(fields) + "\n")
            out.write("\t".join(str(v) for v in fields.values()) + "\n")

    # ------------------------------------------------------------------ GPU path
    def _pack(self):
        """dict -> packed buffers of the C ABI.  One byte per character (latin-1):
        byte order then equals the code-point order ``sorted()`` uses (kmer.py:172)."""
        packed = getattr(self.sequences, "packed", None)
        if callable(packed):
            got = packed()                     # came from karma_b200.fasta.read_fasta_file, unmodified
            if got is not None:
                return got
        seqs = list(self.sequences.values())
        try:
            raw = "".join(seqs).encode("latin-1")
        except UnicodeEncodeError as e:
            raise ValueError("karma_b200: sequences must be single-byte characters") from e
        lens = np.fromiter((len(s) for s in seqs), dtype=np.int64, count=len(seqs))
        offsets = np.zeros(len(seqs) + 1, dtype=np.int64)
        np.cumsum(lens, out=offsets[1:])
        bases = np.frombuffer(raw, dtype=np.uint8)
        key_len = np.fromiter((len(k) for k in self.sequences), dtype=np.int32, count=len(seqs))
        return bases, offsets, key_len

    def _get_engine(self):
        if self._engine is None:
            from .engine import Engine
            self._engine = Engine()
        return self._engine

    def __calc_kmer_profile(self, n_neighbors=None, host_profile=True):
        """kmer.py:199-264 on the GPU.  Returns the float64 (N, D) profile; sets
        ``self.kmers`` ({kmer: column}) like the reference.  With ``n_neighbors``
        the exact kNN graph is computed in the same pass and left in
        ``self.knn_indices`` / ``self.knn_dists``.  With ``host_profile=False`` the
        profile is returned as a device tensor and the device k-lists are left in
        ``self._d_knn``."""
        from .engine import ZeroRowError, profile_and_knn
        logger.info("Extracting kmers from contigs.")               # kmer.py:152
        if self.kmer_size != "5p6":
            logger.info(f"Accounting only {self.kmer_size}-mers.")  # kmer.py:167
        if len(self.sequences) == 0:
            self.kmers = {}
            return np.zeros((0, 0), dtype=np.float64)
        bases, offsets, key_len = self._pack()
        try:
            res = profile_and_knn(self._get_engine(), bases, offsets, key_len, self.kmer_size,
                                  n_neighbors=n_neighbors, host_profile=host_profile)
        except ZeroRowError as e:
            # the column dictionary exists by the time the reference fails (kmer.py:202)
            logger.error(f"Values of row {e.row} are all zero, which should not be the case.")  # kmer.py:255-258
            sys.exit(1)
        self.sorted_kmer_set = list(res["columns"])
        self.kmers = {kmer: i for i, kmer in enumerate(self.sorted_kmer_set)}   # kmer.py:175-177
        self.knn_indices, self.knn_dists = res["knn_idx"], res["knn_dist"]
        kmer_profile = res["profile"] if host_profile else res["d_profile"]
        if not host_profile:
            self._d_knn = (res["d_idx"], res["d_dist"])
        self.sorted_kmer_set.clear()                                            # kmer.py:259
        logger.debug(f"KMER-PROFILE - Size: {sys.getsizeof(kmer_profile)}, Shape: {kmer_profile.shape}")
        return kmer_profile

    def __cluster_on_device(self, neighbors, components, dist, r_state, min_cluster_size):
        """The pass with the profile and k-lists kept on the device, then ``cluster_from_lists``.  Returns
        (labels, probabilities); sets ``embedding`` (host float32), ``stage_ms`` and ``spectral_stats``."""
        from .cluster import check_arguments, cluster_from_lists
        k = check_arguments(len(self.sequences), neighbors, components, min_cluster_size)
        logger.info("Calculate kmer profiles.")
        t0 = time.perf_counter()
        d_profile = self.__calc_kmer_profile(n_neighbors=k, host_profile=False)
        pass_ms = (time.perf_counter() - t0) * 1e3
        d_idx, d_dist = self._d_knn
        self._d_knn = None
        # UMAP and HDBSCAN are one device call here: both messages come before it
        logger.info("Dimension reduction with UMAP.")
        logger.info(f"Perform clustering with HDBSCAN. (min_cluster_size: {min_cluster_size})")
        out = cluster_from_lists(self._get_engine(), d_idx, d_dist, d_profile, components, dist, r_state,
                                 min_cluster_size)
        self.umap_route = "device"
        self.embedding = out["embedding"].cpu().numpy()
        self.stage_ms = {"pass": pass_ms, **out["ms"]}
        self.spectral_stats = out["spectral"]
        return out["labels"], out["probabilities"]

    def run(self, neighbors, components, dist, r_state, min_cluster_size):
        """kmer.py:274-325: resume from cluster.txt if present, else profile (+ kNN) on the GPU,
        UMAP, HDBSCAN, write cluster.txt / eval.txt.  UMAP and HDBSCAN run where ``cluster_on`` says."""
        if os.path.isfile(self.output_file):
            logger.info(f"Read from previous calculation: {self.output_file}")
            self.__read_clusters()
            self.__fix_fasta_headers()
            return
        if self.cluster_on == "device":
            labels, probabilities = self.__cluster_on_device(neighbors, components, dist, r_state, min_cluster_size)
            t0 = time.perf_counter()
            self.__write_results(labels, probabilities, neighbors, components, dist, r_state, min_cluster_size)
            self.stage_ms["files"] = (time.perf_counter() - t0) * 1e3
            return

        logger.info("Calculate kmer profiles.")
        # the exact kNN graph comes out of the same GPU pass when it can replace UMAP's own neighbour search:
        # an integer n_neighbors below the number of contigs (UMAP truncates it itself otherwise)
        want_graph = isinstance(neighbors, (int, np.integer)) and not isinstance(neighbors, bool) and \
            1 <= neighbors < len(self.sequences)
        profile = self.__calc_kmer_profile(n_neighbors=int(neighbors) if want_graph else None)

        logger.info("Dimension reduction with UMAP.")
        umap_args = {"n_neighbors": neighbors, "n_components": components, "min_dist": dist, "random_state": r_state}
        embedding, self.umap_route = umap_embedding(profile, self.knn_indices, self.knn_dists, umap_args)
        if self.umap_route == "stock":
            logger.debug("UMAP computed its own neighbour graph (no hand-off route in this umap-learn).")

        logger.info(f"Perform clustering with HDBSCAN. (min_cluster_size: {min_cluster_size})")
        import hdbscan
        hdb_args = {"allow_single_cluster": True} if min_cluster_size == 1 else {"min_cluster_size": min_cluster_size}
        clusterer = hdbscan.HDBSCAN(**hdb_args).fit(embedding)
        self.__write_results(clusterer.labels_, clusterer.probabilities_, neighbors, components, dist, r_state,
                             min_cluster_size)

    def __write_results(self, labels, probabilities, neighbors, components, dist, r_state, min_cluster_size):
        """The end of kmer.py's run: groups, cluster.txt, eval.txt, then the header fix."""
        self.clusters, self.unlabeled_cluster = self.__mask_list(self.sequences, labels)
        self.__save_groups_to_file()
        self.__write_eval_information(
            kmer_size=self.kmer_size, n_neighbors=neighbors, n_components=components, min_dist=dist,
            random_state=r_state, min_cluster_size=min_cluster_size,
            unlabeled=list(labels).count(-1), no_groups=max(labels) + 1,
            mean_probability=np.mean(probabilities))
        self.__fix_fasta_headers()
