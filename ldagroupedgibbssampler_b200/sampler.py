"""Host-side mirror of the reference's sampler interface over libldagpu.so.

The reference picks a sampler by the ``scheme`` string (topics/tui/ParallelLDA.java:401-490); a sampler
is any class implementing ``LDAGibbsSampler`` (topics/LDAGibbsSampler.java:10-47) and, for the
Phi-based ones, ``LDASamplerWithPhi`` (topics/LDASamplerWithPhi.java:5-12).  ``GpuLDASampler`` keeps
those method names, argument meanings and error behaviour for the two new schemes ``gpu_ggs`` and
``gpu_pcgs``; every method is a thin call into the C ABI (include/ldagpu.h) -- the sweep itself runs
inside the library.  The Java twin of this class is java/cc/mallet/topics/GpuLDASampler.java
(INTEGRATION.md); there is no JDK in the build image, so Python carries the host side here.
"""
from __future__ import annotations

import configparser
import ctypes as C
import os
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np

from . import _lib
from ._lib import LdaGpuError, ptr
from .corpus import InstanceList

# gpu_spalias = PCGS with the reference's sparse z-step (scheme "spalias", topics/tui/ParallelLDA.java:401-490)
# gpu_polyaurn = the sparse z-step with the Poisson Polya-urn Phi draw (scheme "polyaurn", ParallelLDA.java:444-446 ->
# topics/PolyaUrnSpaliasLDA.java)
SCHEMES = {"gpu_ggs": 0, "gpu_pcgs": 1, "gpu_spalias": 2, "gpu_polyaurn": 2}


@dataclass
class LDAConfiguration:
    """The configuration keys the hot path reads (configuration/LDAConfiguration.java:8-246,
    configuration/ParsedLDAConfiguration.java:47-550); defaults as in LDAConfiguration.java:12-51."""

    scheme: str = "gpu_ggs"
    topics: int = 10                      # NO_TOPICS_DEFAULT
    alpha: float = -1.0                   # < 0: ALPHA_DEFAULT = 50 / topics
    beta: float = 0.01                    # BETA_DEFAULT
    iterations: int = 200
    seed: int = 0                         # 0 = clock in the reference (ParsedLDAConfiguration.java:137-141)
    start_diagnostic: int = -1
    compute_likelihood: bool = False
    topic_interval: int = 10
    save_phi_mean: bool = False           # the code reads save_phi_mean, the shipped cfgs write save_phi_means
    phi_mean_burnin: int = 0              # percent of iterations (UPL:206-207)
    phi_mean_thin: int = 1
    exec_time: float = 10.0               # seconds of cumulative sampling time (LDAConfiguration.java:35)
    dataset: Optional[str] = None
    test_dataset: Optional[str] = None    # held-out documents: getHeldOutLogLikelihood on the topic_interval grid
    stoplist: Optional[str] = None        # file with one stop word per line (ParsedLDAConfiguration.java:298-304)
    rare_threshold: int = 0               # RARE_WORD_THRESHOLD (LDAConfiguration.java:16)
    keep_numbers: bool = False            # ParsedLDAConfiguration.java:307-310
    keep_connecting_punctuation: bool = False   # KEEP_CONNECTING_PUNCTUATION (LDAConfiguration.java:40)
    tfidf_vocab_size: int = -1            # TF_IDF_VOCAB_SIZE_DEFAULT (LDAConfiguration.java:37)
    max_doc_buf_size: int = 10000         # token buffer of the tokenizers (ParsedLDAConfiguration.java:402-404)
    logging_path: Optional[str] = None    # run directory of the reference's LoggingUtils (util/LoggingUtils.java:43-109):
                                          # log-likelihood.txt / log-posterior.txt are appended there when set
    save_phi: bool = False                # Phi_KxV_<K>_<V>_<iter>.csv in every diagnostic iteration (UPL:564,806-815)
    print_ndocs_interval: Sequence[int] = (-1,)   # iteration ranges [a1, b1, a2, b2, ...] for the Theta dump (UPL:555,757-775)
    print_ndocs_cnt: int = 0              # rows of theta written by that dump (ParsedLDAConfiguration.java:242-244)
    alias_poisson_threshold: int = 100    # ALIAS_POISSON_DEFAULT_THRESHOLD (types/PoissonFixedCoeffSampler.java:26-51)
    hyperparam_optim_interval: int = -1   # HYPERPARAM_OPTIM_INTERVAL_DEFAULT: off (UPL:214,891-894)
    symmetric_alpha: bool = True          # the GPU path keeps alpha symmetric when it is optimised (MSL:812-858)
    gpu_device: int = 0                   # new key
    gpu_devices: Optional[str] = None     # new key: "0,1,2,3" = shard the corpus over these GPUs from this one process

    def getNoTopics(self, default: int = 10) -> int:
        return self.topics

    def getAlpha(self, default: float = 0.0) -> float:
        return self.alpha if self.alpha > 0 else 50.0 / self.topics

    def getBeta(self, default: float = 0.01) -> float:
        return self.beta

    def getNoIterations(self, default: int = 200) -> int:
        return self.iterations

    def getSeed(self, default: int = 0) -> int:
        return self.seed

    def getScheme(self) -> str:
        return self.scheme

    def loadDataset(self, dataset_fn: Optional[str] = None, alphabet=None, stoplist_dir: Optional[str] = None):
        """``LDAUtils.loadDataset(config, dataset_fn[, alphabet])`` (util/LDAUtils.java:136-182) with this
        configuration's ingest keys.  A relative stop-list name is looked up beside the data set (or in
        ``stoplist_dir``); a missing or empty file means no stop words."""
        from .corpus import load_dataset
        fn = dataset_fn or self.dataset
        stop = None
        if self.stoplist:
            cand = self.stoplist if os.path.isabs(self.stoplist) else os.path.join(
                stoplist_dir or os.path.dirname(os.path.abspath(fn)), self.stoplist)
            stop = cand if os.path.exists(cand) else None
        return load_dataset(fn, stoplist=stop, keep_numbers=self.keep_numbers, alphabet=alphabet,
                            rare_threshold=self.rare_threshold, keep_connectors=self.keep_connecting_punctuation,
                            tfidf_vocab_size=self.tfidf_vocab_size, max_token_buffer=self.max_doc_buf_size)

    def loadTestDataset(self, alphabet, dataset_fn: Optional[str] = None, stoplist_dir: Optional[str] = None):
        """The test set (``test_dataset``) read with the TRAINING alphabet frozen: words the training set does not hold
        are dropped, as MALLET's pipes drop them once the alphabet is frozen."""
        from .corpus import load_dataset
        fn = dataset_fn or self.test_dataset
        if not fn:
            raise ValueError("no test_dataset configured")
        stop = None
        if self.stoplist:
            cand = self.stoplist if os.path.isabs(self.stoplist) else os.path.join(
                stoplist_dir or os.path.dirname(os.path.abspath(fn)), self.stoplist)
            stop = cand if os.path.exists(cand) else None
        return load_dataset(fn, stoplist=stop, keep_numbers=self.keep_numbers, alphabet=alphabet,
                            keep_connectors=self.keep_connecting_punctuation, max_token_buffer=self.max_doc_buf_size,
                            frozen_alphabet=True)

    @staticmethod
    def from_cfg(path: str, subconfig: Optional[str] = None, **overrides) -> "LDAConfiguration":
        """Parse a reference .cfg: global keys, then the [subconfig] section wins
        (configuration/SubConfig.java:57-67), then command-line style overrides
        (configuration/LDACommandLineParser.java:45-64)."""
        text = open(path, "r", encoding="utf-8").read()
        cp = configparser.ConfigParser(inline_comment_prefixes=("#",), interpolation=None, strict=False)
        cp.read_string("[__global__]\n" + text)
        vals = dict(cp["__global__"])
        if subconfig:
            if subconfig not in cp:
                raise KeyError(f"no sub-configuration [{subconfig}] in {path}")
            vals.update(dict(cp[subconfig]))
        vals.update({k: str(v) for k, v in overrides.items()})
        c = LDAConfiguration()

        def boolean(s):
            return str(s).strip().lower() in ("true", "1", "yes")

        for key, conv in (("scheme", str), ("topics", int), ("alpha", float), ("beta", float),
                          ("iterations", int), ("seed", int), ("start_diagnostic", int),
                          ("compute_likelihood", boolean), ("topic_interval", int),
                          ("save_phi_mean", boolean), ("phi_mean_burnin", int), ("phi_mean_thin", int),
                          ("exec_time", float), ("dataset", str), ("test_dataset", str), ("stoplist", str),
                          ("rare_threshold", int),
                          ("keep_numbers", boolean), ("keep_connecting_punctuation", boolean),
                          ("tfidf_vocab_size", int), ("max_doc_buf_size", int), ("logging_path", str),
                          ("alias_poisson_threshold", int), ("hyperparam_optim_interval", int), ("save_phi", boolean),
                          ("print_ndocs_interval", lambda v: tuple(int(x) for x in v.replace(";", ",").split(",") if x.strip())),
                          ("print_ndocs_cnt", int),
                          ("gpu_device", int), ("gpu_devices", str)):
            if key in vals:
                setattr(c, key, conv(vals[key].strip()))
        return c


def in_range_interval(index: int, range_pairs: Sequence[int]) -> bool:
    """LDAUtils.inRangeInterval (util/LDAUtils.java:1624-1632)."""
    if len(range_pairs) < 2:
        raise ValueError("Range must be at least 2 long!")
    if len(range_pairs) % 2:
        raise ValueError("Range must contain an even number of pairs!")
    return any(range_pairs[i] <= index <= range_pairs[i + 1] for i in range(0, len(range_pairs), 2))


def format_double(d: float, no_digits: int = 4) -> str:
    """LDAUtils.formatDouble (util/LDAUtils.java:1203-1210): ``%.4f``, except that a non-zero value below 1e-4 in
    magnitude goes through java.text.DecimalFormat("00.###E0") -- two integer digits, at most three fraction digits
    (HALF_EVEN), the exponent adjusted to match: 1.2345e-5 -> "12.345E-6"."""
    if d == 0.0 or abs(d) >= 0.0001:
        return "%.*f" % (no_digits, d)
    from decimal import ROUND_HALF_EVEN, Decimal
    x = Decimal(repr(float(abs(d))))
    e = x.adjusted() - 1                       # mantissa in [10, 100)
    m = (x.scaleb(-e)).quantize(Decimal("0.001"), rounding=ROUND_HALF_EVEN)
    if m >= 100:
        m, e = (m / 10).quantize(Decimal("0.001"), rounding=ROUND_HALF_EVEN), e + 1
    txt = format(m, "f").rstrip("0").rstrip(".")
    return ("-" if d < 0 else "") + txt + "E" + str(e)


def write_ascii_double_matrix(matrix: np.ndarray, fn: str, sep: str = ","):
    """LDAUtils.writeASCIIDoubleMatrix (util/LDAUtils.java:1223-1254): one row per line, formatDouble cells."""
    with open(fn, "w") as f:
        for row in np.asarray(matrix, np.float64):
            f.write(sep.join(format_double(float(v)) for v in row) + "\n")


def format_top_words_as_csv(top_words: Sequence[Sequence[str]]) -> str:
    """LDAUtils.formatTopWordsAsCsv (util/LDAUtils.java:1429-1443)."""
    return "\n".join(",".join(row) for row in top_words)


def format_top_words(top_words: Sequence[Sequence[str]]) -> str:
    """LDAUtils.formatTopWords (util/LDAUtils.java:1445-1460)."""
    return "\n".join("Topic %d: %s" % (i + 1, " ".join(row)) for i, row in enumerate(top_words))


def digamma(z: float) -> float:
    """Digamma by recurrence up to z >= 6 and the asymptotic series (what MALLET's Dirichlet.digamma does)."""
    import math
    psi = 0.0
    while z < 6.0:
        psi -= 1.0 / z
        z += 1.0
    inv = 1.0 / z
    inv2 = inv * inv
    return psi + math.log(z) - 0.5 * inv - inv2 * (1.0 / 12.0 - inv2 * (1.0 / 120.0 - inv2 * (1.0 / 252.0 - inv2 * (
        1.0 / 240.0 - inv2 * (1.0 / 132.0)))))


def learn_symmetric_concentration(count_histogram, observation_lengths, num_dimensions: int, current_value: float,
                                  iterations: int = 200) -> float:
    """MALLET 2.0.8 ``Dirichlet.learnSymmetricConcentration`` (the jar is not in the reference tree, pom.xml:130-141;
    restated from its published source): Minka's fixed point for the concentration alpha_sum of a symmetric
    Dirichlet-multinomial from two histograms -- ``count_histogram[c]`` = number of (observation, dimension) pairs
    with count c, ``observation_lengths[n]`` = number of observations of length n.  Called by
    ModifiedSimpleLDA.optimizeAlpha / optimizeBeta (MSL:847-852,897-901)."""
    ch = np.asarray(count_histogram, np.float64)
    ol = np.asarray(observation_lengths, np.float64)
    largest = int(np.max(np.nonzero(ch)[0])) if np.any(ch[1:] > 0) else 0
    lengths = np.nonzero(ol)[0]
    idx = np.arange(1, largest + 1, dtype=np.float64)
    value = float(current_value)
    for _ in range(iterations):
        param = value / num_dimensions
        # numerator: sum_c hist[c] * sum_{i<c} 1 / (param + i)
        num = float(np.dot(ch[1:largest + 1], np.cumsum(1.0 / (param + idx - 1.0)))) if largest else 0.0
        # denominator: sum_n lengths[n] * (digamma(value + n) - digamma(value))
        base = digamma(value)
        den = float(sum(ol[n] * (digamma(value + float(n)) - base) for n in lengths if n > 0))
        if not (num > 0.0 and den > 0.0):
            break
        value = param * num / den
    return value


@dataclass
class TopicAssignment:
    """MALLET's cc.mallet.topics.TopicAssignment as the samplers use it: the document's type ids
    (``instance``, a FeatureSequence's features) and its topic indicators (``topicSequence``)."""

    instance: np.ndarray
    topicSequence: np.ndarray


class GpuLDASampler:
    """``LDAGibbsSampler`` + ``LDASamplerWithPhi`` for ``scheme = gpu_ggs | gpu_pcgs``."""

    def __init__(self, config: LDAConfiguration, scheme: Optional[str] = None, device: Optional[int] = None,
                 devices: Optional[Sequence[int]] = None):
        self._L = _lib.load()
        self.config = config
        self.scheme = scheme or config.getScheme()
        if self.scheme not in SCHEMES:
            raise ValueError(f"unknown scheme {self.scheme!r}: expected one of {sorted(SCHEMES)}")
        self.device = config.gpu_device if device is None else device
        # several GPUs driven from this one process (ldagpu_create_multi): `devices`, or the gpu_devices key
        if devices is None and config.gpu_devices:
            devices = [int(x) for x in str(config.gpu_devices).replace(";", ",").split(",") if x.strip()]
        self.devices = [int(d) for d in devices] if devices is not None and len(devices) >= 1 else None
        self.numTopics = config.getNoTopics()
        a = config.getAlpha()
        self.alpha = np.full(self.numTopics, a, np.float64)     # MSL:139-143 symmetric alpha
        self.beta = float(config.getBeta())
        self.startSeed = int(config.getSeed())
        self._h = C.c_void_p()
        self._data: Optional[InstanceList] = None
        self._doc_off = None
        self._tokens = None
        self.loglikelihood: List[float] = []
        self.heldout_loglikelihood: List[float] = []
        self._test_doc_off: Optional[np.ndarray] = None   # this process's test documents (None: no test set)
        self._rank, self._world = 0, 1
        self._doc_base = self._token_base = 0

    # ---- plumbing ---------------------------------------------------------------------------
    def _ck(self, rc: int):
        if rc:
            msg = self._L.ldagpu_last_error(self._h if self._h else None)
            raise LdaGpuError(msg.decode() if msg else "libldagpu error")

    def _need(self):
        if not self._h:
            raise LdaGpuError("addInstances has not been called")

    def close(self):
        if self._h:
            self._L.ldagpu_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- LDAGibbsSampler ---------------------------------------------------------------------
    def setConfiguration(self, config: LDAConfiguration):
        self.config = config

    def getConfiguration(self) -> LDAConfiguration:
        return self.config

    def setRandomSeed(self, seed: int):
        """MSL:153-156.  Also re-keys the in-sweep Philox stream when called before addInstances."""
        self.startSeed = int(seed)

    def getStartSeed(self) -> int:
        return self.startSeed

    def addInstances(self, training: InstanceList, *, rank: int = 0, world: int = 1,
                     comm_id: Optional[bytes] = None, init_z: bool = True,
                     presharded: Optional[tuple] = None):
        """UPL:357-456: upload the corpus, draw the initial z from java.util.Random(seed) in document
        order (UPL:398-406), build the counts and draw the initial Phi (UPL:450).  With world > 1 this
        rank keeps a token-balanced contiguous shard of the documents."""
        from .corpus import shard_documents_by_tokens, take_shard
        self.close()
        self._data = training
        off, tokens = training.to_csr()
        self.numTypes = training.getNumTypes()
        self._global_doc_off = off
        self._doc_base = self._token_base = 0
        if presharded is not None:
            # the caller already holds only this rank's documents: (doc_base, token_base, corpus tokens)
            self._doc_base, self._token_base, total = presharded
            self._global_doc_off = np.array([0, total], np.int64)
        elif world > 1:
            d0, d1 = shard_documents_by_tokens(off, world)[rank]
            off, tokens, self._doc_base, self._token_base = take_shard(off, tokens, d0, d1)
        self._doc_off, self._tokens = np.ascontiguousarray(off, np.int64), np.ascontiguousarray(tokens, np.int32)
        self._rank, self._world = rank, world
        if self.devices is not None:
            if world > 1:
                raise ValueError("gpu_devices (one process, several GPUs) and world > 1 (one process per GPU) exclude each other")
            dev = np.ascontiguousarray(self.devices, np.int32)
            self._ck(self._L.ldagpu_create_multi(self.numTopics, self.numTypes, len(off) - 1, ptr(self._doc_off),
                                                 ptr(self._tokens) if len(tokens) else None, ptr(self.alpha), self.beta,
                                                 self.startSeed & 0xFFFFFFFFFFFFFFFF, SCHEMES[self.scheme], len(dev),
                                                 ptr(dev), C.byref(self._h)))
        else:
            self._ck(self._L.ldagpu_create(self.numTopics, self.numTypes, len(off) - 1, ptr(self._doc_off),
                                           ptr(self._tokens) if len(tokens) else None, ptr(self.alpha), self.beta,
                                           self.startSeed & 0xFFFFFFFFFFFFFFFF, SCHEMES[self.scheme], self.device,
                                           self._doc_base, self._token_base, C.byref(self._h)))
        if self.scheme == "gpu_polyaurn":
            self._ck(self._L.ldagpu_set_phi_sampler(self._h, 1, int(self.config.alias_poisson_threshold)))
        if world > 1:
            if comm_id is None:
                raise ValueError("world > 1 needs the 128-byte communicator id (GpuLDASampler.make_comm_id on rank 0)")
            buf = (C.c_char * 128).from_buffer_copy(comm_id)
            self._ck(self._L.ldagpu_comm_init(self._h, rank, world, buf))
        if init_z:
            java_seed = ((self.startSeed + 2 ** 31) % 2 ** 32) - 2 ** 31     # Java int
            self._ck(self._L.ldagpu_init_z_java_random(self._h, java_seed))
        self.loglikelihood = []
        self.heldout_loglikelihood = []
        self._test_doc_off = None

    @staticmethod
    def make_comm_id() -> bytes:
        buf = (C.c_char * 128)()
        if _lib.load().ldagpu_comm_unique_id(buf):
            raise LdaGpuError("ldagpu_comm_unique_id failed (is libnccl.so.2 loadable?)")
        return bytes(buf)

    def addTestInstances(self, testSet: InstanceList):
        """LGS addTestInstances: upload the test set (type ids of the training alphabet, e.g. from
        ``LDAConfiguration.loadTestDataset``).  With world > 1 this rank keeps the token-balanced shard of the test
        documents that matches its rank, as for the training set; several GPUs of one process shard it themselves.
        An empty test set removes it.  K <= 1024 only (DESIGN.md 4.8)."""
        from .corpus import shard_documents_by_tokens, take_shard
        self._need()
        off, tokens = testSet.to_csr()
        doc_base = token_base = 0
        if self._world > 1:
            d0, d1 = shard_documents_by_tokens(off, self._world)[self._rank]
            off, tokens, doc_base, token_base = take_shard(off, tokens, d0, d1)
        off = np.ascontiguousarray(off, np.int64)
        tokens = np.ascontiguousarray(tokens, np.int32)
        D = len(off) - 1 if testSet.size() else 0
        self._ck(self._L.ldagpu_set_test_documents(self._h, D, ptr(off), ptr(tokens) if len(tokens) else None,
                                                   doc_base, token_base))
        self._test_doc_off = off if testSet.size() else None
        self.heldout_loglikelihood = []

    def heldOutLogLikelihood(self, n_particles: int = 10):
        """MarginalProbEstimatorPlain.evaluateLeftToRight (UPL:604-611,840-844) on the current counts: MALLET's
        left-to-right estimator with ``n_particles`` particles (MALLET's default 10) and no resampling.  Returns
        (total over the whole test set, float64 array of ln p(w_d) for this process's test documents)."""
        self._need()
        if self._test_doc_off is None:
            raise LdaGpuError("addTestInstances has not been called")
        out = np.zeros(max(len(self._test_doc_off) - 1, 1), np.float64)
        total = C.c_double(0)
        self._ck(self._L.ldagpu_heldout_log_likelihood(self._h, int(n_particles), ptr(out), C.byref(total)))
        return total.value, out[: len(self._test_doc_off) - 1]

    SWEEPS_PER_CALL = 10   # the abort flag and the exec_time budget are looked at between library calls

    def sample(self, iterations: int, z_out: Optional[np.ndarray] = None, chunk: Optional[int] = None):
        """UPL:552-943: `iterations` sweeps; log-likelihood every topic_interval sweeps when
        compute_likelihood is set (UPL:587-593,838-853).  ``z_out`` (int32[N] or uint16[N], ideally pinned):
        receives the topic indicators after the last sweep, copied while that sweep's Phi draw still runs
        (``ldagpu_sweep_get_z``) -- what the Java shim does after every sample() call.
        The reference looks at ``abort`` and at ``zSamplingTimeCum + phiSamplingTimeCum >= exec_time`` after every
        iteration (UPL:645,926-928).  Here at most ``chunk`` sweeps (default SWEEPS_PER_CALL) go into one library
        call and both are checked between calls, with the timers counted from the start of THIS sample() call;
        ``chunk=0`` puts everything into one call (benchmarks that time a fixed number of sweeps)."""
        self._need()
        cfg = self.config
        z_filled = False
        if z_out is not None and (z_out.dtype not in (np.int32, np.uint16) or not z_out.flags.c_contiguous
                                  or z_out.size < len(self._tokens)):
            raise ValueError("z_out must be a contiguous int32 (or uint16) array of at least N elements")
        z16 = z_out is not None and z_out.dtype == np.uint16
        if cfg.save_phi_mean:
            burn = int(cfg.phi_mean_burnin / 100.0 * iterations)          # UPL:206-207
            self._ck(self._L.ldagpu_set_phi_mean_schedule(self._h, burn, cfg.phi_mean_thin))
        self.preSample()
        # the log-likelihood grid: every topic_interval sweeps when compute_likelihood is set or a test set is present
        held_out = self._test_doc_off is not None
        grid = cfg.compute_likelihood or held_out
        if cfg.compute_likelihood:
            self.loglikelihood.append(self.modelLogLikelihood())
        if held_out:
            self.heldout_loglikelihood.append(self.heldOutLogLikelihood()[0])
        hooked = any(getattr(type(self), n) is not getattr(GpuLDASampler, n)
                     for n in ("preIteration", "postIteration", "preZ", "postZ", "prePhi", "postPhi"))
        per_call = self.SWEEPS_PER_CALL if chunk is None else chunk
        step = max(1, cfg.topic_interval) if grid else iterations
        if per_call > 0:
            step = min(step, per_call)
        t_start = sum(self.getTimers())
        done_total = 0
        while done_total < iterations and not self.getAbort():
            n = min(step, iterations - done_total)
            if grid:   # keep the log-likelihood on its topic_interval grid
                n = min(n, max(1, cfg.topic_interval) - done_total % max(1, cfg.topic_interval))
            if cfg.hyperparam_optim_interval > 1:   # stop where alpha and beta are re-estimated (UPL:891-894)
                it = self.getCurrentIteration()
                n = min(n, cfg.hyperparam_optim_interval - it % cfg.hyperparam_optim_interval)
            if cfg.start_diagnostic > 0:
                # the diagnostic block runs after every sweep from start_diagnostic on (UPL:707-823)
                it = self.getCurrentIteration()
                n = 1 if it + 1 >= cfg.start_diagnostic else min(n, cfg.start_diagnostic - 1 - it)
            if hooked:
                for _ in range(n):
                    self._one_hooked_sweep()
                done = n
            else:
                d = C.c_int32(0)
                if z_out is not None and done_total + n >= iterations:
                    fn = self._L.ldagpu_sweep_get_z16 if z16 else self._L.ldagpu_sweep_get_z
                    self._ck(fn(self._h, n, C.byref(d), ptr(z_out)))
                    z_filled = True
                else:
                    self._ck(self._L.ldagpu_sweep(self._h, n, C.byref(d)))
                done = d.value
            done_total += done
            if cfg.start_diagnostic > 0 and done == n and self.getCurrentIteration() >= cfg.start_diagnostic:
                self._log_posterior_to_file(self.computeLogPosterior())                       # UPL:820-821
                self._diagnostic_dumps(theta_ready=True)                                      # UPL:757-775,806-815
            if cfg.compute_likelihood and done == n and done_total % max(1, cfg.topic_interval) == 0:
                self.loglikelihood.append(self.modelLogLikelihood())
                self._log_likelihood_to_file(self.loglikelihood[-1])                          # UPL:846-850
            if held_out and done == n and done_total % max(1, cfg.topic_interval) == 0:
                self.heldout_loglikelihood.append(self.heldOutLogLikelihood()[0])            # UPL:840-844
            if done < n:
                break
            if cfg.hyperparam_optim_interval > 1 and self.getCurrentIteration() % cfg.hyperparam_optim_interval == 0:
                self.optimizeAlpha()
                self.optimizeBeta()
            if (sum(self.getTimers()) - t_start) / 1000.0 >= cfg.exec_time > 0:        # UPL:926-928
                break
        if z_out is not None and not z_filled:
            self._ck((self._L.ldagpu_get_z16 if z16 else self._L.ldagpu_get_z)(self._h, ptr(z_out)))
        self.postSample()

    def _one_hooked_sweep(self):
        L, h = self._L, self._h
        self._ck(L.ldagpu_next_iteration(h))
        self.preIteration()
        self.preZ()
        if self.scheme == "gpu_ggs":
            self._ck(L.ldagpu_sample_theta(h))
        self._ck(L.ldagpu_sample_z(h))
        self._ck(L.ldagpu_rebuild_counts(h))
        self.postZ()
        self.prePhi()
        self._ck(L.ldagpu_sample_phi(h))
        self.postPhi()
        self.postIteration()

    def sampleZGivenPhi(self, iterations: int):
        """LSWP:11, UPL:975-1014: z-only sweeps with Phi frozen."""
        self._need()
        d = C.c_int32(0)
        self._ck(self._L.ldagpu_sample_z_given_phi(self._h, iterations, C.byref(d)))

    def getNoTopics(self) -> int:
        return self.numTopics

    getNumTopics = getNoTopics

    def getNoTypes(self) -> int:
        return self.numTypes

    def getCurrentIteration(self) -> int:
        self._need()
        it = C.c_int32(0)
        self._ck(self._L.ldagpu_get_iteration(self._h, C.byref(it)))
        return it.value

    def get_z_flat(self) -> np.ndarray:
        self._need()
        z = np.zeros(len(self._tokens), np.int32)
        self._ck(self._L.ldagpu_get_z(self._h, ptr(z)))
        return z

    def set_z_flat(self, z: np.ndarray, redraw_phi: bool = True):
        self._need()
        z = np.ascontiguousarray(z, np.int32)
        if len(z) != len(self._tokens):
            # UPL:1828-1830
            raise ValueError(f"Count does not sum to nr. types! Sumtotal: {len(z)} no.types: {len(self._tokens)}")
        self._ck(self._L.ldagpu_set_z(self._h, ptr(z), 1 if redraw_phi else 0))

    def set_z16_flat(self, z: np.ndarray, redraw_phi: bool = True):
        """setZIndicators with the indicators held as uint16 on the host (K <= 65 536): half the PCIe bytes."""
        self._need()
        z = np.ascontiguousarray(z, np.uint16)
        if len(z) != len(self._tokens):
            raise ValueError(f"Count does not sum to nr. types! Sumtotal: {len(z)} no.types: {len(self._tokens)}")
        self._ck(self._L.ldagpu_set_z16(self._h, ptr(z), 1 if redraw_phi else 0))

    def getZIndicators(self) -> List[np.ndarray]:
        """MSL:464-477: int[D][] (local documents)."""
        z, off = self.get_z_flat(), self._doc_off
        return [z[off[d]: off[d + 1]].copy() for d in range(len(off) - 1)]

    def setZIndicators(self, zIndicators: Sequence[Sequence[int]]):
        """UPL:1797-1843: replace z, rebuild the counts, redraw Phi."""
        flat = (np.concatenate([np.asarray(d, np.int32) for d in zIndicators])
                if len(zIndicators) else np.zeros(0, np.int32))
        lens = np.fromiter((len(d) for d in zIndicators), np.int64, len(zIndicators))
        if len(lens) != len(self._doc_off) - 1 or np.any(lens != np.diff(self._doc_off)):
            raise ValueError("zIndicators do not match the document lengths")
        self.set_z_flat(flat, True)

    def getDocumentTopicMatrix(self) -> np.ndarray:
        """MSL:536-547: int[D][K]."""
        self._need()
        out = np.zeros((len(self._doc_off) - 1, self.numTopics), np.int32)
        self._ck(self._L.ldagpu_get_doc_topic_counts(self._h, ptr(out)))
        return out

    def getZbar(self) -> np.ndarray:
        """MSL:620-668: n_dk / N_d (zero rows for empty documents)."""
        ndk = self.getDocumentTopicMatrix().astype(np.float64)
        lens = np.diff(self._doc_off).astype(np.float64)
        return np.divide(ndk, lens[:, None], out=np.zeros_like(ndk), where=lens[:, None] > 0)

    def getThetaEstimate(self) -> np.ndarray:
        """MSL:709-753: (n_dk + alpha_k) / sum_k (n_dk + alpha_k)."""
        p = self.getDocumentTopicMatrix().astype(np.float64) + self.alpha[None, :]
        return p / p.sum(axis=1, keepdims=True)

    def getTypeTopicMatrix(self) -> np.ndarray:
        """LGS:32 / UPL:226-234: int[V][K]."""
        self._need()
        out = np.zeros((self.numTypes, self.numTopics), np.int32)
        self._ck(self._L.ldagpu_get_type_topic_counts(self._h, ptr(out)))
        return out

    getTypeTopicCounts = getTypeTopicMatrix

    def getTopicTotals(self) -> np.ndarray:
        """MSL:971-976: int[K]."""
        self._need()
        out = np.zeros(self.numTopics, np.int32)
        self._ck(self._L.ldagpu_get_topic_totals(self._h, ptr(out)))
        return out

    def getDeltaStatistics(self):
        raise NotImplementedError("per-sweep deltas are only read by the random-scan builders (SURVEY App. A)")

    def getBeta(self) -> float:
        return self.beta

    def getAlpha(self) -> np.ndarray:
        return self.alpha

    def getDataset(self) -> InstanceList:
        return self._data

    def getData(self) -> List["TopicAssignment"]:
        """LGS:26, MSL:42: one TopicAssignment (instance tokens + topicSequence) per local document, with the
        CURRENT topic indicators -- the copy back into each document's LabelSequence that the Java shim does
        after every sample() call (util/LDAUtils.java:1552-1571 and MSL:464-477,536-547 read z from there)."""
        self._need()
        z, off = self.get_z_flat(), self._doc_off
        return [TopicAssignment(self._tokens[off[d]: off[d + 1]], z[off[d]: off[d + 1]]) for d in range(len(off) - 1)]

    def getAlphabet(self):
        return self._data.getDataAlphabet()

    def getCorpusSize(self) -> int:
        return int(self._global_doc_off[-1])

    def getTypeFrequencies(self) -> np.ndarray:
        return np.bincount(self._tokens, minlength=self.numTypes).astype(np.int32)

    def getTopTypeFrequencyIndices(self) -> np.ndarray:
        return np.argsort(-self.getTypeFrequencies(), kind="stable").astype(np.int32)

    def getTypeMassCumSum(self) -> np.ndarray:
        f = self.getTypeFrequencies()[self.getTopTypeFrequencyIndices()].astype(np.float64)
        return np.cumsum(f / max(f.sum(), 1.0))

    def getLogLikelihood(self) -> List[float]:
        return list(self.loglikelihood)

    def getHeldOutLogLikelihood(self) -> List[float]:
        """The held-out log-likelihood series of sample() (empty without a test set)."""
        return list(self.heldout_loglikelihood)

    def modelLogLikelihood(self) -> float:
        """UPL:1644-1758."""
        self._need()
        v = C.c_double(0)
        self._ck(self._L.ldagpu_log_likelihood(self._h, C.byref(v)))
        return v.value

    def computeLogPosterior(self) -> float:
        """UPL:1573-1634.  GGS evaluates it with the sweep's own theta (UPL:716-720); the other schemes draw a
        diagnostic theta ~ Dir(n_d + alpha) first (UPL:710-714, util/LDAUtils.java:1662-1673) -- here with the
        library's theta kernel (counter = current iteration) instead of MALLET's Dirichlet.nextDistribution."""
        self._need()
        if self.scheme != "gpu_ggs":
            self._ck(self._L.ldagpu_sample_theta(self._h))
        v = C.c_double(0)
        self._ck(self._L.ldagpu_log_posterior(self._h, C.byref(v)))
        return v.value

    # ---- outputs of the driver and of the diagnostic block ---------------------------------------------------------
    def getTopWordIndices(self, noWords: int) -> np.ndarray:
        """LDAUtils.getTopWordIndices (util/LDAUtils.java:896-912): per topic the types sorted by n_wk descending (a
        stable sort: ties keep the type order, as Arrays.sort on IDSorter objects does): int[K][noWords]."""
        if noWords > self.numTypes:
            raise ValueError(f"Asked for more words ({noWords}) than there are types (unique words = noTypes = {self.numTypes}).")
        n_wk = self.getTypeTopicMatrix()
        return np.stack([np.argsort(-n_wk[:, k], kind="stable")[:noWords] for k in range(self.numTopics)]).astype(np.int32)

    def getTopWords(self, noWords: int) -> List[List[str]]:
        """LDAUtils.getTopWords (util/LDAUtils.java:874-894) on this sampler's counts and alphabet."""
        alph = self.getAlphabet()
        return [[str(alph.lookupObject(int(t))) for t in row] for row in self.getTopWordIndices(noWords)]

    def writeTopWords(self, path: str, noWords: int = 20):
        """TopWords.txt as the driver writes it (topics/tui/ParallelLDA.java:56,268-282)."""
        with open(path, "w") as f:
            f.write(format_top_words_as_csv(self.getTopWords(min(noWords, self.numTypes))) + "\n")

    def _diagnostic_dumps(self, theta_ready: bool):
        """The file outputs of the diagnostic block (UPL:707-823) besides log-posterior.txt: Theta_DxK_<n>_<K>_<iter>.csv
        for iterations inside print_ndocs_interval (first print_ndocs_cnt documents, UPL:757-775) and
        Phi_KxV_<K>_<V>_<iter>.csv when save_phi is set (UPL:806-815), both under <logging_path>/ascii (UPL:572-574)."""
        cfg = self.config
        if not cfg.logging_path or self._rank != 0:
            return
        it = self.getCurrentIteration()
        asc = os.path.join(cfg.logging_path, "ascii")
        want_theta = len(cfg.print_ndocs_interval) > 1 and in_range_interval(it, cfg.print_ndocs_interval)
        if want_theta or cfg.save_phi:
            os.makedirs(asc, exist_ok=True)
        if want_theta:
            if not theta_ready and self.scheme != "gpu_ggs":
                self._ck(self._L.ldagpu_sample_theta(self._h))
            theta = self.getTheta()
            n = cfg.print_ndocs_cnt
            rows = theta[:n] if len(theta) > n else theta
            write_ascii_double_matrix(rows, os.path.join(asc, "Theta_DxK_%d_%d_%05d.csv" % (n, self.numTopics, it)))
        if cfg.save_phi:
            write_ascii_double_matrix(self.getPhi(), os.path.join(asc, "Phi_KxV_%d_%d_%05d.csv" % (self.numTopics, self.numTypes, it)))

    # ---- hyper-parameter optimisation (MSL:812-905; UPL:891-894 every hyperparam_optim_interval sweeps) -----------
    def _count_histograms(self):
        """(doc_topic_hist, type_topic_hist, doc_length_hist, topic_size_hist) -- the sufficient statistics of
        MSL:815-846 (documentTopicHistogram merged over topics, the symmetric case), :860-875, :419-431, :877-889."""
        self._need()
        lens = np.diff(self._doc_off)
        max_len = int(lens.max()) if len(lens) else 0
        type_freq = np.bincount(self._tokens, minlength=self.numTypes)
        max_type = int(type_freq.max()) if len(type_freq) else 0
        dh = np.zeros(max_len + 1, np.int64)
        th = np.zeros(max_type + 1, np.int64)
        self._ck(self._L.ldagpu_get_count_histograms(self._h, len(dh), ptr(dh), len(th), ptr(th)))
        n_k = self.getTopicTotals()
        return dh, th, np.bincount(lens, minlength=max_len + 1), np.bincount(n_k, minlength=int(n_k.max()) + 1)

    def optimizeAlpha(self):
        """MSL:812-858 for a symmetric alpha (the GPU path keeps alpha symmetric): alphaSum by the fixed point over
        the histogram of n_dk, then alpha_k = alphaSum / K, pushed into the library."""
        dh, _, doc_len_hist, _ = self._count_histograms()
        alpha_sum = learn_symmetric_concentration(dh, doc_len_hist, self.numTopics, float(self.alpha.sum()))
        self.alpha = np.full(self.numTopics, alpha_sum / self.numTopics, np.float64)
        self._ck(self._L.ldagpu_set_alpha(self._h, ptr(self.alpha)))

    def optimizeBeta(self):
        """MSL:860-905: betaSum by the same fixed point over the histogram of n_wk and of the topic sizes."""
        _, th, _, topic_size_hist = self._count_histograms()
        beta_sum = learn_symmetric_concentration(th, topic_size_hist, self.numTypes, self.beta * self.numTypes)
        self.beta = beta_sum / self.numTypes
        self._ck(self._L.ldagpu_set_beta(self._h, self.beta))

    def _log_posterior_to_file(self, lp: float):
        """util/LDAUtils.java:955-968: `iteration<TAB>logPosterior (6 decimals)<TAB>millis` appended to log-posterior.txt"""
        if self.config.logging_path and self._rank == 0:
            import time
            os.makedirs(self.config.logging_path, exist_ok=True)
            with open(os.path.join(self.config.logging_path, "log-posterior.txt"), "a") as f:
                f.write("%d\t%.6f\t%d\n" % (self.getCurrentIteration(), lp, int(time.time() * 1000)))

    def _log_likelihood_to_file(self, ll: float):
        """util/LDAUtils.java:971-979: `iteration<TAB>logLik` appended to log-likelihood.txt"""
        if self.config.logging_path and self._rank == 0:
            os.makedirs(self.config.logging_path, exist_ok=True)
            with open(os.path.join(self.config.logging_path, "log-likelihood.txt"), "a") as f:
                f.write("%d\t%r\n" % (self.getCurrentIteration(), ll))

    # hooks (MSL:783-810): no-ops; subclasses override, sample() then runs step-wise
    def preSample(self): pass
    def postSample(self): pass
    def preIteration(self): pass
    def postIteration(self): pass
    def preZ(self): pass
    def postZ(self): pass
    def prePhi(self): pass
    def postPhi(self): pass

    # ---- AbortableSampler -------------------------------------------------------------------
    def abort(self):
        if self._h:
            self._L.ldagpu_abort(self._h)

    def getAbort(self) -> bool:
        if not self._h:
            return False
        v = C.c_int32(0)
        self._L.ldagpu_get_abort(self._h, C.byref(v))
        return bool(v.value)

    # ---- LDASamplerWithPhi -------------------------------------------------------------------
    def getPhi(self) -> np.ndarray:
        """UPL:1946-1948: double[K][V]."""
        self._need()
        out = np.zeros((self.numTopics, self.numTypes), np.float64)
        self._ck(self._L.ldagpu_get_phi(self._h, ptr(out)))
        return out

    def setPhi(self, phi: np.ndarray, dataAlphabet=None, targetAlphabet=None):
        """UPL:1897-1926."""
        self._need()
        if dataAlphabet is not None and self._data.alphabet.size() and not dataAlphabet == self.getAlphabet():
            raise ValueError("Vocabularies does not match!")
        phi = np.ascontiguousarray(phi, np.float64)
        if phi.shape != (self.numTopics, self.numTypes):
            raise ValueError(f"phi must be [{self.numTopics}][{self.numTypes}]")
        self._ck(self._L.ldagpu_set_phi(self._h, ptr(phi)))

    def getPhiMeans(self) -> Optional[np.ndarray]:
        """UPL:1954-1966: None until a Phi has been accumulated."""
        self._need()
        out = np.zeros((self.numTopics, self.numTypes), np.float64)
        n = C.c_int32(0)
        self._ck(self._L.ldagpu_get_phi_mean(self._h, ptr(out), C.byref(n)))
        return out if n.value > 0 else None

    def getTheta(self) -> np.ndarray:
        """thetaMatrix of the last sweep (UPL:78, GGS:72): double[D][K]."""
        self._need()
        out = np.zeros((len(self._doc_off) - 1, self.numTopics), np.float64)
        self._ck(self._L.ldagpu_get_theta(self._h, ptr(out)))
        return out

    def setTheta(self, theta: np.ndarray):
        self._need()
        theta = np.ascontiguousarray(theta, np.float64)
        self._ck(self._L.ldagpu_set_theta(self._h, ptr(theta)))

    # ---- timers (the reference prints these, UPL:931-939) -----------------------------------
    def getTimers(self):
        v = [C.c_double(0) for _ in range(4)]
        self._L.ldagpu_get_timers(self._h, *[C.byref(x) for x in v])
        return tuple(x.value for x in v)

    def getLastCallStats(self):
        """(device ms of the last sample()/sampleZGivenPhi() library call, ms in the z-step kernel,
        z-step launches, all kernel launches)"""
        cm, ms, zl, tl = C.c_double(0), C.c_double(0), C.c_int64(0), C.c_int64(0)
        self._L.ldagpu_get_last_call_stats(self._h, C.byref(cm), C.byref(ms), C.byref(zl), C.byref(tl))
        return cm.value, ms.value, zl.value, tl.value

    def getExchangeMode(self) -> str:
        """How the ranks exchange counts and Phi: "single", "nccl" (collectives around the Phi kernels) or
        "p2p" (the Phi kernels read/write the other ranks' memory over NVLink themselves)."""
        m = C.c_int32(0)
        self._L.ldagpu_get_exchange_mode(self._h, C.byref(m))
        return ("single", "nccl", "p2p")[m.value]

    # step-wise access for tests
    def _step(self, name: str):
        self._need()
        self._ck(getattr(self._L, "ldagpu_" + name)(self._h))


def createModel(config: LDAConfiguration, scheme: Optional[str] = None) -> GpuLDASampler:
    """The two new `case` labels of ParallelLDA.createModel (topics/tui/ParallelLDA.java:401-490)."""
    return GpuLDASampler(config, scheme or config.getScheme())
