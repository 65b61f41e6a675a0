package cc.mallet.topics;

// Reference-side binding of libldagpu.so (include/ldagpu.h) -- the class a maintainer of
// clintpgeorge/LDAGroupedGibbsSampler would add for `scheme = gpu_ggs | gpu_pcgs | gpu_spalias | gpu_polyaurn`.
// NOT compiled in this repository's build image (no JDK there); written against
//   * the reference's ModifiedSimpleLDA (accessors, data, alphabet; topics/ModifiedSimpleLDA.java)
//   * the interfaces LDAGibbsSampler (topics/LDAGibbsSampler.java:10-47) and LDASamplerWithPhi
//     (topics/LDASamplerWithPhi.java:5-12)
//   * the Panama Foreign Function & Memory API (JDK 22+).  On JDK 8-21 the same calls go through a
//     ~60-line JNI stub; the C signatures are identical.
// Factory wiring: two `case` labels in topics/tui/ParallelLDA.java:401-490, see INTEGRATION.md.

import java.io.File;
import java.io.IOException;
import java.lang.foreign.*;
import java.lang.invoke.MethodHandle;

import cc.mallet.configuration.LDAConfiguration;
import cc.mallet.types.Alphabet;
import cc.mallet.types.Dirichlet;
import cc.mallet.types.FeatureSequence;
import cc.mallet.types.InstanceList;
import cc.mallet.types.LabelSequence;
import cc.mallet.util.LDAUtils;
import cc.mallet.util.LoggingUtils;

import static java.lang.foreign.ValueLayout.*;

public class GpuLDASampler extends ModifiedSimpleLDA implements LDAGibbsSampler, LDASamplerWithPhi {
    private static final long serialVersionUID = 1L;
    private static final java.util.logging.Logger LOG = java.util.logging.Logger.getLogger(GpuLDASampler.class.getName());

    // ---- C ABI --------------------------------------------------------------------------------
    private static final Linker LINKER = Linker.nativeLinker();
    private static final SymbolLookup LIB = SymbolLookup.libraryLookup(
            System.getProperty("ldagpu.library", "libldagpu.so"), Arena.global());

    private static MethodHandle fn(String name, FunctionDescriptor d) {
        return LINKER.downcallHandle(LIB.find(name).orElseThrow(), d);
    }

    private static final MethodHandle CREATE = fn("ldagpu_create", FunctionDescriptor.of(JAVA_INT,
            JAVA_INT, JAVA_INT, JAVA_LONG, ADDRESS, ADDRESS, ADDRESS, JAVA_DOUBLE, JAVA_LONG, JAVA_INT, JAVA_INT,
            JAVA_LONG, JAVA_LONG, ADDRESS));
    // one JVM, several GPUs: the reference has ONE coordinator thread (tui/ParallelLDA.java:173-202 -> UPL:552-943)
    private static final MethodHandle CREATE_MULTI = fn("ldagpu_create_multi", FunctionDescriptor.of(JAVA_INT,
            JAVA_INT, JAVA_INT, JAVA_LONG, ADDRESS, ADDRESS, ADDRESS, JAVA_DOUBLE, JAVA_LONG, JAVA_INT, JAVA_INT,
            ADDRESS, ADDRESS));
    private static final MethodHandle SET_PHI_SAMPLER = fn("ldagpu_set_phi_sampler", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, JAVA_INT));
    private static final MethodHandle GET_TIMERS = fn("ldagpu_get_timers", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS));
    private static final MethodHandle DESTROY = fn("ldagpu_destroy", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    private static final MethodHandle LAST_ERROR = fn("ldagpu_last_error", FunctionDescriptor.of(ADDRESS, ADDRESS));
    private static final MethodHandle INIT_Z = fn("ldagpu_init_z_java_random", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT));
    private static final MethodHandle SET_Z = fn("ldagpu_set_z", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_INT));
    private static final MethodHandle GET_Z = fn("ldagpu_get_z", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
    private static final MethodHandle SWEEP = fn("ldagpu_sweep", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, ADDRESS));
    private static final MethodHandle Z_GIVEN_PHI = fn("ldagpu_sample_z_given_phi", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, ADDRESS));
    private static final MethodHandle GET_NWK = fn("ldagpu_get_type_topic_counts", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
    private static final MethodHandle GET_NK = fn("ldagpu_get_topic_totals", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
    private static final MethodHandle GET_PHI = fn("ldagpu_get_phi", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
    private static final MethodHandle SET_PHI = fn("ldagpu_set_phi", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
    private static final MethodHandle GET_PHI_MEAN = fn("ldagpu_get_phi_mean", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS));
    private static final MethodHandle SET_MEAN_SCHEDULE = fn("ldagpu_set_phi_mean_schedule", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, JAVA_INT));
    private static final MethodHandle GET_THETA = fn("ldagpu_get_theta", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
    private static final MethodHandle LOG_LIKELIHOOD = fn("ldagpu_log_likelihood", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
    private static final MethodHandle LOG_POSTERIOR = fn("ldagpu_log_posterior", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
    private static final MethodHandle ABORT = fn("ldagpu_abort", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    private static final MethodHandle SAMPLE_THETA = fn("ldagpu_sample_theta", FunctionDescriptor.of(JAVA_INT, ADDRESS));
    // hyper-parameter optimisation hooks (ModifiedSimpleLDA.java:812-905, UncollapsedParallelLDA.java:891-894)
    private static final MethodHandle GET_HISTOGRAMS = fn("ldagpu_get_count_histograms", FunctionDescriptor.of(JAVA_INT,
            ADDRESS, JAVA_INT, ADDRESS, JAVA_INT, ADDRESS));
    private static final MethodHandle SET_ALPHA = fn("ldagpu_set_alpha", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
    private static final MethodHandle SET_BETA = fn("ldagpu_set_beta", FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_DOUBLE));
    private static final MethodHandle SET_TEST_DOCS = fn("ldagpu_set_test_documents", FunctionDescriptor.of(JAVA_INT,
            ADDRESS, JAVA_LONG, ADDRESS, ADDRESS, JAVA_LONG, JAVA_LONG));
    private static final MethodHandle HELDOUT_LL = fn("ldagpu_heldout_log_likelihood", FunctionDescriptor.of(JAVA_INT,
            ADDRESS, JAVA_INT, ADDRESS, ADDRESS));

    private final Arena arena = Arena.ofShared();
    private MemorySegment handle = MemorySegment.NULL;
    private final int scheme;             // 0 = gpu_ggs, 1 = gpu_pcgs, 2 = gpu_spalias / gpu_polyaurn (sparse z-step)
    private final boolean polyaUrn;       // gpu_polyaurn: Poisson Polya-urn Phi draw (topics/PolyaUrnSpaliasLDA.java)
    private static final int SWEEPS_PER_CALL = 10;   // abort and exec_time are looked at between library calls
    private long[] docOffsets;
    private int numTokens;
    private int noSampledPhi = 0;

    public GpuLDASampler(LDAConfiguration config, boolean grouped) {
        this(config, grouped ? "gpu_ggs" : "gpu_pcgs");
    }

    /** scheme: gpu_ggs | gpu_pcgs | gpu_spalias | gpu_polyaurn (the new `case` labels of ParallelLDA.createModel) */
    public GpuLDASampler(LDAConfiguration config, String schemeName) {
        super(config);
        switch (schemeName) {
        case "gpu_ggs": scheme = 0; polyaUrn = false; break;
        case "gpu_pcgs": scheme = 1; polyaUrn = false; break;
        case "gpu_spalias": scheme = 2; polyaUrn = false; break;
        case "gpu_polyaurn": scheme = 2; polyaUrn = true; break;
        default: throw new IllegalArgumentException("unknown GPU scheme " + schemeName);
        }
    }

    /** new key `gpu_devices = 0,1,2,3`: shard the corpus over these GPUs from this one JVM (default: gpu_device only) */
    private int[] gpuDevices() {
        String v = config.getStringProperty("gpu_devices");
        if (v == null || v.trim().isEmpty()) return new int[] { config.getIntProperty("gpu_device", 0) };
        String[] parts = v.split("[,;]");
        int[] out = new int[parts.length];
        for (int i = 0; i < parts.length; i++) out[i] = Integer.parseInt(parts[i].trim());
        return out;
    }

    private void ck(int rc) {
        if (rc == 0) return;
        try {
            MemorySegment msg = (MemorySegment) LAST_ERROR.invokeExact(handle);
            // the reference throws IllegalStateException / IllegalArgumentException on invariant breaks
            // (UncollapsedParallelLDA.java:475-481,1496-1497,1529-1531,1828-1830)
            throw new IllegalStateException("libldagpu: " + msg.reinterpret(512).getString(0));
        } catch (RuntimeException e) {
            throw e;
        } catch (Throwable t) {
            throw new IllegalStateException(t);
        }
    }

    /** UncollapsedParallelLDA.java:357-456: flatten the InstanceList to CSR and upload it. */
    @Override
    public void addInstances(InstanceList training) {
        alphabet = training.getDataAlphabet();
        numTypes = alphabet.size();
        int D = training.size();
        docOffsets = new long[D + 1];
        for (int d = 0; d < D; d++)
            docOffsets[d + 1] = docOffsets[d] + ((FeatureSequence) training.get(d).getData()).getLength();
        numTokens = (int) docOffsets[D];
        int[] tokens = new int[numTokens];
        int longestDoc = 0;
        for (int d = 0; d < D; d++) {
            FeatureSequence fs = (FeatureSequence) training.get(d).getData();
            // the backing array may be longer than getLength() (TestInitialization.java:346-349)
            System.arraycopy(fs.getFeatures(), 0, tokens, (int) docOffsets[d], fs.getLength());
            data.add(new TopicAssignment(training.get(d), new LabelSequence(topicAlphabet, new int[fs.getLength()])));
            longestDoc = Math.max(longestDoc, fs.getLength());
        }
        // sufficient statistics of the hyper-parameter optimisation that do not change with z
        // (UncollapsedParallelLDA.java:408-431): histogram of document lengths, largest corpus frequency of a type
        docLengthCounts = new int[longestDoc + 1];
        for (int d = 0; d < D; d++) docLengthCounts[(int) (docOffsets[d + 1] - docOffsets[d])]++;
        int[] typeTotals = new int[numTypes];
        for (int t : tokens) typeTotals[t]++;
        maxTypeCount = 0;
        for (int c : typeTotals) maxTypeCount = Math.max(maxTypeCount, c);
        try {
            MemorySegment out = arena.allocate(ADDRESS);
            int[] devices = gpuDevices();
            // the library shards the documents by token count over the devices and exchanges counts / Phi between
            // them over NVLink peer memory; with one device this is the plain single-GPU handle
            ck((int) CREATE_MULTI.invokeExact(numTopics, numTypes, (long) D,
                    arena.allocateFrom(JAVA_LONG, docOffsets), arena.allocateFrom(JAVA_INT, tokens),
                    arena.allocateFrom(JAVA_DOUBLE, alpha), beta, (long) getStartSeed(), scheme,
                    devices.length, arena.allocateFrom(JAVA_INT, devices), out));
            handle = out.get(ADDRESS, 0);
            if (polyaUrn)   // before the first Phi is drawn (UPL:450 -> PolyaUrnSpaliasLDA.loopOverTopics)
                ck((int) SET_PHI_SAMPLER.invokeExact(handle, 1, config.getAliasPoissonThreshold(LDAConfiguration.ALIAS_POISSON_DEFAULT_THRESHOLD)));
            ck((int) INIT_Z.invokeExact(handle, getStartSeed()));   // Randoms(seed).nextInt(K), UPL:398-406
        } catch (RuntimeException e) {
            throw e;
        } catch (Throwable t) {
            throw new IllegalStateException(t);
        }
        pullZ();
    }

    /** copy z back into each document's LabelSequence: getData(), getZIndicators(), LDAUtils.getDocumentTopicCounts
     *  (util/LDAUtils.java:1552-1571) and ModifiedSimpleLDA.java:464-477,536-547 read it from there. */
    private void pullZ() {
        try (Arena a = Arena.ofConfined()) {
            MemorySegment z = a.allocate(JAVA_INT, Math.max(numTokens, 1));
            ck((int) GET_Z.invokeExact(handle, z));
            for (int d = 0; d < data.size(); d++) {
                int[] dst = ((LabelSequence) data.get(d).topicSequence).getFeatures();
                MemorySegment.copy(z, JAVA_INT, docOffsets[d] * 4, dst, 0, dst.length);
            }
            int[] nk = new int[numTopics];
            MemorySegment nkSeg = a.allocate(JAVA_INT, numTopics);
            ck((int) GET_NK.invokeExact(handle, nkSeg));
            MemorySegment.copy(nkSeg, JAVA_INT, 0, nk, 0, numTopics);
            tokensPerTopic = nk;
        } catch (RuntimeException e) {
            throw e;
        } catch (Throwable t) {
            throw new IllegalStateException(t);
        }
    }

    /** UncollapsedParallelLDA.java:552-943.  Diagnostics (log-posterior / log-likelihood files, Phi / Theta dumps,
     *  UPL:707-853) stay in Java -- written by the reference's LDAUtils -- and read their inputs from the library. */
    @Override
    public void sample(int iterations) throws IOException {
        preSample();
        int interval = config.computeLikelihood() ? Math.max(1, config.getTopicInterval(10)) : iterations;
        if (config.savePhiMeans(false)) {
            int burn = (int) (config.getPhiBurnInPercent(0) / 100.0 * iterations);      // UPL:206-207
            try { ck((int) SET_MEAN_SCHEDULE.invokeExact(handle, burn, config.getPhiMeanThin(1))); }
            catch (RuntimeException e) { throw e; } catch (Throwable t) { throw new IllegalStateException(t); }
        }
        // UPL:555-581: the diagnostic block's settings and output directories
        int startDiagnostic = config.getStartDiagnostic(LDAConfiguration.START_DIAG_DEFAULT);
        int[] printFirstNDocs = config.getPrintNDocsInterval();
        int nDocs = config.getPrintNDocs();
        boolean savePhi = config.getSavePhi();
        String loggingPath = config.getLoggingUtil().getLogDir().getAbsolutePath();
        File asciiOutput = LoggingUtils.checkCreateAndCreateDir(loggingPath + "/ascii");
        // UPL:214,891-894: alpha and beta are re-estimated every hyperparam_optim_interval sweeps (off by default)
        int hyperInterval = config.getHyperparamOptimInterval(LDAConfiguration.HYPERPARAM_OPTIM_INTERVAL_DEFAULT);
        int done = 0;
        // UPL:577,926-928: stop when zSamplingTimeCum + phiSamplingTimeCum reaches exec_time (default 10 s,
        // LDAConfiguration.java:35), counted from the start of THIS call; the abort flag is checked as often (UPL:645)
        double maxExecTimeMillis = config.getMaxExecTimeSeconds(LDAConfiguration.EXEC_TIME_DEFAULT) * 1000.0;
        try (Arena a = Arena.ofConfined()) {
            MemorySegment n = a.allocate(JAVA_INT);
            double t0 = samplingMillis(a);
            while (done < iterations && !abort) {
                int step = Math.min(Math.min(interval, SWEEPS_PER_CALL), iterations - done);
                if (config.computeLikelihood()) step = Math.min(step, interval - done % interval);
                if (hyperInterval > 1) step = Math.min(step, hyperInterval - done % hyperInterval);
                // the diagnostic block runs after EVERY sweep from start_diagnostic on (UPL:706-823): one sweep per call
                // there, and the last call before it must stop right at start_diagnostic - 1
                if (startDiagnostic > 0) step = done + 1 >= startDiagnostic ? 1 : Math.min(step, startDiagnostic - 1 - done);
                preIteration();
                ck((int) SWEEP.invokeExact(handle, step, n));
                done += n.get(JAVA_INT, 0);
                currentIteration = done;
                if (config.computeLikelihood() && done % interval == 0) loglikelihood.add(modelLogLikelihood());
                if (startDiagnostic > 0 && done >= startDiagnostic && n.get(JAVA_INT, 0) > 0)
                    diagnostics(done, printFirstNDocs, nDocs, savePhi, asciiOutput, loggingPath);
                if (hyperInterval > 1 && done % hyperInterval == 0) {
                    pullZ();              // tokensPerTopic for the topic-size histogram
                    optimizeAlpha();
                    optimizeBeta();
                }
                postIteration();
                if (n.get(JAVA_INT, 0) < step) break;
                if (maxExecTimeMillis > 0 && samplingMillis(a) - t0 >= maxExecTimeMillis) break;
            }
        } catch (RuntimeException | IOException e) {
            throw e;
        } catch (Throwable t) {
            throw new IllegalStateException(t);
        }
        pullZ();
        postSample();
    }

    /** The diagnostic block of UPL:706-823, fed from the library: `Theta_DxK_<n>_<K>_<iter>.csv` for the first n
     *  documents when the iteration lies in print_ndocs_interval, `Phi_KxV_<K>_<V>_<iter>.csv` when save_phi is set,
     *  and one line of log-posterior.txt -- written by the reference's own LDAUtils (util/LDAUtils.java:955-968,
     *  1223-1254), so formats are the reference's by construction. */
    private void diagnostics(int iteration, int[] printFirstNDocs, int nDocs, boolean savePhi, File asciiOutput,
                             String loggingPath) throws IOException {
        if (printFirstNDocs.length > 1 && LDAUtils.inRangeInterval(iteration, printFirstNDocs)) {
            // GGS: the sweep's own theta (UPL:716-720); the other schemes: theta ~ Dir(n_d + alpha) from the current z
            // (UPL:710-714) -- the draw is keyed by (sweep, document, topic), so computeLogPosterior() below sees the same one
            double[][] theta = diagnosticTheta();
            double[][] head = java.util.Arrays.copyOf(theta, Math.min(nDocs, theta.length));
            LDAUtils.writeASCIIDoubleMatrix(head, String.format(asciiOutput.getAbsolutePath() + "/Theta_DxK_" + nDocs + "_"
                    + numTopics + "_%05d.csv", iteration), ",");
        }
        if (savePhi)
            LDAUtils.writeASCIIDoubleMatrix(getPhi(), String.format(asciiOutput.getAbsolutePath() + "/Phi_KxV_" + numTopics
                    + "_" + numTypes + "_%05d.csv", iteration), ",");
        LDAUtils.logPosteriorToFile(computeLogPosterior(), iteration, loggingPath, LOG);
    }

    /** double[D][K]: GGS thetaMatrix of the last sweep, or the diagnostic theta of the other schemes */
    public double[][] diagnosticTheta() {
        int D = data.size();
        double[][] out = new double[D][numTopics];
        try (Arena a = Arena.ofConfined()) {
            if (scheme != 0) ck((int) SAMPLE_THETA.invokeExact(handle));
            MemorySegment m = a.allocate(JAVA_DOUBLE, (long) D * numTopics);
            ck((int) GET_THETA.invokeExact(handle, m));
            for (int d = 0; d < D; d++) MemorySegment.copy(m, JAVA_DOUBLE, (long) d * numTopics * 8, out[d], 0, numTopics);
        } catch (RuntimeException e) { throw e; } catch (Throwable t) { throw new IllegalStateException(t); }
        return out;
    }

    /** z + count merge + Phi + exchange time so far, in ms (the reference's zSamplingTimeCum + phiSamplingTimeCum) */
    private double samplingMillis(Arena a) throws Throwable {
        MemorySegment t = a.allocate(JAVA_DOUBLE, 4);
        ck((int) GET_TIMERS.invokeExact(handle, t.asSlice(0, 8), t.asSlice(8, 8), t.asSlice(16, 8), t.asSlice(24, 8)));
        return t.getAtIndex(JAVA_DOUBLE, 0) + t.getAtIndex(JAVA_DOUBLE, 1) + t.getAtIndex(JAVA_DOUBLE, 2) + t.getAtIndex(JAVA_DOUBLE, 3);
    }

    @Override
    public void sampleZGivenPhi(int iterations) {
        try (Arena a = Arena.ofConfined()) {
            ck((int) Z_GIVEN_PHI.invokeExact(handle, iterations, a.allocate(JAVA_INT)));
        } catch (RuntimeException e) { throw e; } catch (Throwable t) { throw new IllegalStateException(t); }
        pullZ();
    }

    @Override
    public void setZIndicators(int[][] zIndicators) {
        int[] flat = new int[numTokens];
        int sum = 0;
        for (int d = 0; d < zIndicators.length; d++) {
            System.arraycopy(zIndicators[d], 0, flat, (int) docOffsets[d], zIndicators[d].length);
            sum += zIndicators[d].length;
        }
        if (sum != numTokens)   // UPL:1828-1830
            throw new IllegalArgumentException("Count does not sum to nr. types! Sumtotal: " + sum + " no.types: " + numTokens);
        try (Arena a = Arena.ofConfined()) {
            ck((int) SET_Z.invokeExact(handle, a.allocateFrom(JAVA_INT, flat), 1));
        } catch (RuntimeException e) { throw e; } catch (Throwable t) { throw new IllegalStateException(t); }
        pullZ();
    }

    @Override
    public int[][] getTypeTopicMatrix() {
        int[][] out = new int[numTypes][numTopics];
        try (Arena a = Arena.ofConfined()) {
            MemorySegment m = a.allocate(JAVA_INT, (long) numTypes * numTopics);
            ck((int) GET_NWK.invokeExact(handle, m));
            for (int w = 0; w < numTypes; w++) MemorySegment.copy(m, JAVA_INT, (long) w * numTopics * 4, out[w], 0, numTopics);
        } catch (RuntimeException e) { throw e; } catch (Throwable t) { throw new IllegalStateException(t); }
        return out;
    }

    public int[][] getTypeTopicCounts() { return getTypeTopicMatrix(); }   // UPL:226-234

    @Override
    public double[][] getPhi() {
        double[][] out = new double[numTopics][numTypes];
        try (Arena a = Arena.ofConfined()) {
            MemorySegment m = a.allocate(JAVA_DOUBLE, (long) numTopics * numTypes);
            ck((int) GET_PHI.invokeExact(handle, m));
            for (int k = 0; k < numTopics; k++) MemorySegment.copy(m, JAVA_DOUBLE, (long) k * numTypes * 8, out[k], 0, numTypes);
        } catch (RuntimeException e) { throw e; } catch (Throwable t) { throw new IllegalStateException(t); }
        return out;
    }

    @Override
    public void setPhi(double[][] phi, Alphabet dataAlphabet, Alphabet targetAlphabet) {
        if (!dataAlphabet.equals(getAlphabet())) throw new IllegalArgumentException("Vocabularies does not match!");   // UPL:1913-1915
        try (Arena a = Arena.ofConfined()) {
            MemorySegment m = a.allocate(JAVA_DOUBLE, (long) numTopics * numTypes);
            for (int k = 0; k < numTopics; k++) MemorySegment.copy(phi[k], 0, m, JAVA_DOUBLE, (long) k * numTypes * 8, numTypes);
            ck((int) SET_PHI.invokeExact(handle, m));
        } catch (RuntimeException e) { throw e; } catch (Throwable t) { throw new IllegalStateException(t); }
    }

    @Override
    public double[][] getPhiMeans() {
        double[][] out = new double[numTopics][numTypes];
        try (Arena a = Arena.ofConfined()) {
            MemorySegment m = a.allocate(JAVA_DOUBLE, (long) numTopics * numTypes);
            MemorySegment n = a.allocate(JAVA_INT);
            ck((int) GET_PHI_MEAN.invokeExact(handle, m, n));
            noSampledPhi = n.get(JAVA_INT, 0);
            if (noSampledPhi == 0) return null;                      // UPL:1955-1958
            for (int k = 0; k < numTopics; k++) MemorySegment.copy(m, JAVA_DOUBLE, (long) k * numTypes * 8, out[k], 0, numTypes);
        } catch (RuntimeException e) { throw e; } catch (Throwable t) { throw new IllegalStateException(t); }
        return out;
    }

    /** LDAGibbsSampler.addTestInstances: the test set (type ids of the training alphabet) goes to the library once and
     *  stays resident; the library shards it over the GPUs of this handle.  K <= 1024 only. */
    @Override
    public void addTestInstances(InstanceList testSet) {
        int D = testSet.size();
        long[] off = new long[D + 1];
        for (int d = 0; d < D; d++) off[d + 1] = off[d] + ((FeatureSequence) testSet.get(d).getData()).getLength();
        int[] tokens = new int[(int) off[D]];
        for (int d = 0; d < D; d++) {
            FeatureSequence fs = (FeatureSequence) testSet.get(d).getData();
            System.arraycopy(fs.getFeatures(), 0, tokens, (int) off[d], fs.getLength());
        }
        try (Arena a = Arena.ofConfined()) {
            ck((int) SET_TEST_DOCS.invokeExact(handle, (long) D, a.allocateFrom(JAVA_LONG, off),
                    a.allocateFrom(JAVA_INT, tokens), 0L, 0L));
        } catch (RuntimeException e) { throw e; } catch (Throwable t) { throw new IllegalStateException(t); }
    }

    /** MarginalProbEstimatorPlain.evaluateLeftToRight (UPL:604-611,840-844): MALLET's left-to-right estimator without
     *  resampling on the current counts, nParticles particles (MALLET's default 10) */
    public double heldOutLogLikelihood(int nParticles) {
        try (Arena a = Arena.ofConfined()) {
            MemorySegment v = a.allocate(JAVA_DOUBLE);
            ck((int) HELDOUT_LL.invokeExact(handle, nParticles, MemorySegment.NULL, v));
            return v.get(JAVA_DOUBLE, 0);
        } catch (RuntimeException e) { throw e; } catch (Throwable t) { throw new IllegalStateException(t); }
    }

    @Override
    public double modelLogLikelihood() {
        try (Arena a = Arena.ofConfined()) {
            MemorySegment v = a.allocate(JAVA_DOUBLE);
            ck((int) LOG_LIKELIHOOD.invokeExact(handle, v));
            return v.get(JAVA_DOUBLE, 0);
        } catch (RuntimeException e) { throw e; } catch (Throwable t) { throw new IllegalStateException(t); }
    }

    /** replaces the `whichModel.equals("ggs")` test of UPL:710: the GPU sampler owns its diagnostic theta */
    public double computeLogPosterior() {
        try (Arena a = Arena.ofConfined()) {
            // PCGS / sparse PCGS: diagnostic theta ~ Dir(n_d + alpha) from the current z first (UPL:710-714,
            // util/LDAUtils.java:1662-1673); GGS keeps the sweep's own theta (UPL:716-720)
            if (scheme != 0) ck((int) SAMPLE_THETA.invokeExact(handle));
            MemorySegment v = a.allocate(JAVA_DOUBLE);
            ck((int) LOG_POSTERIOR.invokeExact(handle, v));
            return v.get(JAVA_DOUBLE, 0);
        } catch (RuntimeException e) { throw e; } catch (Throwable t) { throw new IllegalStateException(t); }
    }

    /** ModifiedSimpleLDA.java:812-858, symmetric alpha (the GPU path keeps alpha symmetric).  The reference fills
     *  documentTopicHistogram inside its z-step (UPL:1382-1401); here the library counts the (document, topic)
     *  pairs with n_dk = c from the current z, and MALLET's fixed point runs on the host as before. */
    @Override
    public void optimizeAlpha() {
        int bins = docLengthCounts.length;
        try (Arena a = Arena.ofConfined()) {
            MemorySegment dh = a.allocate(JAVA_LONG, bins);
            ck((int) GET_HISTOGRAMS.invokeExact(handle, bins, dh, 0, MemorySegment.NULL));
            int[] hist = new int[bins];
            for (int c = 0; c < bins; c++) hist[c] = (int) dh.getAtIndex(JAVA_LONG, c);
            alphaSum = Dirichlet.learnSymmetricConcentration(hist, docLengthCounts, numTopics, alphaSum);
            java.util.Arrays.fill(alpha, alphaSum / numTopics);
            ck((int) SET_ALPHA.invokeExact(handle, a.allocateFrom(JAVA_DOUBLE, alpha)));
        } catch (RuntimeException e) { throw e; } catch (Throwable t) { throw new IllegalStateException(t); }
    }

    /** ModifiedSimpleLDA.java:860-905: the histogram of n_wk comes from the library, the topic sizes from tokensPerTopic */
    @Override
    public void optimizeBeta() {
        int bins = maxTypeCount + 1;
        try (Arena a = Arena.ofConfined()) {
            MemorySegment th = a.allocate(JAVA_LONG, bins);
            ck((int) GET_HISTOGRAMS.invokeExact(handle, 0, MemorySegment.NULL, bins, th));
            int[] countHistogram = new int[bins];
            for (int c = 0; c < bins; c++) countHistogram[c] = (int) Math.min(th.getAtIndex(JAVA_LONG, c), Integer.MAX_VALUE);
            int maxTopicSize = 0;
            for (int k = 0; k < numTopics; k++) maxTopicSize = Math.max(maxTopicSize, tokensPerTopic[k]);
            int[] topicSizeHistogram = new int[maxTopicSize + 1];
            for (int k = 0; k < numTopics; k++) topicSizeHistogram[tokensPerTopic[k]]++;
            betaSum = Dirichlet.learnSymmetricConcentration(countHistogram, topicSizeHistogram, numTypes, betaSum);
            beta = betaSum / numTypes;
            ck((int) SET_BETA.invokeExact(handle, beta));
        } catch (RuntimeException e) { throw e; } catch (Throwable t) { throw new IllegalStateException(t); }
    }

    @Override
    public void abort() {   // may arrive from the shutdown-hook thread (tui/ParallelLDA.java:82-101)
        super.abort();
        try { int rc = (int) ABORT.invokeExact(handle); } catch (Throwable t) { /* best effort */ }
    }

    @Override public void prePhi() { }
    @Override public void postPhi() { }

    public void close() {
        try { if (!handle.equals(MemorySegment.NULL)) { int rc = (int) DESTROY.invokeExact(handle); } }
        catch (Throwable t) { /* ignore */ }
        handle = MemorySegment.NULL;
        arena.close();
    }
}
