/*
 * GpuAlignerExtension.cpp -- the reference-side binding of libsnapgpu: an AlignerExtension (reference
 * SNAPLib/AlignerContext.h:145-180) whose runIterationThread() overloads take over a SNAP worker thread's share of the
 * input (call sites SingleAligner.cpp:102, PairedAligner.cpp:503) and run it through the C ABI of include/snapgpu.h, plus the
 * main() of `snap-aligner-gpu`, which is stock SNAP with this extension installed (SingleAlignerContext(AlignerExtension *),
 * SingleAligner.cpp:43; PairedAlignerContext(AlignerExtension *), PairedAligner.cpp:366).
 *
 * This file is the ONLY code that touches SNAP types; below it everything is plain C (pointers, sizes, POD structs).  It is
 * compiled against the reference headers where they lie and linked with the UNMODIFIED SNAPLib objects and -lsnapgpu by
 * oracle/Makefile.  Must compile as C++98 like the reference.
 *
 * Threading contract (the reference: one BaseAligner per worker thread, "NOT thread safe", BaseAligner.h:19-20).  A GPU aligner
 * handle owns tens of GB of per-warp arenas, so it is NOT per SNAP thread: there is ONE engine (index image + one single-end
 * or paired-end handle) PER CUDA DEVICE, shared by the worker threads mapped to that device (thread t -> device t mod D).
 * A worker thread collects a batch of its supplier's reads (copies: a Read is only valid until the next getNextRead(),
 * Read.h:176), takes the device's lock, aligns the batch, releases the lock and then writes / counts the results itself -- so
 * with -t N the N threads parse FASTQ and format SAM concurrently while the devices align, and `-t 8` on an 8-GPU box is one
 * feeder thread per GPU.  Results do not depend on the batching or on N (each read is aligned independently).
 *
 * What the stock loop does per read and this file does per batch, in the same order:
 *   single: SingleAligner.cpp:197-338 (pre-filter :213, AlignRead :250, passFilter + writeReads :296-322, updateStats :354-374)
 *   paired: PairedAligner.cpp:654-927 (id check :664, useful0/1 :676-678, align :727, forceSpacing :822, passFilter :832-850,
 *           writePairs :870, updateStats :962-1010)
 * Not supported (fails loudly, never falls back to the CPU aligner): secondary alignments (-om) of `paired`, 64-bit indexes, -ins.
 */
#include "stdafx.h"
#include "Compat.h"
#include "BigAlloc.h"
#include "Genome.h"
#include "GenomeIndex.h"
#include "Read.h"
#include "AlignerContext.h"
#include "AlignerOptions.h"
#include "AlignerStats.h"
#include "SingleAligner.h"
#include "PairedAligner.h"
#include "AlignmentResult.h"
#include "SeedSequencer.h"
#include "exit.h"
#include "Error.h"

#include <pthread.h>
#include <string.h>
#include <stdio.h>
#include <stdlib.h>
#include <new>
#include <vector>

#include "../include/snapgpu.h"

// ------------------------------------------------------------------------------------------------------------------------------
// One engine per CUDA device, shared by the SNAP worker threads mapped to it.
// ------------------------------------------------------------------------------------------------------------------------------
struct GpuEngine {
    int              device;
    snapgpu_index   *index;
    snapgpu_aligner *aligner;        // single-end or paired-end handle, created by the first thread that needs it
    pthread_mutex_t  lock;           // a handle is not thread safe (like BaseAligner): one batch at a time per device
};

struct GpuShared {
    pthread_mutex_t  lock;
    snapgpu_group   *group;          // NCCL communicators over the devices (index broadcast, statistics all-reduce)
    snapgpu_counters *counters;      // [nDevices] work counters of each device's batches
    int              nDevices;
    GpuEngine       *engines;
    int              nextThread;     // worker threads are numbered in the order they arrive
    bool             opened;
    _int64           batchReads;     // reads per batch and per call into the engine
    int              refs;
};

static void gpuFatal(const char *what)
{
    WriteErrorMessage("snap-aligner-gpu: %s: %s\n", what, snapgpu_last_error());
    soft_exit(1);
}

// snapgpu_single_result -> SingleAlignmentResult, field for field (AlignmentResult.h:49-77).
static void toSnap(const snapgpu_single_result &g, SingleAlignmentResult *s)
{
    s->status = (AlignmentResult)g.status;
    s->location = GenomeLocation(g.location);
    s->origLocation = GenomeLocation(g.origLocation);
    s->direction = (Direction)g.direction;
    s->score = g.score;
    s->scorePriorToClipping = g.scorePriorToClipping;
    s->mapq = g.mapq;
    s->clippingForReadAdjustment = g.clippingForReadAdjustment;
    s->usedAffineGapScoring = g.usedAffineGapScoring != 0;
    s->basesClippedBefore = g.basesClippedBefore;
    s->basesClippedAfter = g.basesClippedAfter;
    s->agScore = g.agScore;
    s->supplementary = g.supplementary != 0;
    s->seedOffset = g.seedOffset;
    s->matchProbability = g.matchProbability;
    s->probabilityAllCandidates = g.probabilityAllCandidates;
    s->popularSeedsSkipped = g.popularSeedsSkipped;
    s->alignmentTimeInNanoseconds = 0;
    if (s->status == NotFound) {
        s->location = InvalidGenomeLocation;
    }
}

// snapgpu_paired_result -> PairedAlignmentResult (AlignmentResult.h:86-129).
static void toSnap(const snapgpu_paired_result &g, PairedAlignmentResult *s)
{
    for (int r = 0; r < NUM_READS_PER_PAIR; r++) {
        s->status[r] = (AlignmentResult)g.status[r];
        s->location[r] = GenomeLocation(g.location[r]);
        s->origLocation[r] = GenomeLocation(g.origLocation[r]);
        s->direction[r] = (Direction)g.direction[r];
        s->score[r] = g.score[r];
        s->scorePriorToClipping[r] = g.scorePriorToClipping[r];
        s->mapq[r] = g.mapq[r];
        s->clippingForReadAdjustment[r] = g.clippingForReadAdjustment[r];
        s->usedAffineGapScoring[r] = g.usedAffineGapScoring[r] != 0;
        s->basesClippedBefore[r] = g.basesClippedBefore[r];
        s->basesClippedAfter[r] = g.basesClippedAfter[r];
        s->agScore[r] = g.agScore[r];
        s->supplementary[r] = g.supplementary[r] != 0;
        s->seedOffset[r] = g.seedOffset[r];
        s->lvIndels[r] = g.lvIndels[r];
        s->matchProbability[r] = g.matchProbability[r];
        s->popularSeedsSkipped[r] = g.popularSeedsSkipped[r];
        s->usedGaplessClipping[r] = g.usedGaplessClipping[r] != 0;
        s->refSpan[r] = g.refSpan[r];
        s->liftover[r] = g.liftover[r] != 0;
        if (s->status[r] == NotFound) {
            s->location[r] = InvalidGenomeLocation;
        }
    }
    s->probabilityAllPairs = g.probabilityAllPairs;
    s->alignedAsPair = g.alignedAsPair != 0;
    s->agForcedSingleAlignerCall = g.agForcedSingleAlignerCall != 0;
    s->nanosInAlignTogether = 0;
    s->alignmentTimeInNanoseconds = 0;
    s->nLVCalls = 0;
    s->nSmallHits = 0;
}

// The AlignerContext / AlignerOptions fields the hot path reads (AlignerContext.h:102-131) -> snapgpu_params.
static void paramsFromContext(AlignerContext *c, bool paired, snapgpu_params *p)
{
    snapgpu_params_default(p);
    p->maxHits = (uint32_t)c->maxHits;
    p->maxDist = c->maxDist;
    p->numSeedsFromCommandLine = c->numSeedsFromCommandLine;
    p->seedCoverage = c->seedCoverage;
    p->minWeightToCheck = c->minWeightToCheck;
    p->extraSearchDepth = c->extraSearchDepth;
    p->minReadLength = c->minReadLength;
    p->useAffineGap = c->useAffineGap ? 1 : 0;
    p->matchReward = (int32_t)c->matchReward;
    p->subPenalty = (int32_t)c->subPenalty;
    p->gapOpenPenalty = (int32_t)c->gapOpenPenalty;
    p->gapExtendPenalty = (int32_t)c->gapExtendPenalty;
    p->fivePrimeEndBonus = (int32_t)c->fivePrimeEndBonus;
    p->threePrimeEndBonus = (int32_t)c->threePrimeEndBonus;
    p->noUkkonen = c->disabledOptimizations.noUkkonen ? 1 : 0;
    p->noOrderedEvaluation = c->disabledOptimizations.noOrderedEvaluation ? 1 : 0;
    p->noTruncation = c->disabledOptimizations.noTruncation ? 1 : 0;
    p->noEditDistance = c->disabledOptimizations.noEditDistance ? 1 : 0;
    p->noBandedAffineGap = c->disabledOptimizations.noBandedAffineGap ? 1 : 0;
    p->altAwareness = c->altAwareness ? 1 : 0;
    p->maxScoreGapToPreferNonAltAlignment = c->maxScoreGapToPreferNonALTAlignment;
    p->explorePopularSeeds = c->options->explorePopularSeeds ? 1 : 0;
    p->stopOnFirstHit = c->options->stopOnFirstHit ? 1 : 0;
    p->maxSecondaryAlignmentAdditionalEditDistance = c->maxSecondaryAlignmentAdditionalEditDistance;
    p->ignoreAlignmentAdjustmentsForOm = c->ignoreAlignmentAdjustmentForOm ? 1 : 0;
    (void)paired;
}

// The per-thread batch: copies of the supplier's reads (ReadWithOwnMemory, Read.h:862-980 -- the reference's own class for
// keeping a Read past its supplier's lifetime) and the concatenated clipped views the C ABI takes.
struct ReadBatchCopy {
    _int64              capacity, n;
    ReadWithOwnMemory  *reads;       // raw storage, constructed in place
    char               *bases, *quals;
    uint64_t           *offsets;
    uint32_t           *lens;
    size_t              used, basesCapacity;

    void init(_int64 cap)
    {
        capacity = cap; n = 0; used = 0;
        reads = (ReadWithOwnMemory *)BigAlloc((size_t)cap * sizeof(ReadWithOwnMemory));
        basesCapacity = (size_t)cap * 400;
        bases = (char *)snapgpu_host_alloc(basesCapacity);
        quals = (char *)snapgpu_host_alloc(basesCapacity);
        offsets = (uint64_t *)snapgpu_host_alloc((size_t)cap * sizeof(uint64_t));
        lens = (uint32_t *)snapgpu_host_alloc((size_t)cap * sizeof(uint32_t));
        if (!reads || !bases || !quals || !offsets || !lens) gpuFatal("allocating the read batch");
    }
    bool full(unsigned nextLen) const { return n >= capacity || used + nextLen > basesCapacity; }
    Read *add(const Read *r)
    {
        ReadWithOwnMemory *copy = new (&reads[n]) ReadWithOwnMemory(*r);
        const unsigned len = copy->getDataLength();
        memcpy(bases + used, copy->getData(), len);
        memcpy(quals + used, copy->getQuality(), len);
        offsets[n] = used; lens[n] = len;
        used += len;
        n++;
        return copy;
    }
    void clear()
    {
        for (_int64 i = 0; i < n; i++) reads[i].dispose();
        n = 0; used = 0;
    }
    void destroy()
    {
        clear();
        BigDealloc(reads);
        snapgpu_host_free(bases); snapgpu_host_free(quals); snapgpu_host_free(offsets); snapgpu_host_free(lens);
    }
};

class GpuAlignerExtension : public AlignerExtension
{
public:
    GpuAlignerExtension() : shared(new GpuShared), threadNo(-1)
    {
        pthread_mutex_init(&shared->lock, NULL);
        shared->nDevices = 0; shared->engines = NULL; shared->nextThread = 0; shared->opened = false; shared->refs = 1;
        shared->group = NULL; shared->counters = NULL;
        shared->batchReads = 65536;
        if (const char *e = getenv("SNAPGPU_EXT_BATCH_READS")) { if (atoll(e) >= 2) shared->batchReads = atoll(e) / 2 * 2; }
    }
    GpuAlignerExtension(GpuShared *s) : shared(s), threadNo(-1)
    {
        pthread_mutex_lock(&shared->lock); shared->refs++; pthread_mutex_unlock(&shared->lock);
    }
    virtual ~GpuAlignerExtension()
    {
        pthread_mutex_lock(&shared->lock);
        const int left = --shared->refs;
        pthread_mutex_unlock(&shared->lock);
        if (left == 0) {
            for (int d = 0; d < shared->nDevices; d++) {
                if (shared->engines[d].aligner) snapgpu_aligner_destroy(shared->engines[d].aligner);
                if (shared->engines[d].index) snapgpu_index_close(shared->engines[d].index);
                pthread_mutex_destroy(&shared->engines[d].lock);
            }
            delete[] shared->engines;
            delete[] shared->counters;
            if (shared->group) snapgpu_group_destroy(shared->group);
            pthread_mutex_destroy(&shared->lock);
            delete shared;
        }
    }

    // AlignerContext::initializeThread (AlignerContext.cpp:226): one copy per worker thread, all sharing the engines
    virtual AlignerExtension *copy() { return new GpuAlignerExtension(shared); }

    virtual bool runIterationThread(ReadSupplier *supplier, AlignerContext *context);
    virtual bool runIterationThread(PairedReadSupplier *supplier, AlignerContext *context);

    // AlignerContext::printStats (AlignerContext.cpp:670): the engine's own work counters, summed over the devices with ncclAllReduce
    virtual void printStats()
    {
        if (!shared->opened) return;
        if (shared->group != NULL && snapgpu_counters_allreduce(shared->group, shared->counters)) gpuFatal("reducing the counters");
        const snapgpu_counters &c = shared->counters[0];
        WriteStatusMessage("snap-aligner-gpu: %d device%s: %lld hash lookups (%.1f slots examined each), %lld locations scored with Landau-Vishkin, %lld with affine gap\n",
                           shared->nDevices, shared->nDevices == 1 ? "" : "s", (long long)c.nHashTableLookups,
                           c.nHashTableLookups ? (double)c.nHashEntriesProbed / (double)c.nHashTableLookups : 0.0, (long long)c.lvCalls, (long long)c.affineGapCalls);
    }

private:
    GpuShared *shared;
    int        threadNo;

    void addCounters(GpuEngine *engine, const snapgpu_counters &c)
    {
        pthread_mutex_lock(&shared->lock);
        _int64 *dst = (_int64 *)&shared->counters[engine->device];
        const _int64 *src = (const _int64 *)&c;
        for (size_t k = 0; k < sizeof(snapgpu_counters) / sizeof(_int64); k++) dst[k] += src[k];
        pthread_mutex_unlock(&shared->lock);
    }

    // Opens the index image on every device on first use (AlignerExtension::initialize() gets no context, so this is where the
    // index directory is first known) and creates this thread's device's aligner handle.  Returns the thread's engine.
    GpuEngine *engineForThisThread(AlignerContext *context, bool paired);
};

GpuEngine *GpuAlignerExtension::engineForThisThread(AlignerContext *context, bool paired)
{
    pthread_mutex_lock(&shared->lock);
    if (!shared->opened) {
        if (context->maxSecondaryAlignmentAdditionalEditDistance >= 0 && paired) {
            WriteErrorMessage("snap-aligner-gpu: secondary alignments (-om) are supported for `single` only\n");
            soft_exit(1);
        }
        if (context->index == NULL || context->index->doesGenomeIndexHave64BitLocations()) {
            WriteErrorMessage("snap-aligner-gpu: needs an index with 4-byte genome locations (the lookupSeed32 path)\n");
            soft_exit(1);
        }
        int nDev = snapgpu_device_count();
        if (nDev < 1) gpuFatal("no CUDA device");
        if (const char *e = getenv("SNAPGPU_EXT_DEVICES")) { if (atoi(e) >= 1 && atoi(e) < nDev) nDev = atoi(e); }
        if (nDev > (int)context->options->numThreads) nDev = (int)context->options->numThreads;       // a device needs a thread to feed it
        shared->engines = new GpuEngine[nDev];
        for (int d = 0; d < nDev; d++) {
            shared->engines[d].device = d; shared->engines[d].index = NULL; shared->engines[d].aligner = NULL;
            pthread_mutex_init(&shared->engines[d].lock, NULL);
        }
        // one upload from the index directory, then ncclBroadcast to the other devices over NVLink / NVSwitch (SURVEY 8e)
        if (snapgpu_index_open(context->options->indexDir, 0, &shared->engines[0].index)) gpuFatal("loading the index onto device 0");
        shared->counters = new snapgpu_counters[nDev];
        memset(shared->counters, 0, sizeof(snapgpu_counters) * nDev);
        if (nDev > 1) {
            int *devs = new int[nDev];
            snapgpu_index **copies = new snapgpu_index *[nDev];
            for (int d = 0; d < nDev; d++) devs[d] = d;
            if (snapgpu_group_create(devs, nDev, &shared->group)) gpuFatal("creating the device group (NCCL)");
            if (snapgpu_index_broadcast(shared->group, shared->engines[0].index, copies)) gpuFatal("broadcasting the index");
            for (int d = 1; d < nDev; d++) shared->engines[d].index = copies[d];
            delete[] devs; delete[] copies;
        }
        shared->nDevices = nDev;
        shared->opened = true;
        WriteStatusMessage("snap-aligner-gpu: index resident on %d CUDA device%s; %d worker thread%s feed%s them in batches of %lld reads\n", nDev,
                           nDev == 1 ? "" : "s", (int)context->options->numThreads, context->options->numThreads == 1 ? "" : "s",
                           context->options->numThreads == 1 ? "s" : "", (long long)shared->batchReads);
    }
    if (threadNo < 0) threadNo = shared->nextThread++;
    GpuEngine *e = &shared->engines[threadNo % shared->nDevices];
    pthread_mutex_unlock(&shared->lock);

    pthread_mutex_lock(&e->lock);
    if (e->aligner == NULL) {
        snapgpu_params p;
        paramsFromContext(context, paired, &p);
        if (!paired) {
            if (snapgpu_aligner_create(e->index, &p, shared->batchReads, &e->aligner)) gpuFatal("creating the single-end aligner");
        } else {
            PairedAlignerOptions *po = (PairedAlignerOptions *)context->options;
            snapgpu_paired_params pp;
            snapgpu_paired_params_default(&pp);
            pp.minSpacing = po->minSpacing; pp.maxSpacing = (uint32_t)po->maxSpacing;
            pp.intersectingAlignerMaxHits = po->intersectingAlignerMaxHits; pp.maxCandidatePoolSize = po->maxCandidatePoolSize;
            pp.maxSeedsSingleEnd = (uint32_t)po->maxSeedsSingleEnd; pp.maxDistForIndels = context->maxDistForIndels;
            pp.forceSpacing = po->forceSpacing ? 1 : 0;
            pp.minScoreRealignment = po->minScoreRealignment; pp.minScoreGapRealignmentALT = po->minScoreGapRealignmentALT;
            pp.minAGScoreImprovement = context->options->useSoftClipping ? po->minAGScoreImprovement : 15;       // PairedAligner.cpp:388
            pp.enableHammingScoringBaseAligner = po->enableHammingScoringBaseAligner ? 1 : 0;
            pp.useSoftClipping = context->options->useSoftClipping ? 1 : 0;
            pp.flattenMAPQAtOrBelow = context->options->flattenMAPQAtOrBelow;
            if (po->inferSpacing) {
                WriteErrorMessage("snap-aligner-gpu: -ins (insert size inference makes results depend on the thread partition) is not supported\n");
                soft_exit(1);
            }
            if (snapgpu_paired_aligner_create(e->index, &p, &pp, shared->batchReads / 2, &e->aligner)) gpuFatal("creating the paired-end aligner");
        }
    }
    pthread_mutex_unlock(&e->lock);
    return e;
}

// SingleAlignerContext::updateStats (SingleAligner.cpp:354-374; a protected member there)
static void updateSingleStats(AlignerStats *stats, AlignmentResult result, int mapq)
{
    if (isOneLocation(result)) {
        stats->singleHits++;
    } else if (result == MultipleHits) {
        stats->multiHits++;
    } else {
        stats->notFound++;
    }
    if (result != NotFound && mapq >= 0 && mapq <= (int)AlignerStats::maxMapq) {
        stats->mapqHistogram[mapq]++;
    }
}

bool GpuAlignerExtension::runIterationThread(ReadSupplier *supplier, AlignerContext *context)
{
    GpuEngine *engine = engineForThisThread(context, false);
    AlignerStats *stats = context->stats;
    AlignerOptions *options = context->options;
    ReadWriter *readWriter = context->readWriter;
    ReadBatchCopy batch;
    batch.init(shared->batchReads);
    snapgpu_single_result *results = (snapgpu_single_result *)snapgpu_host_alloc((size_t)shared->batchReads * sizeof(snapgpu_single_result));
    if (!results) gpuFatal("allocating the result batch");
    snapgpu_counters counters;
    memset(&counters, 0, sizeof(counters));
    const bool om = context->maxSecondaryAlignmentAdditionalEditDistance >= 0;
    _int64 secCap = 31;              // SingleAligner.cpp:141: a buffer of 32 results, the first being the primary
    snapgpu_single_result *secondary = NULL;
    int32_t *nSecondary = NULL;
    std::vector<SingleAlignmentResult> alignmentResults(1);
    if (om) {
        secondary = (snapgpu_single_result *)snapgpu_host_alloc((size_t)shared->batchReads * (size_t)secCap * sizeof(snapgpu_single_result));
        nSecondary = (int32_t *)snapgpu_host_alloc((size_t)shared->batchReads * sizeof(int32_t));
        if (!secondary || !nSecondary) gpuFatal("allocating the secondary-result batch");
    }

    Read *read = supplier->getNextRead();
    while (read != NULL) {
        // fill a batch with copies of this thread's next reads
        while (read != NULL && !batch.full(read->getDataLength())) {
            batch.add(read);
            read = supplier->getNextRead();
        }
        pthread_mutex_lock(&engine->lock);
        int rc;
        if (om) {
            // -om: the primary results plus, per read, up to secCap secondary ones; a read with more reports minus its count and the
            // batch is aligned again with room for it (SingleAligner.cpp:250-263 doubles its buffer per read)
            for (;;) {
                snapgpu_counters c;
                memset(&c, 0, sizeof(c));
                rc = snapgpu_align_single_secondary(engine->aligner, batch.n, batch.bases, batch.quals, batch.offsets, batch.lens, results,
                                                    context->maxSecondaryAlignments, context->maxSecondaryAlignmentsPerContig, secCap, secondary, nSecondary, &c);
                if (rc) break;
                _int64 need = 0;
                for (_int64 i = 0; i < batch.n; i++) if (-(_int64)nSecondary[i] > need) need = -(_int64)nSecondary[i];
                if (need == 0) {
                    _int64 *dst = (_int64 *)&counters; const _int64 *src = (const _int64 *)&c;
                    for (size_t k = 0; k < sizeof(c) / sizeof(_int64); k++) dst[k] += src[k];
                    break;
                }
                while (secCap < need) secCap *= 2;
                snapgpu_host_free(secondary);
                secondary = (snapgpu_single_result *)snapgpu_host_alloc((size_t)shared->batchReads * (size_t)secCap * sizeof(snapgpu_single_result));
                if (!secondary) gpuFatal("allocating the secondary-result batch");
            }
        } else {
            rc = snapgpu_align_single(engine->aligner, batch.n, batch.bases, batch.quals, batch.offsets, batch.lens, results, &counters);
        }
        pthread_mutex_unlock(&engine->lock);
        if (rc) gpuFatal(om ? "snapgpu_align_single_secondary" : "snapgpu_align_single");

        for (_int64 i = 0; i < batch.n; i++) {
            Read *r = &batch.reads[i];
            stats->totalReads++;
            SingleAlignmentResult result;
            memset(&result, 0, sizeof(result));
            if (r->getDataLength() < context->minReadLength || r->countOfNs() > (int)context->maxDist) {
                // SingleAligner.cpp:213-233 (the engine applied the same pre-filter and reported NotFound)
                if (!options->passFilter(r, NotFound, true, false)) {
                    stats->filtered++;
                } else {
                    if (NULL != readWriter) {
                        result.status = NotFound; result.location = InvalidGenomeLocation; result.mapq = 0; result.direction = FORWARD;
                        result.clippingForReadAdjustment = 0; result.usedAffineGapScoring = false; result.basesClippedBefore = 0;
                        result.basesClippedAfter = 0; result.supplementary = false;
                        readWriter->writeReads(context->readerContext, r, &result, 1, true, context->useAffineGap);
                    }
                    stats->uselessReads++;
                }
                continue;
            }
            toSnap(results[i], &result);
            bool containsPrimary = true;
            if (om) {
                // SingleAligner.cpp:292-322: every result through the filter (the last one moves into a hole), then one writeReads call
                _int64 nSec = nSecondary[i];
                alignmentResults.resize((size_t)nSec + 1);
                alignmentResults[0] = result;
                for (_int64 k = 0; k < nSec; k++) {
                    memset(&alignmentResults[(size_t)k + 1], 0, sizeof(SingleAlignmentResult));
                    toSnap(secondary[i * secCap + k], &alignmentResults[(size_t)k + 1]);
                }
                if (NULL != readWriter) {
                    for (_int64 k = 0; k <= nSec; k++) {
                        if (!options->passFilter(r, alignmentResults[(size_t)k].status, false, k != 0 || !containsPrimary)) {
                            if (k == 0) containsPrimary = false;
                            alignmentResults[(size_t)k] = alignmentResults[(size_t)nSec];
                            nSec--;
                            k--;
                        }
                    }
                    stats->extraAlignments += nSec + (containsPrimary ? 0 : 1);
                    readWriter->writeReads(context->readerContext, r, alignmentResults.data(), nSec + 1, containsPrimary, context->useAffineGap);
                }
                if (containsPrimary) {
                    updateSingleStats(stats, result.status, result.mapq);          // :330-334 (alignmentResults[0] is still the primary when containsPrimary)
                } else {
                    stats->filtered++;
                }
                this->writeRead(r, &result);
                continue;
            }
            if (NULL != readWriter) {
                // SingleAligner.cpp:296-322 with nSecondaryResults == 0
                if (!options->passFilter(r, result.status, false, false)) {
                    containsPrimary = false;
                } else {
                    readWriter->writeReads(context->readerContext, r, &result, 1, true, context->useAffineGap);
                }
            }
            if (containsPrimary) {
                updateSingleStats(stats, result.status, result.mapq);
            } else {
                stats->filtered++;
            }
            this->writeRead(r, &result);
        }
        batch.clear();
    }
    stats->lvCalls = counters.lvCalls;
    stats->affineGapCalls = counters.affineGapCalls;
    addCounters(engine, counters);
    batch.destroy();
    snapgpu_host_free(results);
    snapgpu_host_free(secondary);
    snapgpu_host_free(nSecondary);
    return true;             // this thread's share is consumed: the stock loop is skipped (SingleAligner.cpp:102-105)
}

bool GpuAlignerExtension::runIterationThread(PairedReadSupplier *supplier, AlignerContext *context)
{
    GpuEngine *engine = engineForThisThread(context, true);
    AlignerStats *stats = context->stats;
    AlignerOptions *options = context->options;
    PairedAlignerOptions *po = (PairedAlignerOptions *)options;
    ReadWriter *readWriter = context->readWriter;
    ReadBatchCopy batch;
    batch.init(shared->batchReads);
    snapgpu_paired_result *results = (snapgpu_paired_result *)snapgpu_host_alloc((size_t)(shared->batchReads / 2) * sizeof(snapgpu_paired_result));
    if (!results) gpuFatal("allocating the result batch");
    snapgpu_counters counters;
    memset(&counters, 0, sizeof(counters));
    const int maxDist = (int)context->maxDist;

    Read *reads[NUM_READS_PER_PAIR] = {NULL, NULL};
    bool more = supplier->getNextReadPair(&reads[0], &reads[1]);
    while (more) {
        while (more && batch.n + 2 <= batch.capacity && !batch.full(reads[0]->getDataLength() + reads[1]->getDataLength())) {
            if (!po->ignoreMismatchedIDs) {
                Read::checkIdMatch(reads[0], reads[1]);          // PairedAligner.cpp:664-666
            }
            batch.add(reads[0]);
            batch.add(reads[1]);
            more = supplier->getNextReadPair(&reads[0], &reads[1]);
        }
        const _int64 nPairs = batch.n / 2;
        pthread_mutex_lock(&engine->lock);
        const int rc = snapgpu_align_paired(engine->aligner, nPairs, batch.bases, batch.quals, batch.offsets, batch.lens, results, &counters);
        pthread_mutex_unlock(&engine->lock);
        if (rc) gpuFatal("snapgpu_align_paired");

        for (_int64 i = 0; i < nPairs; i++) {
            Read *pr[NUM_READS_PER_PAIR] = {&batch.reads[2 * i], &batch.reads[2 * i + 1]};
            _int64 nSingleResults[2] = {0, 0};
            stats->totalReads += 2;
            const bool useful0 = pr[0]->getDataLength() >= context->minReadLength && (int)pr[0]->countOfNs() <= maxDist;
            const bool useful1 = pr[1]->getDataLength() >= context->minReadLength && (int)pr[1]->countOfNs() <= maxDist;
            PairedAlignmentResult result;
            memset(&result, 0, sizeof(result));
            if (!useful0 && !useful1) {
                // PairedAligner.cpp:679-708
                result.status[0] = result.status[1] = NotFound;
                result.location[0] = result.location[1] = InvalidGenomeLocation;
                const bool pass0 = options->passFilter(pr[0], result.status[0], true, false);
                const bool pass1 = options->passFilter(pr[1], result.status[1], true, false);
                const bool pass = (options->filterFlags & AlignerOptions::FilterBothMatesMatch) ? (pass0 && pass1) : (pass0 || pass1);
                if (pass) {
                    if (NULL != readWriter) {
                        readWriter->writePairs(context->readerContext, pr, &result, 1, NULL, nSingleResults, true, context->useAffineGap);
                    }
                    stats->uselessReads += 2;
                } else {
                    stats->filtered += 2;
                }
                continue;
            }
            toSnap(results[i], &result);
            if (po->forceSpacing && isOneLocation(result.status[0]) != isOneLocation(result.status[1])) {
                // either both align or neither do (PairedAligner.cpp:822-830)
                result.status[0] = result.status[1] = NotFound;
                result.location[0] = result.location[1] = InvalidGenomeLocation;
                result.usedAffineGapScoring[0] = result.usedAffineGapScoring[1] = false;
                result.basesClippedBefore[0] = result.basesClippedBefore[1] = 0;
                result.basesClippedAfter[0] = result.basesClippedAfter[1] = 0;
                result.agScore[0] = result.agScore[1] = 0;
            }
            const bool pass0 = options->passFilter(pr[0], result.status[0], !useful0, false);
            const bool pass1 = options->passFilter(pr[1], result.status[1], !useful1, false);
            const bool firstIsPrimary = (options->filterFlags & AlignerOptions::FilterBothMatesMatch) ? (pass0 && pass1) : (pass0 || pass1);
            if (NULL != readWriter && firstIsPrimary) {
                SingleAlignmentResult *singleResults[2] = {NULL, NULL};
                readWriter->writePairs(context->readerContext, pr, &result, 1, singleResults, nSingleResults, true, context->useAffineGap);
            }
            if (firstIsPrimary) {
                // PairedAlignerContext::updateStats (PairedAligner.cpp:962-1010): the AlignerStats part; the distance / score
                // histograms live in PairedAlignerStats, which the reference defines inside PairedAligner.cpp (no header)
                const bool useful[2] = {useful0, useful1};
                for (int r = 0; r < 2; r++) {
                    if (useful[r]) {
                        updateSingleStats(stats, result.status[r], result.mapq[r]);
                    } else {
                        stats->uselessReads++;
                    }
                }
                if (result.direction[0] == result.direction[1]) stats->sameComplement++;
                if (result.alignedAsPair) stats->alignedAsPairs += 2;
                if (result.agForcedSingleAlignerCall) {
                    stats->agForcedSingleEndAlignment += 2;
                    if (!result.alignedAsPair) stats->agUsedSingleEndAlignment += 2;
                }
            } else {
                stats->filtered += 2;
            }
            this->writePair(pr[0], pr[1], &result);
        }
        batch.clear();
    }
    stats->lvCalls = counters.lvCalls;
    stats->affineGapCalls = counters.affineGapCalls;
    addCounters(engine, counters);
    batch.destroy();
    snapgpu_host_free(results);
    return true;
}

// ------------------------------------------------------------------------------------------------------------------------------
// snap-aligner-gpu: `single` and `paired` with the extension installed; `index` is stock.
// ------------------------------------------------------------------------------------------------------------------------------
#ifndef SNAPGPU_EXTENSION_NO_MAIN
static const char *GPU_VERSION = "2.0.5-snapgpu";

int main(int argc, const char **argv)
{
    if (argc < 2) {
        fprintf(stderr, "Usage: snap-aligner-gpu <index|single|paired> [<options>]   (options as for snap-aligner)\n");
        return 1;
    }
    InitializeSeedSequencers();
    if (strcmp(argv[1], "index") == 0) {
        GenomeIndex::runIndexer(argc - 2, argv + 2);
        return 0;
    }
    for (int i = 1; i < argc; ) {
        unsigned nArgsConsumed = 0;
        if (strcmp(argv[i], "single") == 0) {
            SingleAlignerContext single(new GpuAlignerExtension());
            single.runAlignment(argc - i, argv + i, GPU_VERSION, &nArgsConsumed);
        } else if (strcmp(argv[i], "paired") == 0) {
            PairedAlignerContext paired(new GpuAlignerExtension());
            paired.runAlignment(argc - i, argv + i, GPU_VERSION, &nArgsConsumed);
        } else {
            fprintf(stderr, "Invalid command: %s\n", argv[i]);
            return 1;
        }
        if (nArgsConsumed == 0) break;
        i += nArgsConsumed;
    }
    return 0;
}
#endif
