/*
 * mb200_host_loop.c -- a host application in C on top of the C-ABI (it links against libmb200.so like
 * any other client; it is not part of the engine).  bench.py drives its timed regions through it, so
 * that the numbers are what a C caller (the reference is C99) gets, not what Python's ctypes adds.
 *
 * R independent replicas of the analysis (one engine instance each: its own chains, its own stream)
 * advance generation by generation, the way the reference's RunChain (src/mcmc.c:16718) advances one:
 *
 *   mb200_host_generation_loop   host structs in, lnL out (the end-to-end path): per generation a host
 *                                thread launches the evaluations of its replicas (mb200_evaluate_begin),
 *                                then collects every result (mb200_evaluate_end) -- nothing of a
 *                                replica's generation g+1 starts before its generation g has returned
 *                                its lnL to the host;
 *   mb200_host_replay_loop       device-resident job descriptors (mb200_replay), timed per generation
 *                                with CUDA events on a control stream, optional L2 flush before each.
 */
#include <stdlib.h>
#include <time.h>
#include <pthread.h>
#include <cuda_runtime_api.h>
#include "mb200.h"

/* steps[r * cycle + i]: evaluations of replica r in step i of the cycle (count each).  order[g] is the
 * cycle step of generation g.  lnL / status: R * count entries, results of the last generation.
 * The replicas are independent analyses, so they are dealt out to `threads` host threads (the
 * reference arm uses every host core; this side needs a handful): each thread advances its own
 * replicas generation by generation.  Returns wall-clock seconds, or a negative engine error code. */
typedef struct
{
    const int *instances; int first, last;          /* replicas [first, last) */
    const mb200_evaluation *const *steps; int cycle, count;
    const int *order; int n_generations;
    double *lnL; int *status; int rc;
} LoopSlice;

static void *run_slice (void *arg)
{
    LoopSlice *s = (LoopSlice *) arg;
    int g, r, rc;

    s->rc = MB200_SUCCESS;
    for (g = 0; g < s->n_generations; g++)
        {
        if (s->last - s->first == 1)
            {
            r = s->first;
            rc = mb200_evaluate (s->instances[r], s->steps[(size_t) r * s->cycle + s->order[g]], s->count,
                                 s->lnL + (size_t) r * s->count, s->status + (size_t) r * s->count);
            if (rc != MB200_SUCCESS) { s->rc = rc; return NULL; }
            continue;
            }
        for (r = s->first; r < s->last; r++)
            {
            rc = mb200_evaluate_begin (s->instances[r], s->steps[(size_t) r * s->cycle + s->order[g]], s->count);
            if (rc != MB200_SUCCESS) { s->rc = rc; return NULL; }
            }
        for (r = s->first; r < s->last; r++)
            {
            rc = mb200_evaluate_end (s->instances[r], s->lnL + (size_t) r * s->count, s->status + (size_t) r * s->count);
            if (rc != MB200_SUCCESS) { s->rc = rc; return NULL; }
            }
        }
    return NULL;
}

double mb200_host_generation_loop (const int *instances, int replicas, const mb200_evaluation *const *steps, int cycle,
                                   int count, const int *order, int n_generations, double *lnL, int *status, int threads)
{
    struct timespec t0, t1;
    LoopSlice slice[64];
    pthread_t tid[64];
    int t, rc = MB200_SUCCESS;

    if (threads < 1) threads = 1;
    if (threads > replicas) threads = replicas;
    if (threads > 64) threads = 64;
    for (t = 0; t < threads; t++)
        {
        LoopSlice *s = &slice[t];
        s->instances = instances; s->first = (int)((long) replicas * t / threads); s->last = (int)((long) replicas * (t + 1) / threads);
        s->steps = steps; s->cycle = cycle; s->count = count; s->order = order; s->n_generations = n_generations;
        s->lnL = lnL; s->status = status; s->rc = MB200_SUCCESS;
        }
    clock_gettime (CLOCK_MONOTONIC, &t0);
    for (t = 1; t < threads; t++)
        if (pthread_create (&tid[t], NULL, run_slice, &slice[t]) != 0)
            return -1.0;
    run_slice (&slice[0]);
    for (t = 1; t < threads; t++)
        pthread_join (tid[t], NULL);
    clock_gettime (CLOCK_MONOTONIC, &t1);
    for (t = 0; t < threads; t++)
        if (slice[t].rc != MB200_SUCCESS) rc = slice[t].rc;
    if (rc != MB200_SUCCESS)
        return (double) rc;
    return (double)(t1.tv_sec - t0.tv_sec) + 1e-9 * (double)(t1.tv_nsec - t0.tv_nsec);
}

/* batches[r * cycle + i]: packed batch of replica r for cycle step i.  Per generation: [flush L2 on the
 * control stream] -> start event -> every replica's stream waits for it and replays its batch ->
 * the control stream waits for all of them -> stop event.  Returns the sum of the per-generation
 * device times in milliseconds, or a negative error code. */
double mb200_host_replay_loop (const int *instances, int replicas, const int *batches, int cycle, const int *order,
                               int n_generations, void *flush_buffer, size_t flush_bytes)
{
    cudaStream_t ctl = NULL, *streams;
    cudaEvent_t *start, *stop, *done;
    double total = 0.0;
    int g, r, rc = 0;

    streams = (cudaStream_t *) calloc ((size_t) replicas, sizeof(cudaStream_t));
    done  = (cudaEvent_t *) calloc ((size_t) replicas, sizeof(cudaEvent_t));
    start = (cudaEvent_t *) calloc ((size_t) n_generations, sizeof(cudaEvent_t));
    stop  = (cudaEvent_t *) calloc ((size_t) n_generations, sizeof(cudaEvent_t));
    if (!streams || !done || !start || !stop) return -1.0;
    for (r = 0; r < replicas; r++)
        {
        void *s = NULL;
        if (mb200_get_stream (instances[r], &s) != MB200_SUCCESS) return -2.0;
        streams[r] = (cudaStream_t) s;
        if (cudaEventCreateWithFlags (&done[r], cudaEventDisableTiming) != cudaSuccess) return -3.0;
        }
    if (cudaStreamCreateWithFlags (&ctl, cudaStreamNonBlocking) != cudaSuccess) return -3.0;
    for (g = 0; g < n_generations; g++)
        if (cudaEventCreate (&start[g]) != cudaSuccess || cudaEventCreate (&stop[g]) != cudaSuccess) return -3.0;

    for (g = 0; g < n_generations && rc == 0; g++)
        {
        if (flush_buffer != NULL)
            cudaMemsetAsync (flush_buffer, g & 0xff, flush_bytes, ctl);
        cudaEventRecord (start[g], ctl);
        for (r = 0; r < replicas; r++)
            {
            cudaStreamWaitEvent (streams[r], start[g], 0);
            if (mb200_replay (instances[r], batches[(size_t) r * cycle + order[g]]) != MB200_SUCCESS) { rc = -4; break; }
            cudaEventRecord (done[r], streams[r]);
            cudaStreamWaitEvent (ctl, done[r], 0);
            }
        cudaEventRecord (stop[g], ctl);
        }
    if (cudaStreamSynchronize (ctl) != cudaSuccess) rc = -5;
    for (r = 0; r < replicas; r++) mb200_synchronize (instances[r]);
    for (g = 0; g < n_generations; g++)
        {
        float ms = 0.0f;
        if (rc == 0 && cudaEventElapsedTime (&ms, start[g], stop[g]) == cudaSuccess) total += ms;
        cudaEventDestroy (start[g]); cudaEventDestroy (stop[g]);
        }
    for (r = 0; r < replicas; r++) cudaEventDestroy (done[r]);
    cudaStreamDestroy (ctl);
    free (streams); free (done); free (start); free (stop);
    return (rc == 0) ? total : (double) rc;
}

/* ------------------------------------------------------------------------------------------------
 * MC^3 generation loop of ONE analysis on this process' GPU (the structure of the reference's RunChain,
 * src/mcmc.c:16704-16958, for the chains SetLocalChainsAndDataSplits gave this process): every
 * generation all local chains are evaluated in ONE launch per data partition (the partitions of a chain
 * in flight together), accepted or rejected, and every swap generation the coordinator
 * (include/mb200_mc3.h) exchanges {lnL, lnPrior} and decides the swaps.  The exchange of generation g
 * is in flight while generation g+1's likelihoods run: a swap changes heats, not states, so only the
 * accept step of g+1 has to wait for it.
 *
 *   parts            engine instances of this process, one per data partition
 *   steps            mode 0: steps[p * cycle + i] -> mb200_evaluation[n_local] (host structs, the C-ABI call)
 *   batches          mode 1: batches[p * cycle + i] = packed batch handle (descriptors resident in HBM)
 *   accept           accept[i * n_local + c]: the proposal of local chain c in cycle step i is accepted
 *   lnprior          lnprior[i * n_local + c]: log prior of that proposal
 *   cur_lnl/cur_lnpr in: state before the first generation; out: state after the last
 *   sums             out: [2] wall-clock seconds, device milliseconds (events on the first partition's stream)
 *   lnl_trace        out, may be NULL: lnl_trace[g * n_local + c] = lnL of local chain c's proposal in generation g
 * Returns 0 or a negative error code.
 */
#include "mb200_mc3.h"

int mb200_host_mc3_loop (mb200_mc3 *mc, const int *parts, int n_parts, int n_local, int mode,
                         const mb200_evaluation *const *steps, const int *batches, int cycle,
                         const unsigned char *accept, const double *lnprior, const int *order, int n_generations,
                         int swap_freq, double *cur_lnl, double *cur_lnpr, double *sums, long long *swaps_accepted,
                         double *lnl_trace)
{
    struct timespec t0, t1;
    cudaEvent_t evA = NULL, evB = NULL;
    cudaStream_t s0 = NULL;
    double *lnl_p, *lnl_new;
    int    *status, g, p, c, rc = 0, swap_pending = 0, acc = 0;
    long long n_acc = 0;
    void   *sv = NULL;
    float   ms = 0.0f;

    if (!mc || !parts || n_parts < 1 || n_local < 1 || !order || !accept || !lnprior || !cur_lnl || !cur_lnpr)
        return -1;
    lnl_p   = (double *) malloc ((size_t) n_local * sizeof(double));
    lnl_new = (double *) malloc ((size_t) n_local * sizeof(double));
    status  = (int *)    malloc ((size_t) n_local * sizeof(int));
    if (!lnl_p || !lnl_new || !status)
        return -1;
    if (mb200_get_stream (parts[0], &sv) != MB200_SUCCESS)
        return -2;
    s0 = (cudaStream_t) sv;
    if (cudaEventCreate (&evA) != cudaSuccess || cudaEventCreate (&evB) != cudaSuccess)
        return -3;
    for (p = 0; p < n_parts; p++)
        mb200_synchronize (parts[p]);
    clock_gettime (CLOCK_MONOTONIC, &t0);
    cudaEventRecord (evA, s0);
    for (g = 0; g < n_generations && rc == 0; g++)
        {
        const int i = order[g];
        /* launch: all local chains of every partition */
        for (p = 0; p < n_parts && rc == 0; p++)
            {
            if (mode == 0)
                rc = mb200_evaluate_begin (parts[p], steps[(size_t) p * cycle + i], n_local);
            else
                rc = mb200_replay_begin (parts[p], batches[(size_t) p * cycle + i]);
            }
        if (rc != 0) break;
        /* the previous generation's exchange has been travelling meanwhile: heats are needed from here on */
        if (swap_pending)
            {
            if ((rc = mb200_mc3_exchange_end (mc)) != 0) break;
            if ((rc = mb200_mc3_attempt_swaps (mc, &acc)) != 0) break;
            n_acc += acc;
            swap_pending = 0;
            }
        /* collect: lnL of a chain = sum over its partitions (src/mcmc.c:7441) */
        for (c = 0; c < n_local; c++) lnl_new[c] = 0.0;
        for (p = 0; p < n_parts && rc == 0; p++)
            {
            if (mode == 0)
                rc = mb200_evaluate_end (parts[p], lnl_p, status);
            else
                rc = mb200_replay_end (parts[p], lnl_p, status);
            for (c = 0; c < n_local; c++)
                lnl_new[c] += lnl_p[c];
            }
        if (rc != 0) break;
        if (lnl_trace)
            for (c = 0; c < n_local; c++) lnl_trace[(size_t) g * n_local + c] = lnl_new[c];
        /* accept / reject (the reference: r = exp (T * (lnL' - lnL) + T * (lnPr' - lnPr) + proposal ratio),
           src/mcmc.c:16865-16890; here the outcome is part of the pre-generated proposal cycle, because a
           rejected proposal's index flips are baked into the next step's evaluation) */
        for (c = 0; c < n_local; c++)
            if (accept[(size_t) i * n_local + c])
                {
                cur_lnl[c]  = lnl_new[c];
                cur_lnpr[c] = lnprior[(size_t) i * n_local + c];
                }
        if (swap_freq > 0 && (g + 1) % swap_freq == 0)
            {
            if ((rc = mb200_mc3_exchange_begin (mc, cur_lnl, cur_lnpr)) != 0) break;
            swap_pending = 1;
            }
        }
    if (rc == 0 && swap_pending)
        {
        rc = mb200_mc3_exchange_end (mc);
        if (rc == 0) rc = mb200_mc3_attempt_swaps (mc, &acc);
        n_acc += acc;
        }
    cudaEventRecord (evB, s0);
    for (p = 0; p < n_parts; p++)
        mb200_synchronize (parts[p]);
    cudaEventSynchronize (evB);
    clock_gettime (CLOCK_MONOTONIC, &t1);
    cudaEventElapsedTime (&ms, evA, evB);
    cudaEventDestroy (evA); cudaEventDestroy (evB);
    if (sums)
        {
        sums[0] = (double)(t1.tv_sec - t0.tv_sec) + 1e-9 * (double)(t1.tv_nsec - t0.tv_nsec);
        sums[1] = (double) ms;
        }
    if (swaps_accepted) *swaps_accepted = n_acc;
    free (lnl_p); free (lnl_new); free (status);
    return rc;
}
