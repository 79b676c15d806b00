/* A C program running the multi-GPU pattern exchange without Python: one thread and one pf_ctx per
 * rank, synthetic batches (pf_synth_fill), pf_submit / pf_collect, then pf_exchange_run over the
 * in-process communicator (pf_comm_local).  Checks that every global pattern has exactly one writer
 * and prints the counts.
 *   usage: exchange_threads <world> <n_samples> <clusters per rank> <seed> <device per rank: 0|1>
 *   (1: rank r runs on device r % device count) */
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <cuda_runtime_api.h>

#include "panfeed_b200.h"

typedef struct {
  uint32_t rank, world, n_samples, clusters;
  uint64_t seed;
  int device;
  pf_comm_local* group;
  int rc;
  pf_exchange_result res;
  uint64_t writers[2];       /* [k-mer, cluster] */
  char err[512];
} rank_job;

static int count_writers(const uint8_t* dev, uint64_t n, uint64_t* out) {
  *out = 0;
  if (n == 0) return 0;
  uint8_t* h = (uint8_t*)malloc(n);
  if (!h || cudaMemcpy(h, dev, n, cudaMemcpyDeviceToHost) != cudaSuccess) { free(h); return -1; }
  for (uint64_t i = 0; i < n; ++i) *out += h[i];
  free(h);
  return 0;
}

static void* run_rank(void* arg) {
  rank_job* j = (rank_job*)arg;
  pf_ctx* ctx = NULL;
  pf_params p;
  memset(&p, 0, sizeof p);
  p.abi_version = PF_ABI_VERSION; p.k = 31; p.n_samples = j->n_samples; p.canonical = 1; p.maf = 0.01;
  j->rc = pf_create(&ctx, j->device, &p);
  if (j->rc) { snprintf(j->err, sizeof j->err, "pf_create: %s", pf_last_error(NULL)); goto out; }
  pf_synth_params sp;
  memset(&sp, 0, sizeof sp);
  sp.seed = j->seed; sp.n_samples = j->n_samples; sp.n_clusters = j->clusters;
  sp.first_cluster = j->rank * j->clusters; sp.gene_len = 600; sp.n_founders = 8;
  sp.founder_div = 0.01f; sp.private_div = 0.001f; sp.core_fraction = 0.6f; sp.paralog_rate = 0.01f;
  sp.total_clusters = j->world * j->clusters;
  uint32_t n_seqs = 0; uint64_t n_words = 0;
  j->rc = pf_synth_plan(&sp, &n_seqs, &n_words);
  if (j->rc) { snprintf(j->err, sizeof j->err, "pf_synth_plan"); goto out; }
  uint32_t W = pf_pattern_words(j->n_samples);
  pf_seq_desc* seqs = calloc(n_seqs ? n_seqs : 1, sizeof *seqs);
  pf_cluster_desc* cl = calloc(j->clusters ? j->clusters : 1, sizeof *cl);
  uint32_t* pres = calloc((size_t)j->clusters * W + 1, 4);
  uint64_t* packed = calloc(n_words ? n_words : 1, 8);
  j->rc = pf_synth_fill(j->device, &sp, seqs, cl, pres, packed);
  if (!j->rc) {
    pf_batch b;
    memset(&b, 0, sizeof b);
    b.packed_bases = packed; b.n_words = n_words; b.seqs = seqs; b.n_seqs = n_seqs;
    b.clusters = cl; b.n_clusters = j->clusters; b.cluster_presence = pres;
    pf_batch_result r;
    j->rc = pf_submit(ctx, &b);
    if (!j->rc) j->rc = pf_collect(ctx, &r);
  }
  free(seqs); free(cl); free(pres); free(packed);
  if (j->rc) { snprintf(j->err, sizeof j->err, "batch: %s", pf_last_error(ctx)); goto out; }
  pf_comm comm;
  pf_comm_local_get(j->group, j->rank, &comm);
  j->rc = pf_exchange_run(ctx, &comm, PF_EXCHANGE_WRITER, &j->res);
  if (j->rc) { snprintf(j->err, sizeof j->err, "pf_exchange_run: %s", pf_last_error(ctx)); goto out; }
  if (count_writers(j->res.kmer.writer, j->res.kmer.n_local, &j->writers[0]) ||
      count_writers(j->res.cluster.writer, j->res.cluster.n_local, &j->writers[1])) {
    j->rc = -2; snprintf(j->err, sizeof j->err, "writer copy failed"); goto out;
  }
  j->rc = pf_exchange_release(ctx, &comm);
  if (j->rc) snprintf(j->err, sizeof j->err, "pf_exchange_release: %s", pf_last_error(ctx));
out:
  if (j->rc) pf_comm_local_abort(j->group);     /* nobody waits for a rank that has failed */
  pf_destroy(ctx);
  return NULL;
}

int main(int argc, char** argv) {
  if (argc < 6) { fprintf(stderr, "usage: %s world n_samples clusters seed spread\n", argv[0]); return 2; }
  uint32_t world = (uint32_t)atoi(argv[1]);
  int n_dev = 1;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev < 1) { fprintf(stderr, "no CUDA device\n"); return 2; }
  pf_comm_local* g = NULL;
  if (pf_comm_local_create(world, &g)) { fprintf(stderr, "pf_comm_local_create failed\n"); return 2; }
  rank_job* jobs = calloc(world, sizeof *jobs);
  pthread_t* th = calloc(world, sizeof *th);
  for (uint32_t r = 0; r < world; ++r) {
    jobs[r].rank = r; jobs[r].world = world; jobs[r].n_samples = (uint32_t)atoi(argv[2]);
    jobs[r].clusters = (uint32_t)atoi(argv[3]); jobs[r].seed = strtoull(argv[4], NULL, 10);
    jobs[r].device = atoi(argv[5]) ? (int)(r % (uint32_t)n_dev) : 0;
    jobs[r].group = g;
    pthread_create(&th[r], NULL, run_rank, &jobs[r]);
  }
  int bad = 0;
  for (uint32_t r = 0; r < world; ++r) pthread_join(th[r], NULL);
  uint64_t w[2] = {0, 0};
  for (uint32_t r = 0; r < world; ++r) {
    if (jobs[r].rc) { fprintf(stderr, "rank %u: %d %s\n", r, jobs[r].rc, jobs[r].err); bad = 1; continue; }
    w[0] += jobs[r].writers[0];
    w[1] += jobs[r].writers[1];
    if (jobs[r].res.kmer.n_global != jobs[0].res.kmer.n_global ||
        jobs[r].res.cluster.n_global != jobs[0].res.cluster.n_global) { fprintf(stderr, "n_global differs\n"); bad = 1; }
  }
  if (!bad) {
    if (w[0] != jobs[0].res.kmer.n_global || w[1] != jobs[0].res.cluster.n_global) {
      fprintf(stderr, "writers %llu/%llu != global patterns %llu/%llu\n", (unsigned long long)w[0],
              (unsigned long long)w[1], (unsigned long long)jobs[0].res.kmer.n_global,
              (unsigned long long)jobs[0].res.cluster.n_global);
      bad = 1;
    }
    printf("world=%u kmer_global=%llu cluster_global=%llu kmer_writers=%llu cluster_writers=%llu\n", world,
           (unsigned long long)jobs[0].res.kmer.n_global, (unsigned long long)jobs[0].res.cluster.n_global,
           (unsigned long long)w[0], (unsigned long long)w[1]);
  }
  pf_comm_local_destroy(g);
  free(jobs); free(th);
  return bad;
}
