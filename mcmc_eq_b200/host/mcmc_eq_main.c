/* mcmc_eq_main.c -- the reference's command line on top of the B200 library (plain C host code, C ABI only).
 *
 *     mcmc_eq <config_eqx.dat> <out> <picks> [-n chains] [-d device] [-s seed] [-r slots] [-q]
 *             [-k checkpoint [-K minutes]] [-R checkpoint] [-D diagnostics] [-x]
 *
 * The first three arguments are the reference's (src/mcmc_eq.c:332-338; it ignores anything after them).
 * With one chain (the default) <out> is written exactly like the reference writes it: a "sta ST" record, a
 * "mod X." record every deci-th accepted model, the "bat BF" record and nine "cnt" lines
 * (src/mcmc_eq.c:763,1163,1196-1207; format of print_model_raw :234-248).  With -n N the N chains that the
 * reference would run as N processes (run/srun_mcmc_eq.sh:13,35) run concurrently on one GPU and each writes
 * its own file: <out> is a printf pattern with one integer conversion ("rjx-%03d.out"); without a conversion
 * the chain number is inserted before the extension ("rjx.out" -> "rjx-001.out", the naming scriptsV2/dispe.sh:29
 * globs for).  Chain numbers start at 1 like the SLURM array index.
 *
 * Seeds: config line 32 first value > 0 seeds chain k with value + k (chain 0 == the configured seed);
 * otherwise /dev/urandom (src/mcmc_eq.c:250-265,393-394).  -s overrides.  The random streams are this
 * library's counter-based generator, not libc rand(): chains are statistically, not bitwise, the reference's.
 *
 * Output path: decimated records wait in a device-side ring (-r slots per chain, default 4); after every chunk of
 * iterations the main thread starts an asynchronous drain (mq_drain_begin: pack kernel + device-to-host copy on a second
 * stream) and goes on stepping, a writer thread waits for the batch and formats the print_model_raw text
 * (src/mcmc_eq.c:234-248) into the per-chain files.  The reference writes and flushes each record from inside the
 * sampling loop (:1163).
 *
 * Checkpoints: with -k <file> the run writes a checkpoint at a chunk boundary every -K minutes (default 30; 0 = after
 * every chunk): every record of the chunks so far is written, the chain files are flushed and fsync'ed, and a header
 * (chain count, seed, iterations done, records lost so far, the length of every chain file) followed by the sampler state
 * of mq_state_save goes to <file>.tmp, which is fsync'ed and renamed over <file>: a process killed at any moment leaves
 * the previous checkpoint intact.  -R <file> resumes: the checkpoint is read and checked before anything else happens,
 * the handle is created with its chain count and seed and loads its state, each chain file is cut back to its recorded
 * length and the run goes on from there (no "sta" record is written again).  A run killed after its first checkpoint and
 * resumed with -R leaves chain files byte-identical to those of the uninterrupted run.  -n must be the checkpoint's (or
 * absent); -d may differ.
 *
 * Diagnostics: -D <file> computes split R-hat and the effective sample size of every posterior quantity on the device
 * (mq_diag_*) from the decimated models after the start phase (burn-in = j_max_start, 16 batch slots), and writes <file>
 * at every checkpoint and at the end of the run: a "#" header line (chains used, burn-in, batches, iterations done), then
 * one line per quantity "name index n_models mean sd rhat ess" (names rms dim noise vp vpvs x y z t pres sres), plus one
 * stderr line with the largest R-hat and the smallest ESS and where they occur.  The accumulators are part of the
 * checkpoint: under -R they continue, and -D with a checkpoint that has none fails before any chain file is touched.
 *
 * Reciprocal tables: -x builds the travel-time tables with the source at each receiver row instead of at each event depth
 * (mq_set_tables, MQ_TABLES_RECIPROCAL): n_rows solves per table instead of nz, at the price of the finite-difference
 * scheme's reciprocity error in every prediction (DESIGN.md section 6).  One stderr line says so.  Under -R the mode is the
 * checkpoint's (its state flags); -x against a checkpoint written with parity tables fails before any chain file is touched.
 *
 * Unlike the reference (which exit(0)s on every error) the exit status is non-zero on failure.
 */
#include <math.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <unistd.h>

#include "../../include/mcmceq_b200.h"
#include "mq_io.h"

typedef struct {
    int n_chains;
    FILE** out;
    const mqio_picks* pk;
    long* written;
} sink_t;

static const char* kind_tag(int kind) { return kind == MQ_REC_MODEL ? "mod" : kind == MQ_REC_BEST ? "bat" : "sta"; }

static int write_record(void* user, const mq_record* r)
{
    sink_t* s = (sink_t*)user;
    char code[3];
    if (r->chain < 0 || r->chain >= s->n_chains) return 1;
    if (r->kind == MQ_REC_MODEL) { code[0] = r->code; code[1] = '.'; }     /* "Q." "P." ... src/mcmc_eq.c:870-1096 */
    else if (r->kind == MQ_REC_BEST) { code[0] = 'B'; code[1] = 'F'; }     /* :1196 */
    else { code[0] = 'S'; code[1] = 'T'; }                                  /* :763  */
    code[2] = 0;
    mqio_write_record(s->out[r->chain], kind_tag(r->kind), code, (long)r->number, (long)r->dim, r->rms, r->noise, r->z,
                      r->vp, r->vpvs, s->pk->view.n_events, r->eq, s->pk->reftime, r->origin, s->pk->view.n_stations,
                      r->pres, r->sres);
    s->written[r->chain]++;
    return 0;
}

/* Start model from model.dat in the working directory (aflag == 3, src/mcmc_eq.c:381,636-731): an analyse_eq result file
 * whose STAN lines give the velocity model (depth, Vp = column 7, Vp/Vs = column 9 of the line), EQ lines the hypocentres,
 * RES lines the station corrections and the NOISE line the eight sigmas; the letters of config line 34 (V Q R N) select
 * which of them replace the random start values -- in every chain, as every reference process would read the same file. */
static int apply_model_dat(const mq_config* cfg, mq_models* m, FILE* log)
{
    FILE* f = fopen("model.dat", "r");
    char line[4096], tag[64];
    const char* sw = cfg->inp_model_switch;
    int c, k, nv = 0, nq = 0;
    float zz[1000], vv[1000], rr[1000];
    if (!f) { fprintf(stderr, "could not open model file\n"); return 1; }
    while (fgets(line, sizeof line, f)) {
        float a[16];
        int di;
        if (sscanf(line, "%63s", tag) != 1 || tag[0] == '#') continue;
        if (!strcmp(tag, "STAN") && strchr(sw, 'V')) {
            if (sscanf(line, "%*s %f %f %f %f %f %f %f %f", &a[0], &a[1], &a[2], &a[3], &a[4], &a[5], &a[6], &a[7]) < 8) continue;
            if (nv >= m->max_dim || nv >= 1000) { fprintf(stderr, "model larger than reserved space, increase 'max # of cells/layers' in config file\n"); fclose(f); return 1; }
            zz[nv] = a[0]; vv[nv] = a[5]; rr[nv] = a[7]; nv++;
        } else if (!strcmp(tag, "EQ") && strchr(sw, 'Q')) {
            if (sscanf(line, "%*s %d %f %f %f", &di, &a[0], &a[1], &a[2]) < 4 || di < 0 || di >= m->n_events) continue;
            for (c = 0; c < m->n_chains; c++)
                for (k = 0; k < 3; k++) m->eq[((size_t)c * m->n_events + di) * 3 + k] = a[k];
            nq++;
        } else if (!strcmp(tag, "RES") && strchr(sw, 'R')) {
            if (sscanf(line, "%*s %d %f %f", &di, &a[0], &a[1]) < 3 || di < 0 || di >= m->n_stations) continue;
            for (c = 0; c < m->n_chains; c++) { m->pres[(size_t)c * m->n_stations + di] = a[0]; m->sres[(size_t)c * m->n_stations + di] = a[1]; }
        } else if (!strcmp(tag, "NOISE") && strchr(sw, 'N')) {
            if (sscanf(line, "%*s %f %f %f %f %f %f %f %f", &a[0], &a[1], &a[2], &a[3], &a[4], &a[5], &a[6], &a[7]) < 8) continue;
            for (c = 0; c < m->n_chains; c++)
                for (k = 0; k < 4; k++) { m->noise[8 * (size_t)c + 2 * k] = a[k]; m->noise[8 * (size_t)c + 2 * k + 1] = a[4 + k]; }   /* file: p0..p3 s0..s3 */
        }
    }
    fclose(f);
    if (strchr(sw, 'V')) {
        if (nv < 1) { fprintf(stderr, "model.dat holds no STAN line\n"); return 1; }
        for (c = 0; c < m->n_chains; c++) {
            m->dim[c] = nv;
            for (k = 0; k < nv; k++) {
                m->z[(size_t)c * m->max_dim + k] = zz[k]; m->vp[(size_t)c * m->max_dim + k] = vv[k]; m->vpvs[(size_t)c * m->max_dim + k] = rr[k];
            }
        }
    }
    if (strchr(sw, 'Q') && nq != m->n_events) { fprintf(stderr, "number of quakes does not fit pick file!\n"); return 1; }
    if (log) fprintf(log, "start model from model.dat (%s): %d layers, %d quakes\n", sw, nv, nq);
    return 0;
}

/* ---- writer thread: takes begun batches from a two-deep queue, waits for their records, writes them ----------------- */
typedef struct {
    pthread_t thread;
    pthread_mutex_t mu;
    pthread_cond_t cv;
    mq_batch* q[2];
    int n_q, stop, failed;
    long lost, records;
    sink_t* sink;
} writer_t;

static void* writer_main(void* arg)
{
    writer_t* w = (writer_t*)arg;
    for (;;) {
        mq_batch* b;
        int n = 0, lost = 0;
        pthread_mutex_lock(&w->mu);
        while (w->n_q == 0 && !w->stop) pthread_cond_wait(&w->cv, &w->mu);
        if (w->n_q == 0) { pthread_mutex_unlock(&w->mu); return NULL; }
        b = w->q[0];
        pthread_mutex_unlock(&w->mu);
        if (mq_batch_wait(b, &n, &lost) != MQ_OK || mq_batch_deliver(b, write_record, w->sink) != MQ_OK) w->failed = 1;
        mq_batch_release(b);
        pthread_mutex_lock(&w->mu);
        w->q[0] = w->q[1]; w->n_q--;
        w->lost += lost; w->records += n;
        pthread_cond_broadcast(&w->cv);
        pthread_mutex_unlock(&w->mu);
    }
}

static void writer_wait_slot(writer_t* w)             /* until one of the handle's two batches is free again */
{
    pthread_mutex_lock(&w->mu);
    while (w->n_q == 2) pthread_cond_wait(&w->cv, &w->mu);
    pthread_mutex_unlock(&w->mu);
}

static void writer_push(writer_t* w, mq_batch* b)
{
    pthread_mutex_lock(&w->mu);
    w->q[w->n_q++] = b;
    pthread_cond_broadcast(&w->cv);
    pthread_mutex_unlock(&w->mu);
}

static void writer_idle(writer_t* w)                  /* until everything pushed so far is on disk */
{
    pthread_mutex_lock(&w->mu);
    while (w->n_q > 0) pthread_cond_wait(&w->cv, &w->mu);
    pthread_mutex_unlock(&w->mu);
}

static unsigned long urandom_seed(void)
{
    unsigned long v = (unsigned long)time(NULL);
    FILE* f = fopen("/dev/urandom", "rb");
    if (f) { if (fread(&v, sizeof v, 1, f) != 1) v = (unsigned long)time(NULL); fclose(f); }
    return v;
}

static void out_name(char* dst, size_t cap, const char* pattern, int n_chains, int chain1)
{
    const char* pct = strchr(pattern, '%');
    if (n_chains == 1 && !pct) { snprintf(dst, cap, "%s", pattern); return; }
    if (pct) { snprintf(dst, cap, pattern, chain1); return; }
    {
        const char* dot = strrchr(pattern, '.');
        const char* slash = strrchr(pattern, '/');
        if (dot && (!slash || dot > slash)) snprintf(dst, cap, "%.*s-%03d%s", (int)(dot - pattern), pattern, chain1, dot);
        else snprintf(dst, cap, "%s-%03d", pattern, chain1);
    }
}

/* ---- checkpoints: CLI header, the length of every chain file, then the mq_state_save blob ------------------------------ */
#define CKPT_MAGIC "MQCKPT1"
typedef struct {
    char magic[8];
    int32_t n_chains, reserved;
    uint64_t seed;
    int64_t iters_done, lost;
    uint64_t state_bytes;
} ckpt_head;

typedef struct {
    ckpt_head head;
    int64_t* file_len;   /* [n_chains] */
    unsigned char* state;
} ckpt_t;

static void ckpt_free(ckpt_t* k) { free(k->file_len); free(k->state); memset(k, 0, sizeof *k); }

/* Reads and checks a checkpoint file; nothing of the library is needed for that.  Returns 0 or 1 (message in err). */
static int ckpt_read(const char* path, ckpt_t* k, char* err, size_t cap)
{
    FILE* f = fopen(path, "rb");
    long size;
    size_t n;
    memset(k, 0, sizeof *k);
    if (!f) { snprintf(err, cap, "checkpoint %s: cannot open", path); return 1; }
    if (fseek(f, 0, SEEK_END) != 0 || (size = ftell(f)) < 0 || fseek(f, 0, SEEK_SET) != 0) { fclose(f); snprintf(err, cap, "checkpoint %s: cannot read", path); return 1; }
    if ((size_t)size < sizeof k->head || fread(&k->head, sizeof k->head, 1, f) != 1 || memcmp(k->head.magic, CKPT_MAGIC, sizeof k->head.magic) != 0) {
        fclose(f); snprintf(err, cap, "checkpoint %s: not a checkpoint of mcmc_eq", path); return 1;
    }
    n = (size_t)(k->head.n_chains > 0 ? k->head.n_chains : 0);
    if (n < 1 || k->head.iters_done < 0 || k->head.lost < 0 || k->head.state_bytes < sizeof(mq_state_header) ||
        (uint64_t)size != sizeof k->head + n * sizeof(int64_t) + k->head.state_bytes) {
        fclose(f); snprintf(err, cap, "checkpoint %s: damaged header or truncated file (%ld bytes)", path, size); return 1;
    }
    k->file_len = (int64_t*)malloc(n * sizeof(int64_t));
    k->state = (unsigned char*)malloc((size_t)k->head.state_bytes);
    if (!k->file_len || !k->state || fread(k->file_len, sizeof(int64_t), n, f) != n ||
        fread(k->state, 1, (size_t)k->head.state_bytes, f) != (size_t)k->head.state_bytes) {
        fclose(f); ckpt_free(k); snprintf(err, cap, "checkpoint %s: cannot read", path); return 1;
    }
    fclose(f);
    if (memcmp(((const mq_state_header*)k->state)->magic, MQ_STATE_MAGIC, 8) != 0) { ckpt_free(k); snprintf(err, cap, "checkpoint %s: no sampler state in it", path); return 1; }
    return 0;
}

/* Writes a checkpoint at a chunk boundary; the caller has waited for the writer (writer_idle). */
static int ckpt_write(const char* path, mq_handle* h, sink_t* sink, uint64_t seed, long iters_done, long lost)
{
    char tmp[4200];
    ckpt_head head;
    int64_t* len = (int64_t*)calloc((size_t)sink->n_chains, sizeof(int64_t));
    unsigned char* state = NULL;
    uint64_t bytes = 0;
    FILE* f = NULL;
    int c, ok = 0;
    if (!len) return 1;
    for (c = 0; c < sink->n_chains; c++) {
        if (fflush(sink->out[c]) != 0 || fsync(fileno(sink->out[c])) != 0 || (len[c] = ftell(sink->out[c])) < 0) {
            fprintf(stderr, "checkpoint: cannot flush chain file %d\n", c + 1); goto out;
        }
    }
    if (mq_state_size(h, &bytes) != MQ_OK || !(state = (unsigned char*)malloc((size_t)bytes)) || mq_state_save(h, state, bytes, &bytes) != MQ_OK) {
        fprintf(stderr, "checkpoint: mq_state_save failed: %s\n", mq_last_error()); goto out;
    }
    memset(&head, 0, sizeof head);
    memcpy(head.magic, CKPT_MAGIC, sizeof head.magic);
    head.n_chains = sink->n_chains; head.seed = seed; head.iters_done = iters_done; head.lost = lost; head.state_bytes = bytes;
    snprintf(tmp, sizeof tmp, "%s.tmp", path);
    f = fopen(tmp, "wb");
    if (!f || fwrite(&head, sizeof head, 1, f) != 1 || fwrite(len, sizeof(int64_t), (size_t)sink->n_chains, f) != (size_t)sink->n_chains ||
        fwrite(state, 1, (size_t)bytes, f) != (size_t)bytes || fflush(f) != 0 || fsync(fileno(f)) != 0) {
        fprintf(stderr, "checkpoint: cannot write %s\n", tmp); goto out;
    }
    if (fclose(f) != 0) { f = NULL; fprintf(stderr, "checkpoint: cannot write %s\n", tmp); goto out; }
    f = NULL;
    if (rename(tmp, path) != 0) { fprintf(stderr, "checkpoint: cannot rename %s to %s\n", tmp, path); goto out; }
    ok = 1;
out:
    if (f) fclose(f);
    free(len); free(state);
    return ok ? 0 : 1;
}

/* ---- diagnostics: the parameters a saved state holds, the report file --------------------------------------------------- */
static int state_diag_params(const unsigned char* state, uint64_t bytes, int64_t* burn_in, int32_t* n_batches)
{
    const mq_state_header* H = (const mq_state_header*)state;
    uint32_t k;
    if (!(H->flags & MQ_STATE_DIAG) || bytes < sizeof *H + H->n_sections * sizeof(mq_state_section)) return 1;
    for (k = 0; k < H->n_sections; k++) {
        mq_state_section sec;
        memcpy(&sec, state + sizeof *H + k * sizeof sec, sizeof sec);
        if (sec.id == MQ_STATE_SEC_DIAG && sec.bytes >= 16 && sec.offset + 16 <= bytes) {
            memcpy(burn_in, state + sec.offset, sizeof *burn_in);
            memcpy(n_batches, state + sec.offset + 8, sizeof *n_batches);
            return 0;
        }
    }
    return 1;
}

/* name and index of quantity q (include/mcmceq_b200.h, mq_diag_*) */
static const char* diag_name(int q, int nz, int ne, int* index)
{
    static const char* ev[4] = {"x", "y", "z", "t"};
    *index = 0;
    if (q == 0) return "rms";
    if (q == 1) return "dim";
    if (q < 10) { *index = q - 2; return "noise"; }
    q -= 10;
    if (q < 2 * nz) { *index = q % nz; return q < nz ? "vp" : "vpvs"; }
    q -= 2 * nz;
    if (q < 4 * ne) { *index = q / 4; return ev[q % 4]; }
    q -= 4 * ne;
    *index = q / 2;
    return q % 2 ? "sres" : "pres";
}

static int diag_write(const char* path, mq_handle* h, int nz, int ne, int ns, int64_t burn_in, int n_batches, long iters_done)
{
    const int Q = 10 + 2 * nz + 4 * ne + 2 * ns;
    double* v = (double*)malloc(4 * (size_t)Q * sizeof(double));
    double *mean = v, *sd = v + Q, *rhat = v + 2 * Q, *ess = v + 3 * Q;
    int64_t n_models = 0;
    int32_t used = 0;
    int q, qr = -1, qe = -1, ir, ie, ok = 0;
    char tmp[4200];
    FILE* f = NULL;
    if (!v) return 1;
    if (mq_diag_summary(h, 0, mean, sd, rhat, ess, &n_models, &used) != MQ_OK) {
        fprintf(stderr, "diagnostics: mq_diag_summary failed: %s\n", mq_last_error()); goto out;
    }
    snprintf(tmp, sizeof tmp, "%s.tmp", path);
    if (!(f = fopen(tmp, "w"))) { fprintf(stderr, "diagnostics: cannot write %s\n", tmp); goto out; }
    fprintf(f, "# chains_used %d burn_in %lld batches %d iterations %ld\n", used, (long long)burn_in, n_batches, iters_done);
    for (q = 0; q < Q; q++) {
        int idx;
        const char* name = diag_name(q, nz, ne, &idx);
        fprintf(f, "%-5s %5d %12lld %.9e %.9e %.6f %.1f\n", name, idx, (long long)n_models, mean[q], sd[q], rhat[q], ess[q]);
        if (!isnan(rhat[q]) && (qr < 0 || rhat[q] > rhat[qr])) qr = q;
        if (!isnan(ess[q]) && (qe < 0 || ess[q] < ess[qe])) qe = q;
    }
    if (fclose(f) != 0) { f = NULL; fprintf(stderr, "diagnostics: cannot write %s\n", tmp); goto out; }
    f = NULL;
    if (rename(tmp, path) != 0) { fprintf(stderr, "diagnostics: cannot rename %s to %s\n", tmp, path); goto out; }
    if (qr >= 0 && qe >= 0) {
        const char* nr = diag_name(qr, nz, ne, &ir);
        const char* ne_ = diag_name(qe, nz, ne, &ie);
        fprintf(stderr, "diagnostics after %ld iterations (%d chains used): max R-hat %.4f (%s %d), min ESS %.1f (%s %d)\n", iters_done,
                used, rhat[qr], nr, ir, ess[qe], ne_, ie);
    } else {
        fprintf(stderr, "diagnostics after %ld iterations (%d chains used): no R-hat yet\n", iters_done, used);
    }
    ok = 1;
out:
    if (f) fclose(f);
    free(v);
    return ok ? 0 : 1;
}

static double now_s(void)
{
    struct timespec t;
    clock_gettime(CLOCK_MONOTONIC, &t);
    return (double)t.tv_sec + 1e-9 * (double)t.tv_nsec;
}

#define FAIL(...) do { fprintf(stderr, __VA_ARGS__); fprintf(stderr, "\n"); rc = 1; goto done; } while (0)
#define MQ(call) do { int rc_ = (call); if (rc_ != MQ_OK) FAIL("%s failed (%d): %s", #call, rc_, mq_last_error()); } while (0)

int main(int argc, char** argv)
{
    int rc = 0, n_chains = 1, device = 0, quiet = 0, i, c, from_file = 0, ring = 0, writer_on = 0, n_given = 0, reciprocal = 0;
    const char *ck_path = NULL, *resume_path = NULL, *diag_path = NULL;
    int64_t diag_burn_in = 0;
    int32_t diag_batches = 16;
    double ck_minutes = 30.0, ck_last;
    ckpt_t ck;
    uint64_t seed_used = 0;
    writer_t wr;
    long seed_arg = -1;
    mq_config cfg;
    mqio_picks pk;
    mq_handle* h = NULL;
    sink_t sink;
    int64_t* counts = NULL;
    double *ll = NULL, *rms = NULL;
    long iters_done = 0;
    const char* env;
    clock_t t0;

    memset(&pk, 0, sizeof pk);
    memset(&sink, 0, sizeof sink);
    memset(&wr, 0, sizeof wr);
    memset(&ck, 0, sizeof ck);
    if (argc < 4) {
        fprintf(stderr, "usage: %s config_eqx.dat outfile picks [-n chains] [-d device] [-s seed] [-r ring slots] [-q] "
                        "[-k checkpoint [-K minutes]] [-R checkpoint] [-D diagnostics] [-x]\n", argv[0]);
        return 2;
    }
    if ((env = getenv("MCMCEQ_CHAINS")) != NULL) { n_chains = atoi(env); n_given = 1; }
    if ((env = getenv("MCMCEQ_DEVICE")) != NULL) device = atoi(env);
    for (i = 4; i < argc; i++) {
        if (!strcmp(argv[i], "-n") && i + 1 < argc) { n_chains = atoi(argv[++i]); n_given = 1; }
        else if (!strcmp(argv[i], "-k") && i + 1 < argc) ck_path = argv[++i];
        else if (!strcmp(argv[i], "-K") && i + 1 < argc) ck_minutes = atof(argv[++i]);
        else if (!strcmp(argv[i], "-R") && i + 1 < argc) resume_path = argv[++i];
        else if (!strcmp(argv[i], "-D") && i + 1 < argc) diag_path = argv[++i];
        else if (!strcmp(argv[i], "-d") && i + 1 < argc) device = atoi(argv[++i]);
        else if (!strcmp(argv[i], "-s") && i + 1 < argc) seed_arg = atol(argv[++i]);
        else if (!strcmp(argv[i], "-r") && i + 1 < argc) ring = atoi(argv[++i]);
        else if (!strcmp(argv[i], "-q")) quiet = 1;
        else if (!strcmp(argv[i], "-x")) reciprocal = 1;
        /* anything else is ignored, as the reference ignores extra arguments */
    }
    if (n_chains < 1) n_chains = 1;
    if (ck_minutes < 0) ck_minutes = 0;
    if (resume_path) {   /* checked before anything else: a garbage file fails before a handle exists or a file is touched */
        char err[4400];
        if (ckpt_read(resume_path, &ck, err, sizeof err)) FAIL("%s", err);
        if (n_given && n_chains != ck.head.n_chains) FAIL("-n %d differs from the checkpoint's %d chains", n_chains, ck.head.n_chains);
        n_chains = ck.head.n_chains;
        if (diag_path && state_diag_params(ck.state, ck.head.state_bytes, &diag_burn_in, &diag_batches))
            FAIL("-D: the checkpoint %s holds no diagnostics (the run was started without -D)", resume_path);
        {   /* the table mode is the checkpoint's; a state without tables (eikonal == 0, aflag == 1) has none */
            const uint32_t flags = ((const mq_state_header*)ck.state)->flags;
            if (reciprocal && (flags & MQ_STATE_TABLES) && !(flags & MQ_STATE_RECIPROCAL))
                FAIL("-x: the checkpoint %s was written with parity tables (the run was started without -x)", resume_path);
            if (flags & MQ_STATE_RECIPROCAL) reciprocal = 1;
        }
    }

    if (mqio_read_config(argv[1], &cfg) != MQ_OK) FAIL("%s", mqio_last_error());
    if (mqio_read_picks(argv[3], &pk) != MQ_OK) FAIL("%s", mqio_last_error());
    if (mqio_check_picks(&cfg, &pk, quiet ? NULL : stderr) != MQ_OK) FAIL("%s", mqio_last_error());
    if (cfg.aflag == 3) { from_file = 1; cfg.aflag = 0; }      /* src/mcmc_eq.c:381 */

    {
        unsigned long seed = resume_path ? (unsigned long)ck.head.seed
                           : seed_arg >= 0 ? (unsigned long)seed_arg : (cfg.true_random > 0 ? (unsigned long)cfg.true_random : urandom_seed());
        seed_used = (uint64_t)seed;
        if (!quiet) fprintf(stderr, "%d chain(s) on device %d, seed %lu, %d events, %d stations, %d picks\n", n_chains, device, seed,
                            pk.view.n_events, pk.view.n_stations, pk.view.n_picks);
        MQ(mq_create(&cfg, &pk.view, n_chains, device, (uint64_t)seed, &h));
        if (reciprocal) {
            MQ(mq_set_tables(h, MQ_TABLES_RECIPROCAL));
            fprintf(stderr, "reciprocal travel-time tables (-x): sources at the receiver rows, not the parity forward\n");
        }
        if (ring > 0) MQ(mq_set_ring(h, ring));
        if (resume_path) MQ(mq_state_load(h, ck.state, ck.head.state_bytes));
        else if (diag_path) {   /* the models of the start phase are burn-in */
            diag_burn_in = cfg.j_max_start;
            MQ(mq_diag_begin(h, diag_burn_in, diag_batches, NULL));
        }
    }

    sink.n_chains = n_chains;
    sink.pk = &pk;
    sink.out = (FILE**)calloc((size_t)n_chains, sizeof(FILE*));
    sink.written = (long*)calloc((size_t)n_chains, sizeof(long));
    counts = (int64_t*)calloc((size_t)n_chains * 20, sizeof(int64_t));
    ll = (double*)calloc((size_t)n_chains, sizeof(double));
    rms = (double*)calloc((size_t)n_chains, sizeof(double));
    if (!sink.out || !sink.written || !counts || !ll || !rms) FAIL("out of memory");
    for (c = 0; c < n_chains; c++) {
        char name[4096];
        out_name(name, sizeof name, argv[2], n_chains, c + 1);
        sink.out[c] = fopen(name, resume_path ? "r+" : "w");
        if (!sink.out[c]) FAIL("Could not open: %s", name);
        if (resume_path) {   /* back to the length the checkpoint recorded: what was written after it is written again */
            long have;
            if (fseek(sink.out[c], 0, SEEK_END) != 0 || (have = ftell(sink.out[c])) < 0) FAIL("Could not read: %s", name);
            if ((int64_t)have < ck.file_len[c]) FAIL("%s holds %ld bytes, fewer than the %lld of the checkpoint", name, have, (long long)ck.file_len[c]);
            if (fflush(sink.out[c]) != 0 || ftruncate(fileno(sink.out[c]), (off_t)ck.file_len[c]) != 0 || fseek(sink.out[c], 0, SEEK_END) != 0)
                FAIL("Could not truncate: %s", name);
        }
    }
    if (resume_path) {
        iters_done = (long)ck.head.iters_done;
        wr.lost = (long)ck.head.lost;
        if (!quiet) fprintf(stderr, "resumed from %s after %ld iterations\n", resume_path, iters_done);
        goto main_loop;
    }

    /* start models + first forward (src/mcmc_eq.c:559-765) */
    t0 = clock();
    MQ(mq_init_chains(h));
    if (from_file) {
        /* the random start values stay for whatever model.dat does not supply (src/mcmc_eq.c:559-630 run before :636) */
        mq_models m;
        const size_t n = (size_t)n_chains, md = (size_t)(cfg.max_dim < 1000 ? cfg.max_dim : 1000), ne = (size_t)pk.view.n_events,
                     ns = (size_t)pk.view.n_stations;
        int bad;
        memset(&m, 0, sizeof m);
        m.n_chains = n_chains; m.max_dim = (int)md; m.n_events = (int)ne; m.n_stations = (int)ns;
        m.dim = (int32_t*)calloc(n, sizeof(int32_t));
        m.z = (float*)calloc(n * md, sizeof(float)); m.vp = (float*)calloc(n * md, sizeof(float)); m.vpvs = (float*)calloc(n * md, sizeof(float));
        m.eq = (float*)calloc(n * ne * 3, sizeof(float)); m.pres = (float*)calloc(n * ns, sizeof(float)); m.sres = (float*)calloc(n * ns, sizeof(float));
        m.noise = (float*)calloc(n * 8, sizeof(float)); m.origin = (float*)calloc(n * ne, sizeof(float));
        bad = !m.dim || !m.z || !m.vp || !m.vpvs || !m.eq || !m.pres || !m.sres || !m.noise || !m.origin;
        if (!bad) bad = mq_get_models(h, &m) != MQ_OK || apply_model_dat(&cfg, &m, quiet ? NULL : stderr) || mq_set_models(h, &m) != MQ_OK ||
                        mq_step(h, 0, NULL) != MQ_OK;      /* a step of zero iterations scores the new start models */
        free(m.dim); free(m.z); free(m.vp); free(m.vpvs); free(m.eq); free(m.pres); free(m.sres); free(m.noise); free(m.origin);
        if (bad) FAIL("start from model.dat failed: %s", mq_last_error());
    }
    MQ(mq_get_stats(h, counts, ll, rms));
    if (!quiet) {
        const long ms = (long)((clock() - t0) * 1000 / CLOCKS_PER_SEC);
        fprintf(stderr, "Time taken %ld seconds %ld milliseconds\n", ms / 1000, ms % 1000);
        for (c = 0; c < n_chains && c < 10; c++)
            fprintf(stderr, "Start model found with loglikelihood %f RMS=%f\n", ll[c], rms[c]);
    }
    MQ(mq_snapshot_all(h, 0, write_record, &sink));

main_loop:
    /* main loop (src/mcmc_eq.c:845-1192): the chain ends after j_max_start + j_max_main ACCEPTED models.  A chain's
     * ring holds `ring` decimated records (at most one per deci iterations), so a chunk of ring/2 * deci iterations
     * between two drains loses nothing even with one drain still in flight. */
    {
        const long target = (long)cfg.j_max_start + (long)cfg.j_max_main;
        const int slots = ring > 0 ? ring : 4;
        long chunk_l = (cfg.deci > 0 ? (long)cfg.deci : 1000L) * (slots > 1 ? slots / 2 : 1);
        int chunk;
        if (chunk_l > 2000) chunk_l = 2000;
        if (cfg.deci > 0 && chunk_l < cfg.deci && cfg.deci <= 2000) chunk_l = cfg.deci;
        chunk = (int)chunk_l;
        wr.sink = &sink;
        pthread_mutex_init(&wr.mu, NULL);
        pthread_cond_init(&wr.cv, NULL);
        if (pthread_create(&wr.thread, NULL, writer_main, &wr) != 0) FAIL("could not start the writer thread");
        writer_on = 1;
        ck_last = now_s();
        for (;;) {
            int running = 0;
            mq_batch* b = NULL;
            MQ(mq_step(h, chunk, NULL));
            iters_done += chunk;
            writer_wait_slot(&wr);
            MQ(mq_drain_begin(h, &b));        /* returns at once; the next chunk runs next to the copy */
            writer_push(&wr, b);
            if (wr.failed) FAIL("writing records failed: %s", mq_last_error());
            MQ(mq_get_stats(h, counts, ll, rms));
            for (c = 0; c < n_chains; c++)
                if (counts[20 * c + 17] < target) running++;
            if (!quiet) {
                double a = 0, r = 0;
                for (c = 0; c < n_chains; c++) { a += (double)counts[20 * c + 17]; r += (double)counts[20 * c + 18]; }
                fprintf(stderr, "Test  %8ld  chains running %d/%d  RMS(chain 1)=%16.10f [s] %5.1f accepted\n", iters_done, running,
                        n_chains, rms[0], 100.0 * a / (a + r > 0 ? a + r : 1));
            }
            if (!running) break;
            if (ck_path && now_s() - ck_last >= 60.0 * ck_minutes) {
                long lost;
                writer_idle(&wr);     /* every record of the chunks so far is in the files and the ring is empty */
                if (wr.failed) FAIL("writing records failed: %s", mq_last_error());
                pthread_mutex_lock(&wr.mu);
                lost = wr.lost;
                pthread_mutex_unlock(&wr.mu);
                if (ckpt_write(ck_path, h, &sink, seed_used, iters_done, lost)) FAIL("could not write the checkpoint %s", ck_path);
                if (diag_path && diag_write(diag_path, h, cfg.grid.nz, pk.view.n_events, pk.view.n_stations, diag_burn_in, diag_batches, iters_done))
                    FAIL("could not write the diagnostics %s", diag_path);
                ck_last = now_s();
            }
        }
    }

    /* best model and diagnostics (src/mcmc_eq.c:1196-1207) */
    writer_idle(&wr);
    if (wr.lost) fprintf(stderr, "warning: %ld decimated record(s) were dropped because a chain's ring was full (-r)\n", wr.lost);
    MQ(mq_snapshot_all(h, 1, write_record, &sink));
    for (c = 0; c < n_chains; c++) mqio_write_counts(sink.out[c], counts + 20 * c);
    if (diag_path && diag_write(diag_path, h, cfg.grid.nz, pk.view.n_events, pk.view.n_stations, diag_burn_in, diag_batches, iters_done))
        FAIL("could not write the diagnostics %s", diag_path);

done:
    if (writer_on) {
        pthread_mutex_lock(&wr.mu);
        wr.stop = 1;
        pthread_cond_broadcast(&wr.cv);
        pthread_mutex_unlock(&wr.mu);
        pthread_join(wr.thread, NULL);
    }
    if (sink.out)
        for (c = 0; c < n_chains; c++)
            if (sink.out[c]) fclose(sink.out[c]);
    free(sink.out); free(sink.written); free(counts); free(ll); free(rms);
    if (h) mq_destroy(h);
    mqio_free_picks(&pk);
    ckpt_free(&ck);
    return rc;
}
