/*
 * ctts_pipeline.c -- ctts_b200_synth_texts (include/ctts_b200.h): the text front end pipelined into the GPU
 * back end.  Plain C + pthreads over the two C-ABI libraries.
 *
 * The reference's ctts_synthesize (ctts.c:3623) does, per utterance, normalisation (:3638-3655), the walk
 * with unit selection (:3689-3871, :1406) and every sample loop in one call on one core.  Here:
 *   planner threads   take small groups of utterances (16) off a shared counter and plan them with the unchanged
 *                     front end (ctts_front_plan_batch_threads(..., 1, ...): re-entrant, the handle is only
 *                     read), at most LOOKAHEAD groups ahead of the device;
 *   the calling thread takes, in order, every plan that is ready -- up to piece_utts utterances -- joins them
 *                     into one piece and submits it to a ctts_gpu_session (asynchronous: several pieces are
 *                     compiled / assembled / copied at any time).  So the first piece reaches the device after
 *                     ~1.5 ms of planning (a group is planned by one thread at ~100 us per utterance, while
 *                     the device->host copy alone consumes an utterance every ~25 us), and once the planners
 *                     are ahead the pieces are large enough to keep the kernels and the copies efficient.
 * Nothing here touches a sample.
 */
#define _POSIX_C_SOURCE 200809L
#include <pthread.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <unistd.h>

#include "ctts_b200.h"

#define LOOKAHEAD 96   /* groups planned ahead of the one being submitted (bounds the memory held in plans) */
#define GROUP_UTTS 16  /* utterances per planner job */

/* ------------------------------------------------------------------ plan cache
 * The plan of an utterance depends on its text alone (and on the front end handle: voice index, config, rules) --
 * the speed travels beside the ops -- so a server that is asked for the same sentences again can skip the text
 * half entirely.  Entries are immutable and never evicted (the cache stops taking entries when it is full), so a
 * reader needs the lock only while it probes the table. */
typedef struct {
    uint64_t hash;
    char* text;
    ctts_plan_op* ops;
    uint32_t n_ops, found, missing;
} cache_entry;

struct ctts_b200_plan_cache {
    pthread_mutex_t mu;
    cache_entry** table;   /* open addressing */
    size_t slots, entries;
    size_t bytes, max_bytes;
    uint64_t hits, misses;
};

static uint64_t fnv1a64(const char* s) {
    uint64_t h = 1469598103934665603ull;
    for (; *s; s++) h = (h ^ (unsigned char)*s) * 1099511628211ull;
    return h;
}

ctts_b200_plan_cache* ctts_b200_plan_cache_create(size_t max_bytes) {
    ctts_b200_plan_cache* c = calloc(1, sizeof *c);
    if (!c) return NULL;
    c->max_bytes = max_bytes;
    c->slots = 1024;
    while (c->slots < max_bytes / 2048) c->slots *= 2;   /* a plan of a 200-character sentence is ~11 KB */
    c->table = calloc(c->slots, sizeof *c->table);
    if (!c->table || pthread_mutex_init(&c->mu, NULL) != 0) {
        free(c->table);
        free(c);
        return NULL;
    }
    return c;
}

void ctts_b200_plan_cache_destroy(ctts_b200_plan_cache* c) {
    if (!c) return;
    for (size_t i = 0; i < c->slots; i++)
        if (c->table[i]) {
            free(c->table[i]->text);
            free(c->table[i]->ops);
            free(c->table[i]);
        }
    free(c->table);
    pthread_mutex_destroy(&c->mu);
    free(c);
}

void ctts_b200_plan_cache_stats(ctts_b200_plan_cache* c, uint64_t* hits, uint64_t* misses, uint64_t* entries, uint64_t* bytes) {
    if (!c) return;
    pthread_mutex_lock(&c->mu);
    if (hits) *hits = c->hits;
    if (misses) *misses = c->misses;
    if (entries) *entries = c->entries;
    if (bytes) *bytes = c->bytes;
    pthread_mutex_unlock(&c->mu);
}

static const cache_entry* cache_lookup(ctts_b200_plan_cache* c, const char* text, uint64_t h) {
    const cache_entry* e = NULL;
    pthread_mutex_lock(&c->mu);
    for (size_t i = h & (c->slots - 1), k = 0; k < c->slots && c->table[i]; i = (i + 1) & (c->slots - 1), k++)
        if (c->table[i]->hash == h && strcmp(c->table[i]->text, text) == 0) {
            e = c->table[i];
            break;
        }
    if (e) c->hits++;
    else c->misses++;
    pthread_mutex_unlock(&c->mu);
    return e;
}

static void cache_insert(ctts_b200_plan_cache* c, const char* text, uint64_t h, const ctts_plan_op* ops, uint32_t n_ops,
                         uint32_t found, uint32_t missing) {
    const size_t need = strlen(text) + 1 + (size_t)n_ops * sizeof *ops + sizeof(cache_entry);
    cache_entry* e = malloc(sizeof *e);
    char* t = strdup(text);
    ctts_plan_op* o = malloc((n_ops ? n_ops : 1) * sizeof *o);
    if (!e || !t || !o) {
        free(e);
        free(t);
        free(o);
        return;
    }
    if (n_ops) memcpy(o, ops, (size_t)n_ops * sizeof *o);
    e->hash = h;
    e->text = t;
    e->ops = o;
    e->n_ops = n_ops;
    e->found = found;
    e->missing = missing;
    int taken = 0;
    pthread_mutex_lock(&c->mu);
    if (c->bytes + need <= c->max_bytes && 2 * (c->entries + 1) <= c->slots) {
        size_t i = h & (c->slots - 1);
        int dup = 0;
        while (c->table[i]) {
            if (c->table[i]->hash == h && strcmp(c->table[i]->text, text) == 0) {
                dup = 1;
                break;
            }
            i = (i + 1) & (c->slots - 1);
        }
        if (!dup) {
            c->table[i] = e;
            c->entries++;
            c->bytes += need;
            taken = 1;
        }
    }
    pthread_mutex_unlock(&c->mu);
    if (!taken) {
        free(e);
        free(t);
        free(o);
    }
}

/* Plan `cnt` texts: cached utterances are copied, the others planned by the front end (one call for all of them)
 * and offered to the cache.  The result is byte-identical to planning all of them. */
static int plan_group(ctts_front* front, ctts_b200_plan_cache* cache, const char* const* texts, const float* speeds,
                      uint32_t cnt, ctts_batch_plan* out, uint32_t* stats) {
    if (!cache) return ctts_front_plan_batch_threads(front, texts, speeds, cnt, 1, out, stats);
    const cache_entry** hit = calloc(cnt ? cnt : 1, sizeof *hit);
    uint64_t* hash = malloc((cnt ? cnt : 1) * sizeof *hash);
    const char** miss_text = malloc((cnt ? cnt : 1) * sizeof *miss_text);
    uint32_t* miss_stats = malloc((cnt ? cnt : 1) * 2 * sizeof *miss_stats);
    uint32_t* begin = malloc(((size_t)cnt + 1) * sizeof *begin);
    float* sp = malloc(((size_t)cnt + 1) * sizeof *sp);
    ctts_batch_plan fresh;
    memset(&fresh, 0, sizeof fresh);
    int rc = (hit && hash && miss_text && miss_stats && begin && sp) ? 0 : CTTS_FRONT_ERR_OUT_OF_MEMORY;
    uint32_t n_miss = 0;
    for (uint32_t u = 0; u < cnt && !rc; u++) {
        if (!texts[u]) {
            rc = CTTS_FRONT_ERR_INVALID_ARG;
            break;
        }
        hash[u] = fnv1a64(texts[u]);
        hit[u] = cache_lookup(cache, texts[u], hash[u]);
        if (!hit[u]) miss_text[n_miss++] = texts[u];
    }
    if (!rc && n_miss) rc = ctts_front_plan_batch_threads(front, miss_text, NULL, n_miss, 1, &fresh, miss_stats);
    ctts_plan_op* ops = NULL;
    if (!rc) {
        uint64_t total = 0;
        for (uint32_t u = 0, m = 0; u < cnt; u++)
            total += hit[u] ? hit[u]->n_ops : fresh.utt_op_begin[m + 1] - fresh.utt_op_begin[m], m += hit[u] ? 0 : 1;
        ops = malloc((total ? total : 1) * sizeof *ops);
        if (!ops || total > 0xffffffffull) rc = CTTS_FRONT_ERR_OUT_OF_MEMORY;
    }
    if (!rc) {
        uint32_t at = 0;
        for (uint32_t u = 0, m = 0; u < cnt; u++) {
            begin[u] = at;
            sp[u] = speeds ? speeds[u] : 1.0f;
            if (hit[u]) {
                if (hit[u]->n_ops) memcpy(ops + at, hit[u]->ops, (size_t)hit[u]->n_ops * sizeof *ops);
                at += hit[u]->n_ops;
                if (stats) {
                    stats[2 * u] = hit[u]->found;
                    stats[2 * u + 1] = hit[u]->missing;
                }
            } else {
                const uint32_t b = fresh.utt_op_begin[m], e = fresh.utt_op_begin[m + 1];
                if (e > b) memcpy(ops + at, fresh.ops + b, (size_t)(e - b) * sizeof *ops);
                cache_insert(cache, texts[u], hash[u], fresh.ops + b, e - b, miss_stats[2 * m], miss_stats[2 * m + 1]);
                at += e - b;
                if (stats) {
                    stats[2 * u] = miss_stats[2 * m];
                    stats[2 * u + 1] = miss_stats[2 * m + 1];
                }
                m++;
            }
        }
        begin[cnt] = at;
        out->n_utts = cnt;
        out->n_ops = at;
        out->utt_op_begin = begin;
        out->speed = sp;
        out->ops = ops;   /* released by ctts_front_plan_free: plain malloc'ed arrays, like the front end's */
    } else {
        free(begin);
        free(sp);
        free(ops);
    }
    if (n_miss) ctts_front_plan_free(&fresh);
    free(hit);
    free(hash);
    free(miss_text);
    free(miss_stats);
    return rc;
}

typedef struct {
    ctts_batch_plan plan;
    int state;   /* 0: not planned, 1: planned, <0: error code */
} piece_slot;

typedef struct {
    ctts_front* front;
    ctts_b200_plan_cache* cache;
    const char* const* texts;
    const float* speeds;
    uint32_t* stats;
    uint32_t n, n_pieces;
    uint32_t* piece_begin;     /* n_pieces + 1: the first pieces are small so that the device starts early */
    piece_slot* slots;
    pthread_mutex_t mu;
    pthread_cond_t cv_ready;   /* a piece became ready */
    pthread_cond_t cv_room;    /* the submitter moved on */
    uint32_t next;             /* next piece to plan */
    uint32_t consumed;         /* pieces the submitter is done with */
    int stop;
    double t0, first_plan_s, all_plans_s;
    uint32_t planned;
} pipeline;

static double now_s(void) {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}

static void* planner(void* arg) {
    pipeline* P = arg;
    for (;;) {
        pthread_mutex_lock(&P->mu);
        while (!P->stop && P->next < P->n_pieces && P->next >= P->consumed + LOOKAHEAD) pthread_cond_wait(&P->cv_room, &P->mu);
        if (P->stop || P->next >= P->n_pieces) {
            pthread_mutex_unlock(&P->mu);
            return NULL;
        }
        const uint32_t i = P->next++;
        pthread_mutex_unlock(&P->mu);
        const uint32_t u0 = P->piece_begin[i], cnt = P->piece_begin[i + 1] - u0;
        ctts_batch_plan pl;
        int rc = plan_group(P->front, P->cache, P->texts + u0, P->speeds ? P->speeds + u0 : NULL, cnt, &pl,
                            P->stats ? P->stats + 2 * (size_t)u0 : NULL);
        pthread_mutex_lock(&P->mu);
        if (rc == 0) {
            P->slots[i].plan = pl;
            P->slots[i].state = 1;
        } else {
            P->slots[i].state = rc < 0 ? rc : -1;
        }
        const double t = now_s() - P->t0;
        if (P->planned++ == 0) P->first_plan_s = t;
        P->all_plans_s = t;
        pthread_cond_broadcast(&P->cv_ready);
        pthread_mutex_unlock(&P->mu);
    }
}

uint64_t ctts_b200_capacity_hint(ctts_front* front, const char* const* texts, const float* speeds, uint32_t n) {
    return ctts_b200_capacity_hint_rate(front, texts, speeds, n, CTTS_PLAN_SAMPLE_RATE);
}

static uint32_t gcd_u32(uint32_t a, uint32_t b) {
    while (b) {
        const uint32_t t = a % b;
        a = b;
        b = t;
    }
    return a;
}

/* the capacity hint of every utterance at output rate hz, in samples (flac == 0) or in bytes of its FLAC file
 * (ctts_gpu_flac_bound, rounded up to 16) */
static uint64_t capacity_hint(ctts_front* front, const char* const* texts, const float* speeds, uint32_t n, uint32_t hz, int flac) {
    if (!front || (n && !texts) || hz == 0) return 0;
    const uint32_t g = gcd_u32(CTTS_PLAN_SAMPLE_RATE, hz), L = hz / g, M = CTTS_PLAN_SAMPLE_RATE / g;
    /* every character yields at most one unit or one pause; pauses are shorter than the longest unit for
     * any sane config, but take the larger of the two anyway */
    uint64_t per_char = ctts_front_max_unit_samples(front);
    if (per_char < 8192) per_char = 8192;
    uint64_t total = 0;
    for (uint32_t u = 0; u < n; u++) {
        uint64_t chars = 8;
        for (const unsigned char* c = (const unsigned char*)(texts[u] ? texts[u] : ""); *c; c++)
            chars += (*c >= '0' && *c <= '9') ? 16 : 1;   /* a digit expands to words ("novecentos e ") */
        uint64_t s = chars * per_char;
        if (speeds && speeds[u] < 1.0f) s *= 2;   /* hop = 128 / speed <= 256 */
        s += 1024;
        s = L == M ? s : (s * L + M - 1) / M + 8;   /* ceil(n L / M) at the output rate, rounded up to 8 */
        total += flac ? (ctts_gpu_flac_bound(s) + 15) & ~15ull : s;
    }
    return total;
}

uint64_t ctts_b200_capacity_hint_rate(ctts_front* front, const char* const* texts, const float* speeds, uint32_t n, uint32_t hz) {
    return capacity_hint(front, texts, speeds, n, hz, 0);
}

uint64_t ctts_b200_capacity_hint_flac(ctts_front* front, const char* const* texts, const float* speeds, uint32_t n, uint32_t hz) {
    return capacity_hint(front, texts, speeds, n, hz, 1);
}

/* what synth_texts delivers: PCM, a FLAC file per utterance, or G.711 bytes of one law */
enum out_kind { OUT_PCM, OUT_FLAC, OUT_ULAW, OUT_ALAW };

/* ctts_b200_synth_texts, ctts_b200_synth_texts_flac and ctts_b200_synth_texts_g711: the same pipeline over a PCM, a
 * FLAC or a G.711 session; byte_out is the output of the last two */
static int synth_texts(ctts_front* front, ctts_gpu_ctx* gpu, const char* const* texts, const float* speeds, uint32_t n,
                       enum out_kind kind, int16_t* pcm_out, uint8_t* byte_out, uint64_t capacity, uint64_t* out_offsets,
                       uint32_t* out_bytes, uint32_t* out_counts, uint32_t* stats, uint64_t* used,
                       const ctts_b200_options* opt, ctts_b200_timing* timing) {
    const int flac = kind == OUT_FLAC;
    if (!front || !gpu || (n && (!texts || !out_offsets || !out_counts || (flac && !out_bytes)))) return CTTS_GPU_ERR_INVALID_ARG;
    pipeline P;
    memset(&P, 0, sizeof P);
    P.front = front;
    P.cache = opt ? opt->cache : NULL;
    P.texts = texts;
    P.speeds = speeds;
    P.stats = stats;
    P.n = n;
    const uint32_t piece_utts = opt && opt->piece_utts ? opt->piece_utts : 192;
    const uint32_t group = piece_utts < GROUP_UTTS ? piece_utts : GROUP_UTTS;
    long cores = sysconf(_SC_NPROCESSORS_ONLN);
    uint32_t T = opt && opt->threads ? opt->threads : (uint32_t)(cores > 1 ? cores - 1 : 1);
    if (T > 32) T = 32;
    if (T < 1) T = 1;
    P.n_pieces = (n + group - 1) / group;
    P.piece_begin = malloc(((size_t)P.n_pieces + 1) * sizeof *P.piece_begin);
    if (!P.piece_begin) return CTTS_GPU_ERR_OUT_OF_MEMORY;
    for (uint32_t i = 0; i <= P.n_pieces; i++) P.piece_begin[i] = (uint64_t)i * group < n ? i * group : n;
    P.t0 = now_s();
    if (T > P.n_pieces) T = P.n_pieces;
    if (T < 1) T = 1;

    ctts_assembly_params prm;
    ctts_front_params(front, &prm);
    ctts_gpu_session* ses = NULL;
    ctts_gpu_chunk_fn on_piece = opt ? opt->on_piece : NULL;
    void* user = opt ? opt->user : NULL;
    int rc = kind == OUT_PCM ? ctts_gpu_session_begin(gpu, &prm, pcm_out, capacity, on_piece, user, &ses)
             : flac          ? ctts_gpu_session_begin_flac(gpu, &prm, byte_out, capacity, on_piece, user, &ses)
                             : ctts_gpu_session_begin_g711(gpu, &prm, kind == OUT_ULAW ? CTTS_GPU_G711_ULAW : CTTS_GPU_G711_ALAW,
                                                           byte_out, capacity, on_piece, user, &ses);
    if (rc) {
        free(P.piece_begin);
        return rc;
    }
    P.slots = calloc(P.n_pieces ? P.n_pieces : 1, sizeof *P.slots);
    pthread_t* tids = calloc(T, sizeof *tids);
    if (!P.slots || !tids) {
        free(P.slots);
        free(tids);
        free(P.piece_begin);
        ctts_gpu_session_end(ses, NULL);
        return CTTS_GPU_ERR_OUT_OF_MEMORY;
    }
    pthread_mutex_init(&P.mu, NULL);
    pthread_cond_init(&P.cv_ready, NULL);
    pthread_cond_init(&P.cv_room, NULL);
    uint32_t started = 0;
    for (; started < T; started++)
        if (pthread_create(&tids[started], NULL, planner, &P) != 0) break;
    double waited = 0.0, all_submitted = 0.0;
    uint32_t n_submitted = 0;
    if (started == 0 && P.n_pieces) rc = CTTS_GPU_ERR_OUT_OF_MEMORY;
    ctts_batch_plan joined;                 /* the piece being submitted when it spans several plans */
    uint32_t* j_begin = NULL;
    float* j_speed = NULL;
    ctts_plan_op* j_ops = NULL;
    size_t j_utts_cap = 0, j_ops_cap = 0;
    for (uint32_t i = 0; i < P.n_pieces && !rc;) {
        const double w0 = now_s();
        pthread_mutex_lock(&P.mu);
        while (P.slots[i].state == 0) pthread_cond_wait(&P.cv_ready, &P.mu);
        /* every further plan that is ready right now, up to piece_utts utterances */
        uint32_t j = i + 1;
        while (j < P.n_pieces && P.slots[j].state != 0 && P.piece_begin[j + 1] - P.piece_begin[i] <= piece_utts) j++;
        int st = 1;
        for (uint32_t k = i; k < j; k++)
            if (P.slots[k].state < 0) st = P.slots[k].state;
        pthread_mutex_unlock(&P.mu);
        waited += now_s() - w0;
        if (st < 0) {
            rc = st;
            break;
        }
        const uint32_t u0 = P.piece_begin[i];
        const ctts_batch_plan* piece = &P.slots[i].plan;
        if (j > i + 1) {
            size_t nu = 0, no = 0;
            for (uint32_t k = i; k < j; k++) {
                nu += P.slots[k].plan.n_utts;
                no += P.slots[k].plan.n_ops;
            }
            if (nu + 1 > j_utts_cap) {
                j_utts_cap = 2 * (nu + 1);
                free(j_begin);
                free(j_speed);
                j_begin = malloc(j_utts_cap * sizeof *j_begin);
                j_speed = malloc(j_utts_cap * sizeof *j_speed);
            }
            if (no + 1 > j_ops_cap) {
                j_ops_cap = 2 * (no + 1);
                free(j_ops);
                j_ops = malloc(j_ops_cap * sizeof *j_ops);
            }
            if (!j_begin || !j_speed || !j_ops || no > 0xffffffffu) {
                rc = CTTS_GPU_ERR_OUT_OF_MEMORY;
                break;
            }
            uint32_t au = 0, ao = 0;
            for (uint32_t k = i; k < j; k++) {
                const ctts_batch_plan* q = &P.slots[k].plan;
                for (uint32_t u = 0; u < q->n_utts; u++) {
                    j_begin[au + u] = ao + q->utt_op_begin[u];
                    j_speed[au + u] = q->speed[u];
                }
                if (q->n_ops) memcpy(j_ops + ao, q->ops, (size_t)q->n_ops * sizeof *j_ops);
                au += q->n_utts;
                ao += q->n_ops;
            }
            j_begin[au] = ao;
            joined.n_utts = au;
            joined.n_ops = ao;
            joined.utt_op_begin = j_begin;
            joined.speed = j_speed;
            joined.ops = j_ops;
            piece = &joined;
        }
        rc = kind == OUT_PCM ? ctts_gpu_session_submit(ses, piece, out_offsets + u0, out_counts + u0)
             : flac          ? ctts_gpu_session_submit_flac(ses, piece, out_offsets + u0, out_bytes + u0, out_counts + u0)
                             : ctts_gpu_session_submit_g711(ses, piece, out_offsets + u0, out_counts + u0);
        for (uint32_t k = i; k < j; k++) {
            ctts_front_plan_free(&P.slots[k].plan);   /* the session keeps nothing of the plan */
            P.slots[k].state = 2;
        }
        pthread_mutex_lock(&P.mu);
        P.consumed = j;
        pthread_cond_broadcast(&P.cv_room);
        pthread_mutex_unlock(&P.mu);
        all_submitted = now_s() - P.t0;
        n_submitted++;
        i = j;
    }
    free(j_begin);
    free(j_speed);
    free(j_ops);
    pthread_mutex_lock(&P.mu);
    P.stop = 1;
    pthread_cond_broadcast(&P.cv_room);
    pthread_mutex_unlock(&P.mu);
    for (uint32_t t = 0; t < started; t++) pthread_join(tids[t], NULL);
    for (uint32_t i = 0; i < P.n_pieces; i++)
        if (P.slots[i].state == 1) ctts_front_plan_free(&P.slots[i].plan);
    const int rc_end = ctts_gpu_session_end(ses, used);
    if (!rc) rc = rc_end;
    if (timing) {
        timing->first_plan_s = P.first_plan_s;
        timing->all_plans_s = P.all_plans_s;
        timing->all_submitted_s = all_submitted;
        timing->done_s = now_s() - P.t0;
        timing->wait_for_plans_s = waited;
        timing->pieces = n_submitted;
    }
    pthread_mutex_destroy(&P.mu);
    pthread_cond_destroy(&P.cv_ready);
    pthread_cond_destroy(&P.cv_room);
    free(P.slots);
    free(tids);
    free(P.piece_begin);
    return rc;
}

int ctts_b200_synth_texts(ctts_front* front, ctts_gpu_ctx* gpu, const char* const* texts, const float* speeds,
                          uint32_t n, int16_t* pcm_out, uint64_t capacity, uint64_t* out_offsets,
                          uint32_t* out_counts, uint32_t* stats, uint64_t* samples_used,
                          const ctts_b200_options* opt, ctts_b200_timing* timing) {
    return synth_texts(front, gpu, texts, speeds, n, OUT_PCM, pcm_out, NULL, capacity, out_offsets, NULL, out_counts, stats,
                       samples_used, opt, timing);
}

int ctts_b200_synth_texts_flac(ctts_front* front, ctts_gpu_ctx* gpu, const char* const* texts, const float* speeds,
                               uint32_t n, uint8_t* out, uint64_t capacity_bytes, uint64_t* out_offsets,
                               uint32_t* out_bytes, uint32_t* out_counts, uint32_t* stats, uint64_t* bytes_used,
                               const ctts_b200_options* opt, ctts_b200_timing* timing) {
    return synth_texts(front, gpu, texts, speeds, n, OUT_FLAC, NULL, out, capacity_bytes, out_offsets, out_bytes,
                       out_counts, stats, bytes_used, opt, timing);
}

int ctts_b200_synth_texts_g711(ctts_front* front, ctts_gpu_ctx* gpu, int law, const char* const* texts,
                               const float* speeds, uint32_t n, uint8_t* out, uint64_t capacity_bytes,
                               uint64_t* out_offsets, uint32_t* out_counts, uint32_t* stats, uint64_t* bytes_used,
                               const ctts_b200_options* opt, ctts_b200_timing* timing) {
    if (law != CTTS_GPU_G711_ULAW && law != CTTS_GPU_G711_ALAW) return CTTS_GPU_ERR_INVALID_ARG;
    return synth_texts(front, gpu, texts, speeds, n, law == CTTS_GPU_G711_ULAW ? OUT_ULAW : OUT_ALAW, NULL, out,
                       capacity_bytes, out_offsets, NULL, out_counts, stats, bytes_used, opt, timing);
}
