/*
 * ctts_b200 -- the `ctts synth` command line (ctts.c:3970-4030) over the B200 back end, in the
 * reference's own language: plain C on top of the two C-ABI libraries, no Python, no CUDA headers.
 *
 *   ctts_b200 synth <database.db> "text" <output.wav|output.flac> [speed] [rate] [lufs=<target> [dbtp=<ceiling>]]
 *                   [g711=ulaw|alaw]
 *   ctts_b200 synth-batch <database.db> <texts.tsv> <out_dir> [rate] [flac] [lufs=<target> [dbtp=<ceiling>]]
 *                         [g711=ulaw|alaw]                                                 lines: speed<TAB>text
 *
 * rate: output sample rate in Hz (default 22050, the voice's own; ctts_gpu_set_output_rate lists the others),
 * written into the WAV header.  An output name ending in ".flac", or synth-batch's "flac", writes lossless FLAC files
 * encoded on the device (ctts_b200_synth_texts_flac) instead of 16-bit WAV.  lufs=<target> normalizes every utterance
 * to <target> LUFS (ITU-R BS.1770-4, in [-60, -5]) with its sample peak held to -1 dBFS (ctts_gpu_set_loudness);
 * dbtp=<ceiling> next to it holds the true peak to <ceiling> dBTP instead (in [-20, 0], ctts_gpu_set_loudness_true_peak).
 * g711=ulaw or g711=alaw writes 8-bit G.711 .wav files (format tag 7 or 6, with a fact chunk) encoded on the device
 * (ctts_b200_synth_texts_g711), for telephony: with rate 8000 they are what IVR systems play.  It does not combine with
 * FLAC output.  The trailing options may come in any order.
 *
 * Like the reference it reads config.yaml and normalization.csv from the working directory
 * (ctts.c:3990, :3636), clamps the speed to [0.5, 2.0] (ctts.c:3976-3981) and takes default_speed
 * from the config when none is given (ctts.c:3993).  ctts_b200_synthesize_batch() below is the
 * glue INTEGRATION.md describes (texts -> ctts_b200_synth_texts: planner threads feeding a device
 * session -> per-utterance PCM); everything that touches samples runs on the GPU, and without a CUDA
 * device it fails.
 */
#include <errno.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>

#include "ctts_b200.h"
#include "g711_wav.h"

#define SAMPLE_RATE CTTS_PLAN_SAMPLE_RATE

/* what the files hold: 16-bit PCM WAV, G.711 WAV of either law, or FLAC */
typedef enum { OUT_WAV = 0, OUT_ULAW = CTTS_GPU_G711_ULAW, OUT_ALAW = CTTS_GPU_G711_ALAW, OUT_FLAC } out_kind;

/* the loudness options: lufs = 0 without lufs=; true_peak when dbtp= was given */
typedef struct {
    float lufs, dbtp;
    int true_peak;
} loudness_arg;

typedef struct {
    void* db;
    size_t db_size;
    ctts_front_config cfg;
    ctts_front* front;
    ctts_gpu_ctx* gpu;
    uint32_t rate;   /* output sample rate */
} engine;

static void engine_close(engine* e) {
    if (e->gpu) ctts_gpu_free(e->gpu);
    if (e->front) ctts_front_close(e->front);
    free(e->db);
    memset(e, 0, sizeof *e);
}

/* ctts_init (ctts.c:1117) + ctts_load_config("config.yaml") + the rule table, for both halves */
static int engine_open(engine* e, const char* db_path, uint32_t rate, const loudness_arg* ld) {
    memset(e, 0, sizeof *e);
    FILE* f = fopen(db_path, "rb");
    if (!f) return -1;
    fseek(f, 0, SEEK_END);
    long n = ftell(f);
    fseek(f, 0, SEEK_SET);
    if (n <= 0) { fclose(f); return -1; }
    e->db = malloc((size_t)n);
    if (!e->db || fread(e->db, 1, (size_t)n, f) != (size_t)n) { fclose(f); free(e->db); e->db = NULL; return -1; }
    fclose(f);
    e->db_size = (size_t)n;
    ctts_front_config_defaults(&e->cfg);
    ctts_front_config_load(&e->cfg, "config.yaml");
    FILE* nf = fopen("normalization.csv", "rb");
    if (nf) fclose(nf);
    int rc = ctts_front_open(&e->front, e->db, e->db_size, &e->cfg, nf ? "normalization.csv" : NULL);
    if (rc) { engine_close(e); return rc; }
    const char* dev = getenv("CTTS_GPU_DEVICE");
    rc = ctts_gpu_init(&e->gpu, e->db, e->db_size, dev ? atoi(dev) : 0);
    if (rc) {
        fprintf(stderr, "ctts_gpu_init: %d (no CPU fallback)\n", rc);
        engine_close(e);
        return rc;
    }
    rc = ctts_gpu_set_output_rate(e->gpu, rate);
    if (rc) {
        fprintf(stderr, "output rate %u Hz: %s\n", rate, ctts_gpu_last_error(e->gpu));
        engine_close(e);
        return rc;
    }
    if (ld->lufs != 0.0f && (rc = ld->true_peak ? ctts_gpu_set_loudness_true_peak(e->gpu, ld->lufs, ld->dbtp)
                                                : ctts_gpu_set_loudness(e->gpu, ld->lufs, -1.0f)) != 0) {
        fprintf(stderr, "loudness target %g LUFS: %s\n", (double)ld->lufs, ctts_gpu_last_error(e->gpu));
        engine_close(e);
        return rc;
    }
    e->rate = rate;
    return 0;
}

/* Optional last arguments lufs=<target>, dbtp=<ceiling> and g711=ulaw|alaw, in any order (after the output argument):
 * taken off the argument list.  ld->lufs = 0 without lufs=; *kind = OUT_WAV without g711=, else OUT_ULAW or OUT_ALAW.
 * -1 when a value is not a number or not a law, an option repeats or dbtp= comes without lufs=
 * (any other value is checked by ctts_gpu_set_loudness(_true_peak)). */
static int take_options(int* argc, char** argv, loudness_arg* ld, out_kind* kind) {
    memset(ld, 0, sizeof *ld);
    *kind = OUT_WAV;
    int have_lufs = 0;
    while (*argc >= 6) {   /* behind the required arguments only */
        const char* a = argv[*argc - 1];
        if (strncmp(a, "g711=", 5) == 0) {
            if (*kind) return -1;
            *kind = strcmp(a + 5, "ulaw") == 0 ? OUT_ULAW : strcmp(a + 5, "alaw") == 0 ? OUT_ALAW : OUT_WAV;
            if (!*kind) return -1;
            (*argc)--;
            continue;
        }
        const int is_lufs = strncmp(a, "lufs=", 5) == 0, is_dbtp = strncmp(a, "dbtp=", 5) == 0;
        if (!is_lufs && !is_dbtp) break;
        if (is_lufs ? have_lufs : ld->true_peak) return -1;
        char* end = NULL;
        const float v = strtof(a + 5, &end);
        if (!a[5] || !end || *end != '\0') return -1;
        if (is_lufs) {
            ld->lufs = v;
            have_lufs = 1;
        } else {
            ld->dbtp = v;
            ld->true_peak = 1;
        }
        (*argc)--;
    }
    return ld->true_peak && !have_lufs ? -1 : 0;
}

/* N texts -> N PCM spans (or N .flac files, or N spans of G.711 codes) of one pinned buffer through
 * ctts_b200_synth_texts(_flac, _g711) (the front end's planner threads feed the device piece by piece): r->out (release
 * with ctts_gpu_host_free), r->off[u], r->bytes[u] (FLAC: file sizes) and r->cnt[u] (malloc'ed, n entries each); stats
 * may be NULL (2n: found, missing).  on_chunk (may be NULL) is called as soon as a range of utterances is in host
 * memory; it finds the arrays through r, which is filled before the device starts. */
typedef struct {
    void* out;   /* int16_t PCM, the FLAC files, or the G.711 codes */
    uint64_t* off;
    uint32_t* bytes;
    uint32_t* cnt;
} batch_result;

static void result_free(batch_result* r) {
    ctts_gpu_host_free(r->out);
    free(r->off);
    free(r->bytes);
    free(r->cnt);
    memset(r, 0, sizeof *r);
}

static int ctts_b200_synthesize_batch(engine* e, const char* const* texts, const float* speeds, uint32_t n, out_kind kind,
                                      batch_result* r, uint32_t* stats, ctts_gpu_chunk_fn on_chunk, void* user) {
    /* replaces the SampleBuffer growth policy; G.711: the sample capacity, read as bytes */
    const uint64_t cap = kind == OUT_FLAC ? ctts_b200_capacity_hint_flac(e->front, texts, speeds, n, e->rate)
                                          : ctts_b200_capacity_hint_rate(e->front, texts, speeds, n, e->rate);
    r->off = malloc(sizeof *r->off * ((size_t)n + 1));
    r->bytes = calloc(n ? n : 1, sizeof *r->bytes);
    r->cnt = calloc(n ? n : 1, sizeof *r->cnt);
    r->out = ctts_gpu_host_alloc((kind == OUT_WAV ? sizeof(int16_t) : 1) * (cap ? cap : 16));
    ctts_b200_options opt;
    memset(&opt, 0, sizeof opt);
    opt.on_piece = on_chunk;
    opt.user = user;
    int rc = !r->off || !r->bytes || !r->cnt || !r->out ? CTTS_GPU_ERR_OUT_OF_MEMORY
           : kind == OUT_FLAC ? ctts_b200_synth_texts_flac(e->front, e->gpu, texts, speeds, n, r->out, cap, r->off, r->bytes, r->cnt, stats, NULL, &opt, NULL)
           : kind != OUT_WAV  ? ctts_b200_synth_texts_g711(e->front, e->gpu, kind, texts, speeds, n, r->out, cap, r->off, r->cnt, stats, NULL, &opt, NULL)
                              : ctts_b200_synth_texts(e->front, e->gpu, texts, speeds, n, r->out, cap, r->off, r->cnt, stats, NULL, &opt, NULL);
    if (rc) {
        fprintf(stderr, "synthesis failed: %d %s\n", rc, ctts_gpu_last_error(e->gpu));
        result_free(r);
    }
    return rc;
}

/* utterance u of r as the file `path`: a WAV file as ctts_write_wav (ctts.c:809) writes it (44-byte RIFF/WAVE header,
 * PCM, mono, 16 bit), a G.711 .wav file (g711_wav.h: the header, the codes and a pad byte when the count is odd) or the
 * .flac file */
static int write_utterance(const char* path, out_kind kind, const batch_result* r, uint32_t u, uint32_t rate) {
    FILE* f = fopen(path, "wb");
    if (!f) return -1;
    const uint8_t* bytes = (const uint8_t*)r->out + r->off[u];
    const uint32_t count = r->cnt[u];
    int ok = 1;
    switch (kind) {
    case OUT_WAV: {
        const uint32_t data = count * (uint32_t)sizeof(int16_t), riff = 36 + data, fmt = 16, sr = rate, br = rate * 2;
        const uint16_t pcm = 1, ch = 1, align = 2, bits = 16;
        fwrite("RIFF", 1, 4, f); fwrite(&riff, 4, 1, f); fwrite("WAVE", 1, 4, f);
        fwrite("fmt ", 1, 4, f); fwrite(&fmt, 4, 1, f);
        fwrite(&pcm, 2, 1, f); fwrite(&ch, 2, 1, f); fwrite(&sr, 4, 1, f); fwrite(&br, 4, 1, f);
        fwrite(&align, 2, 1, f); fwrite(&bits, 2, 1, f);
        fwrite("data", 1, 4, f); fwrite(&data, 4, 1, f);
        fwrite((const int16_t*)r->out + r->off[u], sizeof(int16_t), count, f);
        break;
    }
    case OUT_ULAW:
    case OUT_ALAW: {
        uint8_t h[G711_WAV_HEADER_BYTES];
        const uint8_t pad = 0;
        g711_wav_header(h, kind, rate, count);
        ok = fwrite(h, 1, sizeof h, f) == sizeof h && fwrite(bytes, 1, count, f) == count;
        if (count & 1) ok = ok && fwrite(&pad, 1, 1, f) == 1;
        break;
    }
    case OUT_FLAC: ok = fwrite(bytes, 1, r->bytes[u], f) == r->bytes[u]; break;
    }
    return fclose(f) == 0 && ok ? 0 : -1;
}

static int ends_with(const char* s, const char* tail) {
    const size_t a = strlen(s), b = strlen(tail);
    return a >= b && strcmp(s + a - b, tail) == 0;
}

static float clamp_speed(float s) { return s < 0.5f ? 0.5f : s > 2.0f ? 2.0f : s; }

/* an output rate argument: digits only, else 0 (rejected by ctts_gpu_set_output_rate) */
static uint32_t parse_rate(const char* a) {
    char* end = NULL;
    const unsigned long v = strtoul(a, &end, 10);
    return (end && *end == 0 && end != a && v <= 0xffffffffu) ? (uint32_t)v : 0;
}

static int cmd_synth(int argc, char** argv) {
    loudness_arg ld;
    out_kind kind;
    if (take_options(&argc, argv, &ld, &kind) || argc < 5 || argc > 7 || (kind && ends_with(argv[4], ".flac"))) {
        fprintf(stderr, "Usage: %s synth <database.db> \"text\" <output.wav|output.flac> [speed] [rate] [lufs=<target> [dbtp=<ceiling>]] [g711=ulaw|alaw]\n"
                        "       (g711= writes a G.711 .wav file, not FLAC)\n", argv[0]);
        return 1;
    }
    float speed = 1.0f;
    if (argc > 5) speed = clamp_speed(strtof(argv[5], NULL));
    const uint32_t rate = argc > 6 ? parse_rate(argv[6]) : SAMPLE_RATE;
    engine e;
    if (engine_open(&e, argv[2], rate, &ld)) {
        fprintf(stderr, "Failed to load database: %s\n", argv[2]);
        return 1;
    }
    if (argc <= 5 && e.cfg.default_speed != 1.0f) speed = e.cfg.default_speed;
    printf("Loaded database with %u units\n", ctts_front_unit_count(e.front));
    const char* texts[1] = {argv[3]};
    if (ends_with(argv[4], ".flac")) kind = OUT_FLAC;
    batch_result r;
    uint32_t stats[2] = {0, 0};
    if (ctts_b200_synthesize_batch(&e, texts, &speed, 1, kind, &r, stats, NULL, NULL)) { engine_close(&e); return 1; }
    printf("Synthesized %u samples (%.2f seconds)\n", r.cnt[0], (float)r.cnt[0] / (float)e.rate);
    printf("Units found: %u, missing: %u\n", stats[0], stats[1]);
    int rc = write_utterance(argv[4], kind, &r, 0, e.rate);
    if (rc) fprintf(stderr, "Failed to write %s: %s\n", kind == OUT_FLAC ? "FLAC" : "WAV", argv[4]);
    else printf("Written to %s\n", argv[4]);
    result_free(&r);
    engine_close(&e);
    return rc ? 1 : 0;
}

/* synth-batch writes every WAV file as soon as its utterance has arrived (the device is still
 * working on later ones): state shared with the chunk callback */
typedef struct {
    const char* dir;
    uint32_t rate;
    uint32_t base;   /* first utterance of the group being synthesised */
    out_kind kind;
    const batch_result* r;
    double seconds;
    int rc;
} wav_sink;

static void write_chunk(void* user, uint32_t u0, uint32_t u1) {
    wav_sink* w = user;
    for (uint32_t u = u0; u < u1 && !w->rc; u++) {
        char path[4096];
        snprintf(path, sizeof path, "%s/%06u.%s", w->dir, w->base + u, w->kind == OUT_FLAC ? "flac" : "wav");
        w->rc = write_utterance(path, w->kind, w->r, u, w->rate);
        w->seconds += (double)w->r->cnt[u] / w->rate;
    }
}

static int cmd_synth_batch(int argc, char** argv) {
    loudness_arg ld;
    out_kind kind;
    if (take_options(&argc, argv, &ld, &kind) || argc < 5 || argc > 7 || (argc == 7 && strcmp(argv[6], "flac") != 0) ||
        (kind && argc == 7)) {
        fprintf(stderr, "Usage: %s synth-batch <database.db> <texts.tsv> <out_dir> [rate] [flac] [lufs=<target> [dbtp=<ceiling>]] [g711=ulaw|alaw]\n"
                        "       (g711= writes G.711 .wav files, not FLAC)\n", argv[0]);
        return 1;
    }
    const uint32_t rate = argc > 5 ? parse_rate(argv[5]) : SAMPLE_RATE;
    if (argc == 7) kind = OUT_FLAC;
    FILE* f = fopen(argv[3], "rb");
    if (!f) { fprintf(stderr, "cannot read %s\n", argv[3]); return 1; }
    char** texts = NULL;
    float* speeds = NULL;
    uint32_t n = 0, cap = 0;
    char* line = NULL;
    size_t lcap = 0;
    ssize_t len;
    while ((len = getline(&line, &lcap, f)) > 0) {
        while (len > 0 && (line[len - 1] == '\n' || line[len - 1] == '\r')) line[--len] = 0;
        if (len == 0) continue;
        char* tab = strchr(line, '\t');
        if (!tab) continue;
        *tab = 0;
        if (n == cap) {
            cap = cap ? 2 * cap : 1024;
            texts = realloc(texts, cap * sizeof *texts);
            speeds = realloc(speeds, cap * sizeof *speeds);
            if (!texts || !speeds) { fprintf(stderr, "out of memory\n"); return 1; }
        }
        speeds[n] = clamp_speed(strtof(line, NULL));
        texts[n] = strdup(tab + 1);
        n++;
    }
    free(line);
    fclose(f);
    engine e;
    if (engine_open(&e, argv[2], rate, &ld)) {
        fprintf(stderr, "Failed to load database: %s\n", argv[2]);
        return 1;
    }
    if (mkdir(argv[4], 0777) != 0 && errno != EEXIST) { fprintf(stderr, "cannot create %s\n", argv[4]); engine_close(&e); return 1; }
    batch_result r;
    wav_sink sink = {argv[4], e.rate, 0, kind, &r, 0.0, 0};
    /* groups of 1024 utterances: the pinned buffer is sized from the texts alone (ctts_b200_capacity_hint) */
    int rc = 0;
    for (uint32_t g0 = 0; g0 < n && !rc; g0 += 1024) {
        const uint32_t gn = n - g0 < 1024 ? n - g0 : 1024;
        sink.base = g0;
        rc = ctts_b200_synthesize_batch(&e, (const char* const*)texts + g0, speeds + g0, gn, kind, &r, NULL, write_chunk, &sink);
        if (!rc) {
            rc = sink.rc;
            result_free(&r);
        }
    }
    if (rc) fprintf(stderr, "Failed to write %s files into %s\n", kind == OUT_FLAC ? "FLAC" : "WAV", argv[4]);
    else printf("Synthesized %u utterances (%.1f seconds of audio) into %s\n", n, sink.seconds, argv[4]);
    for (uint32_t u = 0; u < n; u++) free(texts[u]);
    free(texts);
    free(speeds);
    engine_close(&e);
    return rc ? 1 : 0;
}

int main(int argc, char** argv) {
    if (argc >= 2 && strcmp(argv[1], "synth") == 0) return cmd_synth(argc, argv);
    if (argc >= 2 && strcmp(argv[1], "synth-batch") == 0) return cmd_synth_batch(argc, argv);
    fprintf(stderr, "Usage: %s synth <database.db> \"text\" <output.wav|output.flac> [speed] [rate] [lufs=<target> [dbtp=<ceiling>]] [g711=ulaw|alaw]\n"
                    "       %s synth-batch <database.db> <texts.tsv> <out_dir> [rate] [flac] [lufs=<target> [dbtp=<ceiling>]] [g711=ulaw|alaw]\n",
            argv[0], argv[0]);
    return 1;
}
