/*
 * host.c — C host layer of the B200-native Ed25519 / X25519 engine.
 *
 * Implements the public API of include/eddsa.h (the reference's /root/reference/lib/eddsa.h:44-114
 * surface, single operations executed as batches of one) and the batch C-ABI of
 * include/eddsa_batch.h on top of the CUDA launchers in kernels_*.cu.
 *
 *   - one context per device: NSLOT streams, page-locked staging buffers, device buffers, a
 *     stream-ordered memory pool for kernel scratch and a worker thread; created lazily;
 *   - a host-buffer batch is sharded by contiguous index ranges over the devices (one long-lived
 *     worker thread per device, no inter-device traffic) and each shard is streamed in chunks:
 *     stage -> H2D -> kernel -> D2H -> unstage, the slots rotating so copies of one chunk overlap
 *     the kernel of another; caller memory that is already page-locked is used directly;
 *   - staging memory that carried secret keys (or secret outputs) is zeroed as soon as the chunk
 *     retires, on the host and on the device (the reference scrubs after every secret-key call:
 *     /root/reference/lib/ed25519-sha512.c:77,136,255, x25519.c:208,221);
 *   - no CPU fallback anywhere: without a working device the batch calls return an error and the
 *     void single-operation calls abort().
 */
#define _GNU_SOURCE
#include <cuda_runtime_api.h>
#include <pthread.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

#include "eddsa.h"
#include "eddsa_batch.h"
#include "edg_internal.h"

/* Weak: the host layer also links against sets of launchers that only implement the reference's verify rule (the mock kernels
 * of the test suite's CUDA runtime simulator).  There the address is NULL and the other rules are refused (bad_policy);
 * kernels_verify.cu always defines it. */
#pragma weak edg_launch_verify_policy

#define EDG_MAX_DEV 16
#define EDG_NSLOT 3
#define EDG_ALIGN 256
#define EDG_COPY_HELPERS 3              /* helper threads for big staging copies, at most; g_copy_helpers of them are used */

typedef enum { OP_GENPUB, OP_SIGN, OP_VERIFY, OP_X25519, OP_X25519_BASE, OP_PK_CONV, OP_SK_CONV, OP_FE_TEST, OP_SC_TEST } edg_op_t;

/* operations whose first input array is a secret key / scalar, and those whose OUTPUT is secret as well */
static int op_secret_in(edg_op_t op) { return op == OP_GENPUB || op == OP_SIGN || op == OP_X25519 || op == OP_X25519_BASE || op == OP_SK_CONV; }
static int op_secret_out(edg_op_t op) { return op == OP_X25519 || op == OP_SK_CONV; }

typedef struct {
    edg_op_t op;
    size_t n;
    int nin;
    const uint8_t *in[3];
    size_t in_item[3];
    int has_msgs;
    const uint8_t *msgs;
    const size_t *off;
    size_t fixed_len;
    uint8_t *out;
    size_t out_item;
    int policy;                                 /* verify: EDDSA_B200_VERIFY_* */
} edg_job_t;

struct shard;
typedef struct {
    int dev, sm_count, ready;
    pthread_mutex_t lock; /* the host-buffer pipeline of this device is exclusive */
    cudaStream_t stream[EDG_NSLOT];
    cudaEvent_t done[EDG_NSLOT];
    cudaStream_t kstream;                       /* verify: all kernels of the host-buffer pipeline run here, one after the other */
    cudaEvent_t in_ready[EDG_NSLOT], k_done[EDG_NSLOT];
    size_t verify_pass;                         /* signatures per full pass of the verify kernels (whole waves) */
    size_t verify_wave;                         /* one wave of resident threads of the loop kernel */
    uint8_t *h_in[EDG_NSLOT], *h_out[EDG_NSLOT];
    uint8_t *d_in[EDG_NSLOT], *d_out[EDG_NSLOT];
    size_t in_cap, out_cap;
    cudaMemPool_t pool;                         /* kernel scratch (verify records, sign nonces): stream-ordered, reused without synchronising */
    void *wtab;                                 /* verify: window tables of the base point, built at context creation */
    void *comb;                                 /* fixed-base comb table, built at context creation */
    /* worker thread: runs the shards of multi-device jobs on this device */
    pthread_t worker;
    int worker_on, worker_stop;
    pthread_mutex_t q_lock;
    pthread_cond_t q_cond;
    struct shard *q_head, *q_tail;
} edg_dev_t;

typedef struct { pthread_mutex_t m; pthread_cond_t cv; int pending; } job_sync_t;
typedef struct shard { edg_dev_t *c; const edg_job_t *j; size_t lo, hi; int rc; char err[256]; job_sync_t *sync; struct shard *next; } shard_t;

static edg_dev_t g_dev[EDG_MAX_DEV]; /* indexed by CUDA device ordinal */
static int g_list[EDG_MAX_DEV];      /* devices the host-buffer API shards over */
static int g_nlist = 0, g_nactive = 0, g_init_rc = 0, g_no_scrub = 0;
static int g_copy_helpers = 0;       /* helper threads for big staging copies (stage_copy): set once in global_init */
static size_t g_chunk_bytes = (size_t)128 << 20;
static pthread_once_t g_once = PTHREAD_ONCE_INIT;
static pthread_mutex_t g_ctx_lock = PTHREAD_MUTEX_INITIALIZER;
static unsigned long long g_launches = 0;
static __thread char t_err[256];

static int fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(t_err, sizeof t_err, fmt, ap);
    va_end(ap);
    return code ? code : EDDSA_B200_EINVAL;
}

#define CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { \
    rc = fail((int)e_, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); goto out; } } while (0)

static size_t align_up(size_t x) { return (x + EDG_ALIGN - 1) & ~(size_t)(EDG_ALIGN - 1); }

static int env_int(const char *name, int dflt)
{
    const char *v = getenv(name);
    return v && *v ? atoi(v) : dflt;
}

static void global_init(void)
{
    int count = 0, i;
    const char *env = getenv("EDDSA_B200_DEVICES");
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count < 1) {
        g_init_rc = e != cudaSuccess ? (int)e : (int)cudaErrorNoDevice;
        return;
    }
    if (count > EDG_MAX_DEV) count = EDG_MAX_DEV;
    for (i = 0; i < EDG_MAX_DEV; i++) {
        g_dev[i].dev = i;
        pthread_mutex_init(&g_dev[i].lock, NULL);
        pthread_mutex_init(&g_dev[i].q_lock, NULL);
        pthread_cond_init(&g_dev[i].q_cond, NULL);
    }
    if (env && strchr(env, ',')) {
        char buf[128], *tok, *save = NULL;
        snprintf(buf, sizeof buf, "%s", env);
        for (tok = strtok_r(buf, ",", &save); tok && g_nlist < EDG_MAX_DEV; tok = strtok_r(NULL, ",", &save)) {
            int d = atoi(tok);
            if (d >= 0 && d < count) g_list[g_nlist++] = d;
        }
    } else {
        int want = env && *env ? atoi(env) : count;
        if (want < 1 || want > count) want = count;
        for (i = 0; i < want; i++) g_list[g_nlist++] = i;
    }
    if (g_nlist == 0) g_list[g_nlist++] = 0;
    __atomic_store_n(&g_nactive, g_nlist, __ATOMIC_RELEASE);
    if (env_int("EDDSA_B200_CHUNK_MB", 0) > 0) g_chunk_bytes = (size_t)env_int("EDDSA_B200_CHUNK_MB", 0) << 20;
    if (env_int("EDDSA_B200_DEBUG_FULL_SCALARS", 0) > 0) edg_verify_debug_full_scalars(1);
    if (env_int("EDDSA_B200_VERIFY_WAVES", 0) > 0) edg_verify_set_waves(env_int("EDDSA_B200_VERIFY_WAVES", 0));
    g_no_scrub = env_int("EDDSA_B200_DEBUG_NO_SCRUB", 0) > 0;   /* test hook: negative control of the staging-scrub test */
    /* helpers for big staging copies: a quarter of the host's cores per visible device, at most 3 — a host shared by one
     * process per GPU (or by eight device workers of this process, which already copy in parallel) gets fewer or none */
    g_copy_helpers = (int)(sysconf(_SC_NPROCESSORS_ONLN) / (4 * (long)count));
    if (getenv("EDDSA_B200_COPY_THREADS")) g_copy_helpers = env_int("EDDSA_B200_COPY_THREADS", 0);
    if (g_copy_helpers > EDG_COPY_HELPERS) g_copy_helpers = EDG_COPY_HELPERS;
    if (g_copy_helpers < 0) g_copy_helpers = 0;
}

static int engine_ready(void)
{
    pthread_once(&g_once, global_init);
    if (g_init_rc) return fail(g_init_rc, "no usable CUDA device: %s", cudaGetErrorString((cudaError_t)g_init_rc));
    return 0;
}

/* undo a (possibly partially built) context; its device is current */
static void dev_teardown(edg_dev_t *c)
{
    int i;
    for (i = 0; i < EDG_NSLOT; i++) {
        if (c->stream[i]) cudaStreamDestroy(c->stream[i]);
        if (c->done[i]) cudaEventDestroy(c->done[i]);
        if (c->in_ready[i]) cudaEventDestroy(c->in_ready[i]);
        if (c->k_done[i]) cudaEventDestroy(c->k_done[i]);
        c->stream[i] = NULL; c->done[i] = c->in_ready[i] = c->k_done[i] = NULL;
    }
    if (c->kstream) cudaStreamDestroy(c->kstream);
    if (c->wtab) cudaFree(c->wtab);
    if (c->comb) cudaFree(c->comb);
    if (c->pool) cudaMemPoolDestroy(c->pool);
    c->kstream = NULL; c->wtab = c->comb = NULL; c->pool = NULL;
}

/* per-device context without staging buffers (enough for the _dev API) */
static int dev_basic(int dev, edg_dev_t **out_ctx)
{
    edg_dev_t *c;
    int rc = engine_ready();
    if (rc) return rc;
    if (dev < 0 || dev >= EDG_MAX_DEV) return fail(EDDSA_B200_EINVAL, "device ordinal %d out of range", dev);
    c = &g_dev[dev];
    if (!__atomic_load_n(&c->ready, __ATOMIC_ACQUIRE)) {
        pthread_mutex_lock(&g_ctx_lock);
        if (!c->ready) {
            int prev = -1, sms = 0, i;
            struct cudaMemPoolProps props;
            unsigned long long keep = ~0ULL;
            cudaGetDevice(&prev);
            CU(cudaSetDevice(dev));
            CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
            c->sm_count = sms;
            rc = edg_kernels_init();
            if (rc) { rc = fail(rc, "kernel attribute setup failed: %s", cudaGetErrorString((cudaError_t)rc)); goto out; }
            for (i = 0; i < EDG_NSLOT; i++) {
                CU(cudaStreamCreateWithFlags(&c->stream[i], cudaStreamNonBlocking));
                CU(cudaEventCreateWithFlags(&c->done[i], cudaEventDisableTiming));
                CU(cudaEventCreateWithFlags(&c->in_ready[i], cudaEventDisableTiming));
                CU(cudaEventCreateWithFlags(&c->k_done[i], cudaEventDisableTiming));
            }
            CU(cudaStreamCreateWithFlags(&c->kstream, cudaStreamNonBlocking));
            c->verify_pass = edg_verify_pass(sms);
            c->verify_wave = c->verify_pass / edg_verify_waves();
            /* scratch pool: freed blocks stay in the pool (no trimming at synchronisation points), so a steady
             * stream of calls allocates nothing after the first one */
            memset(&props, 0, sizeof props);
            props.allocType = cudaMemAllocationTypePinned;
            props.handleTypes = cudaMemHandleTypeNone;
            props.location.type = cudaMemLocationTypeDevice;
            props.location.id = dev;
            CU(cudaMemPoolCreate(&c->pool, &props));
            CU(cudaMemPoolSetAttribute(c->pool, cudaMemPoolAttrReleaseThreshold, &keep));
            CU(cudaMalloc(&c->wtab, edg_verify_table_bytes()));
            rc = edg_verify_table_init(c->wtab, c->stream[0]);
            if (rc) { rc = fail(rc, "window table build failed: %s", cudaGetErrorString((cudaError_t)rc)); goto out; }
            CU(cudaMalloc(&c->comb, edg_comb_table_bytes()));
            rc = edg_comb_table_init(c->comb, c->stream[0]);
            if (rc) { rc = fail(rc, "comb table build failed: %s", cudaGetErrorString((cudaError_t)rc)); goto out; }
            CU(cudaStreamSynchronize(c->stream[0]));
            __atomic_store_n(&c->ready, 1, __ATOMIC_RELEASE);
        out:
            if (rc) dev_teardown(c);
            if (prev >= 0 && prev != dev) cudaSetDevice(prev);
        }
        pthread_mutex_unlock(&g_ctx_lock);
        if (rc) return rc;
    }
    *out_ctx = c;
    return 0;
}

static void free_staging(edg_dev_t *c, int in, int out)
{
    int i;
    for (i = 0; i < EDG_NSLOT; i++) {
        if (in) {
            if (c->h_in[i]) cudaFreeHost(c->h_in[i]);
            if (c->d_in[i]) cudaFree(c->d_in[i]);
            c->h_in[i] = c->d_in[i] = NULL;
        }
        if (out) {
            if (c->h_out[i]) cudaFreeHost(c->h_out[i]);
            if (c->d_out[i]) cudaFree(c->d_out[i]);
            c->h_out[i] = c->d_out[i] = NULL;
        }
    }
    if (in) c->in_cap = 0;
    if (out) c->out_cap = 0;
}

/* make sure the staging / device buffers of c hold at least the given capacities (device current; buffers are
 * scrubbed when their chunk retires, so nothing secret is freed here) */
static int dev_reserve(edg_dev_t *c, size_t in_need, size_t out_need)
{
    int rc = 0, i;
    if (in_need < ((size_t)1 << 20)) in_need = (size_t)1 << 20;   /* avoid re-allocating for small growing batches */
    if (out_need < ((size_t)1 << 16)) out_need = (size_t)1 << 16;
    if (in_need > c->in_cap) {
        free_staging(c, 1, 0);
        for (i = 0; i < EDG_NSLOT; i++) {
            CU(cudaMallocHost((void **)&c->h_in[i], in_need));
            CU(cudaMalloc((void **)&c->d_in[i], in_need));
        }
        c->in_cap = in_need;
    }
    if (out_need > c->out_cap) {
        free_staging(c, 0, 1);
        for (i = 0; i < EDG_NSLOT; i++) {
            CU(cudaMallocHost((void **)&c->h_out[i], out_need));
            CU(cudaMalloc((void **)&c->d_out[i], out_need));
        }
        c->out_cap = out_need;
    }
out:
    return rc;
}

static int is_pinned(const void *p)
{
    struct cudaPointerAttributes a;
    if (!p) return 0;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return 0; }
    return a.type == cudaMemoryTypeHost;
}

/* Enqueue one operation on `stream` (device of c current).  Kernel scratch comes from the context's stream-ordered
 * pool: allocated and freed on the same stream, so back-to-back calls reuse it without synchronising. */
static int launch(edg_dev_t *c, edg_op_t op, size_t n, uint8_t *d_out, uint8_t *const d_in[3], const uint8_t *d_msgs,
                  const unsigned long long *d_off, size_t fixed_len, int policy, void *stream)
{
    int rc = 0;
    void *scratch = NULL;
    size_t need = 0, records = 0;
    unsigned launches = 0;
    if (n == 0) return 0;
    if (op == OP_VERIFY) { records = n < c->verify_pass ? n : c->verify_pass; need = edg_verify_scratch_bytes(records); }   /* 2.4 KB per signature */
    else if (op == OP_GENPUB || op == OP_SIGN) need = edg_fixedbase_scratch_bytes(op == OP_SIGN, n);
    if (need) CU(cudaMallocFromPoolAsync(&scratch, need, c->pool, (cudaStream_t)stream));
    switch (op) {
    case OP_GENPUB: rc = edg_launch_genpub(n, d_out, d_in[0], scratch, c->comb, c->sm_count, stream, &launches); break;
    case OP_SIGN: rc = edg_launch_sign(n, d_out, d_in[0], d_in[1], d_msgs, d_off, fixed_len, scratch, c->comb, c->sm_count, stream, &launches); break;
    case OP_VERIFY:
        rc = policy == EDDSA_B200_VERIFY_REFERENCE
                 ? edg_launch_verify(n, d_out, d_in[0], d_in[1], d_msgs, d_off, fixed_len, scratch, records, c->wtab, c->sm_count, stream, &launches)
                 : edg_launch_verify_policy(n, d_out, d_in[0], d_in[1], d_msgs, d_off, fixed_len, policy, scratch, records, c->wtab, c->sm_count,
                                            stream, &launches);
        break;
    case OP_X25519: rc = edg_launch_x25519(n, d_out, d_in[0], d_in[1], c->sm_count, stream); launches = 1; break;
    case OP_X25519_BASE: rc = edg_launch_x25519_base(n, d_out, d_in[0], c->comb, c->sm_count, stream); launches = 1; break;
    case OP_PK_CONV: rc = edg_launch_pk_convert(n, d_out, d_in[0], c->sm_count, stream); launches = 1; break;
    case OP_SK_CONV: rc = edg_launch_sk_convert(n, d_out, d_in[0], c->sm_count, stream); launches = 1; break;
    case OP_FE_TEST: rc = edg_launch_fe_selftest(n, d_out, d_in[0], d_in[1], (int)fixed_len, c->sm_count, stream); launches = 1; break;
    case OP_SC_TEST: rc = edg_launch_sc_selftest(n, d_out, d_in[0], d_in[1], d_in[2], (int)fixed_len, c->sm_count, stream); launches = 1; break;
    default: rc = EDDSA_B200_EINVAL; break;
    }
    if (scratch) {
        cudaError_t e = cudaFreeAsync(scratch, (cudaStream_t)stream);
        if (!rc && e != cudaSuccess) rc = (int)e;
    }
    if (rc) return fail(rc, "kernel launch failed: %s", rc == EDDSA_B200_EINVAL ? "unknown operation" : cudaGetErrorString((cudaError_t)rc));
    __atomic_fetch_add(&g_launches, (unsigned long long)launches, __ATOMIC_RELAXED);
out:
    return rc;
}

/* ---- staging copies: callers with ordinary (pageable) memory are bound by one thread's memcpy (~15 GB/s) long before the
 * link (55 GB/s) when messages are large, so big copies into the pinned slots are split over a few helper threads.  One
 * request at a time; a caller that finds the helpers busy (several devices staging at once) copies by itself. ---- */
#define EDG_COPY_PARALLEL_MIN ((size_t)8 << 20)
static struct {
    pthread_mutex_t busy, m;
    pthread_cond_t go, done;
    pthread_t th[EDG_COPY_HELPERS];
    int started, stop, pending;
    unsigned long gen;
    uint8_t *dst;
    const uint8_t *src;
    size_t slice, bytes;
} g_copy = {PTHREAD_MUTEX_INITIALIZER, PTHREAD_MUTEX_INITIALIZER, PTHREAD_COND_INITIALIZER, PTHREAD_COND_INITIALIZER, {0}, 0, 0, 0, 0, NULL, NULL, 0, 0};

static void *copy_helper(void *arg)
{
    const size_t k = (size_t)(uintptr_t)arg;           /* helper k copies slice k + 1 (the caller takes slice 0) */
    unsigned long seen = 0;                            /* helpers are created under g_copy.m by the call that posts their first
                                                        * request, so whatever generation they see first is a live request */
    for (;;) {
        pthread_mutex_lock(&g_copy.m);
        while (g_copy.gen == seen && !g_copy.stop) pthread_cond_wait(&g_copy.go, &g_copy.m);
        if (g_copy.stop) { pthread_mutex_unlock(&g_copy.m); return NULL; }
        seen = g_copy.gen;
        uint8_t *dst = g_copy.dst;
        const uint8_t *src = g_copy.src;
        const size_t lo = (k + 1) * g_copy.slice, hi = lo + g_copy.slice < g_copy.bytes ? lo + g_copy.slice : g_copy.bytes;
        pthread_mutex_unlock(&g_copy.m);
        if (lo < hi) memcpy(dst + lo, src + lo, hi - lo);
        pthread_mutex_lock(&g_copy.m);
        if (--g_copy.pending == 0) pthread_cond_signal(&g_copy.done);
        pthread_mutex_unlock(&g_copy.m);
    }
}

static void stage_copy(uint8_t *dst, const uint8_t *src, size_t bytes)
{
    size_t k;
    if (bytes < EDG_COPY_PARALLEL_MIN || g_copy_helpers < 1 || pthread_mutex_trylock(&g_copy.busy) != 0) { memcpy(dst, src, bytes); return; }
    pthread_mutex_lock(&g_copy.m);
    if (!g_copy.started) {
        g_copy.started = 1;
        for (k = 0; k < (size_t)g_copy_helpers; k++)
            if (pthread_create(&g_copy.th[k], NULL, copy_helper, (void *)(uintptr_t)k) != 0) { g_copy.started = -1; break; }
    }
    if (g_copy.started < 0) {                           /* no helpers: plain copy */
        pthread_mutex_unlock(&g_copy.m);
        pthread_mutex_unlock(&g_copy.busy);
        memcpy(dst, src, bytes);
        return;
    }
    g_copy.dst = dst; g_copy.src = src; g_copy.bytes = bytes;
    g_copy.slice = ((bytes + g_copy_helpers) / ((size_t)g_copy_helpers + 1) + 4095) & ~(size_t)4095;
    g_copy.pending = g_copy_helpers;
    g_copy.gen++;
    pthread_cond_broadcast(&g_copy.go);
    pthread_mutex_unlock(&g_copy.m);
    memcpy(dst, src, g_copy.slice < bytes ? g_copy.slice : bytes);
    pthread_mutex_lock(&g_copy.m);
    while (g_copy.pending > 0) pthread_cond_wait(&g_copy.done, &g_copy.m);
    pthread_mutex_unlock(&g_copy.m);
    pthread_mutex_unlock(&g_copy.busy);
}

static void copy_pool_stop(void)
{
    size_t k;
    pthread_mutex_lock(&g_copy.busy);
    pthread_mutex_lock(&g_copy.m);
    if (g_copy.started > 0) {
        g_copy.stop = 1;
        pthread_cond_broadcast(&g_copy.go);
        pthread_mutex_unlock(&g_copy.m);
        for (k = 0; k < (size_t)g_copy_helpers; k++) pthread_join(g_copy.th[k], NULL);
        pthread_mutex_lock(&g_copy.m);
        g_copy.started = 0; g_copy.stop = 0;
    }
    pthread_mutex_unlock(&g_copy.m);
    pthread_mutex_unlock(&g_copy.busy);
}

static size_t msg_bytes(const edg_job_t *j, size_t lo, size_t hi)
{
    if (!j->has_msgs) return 0;
    return j->off ? j->off[hi] - j->off[lo] : (hi - lo) * j->fixed_len;
}

/* bytes of device input for items [lo, hi): fixed-size arrays + rebased offsets + message bytes */
static size_t chunk_in_bytes(const edg_job_t *j, size_t lo, size_t hi)
{
    size_t b = 0;
    int k;
    for (k = 0; k < j->nin; k++) b += align_up((hi - lo) * j->in_item[k]);
    if (j->has_msgs) {
        if (j->off) b += align_up((hi - lo + 1) * sizeof(unsigned long long));
        b += align_up(msg_bytes(j, lo, hi) + 16);
    }
    return b;
}

typedef struct { int inflight, staged_secret; size_t lo, hi; } slot_t;

/* the chunk in slot s has completed: hand its outputs to the caller and wipe what it staged on the host
 * (the device side is wiped by memsets queued behind the kernel, see run_shard) */
static void retire_slot(edg_dev_t *c, const edg_job_t *j, slot_t *sl, int s, int pin_out, int copy_out)
{
    const size_t m = sl->hi - sl->lo;
    if (!pin_out) {
        if (copy_out) stage_copy(j->out + sl->lo * j->out_item, c->h_out[s], m * j->out_item);
        if (op_secret_out(j->op) && !g_no_scrub) memset(c->h_out[s], 0, m * j->out_item);
    }
    if (sl->staged_secret && !g_no_scrub) memset(c->h_in[s], 0, m * j->in_item[0]);
    sl->inflight = 0;
}

/* Run items [lo, hi) of job j on device context c (chunked, pipelined over EDG_NSLOT slots). */
static int run_shard(edg_dev_t *c, const edg_job_t *j, size_t lo, size_t hi)
{
    int rc = 0, k, s, prev_dev = -1;
    size_t pos, nshard = hi - lo, target, wave, budget;
    int staged = 0, big_items;
    slot_t slot[EDG_NSLOT];
    int pin_in[3] = {0, 0, 0}, pin_msgs = 0, pin_out = 0;
    size_t chunk_no = 0;
    const int secret_in = op_secret_in(j->op) && !g_no_scrub, secret_out = op_secret_out(j->op) && !g_no_scrub;
    if (nshard == 0) return 0;
    memset(slot, 0, sizeof slot);
    pthread_mutex_lock(&c->lock);
    cudaGetDevice(&prev_dev);                   /* the caller's current device is restored on the way out */
    CU(cudaSetDevice(c->dev));
    for (k = 0; k < j->nin; k++) pin_in[k] = is_pinned(j->in[k]);
    pin_msgs = j->has_msgs && is_pinned(j->msgs);
    pin_out = is_pinned(j->out);
    /* aim for >= 4 chunks per shard (copy/compute overlap) but never tiny ones */
    target = (nshard + 3) / 4;
    if (target < 65536) target = 65536;
    /* verify: chunks of whole waves of resident threads, kernels serialised on one stream so that the stages never
     * share an SM (instruction cache) while copies overlap on the slot streams */
    wave = j->op == OP_VERIFY && nshard > c->verify_wave && c->verify_wave >= 8 ? c->verify_wave : 0;
    if (wave) target = c->verify_pass;
    if (target > nshard) target = nshard;
    /* the first chunk's staging and copy are exposed, so chunks start small and grow — but every verify chunk is a pass
     * of three kernels whose tails cost ~0.15 ms, so they double: 1, 2, 4, 8 waves, then whole passes (64-byte messages:
     * a chunk's copy, 0.22 ms per wave alone and 0.5 ms when eight GPUs share the host's links, hides under the previous,
     * half as large chunk's kernels, 1.44 ms per wave; jumping from 2 to 12 waves was 0.7 % faster on one GPU and stalled
     * the ranks on the far side of an 8-GPU host for 1 ms); 1, 1, 2, 4, 8 waves when the inputs have to be staged through
     * the pinned slots (a memcpy the GPU waits for).  The other operations: 65536 items and four times more each chunk
     * when staged. */
    for (k = 0; k < j->nin; k++) staged |= !pin_in[k];
    staged |= j->has_msgs && !pin_msgs;
    big_items = chunk_in_bytes(j, lo, hi) / nshard >= 768;      /* ~1 KB per item and up: the copies take as long as the kernels */
    budget = 2 * g_chunk_bytes;
    for (pos = lo; pos < hi;) {
        static const unsigned ramp_pinned[] = {1, 2, 4, 8}, ramp_staged[] = {1, 1, 2, 4, 8};
        size_t m = target, in_bytes, out_bytes, ofs;
        uint8_t *d_in[3] = {NULL, NULL, NULL};
        const uint8_t *d_msgs = NULL;
        const unsigned long long *d_off = NULL;
        if (wave) {
            const size_t steps = staged ? sizeof ramp_staged / sizeof *ramp_staged : sizeof ramp_pinned / sizeof *ramp_pinned;
            if (big_items) {
                /* copies take as long as the kernels: a chunk larger than its predecessor stalls the GPU for the
                 * difference, so the size stays constant — a sixteenth of the shard, in whole waves */
                m = nshard / (16 * wave);
                m = wave * (m < 1 ? 1 : m);
            } else if (chunk_no < steps) m = wave * (staged ? ramp_staged : ramp_pinned)[chunk_no];
            if (m > c->verify_pass) m = c->verify_pass;
        } else if (staged && chunk_no < 4) {
            m = (size_t)65536 << (2 * chunk_no);
            if (m > target) m = target;
        }
        if (pos + m > hi) m = hi - pos;
        /* shrink the chunk until it fits the staging budget (ragged messages); a single oversized item grows the buffers.
         * Verify chunks stay whole waves as long as they can: 1.6 waves cost the loop kernel as much as 2. */
        while (wave && m > wave && chunk_in_bytes(j, pos, pos + m) > budget) m = (m - 1) / wave * wave;
        while (m > 1 && chunk_in_bytes(j, pos, pos + m) > budget) m = (m + 1) / 2;
        in_bytes = chunk_in_bytes(j, pos, pos + m);
        out_bytes = align_up(m * j->out_item);
        s = (int)(chunk_no % EDG_NSLOT);
        if (slot[s].inflight) { /* retire the chunk that used this slot */
            CU(cudaEventSynchronize(c->done[s]));
            retire_slot(c, j, &slot[s], s, pin_out, 1);
        }
        if (in_bytes > c->in_cap || out_bytes > c->out_cap) {
            /* (re)allocation frees buffers other slots may still use: drain first */
            for (k = 0; k < EDG_NSLOT; k++)
                if (slot[k].inflight) {
                    CU(cudaEventSynchronize(c->done[k]));
                    retire_slot(c, j, &slot[k], k, pin_out, 1);
                }
            rc = dev_reserve(c, in_bytes > c->in_cap ? in_bytes : c->in_cap, out_bytes > c->out_cap ? out_bytes : c->out_cap);
            if (rc) goto out;
        }
        ofs = 0;
        slot[s].staged_secret = 0;
        for (k = 0; k < j->nin; k++) {
            size_t bytes = m * j->in_item[k];
            const uint8_t *src = j->in[k] + pos * j->in_item[k];
            if (!pin_in[k]) {
                stage_copy(c->h_in[s] + ofs, src, bytes);
                src = c->h_in[s] + ofs;
                if (k == 0 && secret_in) slot[s].staged_secret = 1;
            }
            CU(cudaMemcpyAsync(c->d_in[s] + ofs, src, bytes, cudaMemcpyHostToDevice, c->stream[s]));
            d_in[k] = c->d_in[s] + ofs;
            ofs += align_up(bytes);
        }
        if (j->has_msgs) {
            size_t mb = msg_bytes(j, pos, pos + m);
            const uint8_t *src = j->msgs + (j->off ? j->off[pos] : pos * j->fixed_len);
            if (j->off) {
                unsigned long long *ho = (unsigned long long *)(c->h_in[s] + ofs);
                size_t i;
                for (i = 0; i <= m; i++) ho[i] = (unsigned long long)(j->off[pos + i] - j->off[pos]);
                CU(cudaMemcpyAsync(c->d_in[s] + ofs, ho, (m + 1) * sizeof *ho, cudaMemcpyHostToDevice, c->stream[s]));
                d_off = (const unsigned long long *)(c->d_in[s] + ofs);
                ofs += align_up((m + 1) * sizeof *ho);
            }
            if (mb) {
                if (!pin_msgs) { stage_copy(c->h_in[s] + ofs, src, mb); src = c->h_in[s] + ofs; }
                CU(cudaMemcpyAsync(c->d_in[s] + ofs, src, mb, cudaMemcpyHostToDevice, c->stream[s]));
            }
            d_msgs = c->d_in[s] + ofs;
        }
        slot[s].inflight = 1; slot[s].lo = pos; slot[s].hi = pos + m;
        if (j->op == OP_VERIFY) {
            CU(cudaEventRecord(c->in_ready[s], c->stream[s]));
            CU(cudaStreamWaitEvent(c->kstream, c->in_ready[s], 0));
            rc = launch(c, j->op, m, c->d_out[s], d_in, d_msgs, d_off, j->fixed_len, j->policy, c->kstream);
            if (rc) goto out;
            CU(cudaEventRecord(c->k_done[s], c->kstream));
            CU(cudaStreamWaitEvent(c->stream[s], c->k_done[s], 0));
        } else {
            rc = launch(c, j->op, m, c->d_out[s], d_in, d_msgs, d_off, j->fixed_len, j->policy, c->stream[s]);
            if (rc) goto out;
        }
        if (secret_in) CU(cudaMemsetAsync(c->d_in[s], 0, m * j->in_item[0], c->stream[s]));        /* the secret keys of this chunk */
        CU(cudaMemcpyAsync(pin_out ? j->out + pos * j->out_item : c->h_out[s], c->d_out[s], m * j->out_item,
                           cudaMemcpyDeviceToHost, c->stream[s]));
        if (secret_out) CU(cudaMemsetAsync(c->d_out[s], 0, m * j->out_item, c->stream[s]));
        CU(cudaEventRecord(c->done[s], c->stream[s]));
        pos += m;
        chunk_no++;
    }
out:
    if (rc) cudaDeviceSynchronize();            /* error path: nothing may still be reading the staging buffers */
    for (k = 0; k < EDG_NSLOT; k++) {
        s = (int)((chunk_no + k) % EDG_NSLOT); /* oldest first */
        if (slot[s].inflight) {
            cudaError_t e = rc ? cudaSuccess : cudaEventSynchronize(c->done[s]);
            if (e != cudaSuccess && !rc) {
                rc = fail((int)e, "cudaEventSynchronize failed: %s", cudaGetErrorString(e));
                cudaDeviceSynchronize();        /* the younger chunks are not waited for one by one any more: nothing may still
                                                 * be running (or writing to the caller's memory) when the call returns */
            }
            retire_slot(c, j, &slot[s], s, pin_out, !rc);
        }
    }
    if (rc && !g_no_scrub && (op_secret_in(j->op) || op_secret_out(j->op))) {
        /* error path: wipe the device copies the queued memsets may not have reached, and the host slots whole — the
         * chunk that failed had staged its keys but was not in flight yet, so retire_slot never saw it */
        for (k = 0; k < EDG_NSLOT; k++) {
            if (c->d_in[k]) cudaMemset(c->d_in[k], 0, c->in_cap);
            if (c->d_out[k]) cudaMemset(c->d_out[k], 0, c->out_cap);
            if (c->h_in[k]) memset(c->h_in[k], 0, c->in_cap);
            if (c->h_out[k] && op_secret_out(j->op)) memset(c->h_out[k], 0, c->out_cap);
        }
    }
    if (prev_dev >= 0 && prev_dev != c->dev) cudaSetDevice(prev_dev);
    pthread_mutex_unlock(&c->lock);
    return rc;
}

/* ---- per-device worker threads (multi-device jobs) ---- */
static void *worker_main(void *p)
{
    edg_dev_t *c = (edg_dev_t *)p;
    for (;;) {
        shard_t *sh;
        pthread_mutex_lock(&c->q_lock);
        while (!c->q_head && !c->worker_stop) pthread_cond_wait(&c->q_cond, &c->q_lock);
        sh = c->q_head;
        if (sh) { c->q_head = sh->next; if (!c->q_head) c->q_tail = NULL; }
        pthread_mutex_unlock(&c->q_lock);
        if (!sh) return NULL;                  /* stop requested and the queue is empty */
        t_err[0] = 0;
        sh->rc = run_shard(c, sh->j, sh->lo, sh->hi);
        memcpy(sh->err, t_err, sizeof sh->err);
        pthread_mutex_lock(&sh->sync->m);
        if (--sh->sync->pending == 0) pthread_cond_signal(&sh->sync->cv);
        pthread_mutex_unlock(&sh->sync->m);
    }
}

static int worker_post(edg_dev_t *c, shard_t *sh)
{
    int rc = 0;
    pthread_mutex_lock(&c->q_lock);
    if (!c->worker_on) {
        c->worker_stop = 0;
        if (pthread_create(&c->worker, NULL, worker_main, c) != 0) rc = fail(EDDSA_B200_EINVAL, "cannot start the worker thread of device %d", c->dev);
        else c->worker_on = 1;
    }
    if (!rc) {
        sh->next = NULL;
        if (c->q_tail) c->q_tail->next = sh; else c->q_head = sh;
        c->q_tail = sh;
        pthread_cond_signal(&c->q_cond);
    }
    pthread_mutex_unlock(&c->q_lock);
    return rc;
}

static void worker_stop(edg_dev_t *c)
{
    pthread_mutex_lock(&c->q_lock);
    if (!c->worker_on) { pthread_mutex_unlock(&c->q_lock); return; }
    c->worker_stop = 1;
    pthread_cond_signal(&c->q_cond);
    pthread_mutex_unlock(&c->q_lock);
    pthread_join(c->worker, NULL);
    c->worker_on = 0;
}

static int run_job(const edg_job_t *j)
{
    int rc = engine_ready(), g, ndev, k, posted = 0;
    shard_t sh[EDG_MAX_DEV];
    job_sync_t sync;
    if (rc) return rc;
    t_err[0] = 0;
    if (j->n == 0) return 0;
    for (k = 0; k < j->nin; k++)
        if (!j->in[k]) return fail(EDDSA_B200_EINVAL, "NULL input array");
    if (!j->out) return fail(EDDSA_B200_EINVAL, "NULL output array");
    if (j->has_msgs && !j->msgs && msg_bytes(j, 0, j->n) != 0) return fail(EDDSA_B200_EINVAL, "NULL message blob");
    if (j->has_msgs && j->off)
        for (size_t i = 0; i < j->n; i++)
            if (j->off[i + 1] < j->off[i]) return fail(EDDSA_B200_EINVAL, "message offsets must be non-decreasing");
    ndev = __atomic_load_n(&g_nactive, __ATOMIC_ACQUIRE);
    if ((size_t)ndev > (j->n + 16383) / 16384) ndev = (int)((j->n + 16383) / 16384); /* small batches: fewer devices */
    if (ndev < 1) ndev = 1;
    for (g = 0; g < ndev; g++) {
        rc = dev_basic(g_list[g], &sh[g].c);
        if (rc) return rc;
        sh[g].j = j;
        sh[g].lo = j->n * (size_t)g / ndev;
        sh[g].hi = j->n * (size_t)(g + 1) / ndev;
        sh[g].rc = 0;
        sh[g].err[0] = 0;
        sh[g].sync = &sync;
    }
    if (ndev == 1) return run_shard(sh[0].c, j, 0, j->n);
    pthread_mutex_init(&sync.m, NULL);
    pthread_cond_init(&sync.cv, NULL);
    sync.pending = ndev;
    for (g = 0; g < ndev; g++) {
        int e = worker_post(sh[g].c, &sh[g]);
        if (e) {
            if (!rc) rc = e;
            pthread_mutex_lock(&sync.m);
            sync.pending--;
            pthread_mutex_unlock(&sync.m);
        } else posted++;
    }
    pthread_mutex_lock(&sync.m);
    while (sync.pending > 0) pthread_cond_wait(&sync.cv, &sync.m);
    pthread_mutex_unlock(&sync.m);
    pthread_cond_destroy(&sync.cv);
    pthread_mutex_destroy(&sync.m);
    for (g = 0; g < ndev; g++)
        if (sh[g].rc && !rc) { rc = sh[g].rc; memcpy(t_err, sh[g].err, sizeof t_err); }
    (void)posted;
    return rc;
}

/* ---------------------------------------------------------------------------------------------
 * host-buffer batch API
 * --------------------------------------------------------------------------------------------- */
int ed25519_genpub_batch(size_t n, uint8_t *pub, const uint8_t *sec)
{
    edg_job_t j = {OP_GENPUB, n, 1, {sec, NULL, NULL}, {32, 0, 0}, 0, NULL, NULL, 0, pub, 32, 0};
    return run_job(&j);
}

int ed25519_sign_batch(size_t n, uint8_t *sig, const uint8_t *sec, const uint8_t *pub, const uint8_t *msgs,
                       const size_t *off, size_t fixed_len)
{
    edg_job_t j = {OP_SIGN, n, 2, {sec, pub, NULL}, {32, 32, 0}, 1, msgs, off, fixed_len, sig, 64, 0};
    return run_job(&j);
}

static int bad_policy(int policy)
{
    t_err[0] = 0;
    if (policy == EDDSA_B200_VERIFY_REFERENCE) return 0;
    if (policy != EDDSA_B200_VERIFY_STRICT && policy != EDDSA_B200_VERIFY_ZIP215) return fail(EDDSA_B200_EINVAL, "unknown verify policy %d", policy);
    if (!edg_launch_verify_policy) return fail(EDDSA_B200_EINVAL, "verify policy %d: these kernels have no launcher for it", policy);
    return 0;
}

int ed25519_verify_policy_batch(size_t n, uint8_t *ok, const uint8_t *sig, const uint8_t *pub, const uint8_t *msgs,
                                const size_t *off, size_t fixed_len, int policy)
{
    edg_job_t j = {OP_VERIFY, n, 2, {sig, pub, NULL}, {64, 32, 0}, 1, msgs, off, fixed_len, ok, 1, policy};
    return bad_policy(policy) ? EDDSA_B200_EINVAL : run_job(&j);
}

int ed25519_verify_batch(size_t n, uint8_t *ok, const uint8_t *sig, const uint8_t *pub, const uint8_t *msgs,
                         const size_t *off, size_t fixed_len)
{
    return ed25519_verify_policy_batch(n, ok, sig, pub, msgs, off, fixed_len, EDDSA_B200_VERIFY_REFERENCE);
}

int x25519_batch(size_t n, uint8_t *out, const uint8_t *scalar, const uint8_t *point)
{
    edg_job_t j = {OP_X25519, n, 2, {scalar, point, NULL}, {32, 32, 0}, 0, NULL, NULL, 0, out, 32, 0};
    return run_job(&j);
}

int x25519_base_batch(size_t n, uint8_t *out, const uint8_t *scalar)
{
    edg_job_t j = {OP_X25519_BASE, n, 1, {scalar, NULL, NULL}, {32, 0, 0}, 0, NULL, NULL, 0, out, 32, 0};
    return run_job(&j);
}

int pk_ed25519_to_x25519_batch(size_t n, uint8_t *out, const uint8_t *in)
{
    edg_job_t j = {OP_PK_CONV, n, 1, {in, NULL, NULL}, {32, 0, 0}, 0, NULL, NULL, 0, out, 32, 0};
    return run_job(&j);
}

int sk_ed25519_to_x25519_batch(size_t n, uint8_t *out, const uint8_t *in)
{
    edg_job_t j = {OP_SK_CONV, n, 1, {in, NULL, NULL}, {32, 0, 0}, 0, NULL, NULL, 0, out, 32, 0};
    return run_job(&j);
}

/* diagnostic: one GF(2^255-19) operation per item on the device (op: 0 mul, 1 sq, 2 add, 3 sub, 4 x121665,
 * 5 canonical form, 6 inverse, 7 ^((p-5)/8), 8 negate, 9 shared inversion of each group of up to 32 consecutive
 * items); a, b, out: n x 32 bytes, any 256-bit values */
int eddsa_b200_fe_selftest(size_t n, uint8_t *out, const uint8_t *a, const uint8_t *b, int op)
{
    edg_job_t j = {OP_FE_TEST, n, 2, {a, b, NULL}, {32, 32, 0}, 0, NULL, NULL, (size_t)op, out, 32, 0};
    return run_job(&j);
}

/* diagnostic: one scalar operation mod L per item on the device (op: 0 out = (a || b) mod L, the 64-byte value
 * a + 2^256 b; 1 out = a mod L; 2 out = a * b + c mod L; 3 out = tau of the half-size verification scalars
 * (rho, tau) of t = a, a < L; 4 out = |rho| of the same in words 0..5, 1 in word 7 if rho < 0; 5 out = a + 2^15 sum
 * 2^(16 k), the signed 16-bit digits of a < 2^253 as the verify loop reads them); a, b, c, out: n x 32 bytes */
int eddsa_b200_sc_selftest(size_t n, uint8_t *out, const uint8_t *a, const uint8_t *b, const uint8_t *c, int op)
{
    edg_job_t j = {OP_SC_TEST, n, 3, {a, b, c}, {32, 32, 32}, 0, NULL, NULL, (size_t)op, out, 32, 0};
    return run_job(&j);
}

/* ---------------------------------------------------------------------------------------------
 * device-buffer batch API (current device, asynchronous)
 * --------------------------------------------------------------------------------------------- */
static int cur_ctx(edg_dev_t **c)
{
    int dev = 0, rc = engine_ready();
    cudaError_t e;
    if (rc) return rc;
    e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return fail((int)e, "cudaGetDevice failed: %s", cudaGetErrorString(e));
    return dev_basic(dev, c);
}

/* diagnostic: read back the base-point window tables the verify kernels use on the current device */
size_t eddsa_b200_verify_tables(uint8_t *out, size_t cap)
{
    edg_dev_t *c;
    size_t bytes = edg_verify_table_bytes() - 48 * sizeof(uint32_t);   /* without the two base points at the end */
    if (!out || cap < bytes || cur_ctx(&c)) return 0;
    if (cudaMemcpy(out, c->wtab, bytes, cudaMemcpyDeviceToHost) != cudaSuccess) { fail(1, "cudaMemcpy of the window tables failed"); return 0; }
    return bytes;
}

/* diagnostic: read back the fixed-base comb table of the current device (rows x entries x 96 bytes) */
size_t eddsa_b200_comb_table(uint8_t *out, size_t cap)
{
    edg_dev_t *c;
    size_t bytes = edg_comb_table_payload_bytes();
    if (!out || cap < bytes || cur_ctx(&c)) return 0;
    if (cudaMemcpy(out, c->comb, bytes, cudaMemcpyDeviceToHost) != cudaSuccess) { fail(1, "cudaMemcpy of the comb table failed"); return 0; }
    return bytes;
}

/* diagnostic (tests of the secret-scrubbing contract): copies up to len bytes from the start of staging buffer
 * `which` (0 host input, 1 device input, 2 host output, 3 device output) of pipeline slot `slot` on the current
 * device into out; returns the number of bytes copied (0: no such buffer yet). */
size_t eddsa_b200_debug_peek_staging(int which, int slot, uint8_t *out, size_t len)
{
    edg_dev_t *c;
    size_t cap;
    const uint8_t *src;
    if (!out || slot < 0 || slot >= EDG_NSLOT || which < 0 || which > 3 || cur_ctx(&c)) return 0;
    pthread_mutex_lock(&c->lock);
    cap = which < 2 ? c->in_cap : c->out_cap;
    src = which == 0 ? c->h_in[slot] : which == 1 ? c->d_in[slot] : which == 2 ? c->h_out[slot] : c->d_out[slot];
    if (len > cap) len = cap;
    if (!src) len = 0;
    if (len) {
        if (which & 1) { if (cudaMemcpy(out, src, len, cudaMemcpyDeviceToHost) != cudaSuccess) len = 0; }
        else memcpy(out, src, len);
    }
    pthread_mutex_unlock(&c->lock);
    return len;
}

static int misaligned(const void *p) { return ((uintptr_t)p & 15) != 0; }

static int dev_call(edg_op_t op, size_t n, uint8_t *out, const uint8_t *a, const uint8_t *b, const uint8_t *msgs,
                    const uint64_t *off, size_t fixed_len, int policy, void *stream)
{
    edg_dev_t *c;
    uint8_t *d_in[3] = {(uint8_t *)a, (uint8_t *)b, NULL};
    int rc = cur_ctx(&c);
    if (rc) return rc;
    t_err[0] = 0;
    if (n == 0) return 0;
    if (!out || !a || misaligned(a) || (b && misaligned(b)) || (op != OP_VERIFY && misaligned(out)))
        return fail(EDDSA_B200_EINVAL, "device arrays must be non-NULL and 16-byte aligned");
    if ((op == OP_SIGN || op == OP_VERIFY) && !msgs && (off || fixed_len))
        return fail(EDDSA_B200_EINVAL, "NULL message blob");
    return launch(c, op, n, out, d_in, msgs, (const unsigned long long *)off, fixed_len, policy, stream);
}

int ed25519_genpub_batch_dev(size_t n, uint8_t *pub, const uint8_t *sec, void *stream)
{
    return dev_call(OP_GENPUB, n, pub, sec, NULL, NULL, NULL, 0, 0, stream);
}

int ed25519_sign_batch_dev(size_t n, uint8_t *sig, const uint8_t *sec, const uint8_t *pub, const uint8_t *msgs,
                           const uint64_t *off, size_t fixed_len, void *stream)
{
    if (n && !pub) return fail(EDDSA_B200_EINVAL, "NULL pub array");
    return dev_call(OP_SIGN, n, sig, sec, pub, msgs, off, fixed_len, 0, stream);
}

int ed25519_verify_policy_batch_dev(size_t n, uint8_t *ok, const uint8_t *sig, const uint8_t *pub, const uint8_t *msgs,
                                    const uint64_t *off, size_t fixed_len, int policy, void *stream)
{
    if (bad_policy(policy)) return EDDSA_B200_EINVAL;
    if (n && !pub) return fail(EDDSA_B200_EINVAL, "NULL pub array");
    return dev_call(OP_VERIFY, n, ok, sig, pub, msgs, off, fixed_len, policy, stream);
}

int ed25519_verify_batch_dev(size_t n, uint8_t *ok, const uint8_t *sig, const uint8_t *pub, const uint8_t *msgs,
                             const uint64_t *off, size_t fixed_len, void *stream)
{
    return ed25519_verify_policy_batch_dev(n, ok, sig, pub, msgs, off, fixed_len, EDDSA_B200_VERIFY_REFERENCE, stream);
}

int x25519_batch_dev(size_t n, uint8_t *out, const uint8_t *scalar, const uint8_t *point, void *stream)
{
    if (n && !point) return fail(EDDSA_B200_EINVAL, "NULL point array");
    return dev_call(OP_X25519, n, out, scalar, point, NULL, NULL, 0, 0, stream);
}

int x25519_base_batch_dev(size_t n, uint8_t *out, const uint8_t *scalar, void *stream)
{
    return dev_call(OP_X25519_BASE, n, out, scalar, NULL, NULL, NULL, 0, 0, stream);
}

int pk_ed25519_to_x25519_batch_dev(size_t n, uint8_t *out, const uint8_t *in, void *stream)
{
    return dev_call(OP_PK_CONV, n, out, in, NULL, NULL, NULL, 0, 0, stream);
}

int sk_ed25519_to_x25519_batch_dev(size_t n, uint8_t *out, const uint8_t *in, void *stream)
{
    return dev_call(OP_SK_CONV, n, out, in, NULL, NULL, NULL, 0, 0, stream);
}

/* ---------------------------------------------------------------------------------------------
 * engine control
 * --------------------------------------------------------------------------------------------- */
int eddsa_b200_init(void)
{
    edg_dev_t *c;
    int rc = engine_ready(), g;
    if (rc) return rc;
    for (g = 0; g < g_nlist; g++) {
        rc = dev_basic(g_list[g], &c);
        if (rc) return rc;
    }
    return 0;
}

void eddsa_b200_shutdown(void)
{
    int d, prev = -1;
    pthread_once(&g_once, global_init);
    if (g_init_rc || !g_nlist) return;
    cudaGetDevice(&prev);
    for (d = 0; d < EDG_MAX_DEV; d++) {
        edg_dev_t *c = &g_dev[d];
        if (!__atomic_load_n(&c->ready, __ATOMIC_ACQUIRE)) continue;
        worker_stop(c);
        copy_pool_stop();
        pthread_mutex_lock(&g_ctx_lock);
        pthread_mutex_lock(&c->lock);
        cudaSetDevice(d);
        cudaDeviceSynchronize();
        free_staging(c, 1, 1);
        dev_teardown(c);
        __atomic_store_n(&c->ready, 0, __ATOMIC_RELEASE);
        pthread_mutex_unlock(&c->lock);
        pthread_mutex_unlock(&g_ctx_lock);
    }
    if (prev >= 0) cudaSetDevice(prev);
}

int eddsa_b200_device_count(void)
{
    if (engine_ready()) return 0;
    return __atomic_load_n(&g_nactive, __ATOMIC_ACQUIRE);
}

int eddsa_b200_set_device_count(int count)
{
    int rc = engine_ready();
    if (rc) return rc;
    if (count < 0 || count > g_nlist) return fail(EDDSA_B200_EINVAL, "device count %d outside 0..%d", count, g_nlist);
    __atomic_store_n(&g_nactive, count ? count : g_nlist, __ATOMIC_RELEASE);
    return 0;
}

unsigned long long eddsa_b200_launch_count(void) { return __atomic_load_n(&g_launches, __ATOMIC_RELAXED); }

const char *eddsa_b200_last_error(void) { return t_err; }

/* ---------------------------------------------------------------------------------------------
 * eddsa.h single-operation API: a batch of one.  void functions cannot report failure, so a device
 * error is fatal (never silently wrong, never a CPU fallback).
 * --------------------------------------------------------------------------------------------- */
static void must(int rc, const char *what)
{
    if (rc) {
        fprintf(stderr, "libeddsa_b200: %s failed (%d): %s\n", what, rc, t_err);
        abort();
    }
}

void ed25519_genpub(uint8_t pub[32], const uint8_t sec[32]) { must(ed25519_genpub_batch(1, pub, sec), "ed25519_genpub"); }

void ed25519_sign(uint8_t sig[64], const uint8_t sec[32], const uint8_t pub[32], const uint8_t *data, size_t len)
{
    static const uint8_t empty[1] = {0};
    must(ed25519_sign_batch(1, sig, sec, pub, data ? data : empty, NULL, len), "ed25519_sign");
}

bool ed25519_verify(const uint8_t sig[64], const uint8_t pub[32], const uint8_t *data, size_t len)
{
    static const uint8_t empty[1] = {0};
    uint8_t ok = 0;
    must(ed25519_verify_batch(1, &ok, sig, pub, data ? data : empty, NULL, len), "ed25519_verify");
    return ok != 0;
}

void x25519_base(uint8_t out[32], const uint8_t scalar[32]) { must(x25519_base_batch(1, out, scalar), "x25519_base"); }

void x25519(uint8_t out[32], const uint8_t scalar[32], const uint8_t point[32])
{
    must(x25519_batch(1, out, scalar, point), "x25519");
}

void pk_ed25519_to_x25519(uint8_t out[32], const uint8_t in[32]) { must(pk_ed25519_to_x25519_batch(1, out, in), "pk_ed25519_to_x25519"); }
void sk_ed25519_to_x25519(uint8_t out[32], const uint8_t in[32]) { must(sk_ed25519_to_x25519_batch(1, out, in), "sk_ed25519_to_x25519"); }

/* obsolete names (reference ed25519-sha512.c:262-324, x25519.c:236-243) */
void eddsa_genpub(uint8_t pub[32], const uint8_t sec[32]) { ed25519_genpub(pub, sec); }
void eddsa_sign(uint8_t sig[64], const uint8_t sec[32], const uint8_t pub[32], const uint8_t *data, size_t len) { ed25519_sign(sig, sec, pub, data, len); }
bool eddsa_verify(const uint8_t sig[64], const uint8_t pub[32], const uint8_t *data, size_t len) { return ed25519_verify(sig, pub, data, len); }
void DH(uint8_t out[32], const uint8_t sec[32], const uint8_t point[32]) { x25519(out, sec, point); }
void eddsa_pk_eddsa_to_dh(uint8_t out[32], const uint8_t in[32]) { pk_ed25519_to_x25519(out, in); }
void eddsa_sk_eddsa_to_dh(uint8_t out[32], const uint8_t in[32]) { sk_ed25519_to_x25519(out, in); }
