/*
 * dra_oracle.c — plain-C restatement of spec/ALLOCATION.md.  TEST INFRASTRUCTURE ONLY (see dra_oracle.h).
 *
 * PARITY UNPINNED for the claim search: the reference has no implementation of it to follow
 * (SURVEY.md F1).  Every rule the reference DOES fix is cited where it is restated.
 * Written for obviousness, not speed: one GPU at a time, one start at a time, no bit tricks shared with
 * the CUDA kernels (the kernels use SWAR shifts, ballots and monotone "dead profile" shortcuts; this
 * file uses none of them, so agreement between the two is evidence, not tautology).
 */
#include "dra_oracle.h"

#include <pthread.h>
#include <stdlib.h>
#include <string.h>

/* ------------------------------------------------------------------------------------------------ */

static void put(dra_out_rec* o, uint32_t gpu, uint8_t start, uint8_t size, uint8_t profile, uint8_t st)
{
    o->gpu = gpu; o->start = start; o->size = size; o->profile = profile; o->status = st;
}

static uint8_t out_profile(const dra_claim_rec* c)
{
    if (c->kind == DRA_KIND_GPU) return DRA_PROFILE_GPU;
    if (c->kind == DRA_KIND_SHARED) return DRA_PROFILE_SHARED;
    return c->profile;
}

/* ---- selectors, spec §10 ------------------------------------------------------------------------- */
static const dra_gpu_attr* g_attrs; static uint32_t g_nattr;
static const dra_selector* g_sels; static uint32_t g_nsel;

void dra_oracle_set_selectors(const dra_gpu_attr* attrs, uint32_t n_gpu, const dra_selector* sels, uint32_t n_sel)
{
    g_attrs = attrs; g_nattr = n_gpu; g_sels = sels; g_nsel = n_sel;
}

static uint32_t claim_sel(const dra_claim_rec* c)
{
    if (c->kind == DRA_KIND_GPU || c->kind == DRA_KIND_MIG) return c->mem_limit_mib;
    if (c->kind == DRA_KIND_SHARED) return c->group;
    return 0;
}

/* does global GPU `g` pass selector `id` (0 = no selector)?  Postfix program over a boolean stack. */
static int sel_pass(uint32_t id, uint32_t g)
{
    if (id == 0) return 1;
    if (id > g_nsel) return 0;
    dra_gpu_attr a; memset(&a, 0, sizeof a);
    if (g_attrs && g < g_nattr) a = g_attrs[g];
    const dra_selector* s = &g_sels[id - 1];
    int stack[DRA_SEL_MAX_INS + 1]; int sp = 0; int any = 0;
    for (uint32_t i = 0; i < DRA_SEL_MAX_INS; i++) {
        const dra_sel_ins* in = &s->ins[i];
        if (in->op == DRA_SEL_END) break;
        any = 1;
        if (in->op == DRA_SEL_CMP) {
            uint32_t v;
            switch (in->attr) {
                case DRA_ATTR_MEMORY_MIB: v = a.mem_total_mib; break;
                case DRA_ATTR_CC: v = a.cc; break;
                case DRA_ATTR_INDEX: v = a.index; break;
                case DRA_ATTR_PRODUCT: v = a.product; break;
                case DRA_ATTR_DRIVER_MAJOR: v = a.driver_major; break;
                default: return 0;
            }
            int r;
            switch (in->cmp) {
                case DRA_CMP_EQ: r = v == in->value; break;
                case DRA_CMP_NE: r = v != in->value; break;
                case DRA_CMP_LT: r = v < in->value; break;
                case DRA_CMP_LE: r = v <= in->value; break;
                case DRA_CMP_GT: r = v > in->value; break;
                case DRA_CMP_GE: r = v >= in->value; break;
                case DRA_CMP_IN_MASK: r = v < 32 && ((in->value >> v) & 1u); break;
                default: return 0;
            }
            stack[sp++] = r;
        } else if (in->op == DRA_SEL_AND || in->op == DRA_SEL_OR) {
            if (sp < 2) return 0;
            int b = stack[--sp], a_ = stack[--sp];
            stack[sp++] = in->op == DRA_SEL_AND ? (a_ && b) : (a_ || b);
        } else if (in->op == DRA_SEL_NOT) {
            if (sp < 1) return 0;
            stack[sp - 1] = !stack[sp - 1];
        } else return 0;
    }
    if (!any) return 1;
    return sp >= 1 ? stack[sp - 1] : 0;
}

/* spec §3: malformed shape (decides the number of slots) */
static int claim_bad_shape(const dra_claim_rec* c, uint32_t n_node, int have_off)
{
    if (c->kind > DRA_KIND_SHARED) return 1;
    if (c->node >= n_node) return 1;
    if (c->kind == DRA_KIND_GPU) {
        if (c->count == 0 || c->count > DRA_MAX_COUNT) return 1;
        if (!have_off && c->count != 1) return 1;
    }
    if (c->kind == DRA_KIND_MIG && c->profile >= DRA_MAX_PROFILES) return 1;
    return 0;
}

/* spec §3 + §10: INVALID = malformed shape, or a selector id beyond the table (keeps its slots) */
static int claim_invalid(const dra_claim_rec* c, uint32_t n_node, int have_off)
{
    return claim_bad_shape(c, n_node, have_off) || claim_sel(c) > g_nsel;
}

/* spec §1: slots(c) */
static uint32_t claim_slots(const dra_claim_rec* c, uint32_t n_node, int have_off)
{
    if (claim_bad_shape(c, n_node, have_off)) return 1;
    return c->kind == DRA_KIND_GPU ? c->count : 1;
}

static void fail_all(dra_out_rec* o, uint32_t slots, const dra_claim_rec* c, uint8_t st)
{
    for (uint32_t k = 0; k < slots; k++) put(&o[k], DRA_GPU_NONE, 0, 0, out_profile(c), st);
}

/* Lowest start of entry e that fits into `busy`; -1 when none.
 * Overlap rule: a placement occupies memory slices [start, start+size) and two placements conflict iff
 * the ranges intersect — go-nvml nvml.h:9761-9765 and :10079-10082, published per slice by
 * cmd/nvidia-dra-plugin/deviceinfo.go:199-204. */
static int lowest_fit(uint16_t busy, dra_prof_ent e)
{
    for (int s = 0; s < 16; s++) {
        if (!((e.start_mask >> s) & 1u)) continue;
        uint32_t m = ((1u << e.size) - 1u) << s;
        if ((busy & m) == 0) return s;
    }
    return -1;
}

static int gpu_offers(const dra_gpu_rec* g, dra_prof_ent e)
{
    /* MIG devices exist only under MIG-enabled parents: cmd/nvidia-dra-plugin/nvlib.go:316-318 */
    return (g->flags & DRA_GPU_MIG_ENABLED) && !(g->flags & DRA_GPU_UNAVAILABLE) && e.start_mask != 0;
}

typedef struct node_job {
    dra_gpu_rec* gpus;          /* the node's GPUs */
    uint32_t g0, ng;            /* global index of gpus[0], count */
    const dra_profile_tbl* tbl;
    const dra_claim_rec* claims;
    const uint32_t* idx;        /* the node's claims, input order */
    uint32_t cnt;
    uint32_t n_node;
    const uint32_t* out_off;    /* may be NULL */
    dra_out_rec* out;
    int commit;                 /* 0: evaluate only (UnsuitableNodes) — caller passes a scratch copy */
    int all_ok;                 /* out: every slot OK */
    uint32_t node_override;     /* UnsuitableNodes: claim.node := candidate */
    int use_override;
} node_job;

static dra_out_rec* slot_of(const node_job* j, uint32_t ci)
{
    return &j->out[j->out_off ? j->out_off[ci] : ci];
}

/* spec §4 — full GPUs are published only for GPUs that are not MIG-enabled: nvlib.go:152 */
static void do_gpu(node_job* j, uint32_t ci)
{
    const dra_claim_rec* c = &j->claims[ci];
    dra_out_rec* o = slot_of(j, ci);
    uint32_t elig = 0;
    const uint32_t sel = claim_sel(c);
    for (uint32_t g = 0; g < j->ng; g++) {
        const dra_gpu_rec* r = &j->gpus[g];
        if (!(r->flags & (DRA_GPU_MIG_ENABLED | DRA_GPU_FULL_ALLOCATED | DRA_GPU_UNAVAILABLE)) &&
            r->share_cnt == 0 && sel_pass(sel, j->g0 + g)) elig++;
    }
    if (elig < c->count) { fail_all(o, c->count, c, DRA_ST_NO_CAPACITY); j->all_ok = 0; return; }
    uint32_t k = 0;
    for (uint32_t g = 0; g < j->ng && k < c->count; g++) {
        dra_gpu_rec* r = &j->gpus[g];
        if (!(r->flags & (DRA_GPU_MIG_ENABLED | DRA_GPU_FULL_ALLOCATED | DRA_GPU_UNAVAILABLE)) &&
            r->share_cnt == 0 && sel_pass(sel, j->g0 + g)) {
            r->flags |= DRA_GPU_FULL_ALLOCATED;
            put(&o[k++], j->g0 + g, 0, 0, DRA_PROFILE_GPU, DRA_ST_OK);
        }
    }
}

/* spec §5 */
static void do_mig(node_job* j, uint32_t ci)
{
    const dra_claim_rec* c = &j->claims[ci];
    dra_out_rec* o = slot_of(j, ci);
    int any_offer = 0;
    for (uint32_t g = 0; g < j->ng; g++) {
        dra_gpu_rec* r = &j->gpus[g];
        dra_prof_ent e = j->tbl[r->model].ent[c->profile];
        if (!gpu_offers(r, e) || !sel_pass(claim_sel(c), j->g0 + g)) continue;
        any_offer = 1;
        if (r->flags & DRA_GPU_FULL_ALLOCATED) continue;
        int s = lowest_fit(r->busy, e);
        if (s < 0) continue;
        r->busy |= (uint16_t)(((1u << e.size) - 1u) << s);
        put(o, j->g0 + g, (uint8_t)s, e.size, c->profile, DRA_ST_OK);
        return;
    }
    put(o, DRA_GPU_NONE, 0, 0, c->profile, any_offer ? DRA_ST_NO_CAPACITY : DRA_ST_BAD_PROFILE);
    j->all_ok = 0;
}

/* spec §6 — matchAttribute parentUUID: demo/specs/quickstart/gpu-test4.yaml:42-44 */
static void do_group(node_job* j, uint32_t i0, uint32_t i1)
{
    for (uint32_t g = 0; g < j->ng; g++) {
        dra_gpu_rec* r = &j->gpus[g];
        if (!(r->flags & DRA_GPU_MIG_ENABLED)) continue;
        if (r->flags & (DRA_GPU_UNAVAILABLE | DRA_GPU_FULL_ALLOCATED)) continue;
        if (!sel_pass(claim_sel(&j->claims[j->idx[i0]]), j->g0 + g)) continue;   /* first member's selector */
        uint16_t busy = r->busy;
        int starts[DRA_MAX_GROUP];
        int ok = 1;
        for (uint32_t i = i0; i < i1 && ok; i++) {
            const dra_claim_rec* c = &j->claims[j->idx[i]];
            dra_prof_ent e = j->tbl[r->model].ent[c->profile];
            int s = e.start_mask ? lowest_fit(busy, e) : -1;
            if (s < 0) { ok = 0; break; }
            starts[i - i0] = s;
            busy |= (uint16_t)(((1u << e.size) - 1u) << s);
        }
        if (!ok) continue;
        r->busy = busy;
        for (uint32_t i = i0; i < i1; i++) {
            const dra_claim_rec* c = &j->claims[j->idx[i]];
            dra_prof_ent e = j->tbl[r->model].ent[c->profile];
            put(slot_of(j, j->idx[i]), j->g0 + g, (uint8_t)starts[i - i0], e.size, c->profile, DRA_ST_OK);
        }
        return;
    }
    for (uint32_t i = i0; i < i1; i++) {
        const dra_claim_rec* c = &j->claims[j->idx[i]];
        put(slot_of(j, j->idx[i]), DRA_GPU_NONE, 0, 0, c->profile, DRA_ST_GROUP);
    }
    j->all_ok = 0;
}

/* spec §7 (extension) */
static void do_shared(node_job* j, uint32_t ci)
{
    const dra_claim_rec* c = &j->claims[ci];
    dra_out_rec* o = slot_of(j, ci);
    for (uint32_t g = 0; g < j->ng; g++) {
        dra_gpu_rec* r = &j->gpus[g];
        if (r->flags & (DRA_GPU_MIG_ENABLED | DRA_GPU_FULL_ALLOCATED | DRA_GPU_UNAVAILABLE)) continue;
        if (r->share_cnt == 0xFFFFu) continue;
        if (r->mem_free_mib < c->mem_limit_mib) continue;
        if (!sel_pass(claim_sel(c), j->g0 + g)) continue;
        r->mem_free_mib -= c->mem_limit_mib;
        r->share_cnt++;
        put(o, j->g0 + g, 0, 0, DRA_PROFILE_SHARED, DRA_ST_OK);
        return;
    }
    put(o, DRA_GPU_NONE, 0, 0, DRA_PROFILE_SHARED, DRA_ST_MEM_LIMIT);
    j->all_ok = 0;
}

static int in_run(const node_job* j, uint32_t i, uint32_t group, int have_off)
{
    const dra_claim_rec* c = &j->claims[j->idx[i]];
    dra_claim_rec t = *c;
    if (j->use_override) t.node = j->node_override;
    return t.kind == DRA_KIND_MIG && t.group == group && !claim_invalid(&t, j->n_node, have_off);
}

/* spec §2: the node's claims, sequentially, input order */
static void node_process(node_job* j)
{
    int have_off = j->out_off != NULL;
    j->all_ok = 1;
    uint32_t i = 0;
    while (i < j->cnt) {
        uint32_t ci = j->idx[i];
        dra_claim_rec c = j->claims[ci];
        if (j->use_override) c.node = j->node_override;
        if (claim_invalid(&c, j->n_node, have_off)) {
            fail_all(slot_of(j, ci), claim_slots(&c, j->n_node, have_off), &c, DRA_ST_INVALID);
            j->all_ok = 0; i++; continue;
        }
        if (c.kind == DRA_KIND_MIG && c.group != 0) {
            uint32_t e = i + 1;
            while (e < j->cnt && e - i < DRA_MAX_GROUP && in_run(j, e, c.group, have_off)) e++;
            do_group(j, i, e);
            i = e; continue;
        }
        if (c.kind == DRA_KIND_GPU) do_gpu(j, ci);
        else if (c.kind == DRA_KIND_MIG) do_mig(j, ci);
        else do_shared(j, ci);
        i++;
    }
}

/* ------------------------------------------------------------------------------------------------ */

static int check_inventory(const dra_gpu_rec* gpus, uint32_t n_gpu, const uint32_t* node_off,
                           uint32_t n_node, const dra_profile_tbl* tbl)
{
    if (node_off[0] != 0 || node_off[n_node] != n_gpu) return -1;
    for (uint32_t n = 0; n < n_node; n++) {
        if (node_off[n + 1] < node_off[n]) return -1;
        if (node_off[n + 1] - node_off[n] > DRA_MAX_GPUS_PER_NODE) return -1;
        for (uint32_t g = node_off[n]; g < node_off[n + 1]; g++) {
            if (gpus[g].model >= DRA_MAX_MODELS) return -1;
            if (gpus[g].node != n) return -1;
        }
    }
    for (uint32_t m = 0; m < DRA_MAX_MODELS; m++)
        for (uint32_t p = 0; p < DRA_MAX_PROFILES; p++) {
            dra_prof_ent e = tbl[m].ent[p];
            if (!e.start_mask) continue;
            if (e.size < 1 || e.size > 16) return -1;
            int hi = 15; while (!((e.start_mask >> hi) & 1u)) hi--;
            if (hi + e.size > 16) return -1;
        }
    return 0;
}

typedef struct bucketed {
    uint32_t* idx;       /* claim indices, stable by node */
    uint32_t* off;       /* n_node+1 */
} bucketed;

/* stable counting sort of claim indices by node (spec §2); claims with node >= n_node are left out */
static int bucket(const dra_claim_rec* claims, uint32_t n_claim, uint32_t n_node, bucketed* b)
{
    b->off = (uint32_t*)calloc((size_t)n_node + 2, sizeof(uint32_t));
    b->idx = (uint32_t*)malloc(((size_t)n_claim + 1) * sizeof(uint32_t));
    if (!b->off || !b->idx) return -1;
    for (uint32_t i = 0; i < n_claim; i++)
        if (claims[i].node < n_node) b->off[claims[i].node + 1]++;
    for (uint32_t n = 0; n < n_node; n++) b->off[n + 1] += b->off[n];
    uint32_t* cur = (uint32_t*)malloc(((size_t)n_node + 1) * sizeof(uint32_t));
    if (!cur) return -1;
    memcpy(cur, b->off, ((size_t)n_node + 1) * sizeof(uint32_t));
    for (uint32_t i = 0; i < n_claim; i++)
        if (claims[i].node < n_node) b->idx[cur[claims[i].node]++] = i;
    free(cur);
    return 0;
}

typedef struct mt_arg {
    dra_gpu_rec* gpus; const uint32_t* node_off; uint32_t n_node;
    const dra_profile_tbl* tbl; const dra_claim_rec* claims;
    const bucketed* b; const uint32_t* out_off; dra_out_rec* out;
    uint32_t n0, n1;
} mt_arg;

static void run_nodes(const mt_arg* a)
{
    for (uint32_t n = a->n0; n < a->n1; n++) {
        node_job j;
        memset(&j, 0, sizeof j);
        j.gpus = a->gpus + a->node_off[n];
        j.g0 = a->node_off[n];
        j.ng = a->node_off[n + 1] - a->node_off[n];
        j.tbl = a->tbl; j.claims = a->claims;
        j.idx = a->b->idx + a->b->off[n];
        j.cnt = a->b->off[n + 1] - a->b->off[n];
        j.n_node = a->n_node; j.out_off = a->out_off; j.out = a->out; j.commit = 1;
        node_process(&j);
    }
}

/* ---- persistent worker pool for the multi-threaded variant --------------------------------------------
 * Nodes are independent (spec §2), a node costs microseconds: creating threads per call costs more than the
 * batch, so the workers are created once, take nodes one at a time from an atomic counter, and wait for the next
 * batch by spinning briefly before they sleep on a condition variable. */
#include <stdatomic.h>
#include <sched.h>

static struct {
    pthread_t* th; int n;                       /* workers (the caller works too) */
    _Atomic uint64_t gen;                       /* batch generation */
    uint64_t start_gen;                         /* gen when the current workers were created */
    _Atomic uint32_t next, done;                /* next node to take; workers finished with this generation */
    const mt_arg* job;
    _Atomic int stop, sleepers;
    pthread_mutex_t mu; pthread_cond_t cv;
} pool = { .mu = PTHREAD_MUTEX_INITIALIZER, .cv = PTHREAD_COND_INITIALIZER };

static void take_nodes(const mt_arg* a)
{
    for (;;) {
        uint32_t n = atomic_fetch_add_explicit(&pool.next, 1u, memory_order_relaxed);
        if (n >= a->n_node) return;
        mt_arg one = *a; one.n0 = n; one.n1 = n + 1;
        run_nodes(&one);
    }
}

static void* pool_worker(void* unused)
{
    (void)unused;
    uint64_t seen = pool.start_gen;             /* batches before this worker existed are not its business */
    for (;;) {
        uint32_t spins = 0;
        while (atomic_load_explicit(&pool.gen, memory_order_acquire) == seen && !atomic_load(&pool.stop)) {
            if (++spins < 20000u) { __builtin_ia32_pause(); continue; }
            pthread_mutex_lock(&pool.mu);                    /* idle for a while: sleep until the next batch */
            atomic_fetch_add(&pool.sleepers, 1);
            while (atomic_load_explicit(&pool.gen, memory_order_acquire) == seen && !atomic_load(&pool.stop))
                pthread_cond_wait(&pool.cv, &pool.mu);
            atomic_fetch_sub(&pool.sleepers, 1);
            pthread_mutex_unlock(&pool.mu);
        }
        if (atomic_load(&pool.stop)) return NULL;
        seen = atomic_load_explicit(&pool.gen, memory_order_acquire);
        take_nodes(pool.job);
        atomic_fetch_add_explicit(&pool.done, 1u, memory_order_release);
    }
}

static void pool_shutdown(void)
{
    if (!pool.n) return;
    pthread_mutex_lock(&pool.mu);
    atomic_store(&pool.stop, 1);
    pthread_cond_broadcast(&pool.cv);
    pthread_mutex_unlock(&pool.mu);
    for (int t = 0; t < pool.n; t++) pthread_join(pool.th[t], NULL);
    free(pool.th); pool.th = NULL; pool.n = 0;
    atomic_store(&pool.stop, 0);
}

/* a forked child has none of the parent's worker threads: start from an empty pool there */
static void pool_after_fork_child(void)
{
    pool.th = NULL; pool.n = 0;
    atomic_store(&pool.stop, 0); atomic_store(&pool.sleepers, 0);
    pthread_mutex_init(&pool.mu, NULL); pthread_cond_init(&pool.cv, NULL);
}

static int pool_resize(int workers)
{
    if (workers == pool.n) return 0;
    pool_shutdown();
    if (workers <= 0) return 0;
    pool.th = (pthread_t*)malloc(sizeof(pthread_t) * (size_t)workers);
    if (!pool.th) return -1;
    static int at_exit_set;
    if (!at_exit_set) { atexit(pool_shutdown); pthread_atfork(NULL, NULL, pool_after_fork_child); at_exit_set = 1; }
    pool.start_gen = atomic_load(&pool.gen);
    for (int t = 0; t < workers; t++)
        if (pthread_create(&pool.th[t], NULL, pool_worker, NULL)) { pool.n = t; pool_shutdown(); return -1; }
    pool.n = workers;
    return 0;
}

int dra_oracle_allocate_mt(dra_gpu_rec* gpus, uint32_t n_gpu, const uint32_t* node_off, uint32_t n_node,
                           const dra_profile_tbl* tbl,
                           const dra_claim_rec* claims, uint32_t n_claim,
                           const uint32_t* out_off, dra_out_rec* out, uint32_t n_out, int n_threads)
{
    if (check_inventory(gpus, n_gpu, node_off, n_node, tbl)) return -1;
    int have_off = out_off != NULL;
    for (uint32_t i = 0; i < n_claim; i++) {
        uint32_t base = have_off ? out_off[i] : i;
        uint32_t sl = claim_slots(&claims[i], n_node, have_off);
        if (base > n_out || sl > n_out - base) return -1;
    }
    /* claims that name no node of the inventory: INVALID, no state touched (spec §3) */
    for (uint32_t i = 0; i < n_claim; i++)
        if (claims[i].node >= n_node)
            put(&out[have_off ? out_off[i] : i], DRA_GPU_NONE, 0, 0, out_profile(&claims[i]), DRA_ST_INVALID);

    bucketed b;
    if (bucket(claims, n_claim, n_node, &b)) return -1;

    mt_arg base = { gpus, node_off, n_node, tbl, claims, &b, out_off, out, 0, n_node };
    if ((uint32_t)n_threads > n_node) n_threads = (int)n_node;
    if (n_threads <= 1 || n_node < 2 || pool_resize(n_threads - 1)) {
        run_nodes(&base);
    } else {
        /* the caller and n_threads-1 pool workers take nodes one at a time (dynamic balance) */
        pool.job = &base;
        atomic_store_explicit(&pool.next, 0u, memory_order_relaxed);
        atomic_store_explicit(&pool.done, 0u, memory_order_relaxed);
        atomic_fetch_add_explicit(&pool.gen, 1u, memory_order_release);
        if (atomic_load(&pool.sleepers)) {
            pthread_mutex_lock(&pool.mu); pthread_cond_broadcast(&pool.cv); pthread_mutex_unlock(&pool.mu);
        }
        take_nodes(&base);
        while (atomic_load_explicit(&pool.done, memory_order_acquire) != (uint32_t)pool.n) __builtin_ia32_pause();
    }
    free(b.idx); free(b.off);
    return 0;
}

int dra_oracle_allocate(dra_gpu_rec* gpus, uint32_t n_gpu, const uint32_t* node_off, uint32_t n_node,
                        const dra_profile_tbl* tbl,
                        const dra_claim_rec* claims, uint32_t n_claim,
                        const uint32_t* out_off, dra_out_rec* out, uint32_t n_out)
{
    return dra_oracle_allocate_mt(gpus, n_gpu, node_off, n_node, tbl, claims, n_claim, out_off, out,
                                  n_out, 1);
}

/* spec §8 — all-or-nothing per pod on a snapshot of the candidate node (SURVEY App. A) */
int dra_oracle_unsuitable(const dra_gpu_rec* gpus, uint32_t n_gpu, const uint32_t* node_off,
                          uint32_t n_node, const dra_profile_tbl* tbl,
                          const dra_claim_rec* claims, uint32_t n_claim,
                          const uint32_t* pod_off, uint32_t n_pod,
                          const uint32_t* cand_nodes, const uint32_t* cand_off, uint8_t* suitable_bits)
{
    if (check_inventory(gpus, n_gpu, node_off, n_node, tbl)) return -1;
    if (pod_off[n_pod] != n_claim) return -1;
    uint32_t n_pair = cand_off[n_pod];
    memset(suitable_bits, 0, ((size_t)n_pair + 7) / 8);

    /* scratch: per-claim slot offsets (prefix of slots) and a scratch out array */
    uint32_t* soff = (uint32_t*)malloc(((size_t)n_claim + 1) * sizeof(uint32_t));
    uint32_t* idx = (uint32_t*)malloc(((size_t)n_claim + 1) * sizeof(uint32_t));
    if (!soff || !idx) return -1;
    for (uint32_t i = 0; i < n_claim; i++) idx[i] = i;

    for (uint32_t p = 0; p < n_pod; p++) {
        uint32_t c0 = pod_off[p], c1 = pod_off[p + 1];
        for (uint32_t k = cand_off[p]; k < cand_off[p + 1]; k++) {
            uint32_t n = cand_nodes[k];
            if (n >= n_node) continue;                       /* unknown node: unsuitable */
            uint32_t tot = 0;
            for (uint32_t i = c0; i < c1; i++) {
                dra_claim_rec t = claims[i]; t.node = n;
                soff[i] = tot; tot += claim_slots(&t, n_node, 1);
            }
            dra_out_rec* scratch = (dra_out_rec*)malloc(((size_t)tot + 1) * sizeof(dra_out_rec));
            dra_gpu_rec snap[DRA_MAX_GPUS_PER_NODE];
            uint32_t ng = node_off[n + 1] - node_off[n];
            memcpy(snap, gpus + node_off[n], ng * sizeof(dra_gpu_rec));
            node_job j;
            memset(&j, 0, sizeof j);
            j.gpus = snap; j.g0 = node_off[n]; j.ng = ng; j.tbl = tbl; j.claims = claims;
            j.idx = idx + c0; j.cnt = c1 - c0; j.n_node = n_node;
            j.out_off = soff; j.out = scratch;
            j.use_override = 1; j.node_override = n;
            node_process(&j);
            if (j.all_ok) suitable_bits[k >> 3] |= (uint8_t)(1u << (k & 7));
            free(scratch);
        }
    }
    free(soff); free(idx);
    return 0;
}

/* ---- spec §12: pod mode and the exhaustive placement search ------------------------------------------------
 * The enumeration that is searched is the (profile, placement) list deviceLib.getGpuInfo collects per GPU
 * (cmd/nvidia-dra-plugin/nvlib.go:244-295); the multi-request shape is demo/specs/quickstart/gpu-test4.yaml:19-44;
 * the search itself follows the recollected classic mig.allocate (SURVEY App. A) — PARITY UNPINNED. */

typedef struct pod_search {
    dra_gpu_rec* gpus; uint32_t g0, ng;
    const dra_profile_tbl* tbl;
    const dra_claim_rec* claims;        /* the pod's claims */
    const uint32_t* mig; uint32_t k;    /* positions of the MIG claims inside the pod */
    int exhaustive;
    uint32_t descents; int limit_hit;
    int gpu_of[DRA_MAX_POD], start_of[DRA_MAX_POD];     /* per level */
} pod_search;

/* level i: canonical order = GPUs ascending, starts ascending; returns 1 when levels i.. are all placed */
static int pod_dfs(pod_search* ps, uint32_t i)
{
    if (i == ps->k) return 1;
    const dra_claim_rec* c = &ps->claims[ps->mig[i]];
    int want_gpu = -1;                                  /* co-location: the GPU of the first earlier member */
    if (c->group != 0)
        for (uint32_t j = 0; j < i; j++)
            if (ps->claims[ps->mig[j]].group == c->group) { want_gpu = ps->gpu_of[j]; break; }
    for (uint32_t g = 0; g < ps->ng; g++) {
        if (want_gpu >= 0 && (int)g != want_gpu) continue;
        dra_gpu_rec* r = &ps->gpus[g];
        dra_prof_ent e = ps->tbl[r->model].ent[c->profile];
        if (!gpu_offers(r, e) || (r->flags & DRA_GPU_FULL_ALLOCATED)) continue;
        if (!sel_pass(claim_sel(c), ps->g0 + g)) continue;
        for (int s = 0; s < 16; s++) {
            if (!((e.start_mask >> s) & 1u)) continue;
            uint16_t m = (uint16_t)(((1u << e.size) - 1u) << s);
            if (r->busy & m) continue;
            if (ps->descents == DRA_EXH_BUDGET) { ps->limit_hit = 1; return 0; }
            ps->descents++;
            r->busy |= m; ps->gpu_of[i] = (int)g; ps->start_of[i] = s;
            if (pod_dfs(ps, i + 1)) return 1;
            r->busy &= (uint16_t)~m;
            if (ps->limit_hit || !ps->exhaustive) return 0;      /* first-fit: the first branch only */
        }
    }
    return 0;
}

/* Evaluate one pod on the node whose GPUs are gpus[0..ng) (mutated only on success).  claims[0..cnt) are the
 * pod's claims (node already validated / overridden by the caller), slot[i] = first OutRec of claim i in out
 * (out may be NULL: evaluate only).  Returns 1 when the pod was placed. */
static int pod_eval(dra_gpu_rec* gpus, uint32_t g0, uint32_t ng, const dra_profile_tbl* tbl,
                    const dra_claim_rec* claims, uint32_t cnt, uint32_t n_node, int have_off,
                    const uint32_t* slot, dra_out_rec* out, int exhaustive)
{
    dra_out_rec scratch[DRA_MAX_POD * DRA_MAX_COUNT];
    uint32_t sslot[DRA_MAX_POD];
    if (!out) {                                          /* evaluate only: private slots */
        uint32_t t = 0;
        for (uint32_t i = 0; i < cnt; i++) { sslot[i] = t; t += claim_slots(&claims[i], n_node, have_off); }
        out = scratch; slot = sslot;
    }
    int any_invalid = 0;
    for (uint32_t i = 0; i < cnt; i++) if (claim_invalid(&claims[i], n_node, have_off)) any_invalid = 1;
    uint8_t fail_st = DRA_ST_POD;
    int ok = !any_invalid;
    dra_gpu_rec work[DRA_MAX_GPUS_PER_NODE];
    memcpy(work, gpus, ng * sizeof(dra_gpu_rec));
    uint32_t mig[DRA_MAX_POD], k = 0;
    if (ok) {                                            /* step 2: GPU and SHARED claims, in order, §4 / §7 */
        uint32_t idx[DRA_MAX_POD];
        for (uint32_t i = 0; i < cnt; i++) idx[i] = i;
        node_job j; memset(&j, 0, sizeof j);
        j.gpus = work; j.g0 = g0; j.ng = ng; j.tbl = tbl; j.claims = claims; j.idx = idx; j.cnt = cnt;
        j.n_node = n_node; j.out_off = slot; j.out = out; j.all_ok = 1;
        for (uint32_t i = 0; i < cnt && j.all_ok; i++) {
            if (claims[i].kind == DRA_KIND_GPU) do_gpu(&j, i);
            else if (claims[i].kind == DRA_KIND_SHARED) do_shared(&j, i);
            else mig[k++] = i;
        }
        ok = j.all_ok;
    }
    pod_search ps; memset(&ps, 0, sizeof ps);
    for (uint32_t i = 0; ok && i < k; i++) {             /* step 3 pre-check: a claim with no placement at all in S' sinks the pod */
        const dra_claim_rec* c = &claims[mig[i]];
        int any = 0;
        for (uint32_t g = 0; g < ng && !any; g++) {
            dra_prof_ent e = tbl[work[g].model].ent[c->profile];
            if (!gpu_offers(&work[g], e) || (work[g].flags & DRA_GPU_FULL_ALLOCATED) || !sel_pass(claim_sel(c), g0 + g)) continue;
            any = lowest_fit(work[g].busy, e) >= 0;
        }
        if (!any) ok = 0;
    }
    if (ok && k) {                                       /* step 3: the MIG claims, canonical DFS */
        ps.gpus = work; ps.g0 = g0; ps.ng = ng; ps.tbl = tbl; ps.claims = claims; ps.mig = mig; ps.k = k;
        ps.exhaustive = exhaustive;
        ok = pod_dfs(&ps, 0);
        if (!ok && ps.limit_hit) fail_st = DRA_ST_SEARCH_LIMIT;
    }
    if (ok) {
        for (uint32_t i = 0; i < k; i++) {
            const dra_claim_rec* c = &claims[mig[i]];
            dra_prof_ent e = tbl[work[ps.gpu_of[i]].model].ent[c->profile];
            put(&out[slot[mig[i]]], g0 + (uint32_t)ps.gpu_of[i], (uint8_t)ps.start_of[i], e.size, c->profile, DRA_ST_OK);
        }
        memcpy(gpus, work, ng * sizeof(dra_gpu_rec));
        return 1;
    }
    for (uint32_t i = 0; i < cnt; i++) {
        int inv = claim_invalid(&claims[i], n_node, have_off);
        fail_all(&out[slot[i]], claim_slots(&claims[i], n_node, have_off), &claims[i], inv ? DRA_ST_INVALID : fail_st);
    }
    return 0;
}

int dra_oracle_allocate_pods(dra_gpu_rec* gpus, uint32_t n_gpu, const uint32_t* node_off, uint32_t n_node,
                             const dra_profile_tbl* tbl, const dra_claim_rec* claims, uint32_t n_claim,
                             const uint32_t* pod_off, uint32_t n_pod,
                             const uint32_t* out_off, dra_out_rec* out, uint32_t n_out, uint32_t flags)
{
    if (check_inventory(gpus, n_gpu, node_off, n_node, tbl)) return -1;
    if (pod_off[0] != 0 || pod_off[n_pod] != n_claim) return -1;
    int have_off = out_off != NULL;
    uint32_t* slot = (uint32_t*)malloc(((size_t)n_claim + 1) * sizeof(uint32_t));
    if (!slot) return -1;
    for (uint32_t i = 0; i < n_claim; i++) {
        slot[i] = have_off ? out_off[i] : i;
        uint32_t sl = claim_slots(&claims[i], n_node, have_off);
        if (slot[i] > n_out || sl > n_out - slot[i]) { free(slot); return -1; }
    }
    /* pods in input order; a pod touches one node only, so "per node in input order" is just input order */
    for (uint32_t p = 0; p < n_pod; p++) {
        uint32_t c0 = pod_off[p], c1 = pod_off[p + 1];
        if (c1 < c0) { free(slot); return -1; }
        uint32_t cnt = c1 - c0;
        if (cnt == 0) continue;
        uint32_t node = claims[c0].node;
        int malformed = cnt > DRA_MAX_POD || node >= n_node;
        for (uint32_t i = c0; i < c1 && !malformed; i++) if (claims[i].node != node) malformed = 1;
        if (malformed) {
            for (uint32_t i = c0; i < c1; i++)
                fail_all(&out[slot[i]], claim_slots(&claims[i], n_node, have_off), &claims[i], DRA_ST_INVALID);
            continue;
        }
        pod_eval(gpus + node_off[node], node_off[node], node_off[node + 1] - node_off[node], tbl,
                 claims + c0, cnt, n_node, have_off, slot + c0, out, (flags & DRA_F_EXHAUSTIVE) != 0);
    }
    free(slot);
    return 0;
}

/* spec §12: UnsuitableNodes with DRA_F_EXHAUSTIVE — a node is unsuitable only if NO assignment of the pod exists */
int dra_oracle_unsuitable_ex(const dra_gpu_rec* gpus, uint32_t n_gpu, const uint32_t* node_off,
                             uint32_t n_node, const dra_profile_tbl* tbl,
                             const dra_claim_rec* claims, uint32_t n_claim,
                             const uint32_t* pod_off, uint32_t n_pod,
                             const uint32_t* cand_nodes, const uint32_t* cand_off, uint8_t* suitable_bits,
                             uint32_t flags)
{
    if (!(flags & DRA_F_EXHAUSTIVE))
        return dra_oracle_unsuitable(gpus, n_gpu, node_off, n_node, tbl, claims, n_claim, pod_off, n_pod,
                                     cand_nodes, cand_off, suitable_bits);
    if (check_inventory(gpus, n_gpu, node_off, n_node, tbl)) return -1;
    if (pod_off[n_pod] != n_claim) return -1;
    uint32_t n_pair = cand_off[n_pod];
    memset(suitable_bits, 0, ((size_t)n_pair + 7) / 8);
    for (uint32_t p = 0; p < n_pod; p++) {
        uint32_t c0 = pod_off[p], cnt = pod_off[p + 1] - pod_off[p];
        if (cnt > DRA_MAX_POD) continue;                          /* unsuitable everywhere */
        for (uint32_t kk = cand_off[p]; kk < cand_off[p + 1]; kk++) {
            uint32_t n = cand_nodes[kk];
            if (n >= n_node) continue;
            dra_claim_rec pod[DRA_MAX_POD];
            for (uint32_t i = 0; i < cnt; i++) { pod[i] = claims[c0 + i]; pod[i].node = n; }
            dra_gpu_rec snap[DRA_MAX_GPUS_PER_NODE];
            uint32_t ng = node_off[n + 1] - node_off[n];
            memcpy(snap, gpus + node_off[n], ng * sizeof(dra_gpu_rec));
            if (pod_eval(snap, node_off[n], ng, tbl, pod, cnt, n_node, 1, NULL, NULL, 1))
                suitable_bits[kk >> 3] |= (uint8_t)(1u << (kk & 7));
        }
    }
    return 0;
}

/* spec §9 */
int dra_oracle_deallocate(dra_gpu_rec* gpus, uint32_t n_gpu, uint32_t n_node,
                          const dra_claim_rec* claims, uint32_t n_claim,
                          const uint32_t* out_off, const dra_out_rec* out, uint32_t n_out)
{
    int have_off = out_off != NULL;
    for (uint32_t i = 0; i < n_claim; i++) {
        const dra_claim_rec* c = &claims[i];
        uint32_t base = have_off ? out_off[i] : i;
        /* slots(c) of spec §1/§3, the same as Allocate used: an INVALID claim (here: naming no node) has one */
        uint32_t sl = (c->kind == DRA_KIND_GPU && c->node < n_node && c->count >= 1 && c->count <= DRA_MAX_COUNT &&
                       (have_off || c->count == 1)) ? c->count : 1;
        if (base > n_out || sl > n_out - base) return -1;
        for (uint32_t k = 0; k < sl; k++) {
            const dra_out_rec* o = &out[base + k];
            if (o->status != DRA_ST_OK || o->gpu >= n_gpu) continue;
            dra_gpu_rec* r = &gpus[o->gpu];
            if (c->kind == DRA_KIND_GPU) r->flags &= (uint8_t)~DRA_GPU_FULL_ALLOCATED;
            else if (c->kind == DRA_KIND_MIG)
                r->busy &= (uint16_t)~(((1u << o->size) - 1u) << o->start);
            else if (c->kind == DRA_KIND_SHARED) { r->mem_free_mib += c->mem_limit_mib; r->share_cnt--; }
        }
    }
    return 0;
}

/* api/nvidia.com/resource/gpu/v1alpha1/sharing.go:234-237:
 *     v := d.Value() / 1024 / 1024 ; return fmt.Sprintf("%vM", v), v > 0          */
int64_t dra_oracle_megabyte(int64_t bytes, int* valid)
{
    int64_t v = bytes / 1024 / 1024;     /* C99 '/' truncates toward zero, as Go's does */
    if (valid) *valid = v > 0;
    return v;
}

/* cmd/nvidia-dra-controller/imex.go:336-349 */
int32_t dra_oracle_imex_offset(const int32_t* used, uint32_t n_used, int32_t step, int32_t limit)
{
    for (int32_t off = 0; off < limit; off += step) {
        int taken = 0;
        for (uint32_t k = 0; k < n_used; k++) if (used[k] == off) { taken = 1; break; }
        if (!taken) return off;
    }
    return -1;
}
