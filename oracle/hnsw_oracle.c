/*
 *  oracle/hnsw_oracle.c — TEST INFRASTRUCTURE, not product code.
 *
 *  Plain-C restatement ("port") of the reference's HNSW search path, written from the reference's
 *  behaviour, with each routine citing the file:line under /root/reference/include/usearch it
 *  follows. Only tests/, __graft_entry__.smoke() and bench.py's CPU arms may load this library;
 *  the product (usearch_b200/) never links or calls it.
 *
 *  Parity status: PINNED. tests/test_oracle.py checks this port against (a) the tiny known-answer
 *  vectors the reference's own test-suites hold (javascript/usearch.test.js:60-84,161-191;
 *  golang/lib_test.go:835-877; cpp/test.cpp:1071-1099), (b) committed golden fixtures under
 *  tests/golden/ that were produced by running the unmodified reference (oracle/_ref, script
 *  tests/golden/make_golden.py), and (c) the live reference library when oracle/_ref is present.
 *
 *  Input is the reference's own serialised index (v2 format):
 *    index_dense.hpp:994-1062  [u32 rows, u32 cols][rows*cols vector bytes][64-byte head]
 *    index.hpp:3276-3317       [40-byte graph header][int16 levels][node tapes]
 *    index.hpp:2116-2195       node tape = key u64 | level i16 | {u32 n, slot[M0]} | level x {u32 n, slot[M]}
 */
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "metrics_pinned.h"

typedef float (*oracle_metric_t)(void const*, void const*, size_t);

typedef struct oracle_index_t {
    uint8_t const* blob;
    size_t blob_length;
    /* dense head (index_dense.hpp:42-79) */
    uint8_t metric_kind, scalar_kind;
    uint64_t dimensions, count_present, count_deleted;
    size_t bytes_per_vector;
    uint8_t const* vectors; /* slot-major matrix inside the blob */
    /* graph header (index.hpp:1863-1869) */
    uint64_t size, connectivity, connectivity_base, max_level, entry_slot;
    int16_t const* levels;    /* unaligned in the blob: read with memcpy */
    uint64_t* node_offsets;   /* byte offset of every node tape inside the blob */
    size_t neighbors_bytes, neighbors_base_bytes; /* index.hpp:3731-3737 precompute_ */
    oracle_metric_t metric;
    size_t metric_third; /* dimensions, or bytes for b1x8 (index_plugins.hpp:1743-1744) */
    uint64_t free_key;   /* index_dense.hpp:513: default_free_value<u64>() == UINT64_MAX */
    size_t expansion_search;
} oracle_index_t;

/* ---------- metric table ----------------------------------------------------------------- */

#define WRAP(name, type)                                                                         \
    static float wrap_##name(void const* a, void const* b, size_t n) {                           \
        return pinned_##name((type const*)a, (type const*)b, n);                                 \
    }
WRAP(l2sq_f32, float) WRAP(ip_f32, float) WRAP(cos_f32, float)
WRAP(l2sq_f16, uint16_t) WRAP(ip_f16, uint16_t) WRAP(cos_f16, uint16_t)
WRAP(l2sq_bf16, uint16_t) WRAP(ip_bf16, uint16_t) WRAP(cos_bf16, uint16_t)
WRAP(l2sq_i8, int8_t) WRAP(ip_i8, int8_t) WRAP(cos_i8, int8_t)
WRAP(hamming_b1, uint8_t) WRAP(tanimoto_b1, uint8_t) WRAP(sorensen_b1, uint8_t)

/* enum values: index_plugins.hpp:113-159 */
enum { SK_B1 = 1, SK_BF16 = 4, SK_F64 = 10, SK_F32 = 11, SK_F16 = 12, SK_I8 = 23 };

static oracle_metric_t pick_metric(uint8_t m, uint8_t s) {
    switch (s) {
    case SK_F32: return m == 'e' ? wrap_l2sq_f32 : m == 'i' ? wrap_ip_f32 : m == 'c' ? wrap_cos_f32 : NULL;
    case SK_F16: return m == 'e' ? wrap_l2sq_f16 : m == 'i' ? wrap_ip_f16 : m == 'c' ? wrap_cos_f16 : NULL;
    case SK_BF16: return m == 'e' ? wrap_l2sq_bf16 : m == 'i' ? wrap_ip_bf16 : m == 'c' ? wrap_cos_bf16 : NULL;
    case SK_I8: return m == 'e' ? wrap_l2sq_i8 : m == 'i' ? wrap_ip_i8 : m == 'c' ? wrap_cos_i8 : NULL;
    case SK_B1:
        return m == 'b' ? wrap_hamming_b1 : (m == 't' || m == 'j') ? wrap_tanimoto_b1 : m == 's' ? wrap_sorensen_b1 : NULL;
    default: return NULL;
    }
}

static size_t bits_per_scalar(uint8_t s) { /* index_plugins.hpp:237-257 */
    switch (s) {
    case SK_B1: return 1;
    case SK_I8: return 8;
    case SK_F16: case SK_BF16: return 16;
    case SK_F32: return 32;
    case SK_F64: return 64;
    default: return 0;
    }
}

/* ---------- blob parsing ------------------------------------------------------------------ */

static uint64_t rd_u64(uint8_t const* p) { uint64_t v; memcpy(&v, p, 8); return v; }
static uint32_t rd_u32(uint8_t const* p) { uint32_t v; memcpy(&v, p, 4); return v; }
static int16_t rd_i16(uint8_t const* p) { int16_t v; memcpy(&v, p, 2); return v; }

void oracle_close(oracle_index_t* ix) {
    if (!ix) return;
    free(ix->node_offsets);
    free(ix);
}

/* The blob is borrowed (like the reference's `view`, index_dense.hpp:1198-1313): keep it alive. */
oracle_index_t* oracle_open(void const* buffer, size_t length, char const** error) {
    *error = NULL;
    uint8_t const* p = (uint8_t const*)buffer;
    uint8_t const* end = p + length;
    oracle_index_t* ix = (oracle_index_t*)calloc(1, sizeof(*ix));
    if (!ix) { *error = "Out of memory!"; return NULL; }
    ix->blob = p;
    ix->blob_length = length;
    ix->free_key = UINT64_MAX;
    ix->expansion_search = 64; /* index.hpp:1350 default_expansion_search */

    if (length < 8 + 64 + 40) { *error = "File is corrupted and lacks matrix dimensions"; goto fail; }
    uint64_t rows = rd_u32(p), cols = rd_u32(p + 4);
    p += 8;
    if ((uint64_t)(end - p) < rows * cols + 64 + 40) { *error = "File is corrupted and lacks a header"; goto fail; }
    ix->vectors = p;
    p += rows * cols;

    /* 64-byte head: "usearch" magic, 3 x u16 version, metric, scalar, key kind, slot kind,
     * count_present, count_deleted, dimensions, multi */
    if (memcmp(p, "usearch", 7) != 0) { *error = "Magic header mismatch - the file isn't an index"; goto fail; }
    ix->metric_kind = p[13];
    ix->scalar_kind = p[14];
    ix->count_present = rd_u64(p + 17);
    ix->count_deleted = rd_u64(p + 25);
    ix->dimensions = rd_u64(p + 33);
    p += 64;
    ix->bytes_per_vector = (ix->dimensions * bits_per_scalar(ix->scalar_kind) + 7) / 8;
    if (rows && cols != ix->bytes_per_vector) { *error = "Matrix columns do not match bytes per vector"; goto fail; }
    ix->metric = pick_metric(ix->metric_kind, ix->scalar_kind);
    if (!ix->metric) { *error = "Unknown metric kind!"; goto fail; }
    ix->metric_third = ix->scalar_kind == SK_B1 ? (ix->dimensions + 7) / 8 : ix->dimensions;

    ix->size = rd_u64(p);
    ix->connectivity = rd_u64(p + 8);
    ix->connectivity_base = rd_u64(p + 16);
    ix->max_level = rd_u64(p + 24);
    ix->entry_slot = rd_u64(p + 32);
    p += 40;
    if (ix->size != rows) { *error = "Index size and the number of vectors doesn't match"; goto fail; }
    ix->neighbors_bytes = ix->connectivity * 4 + 4;
    ix->neighbors_base_bytes = ix->connectivity_base * 4 + 4;
    if ((uint64_t)(end - p) < ix->size * 2) { *error = "File is corrupted and can't fit all the levels"; goto fail; }
    ix->levels = (int16_t const*)p;
    uint8_t const* levels_bytes = p;
    p += ix->size * 2;
    ix->node_offsets = (uint64_t*)malloc((ix->size + 1) * sizeof(uint64_t));
    if (!ix->node_offsets) { *error = "Out of memory!"; goto fail; }
    for (uint64_t i = 0; i < ix->size; ++i) {
        int16_t level = rd_i16(levels_bytes + 2 * i);
        size_t node_bytes = 10 + ix->neighbors_base_bytes + ix->neighbors_bytes * (size_t)level;
        if ((size_t)(end - p) < node_bytes) { *error = "File is corrupted and can't fit all the nodes"; goto fail; }
        ix->node_offsets[i] = (uint64_t)(p - ix->blob);
        p += node_bytes;
    }
    return ix;
fail:
    oracle_close(ix);
    return NULL;
}

size_t oracle_size(oracle_index_t const* ix) { return ix->size; }
size_t oracle_dimensions(oracle_index_t const* ix) { return ix->dimensions; }
size_t oracle_connectivity(oracle_index_t const* ix) { return ix->connectivity; }
size_t oracle_max_level(oracle_index_t const* ix) { return ix->max_level; }
size_t oracle_bytes_per_vector(oracle_index_t const* ix) { return ix->bytes_per_vector; }
int oracle_metric_kind(oracle_index_t const* ix) { return ix->metric_kind; }
int oracle_scalar_kind(oracle_index_t const* ix) { return ix->scalar_kind; }
void oracle_change_expansion_search(oracle_index_t* ix, size_t ef) { ix->expansion_search = ef; }

float oracle_distance(oracle_index_t const* ix, void const* a, void const* b) {
    return ix->metric(a, b, ix->metric_third);
}

/* ---------- containers -------------------------------------------------------------------- */

typedef struct { float distance; uint32_t slot; } candidate_t; /* index.hpp:2097-2101 */

/* max_heap_gt (index.hpp:664-835) holding {-distance, slot}: compare on distance only */
typedef struct { candidate_t* e; size_t size, capacity; } heap_t;

static size_t ceil2(size_t v) { size_t r = 1; while (r < v) r <<= 1; return r; }

static int heap_reserve(heap_t* h, size_t n) { /* :727-746 */
    if (n < h->capacity) return 1;
    size_t cap = ceil2(n);
    size_t alt = h->capacity * 2 > 16 ? h->capacity * 2 : 16;
    if (cap < alt) cap = alt;
    candidate_t* e = (candidate_t*)realloc(h->e, cap * sizeof(candidate_t));
    if (!e) return 0;
    h->e = e;
    h->capacity = cap;
    return 1;
}
static void heap_shift_up(heap_t* h, size_t i) { /* :808-811: swap while parent < child, strictly */
    for (; i && h->e[(i - 1) / 2].distance < h->e[i].distance; i = (i - 1) / 2) {
        candidate_t t = h->e[(i - 1) / 2]; h->e[(i - 1) / 2] = h->e[i]; h->e[i] = t;
    }
}
static void heap_shift_down(heap_t* h, size_t i) { /* :819-834 */
    for (;;) {
        size_t max_idx = i, left = 2 * i + 1, right = 2 * i + 2;
        if (left < h->size && h->e[max_idx].distance < h->e[left].distance) max_idx = left;
        if (right < h->size && h->e[max_idx].distance < h->e[right].distance) max_idx = right;
        if (max_idx == i) return;
        candidate_t t = h->e[i]; h->e[i] = h->e[max_idx]; h->e[max_idx] = t;
        i = max_idx;
    }
}
static int heap_insert(heap_t* h, candidate_t c) { /* :753-770 */
    if (!heap_reserve(h, h->size + 1)) return 0;
    h->e[h->size++] = c;
    heap_shift_up(h, h->size - 1);
    return 1;
}
static void heap_pop(heap_t* h) { /* :786-794 */
    candidate_t t = h->e[0]; h->e[0] = h->e[h->size - 1]; h->e[h->size - 1] = t;
    h->size--;
    heap_shift_down(h, 0);
}

/* sorted_buffer_gt (index.hpp:845-956), ascending by distance */
typedef struct { candidate_t* e; size_t size, capacity; } sorted_t;

static size_t sorted_lower_bound(sorted_t const* s, float d) { /* std::lower_bound with `<` on distance */
    size_t lo = 0, hi = s->size;
    while (lo < hi) {
        size_t mid = lo + (hi - lo) / 2;
        if (s->e[mid].distance < d) lo = mid + 1; else hi = mid;
    }
    return lo;
}
static void sorted_insert_reserved(sorted_t* s, candidate_t c) { /* :915-923 */
    size_t slot = s->size ? sorted_lower_bound(s, c.distance) : 0;
    memmove(s->e + slot + 1, s->e + slot, (s->size - slot) * sizeof(candidate_t));
    s->e[slot] = c;
    s->size++;
}
static int sorted_insert(sorted_t* s, candidate_t c, size_t limit) { /* :928-939 */
    size_t slot = s->size ? sorted_lower_bound(s, c.distance) : 0;
    if (slot == limit) return 0;
    size_t full = s->size == limit;
    size_t to_move = s->size - slot - full;
    memmove(s->e + slot + 1, s->e + slot, to_move * sizeof(candidate_t));
    s->e[slot] = c;
    s->size += !full;
    return 1;
}

/* growing_hash_set_gt (index.hpp:1084-1211); identity hash, linear probing, 0xFFFFFFFF = empty */
typedef struct { uint32_t* slots; size_t capacity, count; } visits_t;

static void visits_clear(visits_t* v) { if (v->slots) memset(v->slots, 0xFF, v->capacity * 4); v->count = 0; }
static int visits_reserve(visits_t* v, size_t n) { /* :1181-1210 */
    n = n * 5u / 3u;
    if (n <= v->capacity) return 1;
    size_t cap = ceil2(n);
    uint32_t* slots = (uint32_t*)malloc(cap * 4);
    if (!slots) return 0;
    memset(slots, 0xFF, cap * 4);
    for (size_t i = 0; i < v->capacity; ++i) {
        if (v->slots[i] == 0xFFFFFFFFu) continue;
        size_t j = v->slots[i] & (cap - 1);
        while (slots[j] != 0xFFFFFFFFu) j = (j + 1) & (cap - 1);
        slots[j] = v->slots[i];
    }
    free(v->slots);
    v->slots = slots;
    v->capacity = cap;
    return 1;
}
static int visits_set(visits_t* v, uint32_t s) { /* :1163-1175, returns previous membership */
    size_t i = s & (v->capacity - 1);
    while (v->slots[i] != 0xFFFFFFFFu) {
        if (v->slots[i] == s) return 1;
        i = (i + 1) & (v->capacity - 1);
    }
    v->slots[i] = s;
    v->count++;
    return 0;
}

typedef struct { /* context_t (index.hpp:2202-2250) */
    heap_t next;
    sorted_t top;
    visits_t visits;
    uint64_t computed_distances, iteration_cycles;
} context_t;

static void context_free(context_t* c) { free(c->next.e); free(c->top.e); free(c->visits.slots); }

/* ---------- node access ------------------------------------------------------------------- */

static uint8_t const* node_tape(oracle_index_t const* ix, uint32_t slot) { return ix->blob + ix->node_offsets[slot]; }
static uint64_t node_key(oracle_index_t const* ix, uint32_t slot) { return rd_u64(node_tape(ix, slot)); }
static uint8_t const* neighbors_base(oracle_index_t const* ix, uint32_t slot) { return node_tape(ix, slot) + 10; }
static uint8_t const* neighbors_non_base(oracle_index_t const* ix, uint32_t slot, size_t level) { /* :3790-3795 */
    return node_tape(ix, slot) + 10 + ix->neighbors_base_bytes + (level - 1) * ix->neighbors_bytes;
}
static float measure(oracle_index_t const* ix, context_t* c, void const* q, uint32_t slot) { /* :2215-2233 */
    c->computed_distances++;
    return ix->metric(q, ix->vectors + (size_t)slot * ix->bytes_per_vector, ix->metric_third);
}

/* ---------- the search path --------------------------------------------------------------- */

/* The predicate of index_dense_gt (index_dense.hpp:2071-2077): not a removed member and, for filtered_search, a key
 * in the caller's set (sorted ascending; NULL admits every key). */
typedef struct { uint64_t const* keys; size_t count; } allowed_t;

static int admits(oracle_index_t const* ix, allowed_t const* allowed, uint32_t slot) {
    uint64_t key = node_key(ix, slot);
    if (key == ix->free_key) return 0;
    if (!allowed || !allowed->keys) return 1;
    size_t lo = 0, hi = allowed->count;
    while (lo < hi) {
        size_t mid = lo + (hi - lo) / 2;
        if (allowed->keys[mid] < key) lo = mid + 1;
        else hi = mid;
    }
    return lo < allowed->count && allowed->keys[lo] == key;
}

/* search_for_one_ (index.hpp:3963-4003): greedy descent from begin_level down to level 1 */
static uint32_t search_for_one(oracle_index_t const* ix, context_t* c, void const* q, uint32_t closest,
                               int64_t begin_level, int64_t end_level) {
    visits_clear(&c->visits);
    float closest_dist = measure(ix, c, q, closest);
    for (int64_t level = begin_level; level > end_level; --level) {
        int changed;
        do {
            changed = 0;
            uint8_t const* nb = neighbors_non_base(ix, closest, (size_t)level); /* list of the node held at loop entry */
            uint32_t n = rd_u32(nb);
            for (uint32_t i = 0; i < n; ++i) {
                uint32_t cand = rd_u32(nb + 4 + 4 * i);
                float d = measure(ix, c, q, cand);
                if (d < closest_dist) { closest_dist = d; closest = cand; changed = 1; }
            }
            c->iteration_cycles++;
        } while (changed);
    }
    return closest;
}

/* search_to_find_in_base_ (index.hpp:4175-4246): best-first expansion over layer 0 */
static int search_to_find_in_base(oracle_index_t const* ix, context_t* c, void const* q, uint32_t start, size_t expansion,
                                  allowed_t const* allowed) {
    heap_t* next = &c->next;
    sorted_t* top = &c->top;
    visits_t* visits = &c->visits;
    size_t const top_limit = expansion;
    visits_clear(visits);
    next->size = 0;
    top->size = 0;
    if (!visits_reserve(visits, ix->connectivity_base + 1u)) return 0;

    float radius = measure(ix, c, q, start);
    candidate_t seed = {-radius, start};
    next->e[next->size++] = seed; /* insert_reserved into an empty heap */
    visits_set(visits, start);
    if (admits(ix, allowed, start)) {
        candidate_t t = {radius, start};
        sorted_insert_reserved(top, t);
    }

    while (next->size) {
        candidate_t cand = next->e[0];
        if ((-cand.distance) > radius && top->size == top_limit) break;
        heap_pop(next);
        c->iteration_cycles++;

        uint8_t const* nb = neighbors_base(ix, cand.slot);
        uint32_t n = rd_u32(nb);
        if (!visits_reserve(visits, visits->count + n)) return 0;
        for (uint32_t i = 0; i < n; ++i) {
            uint32_t succ = rd_u32(nb + 4 + 4 * i);
            if (visits_set(visits, succ)) continue;
            float d = measure(ix, c, q, succ);
            if (top->size < top_limit || d < radius) {
                candidate_t neg = {-d, succ};
                if (!heap_insert(next, neg)) return 0;
                if (admits(ix, allowed, succ)) {
                    candidate_t pos = {d, succ};
                    sorted_insert(top, pos, top_limit);
                    radius = top->e[top->size - 1].distance;
                }
            }
        }
    }
    return 1;
}

/* search_exact_ (index.hpp:4251-4268) */
static void search_exact(oracle_index_t const* ix, context_t* c, void const* q, size_t count, allowed_t const* allowed) {
    c->top.size = 0;
    for (uint64_t i = 0; i < ix->size; ++i) {
        if (!admits(ix, allowed, (uint32_t)i)) continue;
        candidate_t t = {measure(ix, c, q, (uint32_t)i), (uint32_t)i};
        sorted_insert(&c->top, t, count);
    }
}

static uint32_t const SNAN_BITS = 0x7FA00000u; /* std::numeric_limits<float>::signaling_NaN() */

/* index_gt::search (index.hpp:3016-3075) + search_result_t::dump_to (:2707-2722).
 * The query is already in the index's scalar kind. Returns the number of results found;
 * always writes `wanted` output slots. */
static size_t search_one(oracle_index_t const* ix, context_t* c, void const* q, size_t wanted, size_t expansion_cfg,
                         int exact, allowed_t const* allowed, uint64_t* keys, float* distances, uint64_t* computed,
                         uint64_t* visited) {
    size_t count = 0;
    uint64_t computed0 = c->computed_distances, cycles0 = c->iteration_cycles;
    c->top.size = 0;
    if (wanted && ix->size) {
        if (!expansion_cfg) expansion_cfg = 64;
        if (exact) {
            size_t cap = wanted + 1;
            if (c->top.capacity < cap) { c->top.e = (candidate_t*)realloc(c->top.e, cap * sizeof(candidate_t)); c->top.capacity = cap; }
            search_exact(ix, c, q, wanted, allowed);
        } else {
            size_t expansion = expansion_cfg > wanted ? expansion_cfg : wanted;
            heap_reserve(&c->next, expansion);
            if (c->top.capacity < expansion + 1) {
                c->top.e = (candidate_t*)realloc(c->top.e, (expansion + 1) * sizeof(candidate_t));
                c->top.capacity = expansion + 1;
            }
            uint32_t closest = search_for_one(ix, c, q, (uint32_t)ix->entry_slot, (int64_t)ix->max_level, 0);
            search_to_find_in_base(ix, c, q, closest, expansion, allowed);
        }
        if (c->top.size > wanted) c->top.size = wanted; /* shrink */
        count = c->top.size;
    }
    size_t i = 0;
    for (; i < count; ++i) {
        keys[i] = node_key(ix, c->top.e[i].slot);
        distances[i] = c->top.e[i].distance;
    }
    for (; i < wanted; ++i) {
        keys[i] = 0;
        memcpy(&distances[i], &SNAN_BITS, 4);
    }
    if (computed) *computed = c->computed_distances - computed0;
    if (visited) *visited = c->iteration_cycles - cycles0;
    return count;
}

typedef struct {
    oracle_index_t const* ix;
    uint8_t const* queries;
    size_t nq, stride, wanted, expansion;
    int exact;
    allowed_t allowed;
    uint64_t *keys, *counts, *computed, *visited;
    float* distances;
    size_t begin, end;
} job_t;

static void* worker(void* arg) {
    job_t* j = (job_t*)arg;
    context_t c;
    memset(&c, 0, sizeof(c));
    for (size_t i = j->begin; i < j->end; ++i)
        j->counts[i] = search_one(j->ix, &c, j->queries + i * j->stride, j->wanted, j->expansion, j->exact, &j->allowed,
                                  j->keys + i * j->wanted, j->distances + i * j->wanted,
                                  j->computed ? j->computed + i : NULL, j->visited ? j->visited + i : NULL);
    context_free(&c);
    return NULL;
}

/* Batch driver: contiguous chunks per thread, like executor_stl_t::dynamic (index_plugins.hpp:668-690).
 * `allowed_keys` (sorted ascending) makes it filtered_search (index_dense.hpp:774-779); NULL searches every member. */
void oracle_filtered_search_many(oracle_index_t const* ix, void const* queries, size_t nq, size_t stride_bytes,
                                 size_t wanted, size_t threads, int exact, uint64_t const* allowed_keys, size_t allowed_count,
                                 uint64_t* keys, float* distances, uint64_t* counts, uint64_t* computed, uint64_t* visited) {
    if (threads < 1) threads = 1;
    if (threads > nq) threads = nq ? nq : 1;
    job_t* jobs = (job_t*)calloc(threads, sizeof(job_t));
    pthread_t* tids = (pthread_t*)calloc(threads, sizeof(pthread_t));
    size_t per = (nq + threads - 1) / threads;
    for (size_t t = 0; t < threads; ++t) {
        job_t j = {ix, (uint8_t const*)queries, nq, stride_bytes, wanted, ix->expansion_search, exact,
                   {allowed_keys, allowed_count}, keys, counts, computed, visited, distances, t * per, (t + 1) * per < nq ? (t + 1) * per : nq};
        if (j.begin > nq) j.begin = nq;
        jobs[t] = j;
        if (threads == 1) worker(&jobs[t]);
        else pthread_create(&tids[t], NULL, worker, &jobs[t]);
    }
    if (threads > 1)
        for (size_t t = 0; t < threads; ++t) pthread_join(tids[t], NULL);
    free(jobs);
    free(tids);
}

void oracle_search_many(oracle_index_t const* ix, void const* queries, size_t nq, size_t stride_bytes, size_t wanted,
                        size_t threads, int exact, uint64_t* keys, float* distances, uint64_t* counts,
                        uint64_t* computed, uint64_t* visited) {
    oracle_filtered_search_many(ix, queries, nq, stride_bytes, wanted, threads, exact, NULL, 0, keys, distances, counts,
                                computed, visited);
}

/* exact_search_t (index_plugins.hpp:2071-2164) over raw matrices: metric(dataset row, query) for every pair, the `wanted`
 * smallest distances of each query in ascending order, keys = dataset row numbers (the order among equal distances is
 * unspecified there: std::partial_sort). Returns 0, or -1 for an unknown metric / scalar pair or wanted > n. */
int oracle_exact_search(void const* dataset, size_t n, size_t dataset_stride, void const* queries, size_t nq,
                        size_t queries_stride, int metric_kind, int scalar_kind, size_t dimensions, size_t wanted,
                        uint64_t* keys, float* distances) {
    oracle_metric_t metric = pick_metric((uint8_t)metric_kind, (uint8_t)scalar_kind);
    size_t third = scalar_kind == SK_B1 ? (dimensions + 7) / 8 : dimensions;
    if (!metric || wanted > n) return -1;
    sorted_t top = {(candidate_t*)malloc((wanted + 1) * sizeof(candidate_t)), 0, wanted + 1};
    for (size_t q = 0; q < nq; ++q) {
        void const* query = (uint8_t const*)queries + q * queries_stride;
        top.size = 0;
        for (size_t i = 0; i < n; ++i) {
            candidate_t c = {metric((uint8_t const*)dataset + i * dataset_stride, query, third), (uint32_t)i};
            sorted_insert(&top, c, wanted);
        }
        for (size_t i = 0; i < wanted; ++i) keys[q * wanted + i] = top.e[i].slot, distances[q * wanted + i] = top.e[i].distance;
    }
    free(top.e);
    return 0;
}

/* Query-side casts from f32 (index_plugins.hpp:1105-1224): used to validate the device casts.
 *   → i8  : clamp(x * 127 / ||x||, ±127) computed in f64, truncated toward zero   (:1172-1191)
 *   → b1  : bit set when x > 0, MSB-first within each byte                         (:1139-1158)
 *   → f16 / bf16 : round-to-nearest-even                                            (:473-594) */
size_t oracle_cast_from_f32(int scalar_kind, float const* in, size_t d, void* out) {
    switch (scalar_kind) {
    case SK_F32: memcpy(out, in, d * 4); return d * 4;
    case SK_I8: {
        double magnitude = 0;
        for (size_t i = 0; i < d; ++i) magnitude += (double)in[i] * (double)in[i];
        magnitude = sqrt(magnitude);
        int8_t* o = (int8_t*)out;
        for (size_t i = 0; i < d; ++i) {
            double v = (double)in[i] * 127.0 / magnitude;
            if (v > 127.0) v = 127.0;
            if (v < -127.0) v = -127.0;
            o[i] = (int8_t)v;
        }
        return d;
    }
    case SK_B1: {
        uint8_t* o = (uint8_t*)out;
        size_t bytes = (d + 7) / 8;
        memset(o, 0, bytes);
        for (size_t i = 0; i < d; ++i)
            if (in[i] > 0) o[i / 8] |= (uint8_t)(128 >> (i & 7));
        return bytes;
    }
    default: return 0;
    }
}

/* index_gt::cluster (index.hpp:3092-3125): the descent alone, stopped above `level - 1` (level 0 behaves like level 1),
 * then one more measurement of the winner. Single-threaded batch. */
void oracle_cluster_many(oracle_index_t const* ix, void const* queries, size_t nq, size_t stride_bytes, size_t level,
                         uint64_t* keys, float* distances, uint64_t* computed, uint64_t* visited) {
    context_t c;
    memset(&c, 0, sizeof(c));
    for (size_t i = 0; i < nq && ix->size; ++i) {
        void const* q = (uint8_t const*)queries + i * stride_bytes;
        uint64_t computed0 = c.computed_distances, cycles0 = c.iteration_cycles;
        uint32_t closest = search_for_one(ix, &c, q, (uint32_t)ix->entry_slot, (int64_t)ix->max_level,
                                          level == 0 ? 0 : (int64_t)level - 1);
        keys[i] = node_key(ix, closest);
        distances[i] = measure(ix, &c, q, closest);
        if (computed) computed[i] = c.computed_distances - computed0;
        if (visited) visited[i] = c.iteration_cycles - cycles0;
    }
    context_free(&c);
}
