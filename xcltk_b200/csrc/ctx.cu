// ctx.cu -- context, host<->HBM transfers of read batches, small shared host helpers.
#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include "owner.hpp"

extern "C" void xg_set_host_alloc(void *(*a)(size_t), void (*f)(void *));

namespace {
void *pinned_alloc(size_t n) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, n ? n : 256, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}
void pinned_free(void *p) { cudaFreeHost(p); }
}  // namespace

extern "C" {

const char *xg_version(void) { return "xcltk_b200 0.1 (reference semantics: xcltk 0.5.2)"; }

int xg_create(int32_t device, xg_ctx **out) {
    if (!out) return XG_E_ARG;
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    xg_ctx *ctx = new xg_ctx();
    *out = ctx;   // returned even on failure so that xg_last_error() works
    if (e != cudaSuccess || n <= 0) {
        cudaGetLastError();
        return ctx->fail(XG_E_CUDA, std::string("no CUDA device: ") +
                                        (e != cudaSuccess ? cudaGetErrorString(e) : "device count 0") +
                                        " (this library has no CPU fallback)");
    }
    if (device < 0 || device >= n) return ctx->fail(XG_E_ARG, "device index out of range");
    ctx->device = device;
    XG_CUDA(cudaSetDevice(device));
    XG_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    for (auto &ev : ctx->ev) XG_CUDA(cudaEventCreate(&ev));
    xg_set_host_alloc(pinned_alloc, pinned_free);   // decoded batches become pinned
    return XG_OK;
}

void xg_destroy(xg_ctx *ctx) {
    if (!ctx) return;
    if (ctx->stream) {
        cudaSetDevice(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        for (auto &kv : ctx->scratch)
            if (kv.second.p) cudaFree(kv.second.p);
        for (auto &ev : ctx->ev)
            if (ev) cudaEventDestroy(ev);
        for (auto &ev : ctx->ev_pool) cudaEventDestroy(ev);
        for (cudaStream_t st : {ctx->big_stream, ctx->inflate_stream, ctx->copy_stream, ctx->d2h_stream})
            if (st) cudaStreamDestroy(st);
        for (auto &b : ctx->pinned) cudaFreeHost(b.p);
        for (auto &b : ctx->devbufs) cudaFree(b.p);
        if (ctx->fx_cache && ctx->fx_cache_free) ctx->fx_cache_free(ctx->fx_cache);
        cudaStreamDestroy(ctx->stream);
    }
    delete ctx;
}

int xg_set_option(xg_ctx *ctx, const char *name, int64_t value) {
    if (!ctx || !name) return XG_E_ARG;
    if (std::string(name) == "stream_priority") {
        // 1: the context's stream gets the device's greatest priority -- for a context whose short kernels run
        // beside another context's long ones on the same GPU (their CTAs are scheduled first whenever both wait)
        if (!ctx->stream) return ctx->fail(XG_E_CUDA, "context has no device");
        XG_CUDA(cudaSetDevice(ctx->device));
        int least = 0, greatest = 0;
        XG_CUDA(cudaDeviceGetStreamPriorityRange(&least, &greatest));
        cudaStream_t st = nullptr;
        XG_CUDA(cudaStreamCreateWithPriority(&st, cudaStreamNonBlocking, value ? greatest : least));
        XG_CUDA(cudaStreamSynchronize(ctx->stream));
        cudaStreamDestroy(ctx->stream);
        ctx->stream = st;
        return XG_OK;
    }
    if (std::string(name) == "discover_slice") {
        if (value < 0) return ctx->fail(XG_E_ARG, "discover_slice must be >= 0");
        ctx->discover_slice = value;
        return XG_OK;
    }
    return ctx->fail(XG_E_ARG, std::string("unknown option '") + name + "'");
}

const char *xg_last_error(xg_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

void xg_last_timing(xg_ctx *ctx, double out[16]) {
    for (int i = 0; i < 16; i++) out[i] = ctx->timing[i];
}

int64_t xg_dreads_n(const xg_dreads *d) { return d ? d->n_reads : 0; }

void xg_dreads_info(const xg_dreads *d, int64_t out[8]) {
    const int64_t v[8] = {d->n_reads, d->n_cigar,     d->n_seq_words, d->n_runs,
                          d->n_tiles, d->max_aln_len, d->max_span,    d->bytes};
    for (int i = 0; i < 8; i++) out[i] = v[i];
}

void xg_dreads_index(const xg_dreads *d, xg_run *runs_out, xg_tile *tiles_out) {
    if (runs_out && !d->h_runs.empty()) memcpy(runs_out, d->h_runs.data(), d->h_runs.size() * sizeof(xg_run));
    if (tiles_out && !d->h_tiles.empty()) memcpy(tiles_out, d->h_tiles.data(), d->h_tiles.size() * sizeof(xg_tile));
}

void xg_dreads_free(xg_ctx *ctx, xg_dreads *d) {
    if (!d) return;
    if (ctx) cudaSetDevice(ctx->device);
    void *ps_all[] = {d->pos_end, d->fmq, d->cig_off, d->keys, d->seq_off, d->cigar, d->seq, d->runs, d->tiles};
    void *ps_map[] = {d->pos_end, d->runs, d->tiles};      // mapped batch: the rest is the caller's host memory
    std::vector<void *> ps(d->mapped ? std::begin(ps_map) : std::begin(ps_all),
                           d->mapped ? std::end(ps_map) : std::end(ps_all));
    for (void *p : ps)
        if (p) {
            if (d->pooled && ctx) ctx->dev_put(p); else cudaFree(p);
        }
    if (d->tile_pmax) {
        if (ctx) ctx->dev_put(d->tile_pmax); else cudaFree(d->tile_pmax);
    }
    delete d;
}

int xg_upload_reads(xg_ctx *ctx, const xg_reads *h, xg_dreads **out) {
    if (!ctx || !ctx->stream) return ctx ? ctx->fail(XG_E_CUDA, "context has no device") : XG_E_ARG;
    if (!h || !out) return ctx->fail(XG_E_ARG, "xg_upload_reads: null argument");
    XG_CUDA(cudaSetDevice(ctx->device));
    xg_dreads *d = xg_dreads_new(h);
    size_t n = (size_t)h->n_reads;
    bool seq = h->seq_off != nullptr && h->seq != nullptr;
    struct Cp {
        void **dst;
        const void *src;
        size_t bytes;
    } cps[] = {
        {(void **)&d->pos_end, h->pos_end, n * 8},
        {(void **)&d->fmq, h->fmq, n * 4},
        {(void **)&d->cig_off, h->cig_off, (n + 1) * 4},
        {(void **)&d->keys, h->keys, n * 16},
        {(void **)&d->seq_off, seq ? h->seq_off : nullptr, seq ? n * 4 : 0},
        {(void **)&d->cigar, h->cigar, (size_t)h->n_cigar * 4},
        {(void **)&d->seq, seq ? h->seq : nullptr, seq ? (size_t)h->n_seq_words * 4 : 0},
        {(void **)&d->runs, h->runs, (size_t)h->n_runs * sizeof(xg_run)},
        {(void **)&d->tiles, h->tiles, (size_t)h->n_tiles * sizeof(xg_tile)},
    };
    for (auto &c : cps) {
        if (!c.src) continue;
        *c.dst = ctx->dev_get(c.bytes + 64);      // slack: the kernels load records in aligned pairs / quads
        if (!*c.dst) {
            xg_dreads_free(ctx, d);
            return ctx->fail(XG_E_CUDA, "out of device memory for the read batch");
        }
    }
    cudaEventRecord(ctx->ev[6], ctx->stream);
    for (auto &c : cps) {
        if (!c.src || !c.bytes) continue;
        cudaError_t e = cudaMemcpyAsync(*c.dst, c.src, c.bytes, cudaMemcpyHostToDevice, ctx->stream);
        if (e != cudaSuccess) {
            xg_dreads_free(ctx, d);
            return ctx->fail(XG_E_CUDA, std::string("H2D reads: ") + cudaGetErrorString(e));
        }
        d->bytes += (int64_t)c.bytes;
    }
    cudaEventRecord(ctx->ev[7], ctx->stream);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        xg_dreads_free(ctx, d);
        return ctx->fail(XG_E_CUDA, std::string("H2D reads: ") + cudaGetErrorString(e));
    }
    float ms = 0;
    cudaEventElapsedTime(&ms, ctx->ev[6], ctx->ev[7]);
    d->h2d_ms = ms;
    ctx->timing[3] = ms;
    int rc = xg_make_tile_pmax(ctx, d);
    if (rc) {
        xg_dreads_free(ctx, d);
        return rc;
    }
    *out = d;
    return XG_OK;
}

// Records stay in pinned host memory; only pos/end (+ runs, tiles) are copied to HBM and the
// other arrays are read by the kernels through the mapped host pointers (zero-copy).  For the
// baf pileup, which needs flag / keys / CIGAR / sequence of the few reads that cover a SNP
// only: 8 B per read cross PCIe instead of ~84 B.
int xg_map_reads(xg_ctx *ctx, const xg_reads *h, xg_dreads **out) {
    if (!ctx || !ctx->stream) return ctx ? ctx->fail(XG_E_CUDA, "context has no device") : XG_E_ARG;
    if (!h || !out) return ctx->fail(XG_E_ARG, "xg_map_reads: null argument");
    XG_CUDA(cudaSetDevice(ctx->device));
    const void *must_be_pinned[] = {h->fmq, h->cig_off, h->keys, h->cigar, h->seq_off, h->seq};
    for (const void *p : must_be_pinned) {
        if (!p) continue;
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, p) != cudaSuccess || at.type != cudaMemoryTypeHost) {
            cudaGetLastError();
            return ctx->fail(XG_E_ARG, "xg_map_reads: record arrays must be pinned host memory "
                                       "(xg_decode_bams output after xg_create, or cudaHostRegister)");
        }
    }
    xg_dreads *d = xg_dreads_new(h);
    d->mapped = true;
    size_t n = (size_t)h->n_reads;
    d->pos_end = (int2 *)ctx->dev_get(n * 8 + 16);
    d->runs = (xg_run *)ctx->dev_get((size_t)h->n_runs * sizeof(xg_run) + 16);
    d->tiles = (xg_tile *)ctx->dev_get((size_t)h->n_tiles * sizeof(xg_tile) + 16);
    if (!d->pos_end || !d->runs || !d->tiles) {
        xg_dreads_free(ctx, d);
        return ctx->fail(XG_E_CUDA, "out of device memory for the read batch");
    }
    auto devptr = [](const void *p) -> void * {
        void *q = nullptr;
        if (!p || cudaHostGetDevicePointer(&q, const_cast<void *>(p), 0) != cudaSuccess) {
            cudaGetLastError();
            return nullptr;
        }
        return q;
    };
    d->fmq = (uint32_t *)devptr(h->fmq);
    d->cig_off = (uint32_t *)devptr(h->cig_off);
    d->keys = (ulonglong2 *)devptr(h->keys);
    d->cigar = (uint32_t *)devptr(h->cigar);
    d->seq_off = (uint32_t *)devptr(h->seq_off);
    d->seq = (uint32_t *)devptr(h->seq);
    cudaEventRecord(ctx->ev[6], ctx->stream);
    cudaMemcpyAsync(d->pos_end, h->pos_end, n * 8, cudaMemcpyHostToDevice, ctx->stream);
    cudaMemcpyAsync(d->runs, h->runs, (size_t)h->n_runs * sizeof(xg_run), cudaMemcpyHostToDevice, ctx->stream);
    cudaMemcpyAsync(d->tiles, h->tiles, (size_t)h->n_tiles * sizeof(xg_tile), cudaMemcpyHostToDevice, ctx->stream);
    cudaEventRecord(ctx->ev[7], ctx->stream);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        xg_dreads_free(ctx, d);
        return ctx->fail(XG_E_CUDA, std::string("xg_map_reads: ") + cudaGetErrorString(e));
    }
    float ms = 0;
    cudaEventElapsedTime(&ms, ctx->ev[6], ctx->ev[7]);
    d->h2d_ms = ms;
    d->bytes = (int64_t)(n * 8);
    *out = d;
    return XG_OK;
}

int xg_download_reads(xg_ctx *ctx, const xg_dreads *d, xg_reads **out) {
    if (!ctx || !ctx->stream) return ctx ? ctx->fail(XG_E_CUDA, "context has no device") : XG_E_ARG;
    XG_CUDA(cudaSetDevice(ctx->device));
    xg_reads_owner *o = new xg_reads_owner();   // released by xg_reads_free()
    memset(&o->r, 0, sizeof(o->r));
    o->free_fn = pinned_free;
    size_t n = (size_t)d->n_reads;
    auto dl = [&](const void *src, size_t bytes) -> void * {
        void *p = pinned_alloc(bytes);
        if (!p) return nullptr;
        o->bufs.push_back(p);
        if (bytes) cudaMemcpyAsync(p, src, bytes, cudaMemcpyDeviceToHost, ctx->stream);
        return p;
    };
    o->r.n_reads = d->n_reads;
    o->r.n_cigar = d->n_cigar;
    o->r.n_seq_words = d->n_seq_words;
    o->r.n_runs = d->n_runs;
    o->r.n_tiles = d->n_tiles;
    o->r.max_aln_len = d->max_aln_len;
    o->r.max_span = d->max_span;
    o->r.n_records_seen = d->n_reads;
    o->r.pos_end = (const int32_t *)dl(d->pos_end, n * 8);
    o->r.fmq = (const uint32_t *)dl(d->fmq, n * 4);
    o->r.cig_off = (const uint32_t *)dl(d->cig_off, (n + 1) * 4);
    o->r.keys = (const uint64_t *)dl(d->keys, n * 16);
    o->r.cigar = (const uint32_t *)dl(d->cigar, (size_t)d->n_cigar * 4);
    if (d->seq_off && d->seq) {
        o->r.seq_off = (const uint32_t *)dl(d->seq_off, n * 4);
        o->r.seq = (const uint32_t *)dl(d->seq, (size_t)d->n_seq_words * 4);
    }
    xg_run *runs = (xg_run *)pinned_alloc(sizeof(xg_run) * (d->h_runs.size() + 1));
    xg_tile *tiles = (xg_tile *)pinned_alloc(sizeof(xg_tile) * (d->h_tiles.size() + 1));
    if (runs) o->bufs.push_back(runs);
    if (tiles) o->bufs.push_back(tiles);
    auto drop = [&](int code, const std::string &msg) {      // the owner and what it holds go away on every error path
        cudaStreamSynchronize(ctx->stream);
        for (void *q : o->bufs) pinned_free(q);
        delete o;
        return ctx->fail(code, msg);
    };
    const bool seq_ok = !(d->seq_off && d->seq) || (o->r.seq_off && o->r.seq);
    if (!runs || !tiles || !o->r.pos_end || !o->r.fmq || !o->r.cig_off || !o->r.keys || !o->r.cigar || !seq_ok)
        return drop(XG_E_NOMEM, "out of pinned host memory for the downloaded batch");
    memcpy(runs, d->h_runs.data(), sizeof(xg_run) * d->h_runs.size());
    memcpy(tiles, d->h_tiles.data(), sizeof(xg_tile) * d->h_tiles.size());
    o->r.runs = runs;
    o->r.tiles = tiles;
    const cudaError_t ce = cudaStreamSynchronize(ctx->stream);
    if (ce != cudaSuccess) return drop(XG_E_CUDA, std::string("D2H reads: ") + cudaGetErrorString(ce));
    *out = &o->r;
    return XG_OK;
}

void xg_coo_free(xg_coo *m) {
    if (!m) return;
    xg_coo_owner *o = reinterpret_cast<xg_coo_owner *>(m);
    for (void *p : o->bufs) {
        if (o->ctx) o->ctx->pinned_put(p); else cudaFreeHost(p);
    }
    delete o;
}

}  // extern "C"

xg_dreads *xg_dreads_new(const xg_reads *h) {
    xg_dreads *d = new xg_dreads();
    d->n_reads = h->n_reads;
    d->n_cigar = h->n_cigar;
    d->n_seq_words = h->n_seq_words;
    d->n_runs = h->n_runs;
    d->n_tiles = h->n_tiles;
    d->max_aln_len = h->max_aln_len;
    d->max_span = h->max_span;
    d->h_runs.assign(h->runs, h->runs + h->n_runs);
    d->h_tiles.assign(h->tiles, h->tiles + h->n_tiles);
    d->pooled = true;
    return d;
}

// Prefix max (restarting at every run) of the tiles' max_end: with it "first tile whose records
// can still reach position x" is a binary search.  Built once per batch from the host tile index, with the
// stretches of tiles of one run (basefc plans one window job per stretch and call).
int xg_make_tile_pmax(xg_ctx *ctx, xg_dreads *d) {
    size_t nt = d->h_tiles.size();
    std::vector<int32_t> pm(nt);
    d->h_run_tiles.clear();
    for (size_t t = 0; t < nt; t++) {
        bool first = (t == 0) || d->h_tiles[t - 1].run != d->h_tiles[t].run;
        pm[t] = first ? d->h_tiles[t].max_end : std::max(pm[t - 1], d->h_tiles[t].max_end);
        if (first) d->h_run_tiles.push_back(make_int3(d->h_tiles[t].run, (int)t, (int)t));
        d->h_run_tiles.back().z = (int)t + 1;
    }
    if (d->tile_pmax) ctx->dev_put(d->tile_pmax);
    d->tile_pmax = (int32_t *)ctx->dev_get(nt * 4 + 16);
    if (!d->tile_pmax) return ctx->fail(XG_E_CUDA, "out of device memory for the tile index");
    if (nt) XG_CUDA(cudaMemcpy(d->tile_pmax, pm.data(), nt * 4, cudaMemcpyHostToDevice));
    return XG_OK;
}

// Build the open-addressing cell-barcode table on the host and upload it.
// Replaces the dict lookup `smp in self.cell_cnt` (rdr/fc/mcount.py:119-127).
int xg_build_barcode_table(xg_ctx *ctx, const xg_barcodes *cells, BarcodeTable *out) {
    // the table depends on the key list only: it stays on the device while the caller passes the same list
    const std::initializer_list<xg_input_key::Span> in = {{&cells->n, sizeof cells->n},
                                                          {cells->keys, sizeof(uint64_t) * (size_t)cells->n}};
    uint64_t h = 1469598103934665603ull ^ (uint64_t)cells->n;
    for (int32_t i = 0; i < cells->n; i++) {
        h = (h ^ cells->keys[i]) * 1099511628211ull;
        h ^= h >> 29;
    }
    for (int k = 0; k < 2; k++) {
        xg_ctx::BcCache &c = ctx->bc_cache[k];
        if (c.valid && c.key.matches(h, in)) {
            c.used = ++ctx->bc_clock;
            out->slots = (const ulonglong2 *)c.slots;
            out->mask = c.mask;
            out->shift = c.shift;
            return XG_OK;
        }
    }
    int slot;                                   // an empty entry, else the one used longest ago
    if (!ctx->bc_cache[0].valid) slot = 0;
    else if (!ctx->bc_cache[1].valid) slot = 1;
    else slot = ctx->bc_cache[0].used <= ctx->bc_cache[1].used ? 0 : 1;
    ctx->bc_cache[slot].valid = false;
    uint32_t cap = 16, log2cap = 4;
    while (cap < (uint32_t)cells->n * 2u + 2u) {
        cap <<= 1;
        log2cap++;
    }
    std::vector<ulonglong2> tab(cap, make_ulonglong2(XG_KEY_NONE, 0));
    for (int32_t i = 0; i < cells->n; i++) {
        uint64_t key = cells->keys[i];
        if (key == XG_KEY_NONE || key == XG_KEY_NOMATCH)
            return ctx->fail(XG_E_ARG, "invalid barcode key");
        uint32_t s = barcode_home(key, 32 - log2cap);
        while (tab[s].x != XG_KEY_NONE) {
            if (tab[s].x == key) return ctx->fail(XG_E_ARG, "duplicate barcode key");
            s = (s + 1) & (cap - 1);
        }
        tab[s] = make_ulonglong2(key, (unsigned long long)i);
    }
    XG_GET(dt, ulonglong2, slot ? "bc_slots1" : "bc_slots0", cap);
    XG_CUDA(cudaMemcpyAsync(dt, tab.data(), (size_t)cap * 16, cudaMemcpyHostToDevice, ctx->stream));
    XG_CUDA(cudaStreamSynchronize(ctx->stream));   // tab goes out of scope
    out->slots = dt;
    out->mask = cap - 1;
    out->shift = 32 - log2cap;
    ctx->bc_cache[slot].slots = dt;
    ctx->bc_cache[slot].mask = out->mask;
    ctx->bc_cache[slot].shift = out->shift;
    ctx->bc_cache[slot].key.assign(h, in);
    ctx->bc_cache[slot].used = ++ctx->bc_clock;
    ctx->bc_cache[slot].valid = true;
    return XG_OK;
}
