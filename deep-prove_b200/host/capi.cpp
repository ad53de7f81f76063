// C entry points over the host mirror (for the Python tests / bench; a Rust caller would use its own
// crates above include/deepprove_b200.h instead).  Nothing here touches oracle/.
#include "sumcheck.hpp"

using namespace dp;
static thread_local std::string g_herr;
#define DPH_TRY try {
#define DPH_CATCH } catch (const Error &e) { g_herr = e.what(); return e.code ? e.code : 1; } catch (const std::exception &e) { g_herr = e.what(); return 1; }

extern "C" {

const char *dph_last_error() { return g_herr.c_str(); }

void dph_poseidon2_permute(uint64_t *state) { Poseidon2::permute(state); }
// fast (weak-form) permutation against the canonical formulation on n seeded states, every third one drawn from edge values;
// returns the number of mismatching or non-canonical output words (0 expected)
uint64_t dph_poseidon2_selfcheck(uint64_t n, uint64_t seed) {
    auto sm = [&]() { uint64_t z = (seed += 0x9E3779B97F4A7C15ULL); z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL; z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL; return z ^ (z >> 31); };
    const uint64_t edge[] = {0, 1, 2, P - 1, P - 2, EPS, EPS + 1, 1ULL << 32, 1ULL << 63, (P - 1) / 2, 0xFFFFFFFEFFFFFFFFULL, 7};
    const int ne = sizeof(edge) / 8; uint64_t bad = 0, a[8], b[8], ca[8] = {0}, cb[8] = {0};
    for (uint64_t it = 0; it < n; it++) {
        for (int i = 0; i < 8; i++) a[i] = b[i] = (it % 3 == 0) ? edge[sm() % ne] : canon(sm());
        Poseidon2::permute(a); Poseidon2::permute_canonical(b);
        for (int i = 0; i < 8; i++) if (a[i] != b[i] || a[i] >= P) bad++;
        ca[it & 3] = cb[it & 3] = canon(sm());                       // and a chained (sponge-like) sequence
        Poseidon2::permute(ca); Poseidon2::permute_canonical(cb);
        for (int i = 0; i < 8; i++) if (ca[i] != cb[i]) bad++;
    }
    return bad;
}

// Hasher pair of everything proved from now on: 0 = PoseidonHasher + BasicTranscript (default), 1 = BlakeHasher + BlakeTranscript
// (the reference's cargo feature `blake`: mpcs/src/lib.rs:339-342, zkml/src/bin/bench.rs:29-44).  Process-wide; set it between proofs.
int dph_set_hasher(int kind) { if (kind != 0 && kind != 1) { g_herr = "dph_set_hasher: 0 or 1"; return 1; } if (dp_set_merkle_hasher(kind) != DP_OK) { g_herr = dp_last_error(); return 1; } dp::hasher_mode() = kind; return 0; }
void *dph_transcript_new(const char *label) { return new DynTranscript(label); }
void dph_transcript_free(void *t) { delete (DynTranscript *)t; }
void dph_transcript_append_f(void *t, const uint64_t *f, uint64_t n) { for (uint64_t i = 0; i < n; i++) ((DynTranscript *)t)->append_field_element(f[i]); }
void dph_transcript_append_msg(void *t, const uint8_t *m, uint64_t n) { ((DynTranscript *)t)->append_message(m, n); }
void dph_transcript_append_e(void *t, const uint64_t *e, uint64_t n) { for (uint64_t i = 0; i < n; i++) ((DynTranscript *)t)->append_field_element_ext(Ext(e[2 * i], e[2 * i + 1])); }
void dph_transcript_challenge(void *t, const char *label, uint64_t *out) { Ext c = ((DynTranscript *)t)->get_and_append_challenge(label); out[0] = c.c0; out[1] = c.c1; }

// VirtualPolynomial numbers MLEs by FIRST USE in the products (virtual_poly.rs:168-177), and get_mle_final_evaluations()
// returns them in that order; the C entry points below report final evaluations in the CALLER's `mles` order instead.
// remap[i] = position of caller MLE i in first-use order, UINT32_MAX when no product references it (its slot is zeroed).
static std::vector<uint32_t> first_use_remap(const dp_sc_product *products, uint32_t n_products, uint32_t n_mles) {
    std::vector<uint32_t> remap(n_mles, UINT32_MAX); uint32_t next = 0;
    for (uint32_t p = 0; p < n_products; p++) for (uint32_t j = 0; j < products[p].n_idx; j++) { uint32_t i = products[p].idx[j]; if (i < n_mles && remap[i] == UINT32_MAX) remap[i] = next++; }
    return remap;
}
static void write_finals(const ExtVec &fin, const std::vector<uint32_t> &remap, uint64_t *out_final) {
    for (size_t i = 0; i < remap.size(); i++) {
        Ext v = (remap[i] != UINT32_MAX && remap[i] < fin.size()) ? fin[remap[i]] : Ext::zero();
        out_final[2 * i] = v.c0; out_final[2 * i + 1] = v.c1;
    }
}

// IOPProverState::prove_parallel over device MLE handles with DynTranscript::new(label) (or an
// existing transcript when `transcript` is non-null).  out_msgs: nv x (max_deg+1) x E.
int dph_sumcheck_prove_parallel(dp_mle *const *mles, uint32_t n_mles, const dp_sc_product *products, uint32_t n_products,
                                uint32_t max_nv, const char *label, void *transcript, uint64_t *out_point, uint64_t *out_msgs,
                                uint64_t *out_final, uint32_t *out_max_deg) {
    DPH_TRY
    VirtualPolynomial vp(max_nv);
    std::vector<DeviceMle> views;
    for (uint32_t i = 0; i < n_mles; i++) {
        uint64_t len; int ext; check(dp_mle_info(mles[i], &len, &ext, nullptr));
        views.push_back(DeviceMle::wrap_device(dp_mle_device_ptr(mles[i]), len, ext));
    }
    // register in caller order so final evaluations line up with `mles`
    for (uint32_t p = 0; p < n_products; p++) {
        std::vector<DeviceMle> l;
        for (uint32_t j = 0; j < products[p].n_idx; j++) l.push_back(views.at(products[p].idx[j]));
        vp.add_mle_list(l, Ext(products[p].coef[0], products[p].coef[1]));
    }
    std::vector<uint32_t> remap = first_use_remap(products, n_products, n_mles);
    DynTranscript local(label ? label : "");
    DynTranscript &t = transcript ? *(DynTranscript *)transcript : local;
    auto res = IOPProverState::prove_parallel(std::move(vp), t);
    size_t deg = res.first.proofs.empty() ? 0 : res.first.proofs[0].evaluations.size() - 1;
    *out_max_deg = (uint32_t)deg;
    for (size_t i = 0; i < res.first.point.size(); i++) { out_point[2 * i] = res.first.point[i].c0; out_point[2 * i + 1] = res.first.point[i].c1; }
    size_t k = 0;
    for (auto &m : res.first.proofs) for (auto &e : m.evaluations) { out_msgs[2 * k] = e.c0; out_msgs[2 * k + 1] = e.c1; k++; }
    const ExtVec &fin = res.second.get_mle_final_evaluations();
    write_finals(fin, remap, out_final);
    return 0;
    DPH_CATCH
}

}  // extern "C"

// ---- mpcs (host/mpcs.hpp) ----
#include "mpcs.hpp"
extern "C" {

// Basefold::commit + Basefold::open with BasefoldProof flattened (BasefoldProof::flatten layout)
int dph_pcs_open(dp_mle *poly, uint32_t full_log, const uint64_t *point, const char *label, uint64_t *out, uint64_t cap, uint64_t *out_len, uint64_t *out_root) {
    DPH_TRY
    uint64_t len; int ext; uint32_t nv; check(dp_mle_info(poly, &len, &ext, &nv));
    DeviceMle m = DeviceMle::wrap_device(dp_mle_device_ptr(poly), len, ext);
    BasefoldProverParams pp; pp.full_message_size_log = full_log;
    auto comm = Basefold::commit(pp, m);
    if (out_root) memcpy(out_root, comm.root.v, 32);
    ExtVec pt; for (uint32_t i = 0; i < nv; i++) pt.push_back(Ext(point[2 * i], point[2 * i + 1]));
    DynTranscript t(label);
    BasefoldProof pr = Basefold::open(pp, m, comm, pt, t);
    std::vector<uint64_t> f = pr.flatten();
    *out_len = f.size();
    if (f.size() > cap) { g_herr = "dph_pcs_open: output buffer too small"; return 2; }
    memcpy(out, f.data(), 8 * f.size());
    return 0;
    DPH_CATCH
}

int dph_pcs_batch_open(dp_mle *const *polys, uint32_t n, uint32_t full_log, const uint64_t *points, const char *label, uint64_t *out, uint64_t cap,
                       uint64_t *out_len) {
    DPH_TRY
    BasefoldProverParams pp; pp.full_message_size_log = full_log;
    std::vector<DeviceMle> ms; std::vector<BasefoldCommitmentWithWitness> comms; std::vector<ExtVec> pts; std::vector<Evaluation> evals;
    size_t o = 0;
    for (uint32_t i = 0; i < n; i++) {
        uint64_t len; int ext; uint32_t nv; check(dp_mle_info(polys[i], &len, &ext, &nv));
        ms.push_back(DeviceMle::wrap_device(dp_mle_device_ptr(polys[i]), len, ext));
        comms.push_back(Basefold::commit(pp, ms.back()));
        ExtVec pt; for (uint32_t k = 0; k < nv; k++) pt.push_back(Ext(points[2 * (o + k)], points[2 * (o + k) + 1]));
        o += nv; pts.push_back(pt);
        Evaluation ev; ev.poly = i; ev.point = i; ev.value = ms.back().evaluate(pt);
        evals.push_back(ev);
    }
    DynTranscript t(label);
    BasefoldProof pr = Basefold::batch_open(pp, ms, comms, pts, evals, t);
    std::vector<uint64_t> f = pr.flatten();
    *out_len = f.size();
    if (f.size() > cap) { g_herr = "dph_pcs_batch_open: output buffer too small"; return 2; }
    memcpy(out, f.data(), 8 * f.size());
    return 0;
    DPH_CATCH
}

}  // extern "C"

// ---- zkml MLP prover (host/zkml.hpp) ----
#include "zkml.hpp"
#include <chrono>
namespace {
struct ZkHandle { dp::zkml::Model model; dp::zkml::Context ctx; dp::zkml::DeviceTrace trace; std::vector<dp::zkml::Element> trace_input; };   // the stored trace lives in HBM
}
extern "C" {

// Model = n_layers x [Dense(width x width)+bias -> Requant -> ReLU]; rq = n_layers x {right_shift, fp_scale, fpm, intermediate_bits}.
// Builds the Context: uploads weights/bias/tables and commits them (CommitmentContext::new) -- setup, not proving.
int dph_zkml_context_new(uint32_t n_layers, uint32_t width, const int64_t *weights, const int64_t *bias, const int64_t *rq, void **out) {
    DPH_TRY
    using namespace dp::zkml;
    auto *h = new ZkHandle();
    h->model.input_len = width;
    for (uint32_t l = 0; l < n_layers; l++) {
        Node d; d.op = Op::Dense; d.nrows = d.ncols = width;
        d.weights.assign(weights + (size_t)l * width * width, weights + (size_t)(l + 1) * width * width);
        d.bias.assign(bias + (size_t)l * width, bias + (size_t)(l + 1) * width);
        h->model.nodes.push_back(std::move(d));
        Node r; r.op = Op::Requant; r.rq.right_shift = rq[4 * l]; r.rq.fp_scale = rq[4 * l + 1]; r.rq.fixed_point_multiplier = rq[4 * l + 2]; r.rq.intermediate_bit_size = rq[4 * l + 3];
        h->model.nodes.push_back(r);
        Node a; a.op = Op::Relu; h->model.nodes.push_back(a);
    }
    h->ctx = Context::generate(h->model);
    check(dp_synchronize());
    *out = h;
    return 0;
    DPH_CATCH
}
extern "C" void dph_zkml_pool_free(void *handle);
void dph_zkml_context_free(void *h) { dph_zkml_pool_free(h); delete (ZkHandle *)h; }

// mode 0: inference + Prover::prove + flatten (end to end from the host input buffer)
// mode 1: run inference only and keep the trace in the handle (not proving)
// mode 2: Prover::prove on the stored trace (what zkml/src/bin/bench.rs times), flatten only if out != NULL
int dph_zkml_prove(void *handle, const int64_t *input, int mode, const char *label, uint64_t *out, uint64_t cap, uint64_t *out_len) {
    DPH_TRY
    using namespace dp::zkml;
    ZkHandle *h = (ZkHandle *)handle;
    size_t w = h->model.input_len;
    if (mode == 0 || mode == 1) { h->trace_input.assign(input, input + w); h->trace = run_device(h->ctx, h->trace_input); check(dp_synchronize()); if (mode == 1) return 0; }
    DynTranscript t(label);
    Prover<DynTranscript> prover(h->ctx, t);
    Proof p = prover.prove(h->trace);
    if (out) {
        std::vector<uint64_t> f = p.flatten(h->model.nodes.size());
        *out_len = f.size();
        if (f.size() > cap) { g_herr = "dph_zkml_prove: output buffer too small"; return 2; }
        memcpy(out, f.data(), 8 * f.size());
    }
    return 0;
    DPH_CATCH
}

}  // extern "C"

// ---- concurrent proving: a persistent pool of host threads, each with its own library context (stream + device
// arena) on `device`, proves the stored trace; the GPU runs the threads' small latency-bound kernels side by side.
#include <thread>
#include <mutex>
#include <atomic>
#include <condition_variable>
extern "C" void dp_hostprof_dump(void);
namespace {
struct ZkPool {
    std::vector<std::thread> th; std::mutex mu; std::condition_variable cv, done_cv;
    ZkHandle *h = nullptr; int device = 0; bool stop = false; uint64_t pending = 0, inflight = 0; std::string label, err; bool failed = false; bool e2e = false;
    // Identical proofs started together stay in lockstep: all of them sit in the latency-bound layer sumchecks (GPU nearly idle)
    // and then all of them queue their GPU-filling opening kernels behind each other (CUPTI timeline, profiles/r02k).  So the
    // workers of one call start `stagger_s` apart (one proof duration spread over the workers; the duration is an average over the
    // proofs this pool has already run -- the first call of a pool is not staggered): latency-bound and GPU-bound phases of
    // different proofs then overlap.  The ramp-up and ramp-down this costs are inside the caller's timed region.
    uint32_t active = 0; uint64_t call_gen = 0; double stagger_s = 0.0, avg_proof_s = 0.0; uint64_t n_timed = 0;
    // the proof of the job claimed last in the most recent call; every other proof of a call is dropped
    dp::zkml::Proof last; bool has_last = false;
    void keep_last(dp::zkml::Proof &p) { std::lock_guard<std::mutex> lk(mu); last = std::move(p); has_last = true; }
    void worker(uint32_t idx) {
        bool inited = false; uint64_t seen_gen = 0;
        for (;;) {
            uint64_t gen; double delay = 0.0; bool last_job;
            { std::unique_lock<std::mutex> lk(mu); cv.wait(lk, [&] { return stop || (pending > 0 && idx < active); }); if (stop) break; pending--; inflight++; last_job = pending == 0; gen = call_gen; if (gen != seen_gen) { seen_gen = gen; delay = stagger_s * idx; } }
            try {
                const bool first_ever = !inited;     // grows this thread's device arena: not a representative duration
                if (!inited) { dp::check(dp_init(device)); inited = true; }
                if (delay > 0.0) std::this_thread::sleep_for(std::chrono::duration<double>(delay));
                auto t0 = std::chrono::steady_clock::now();
                struct timespec cts0; clock_gettime(CLOCK_THREAD_CPUTIME_ID, &cts0);
                dp::DynTranscript t(label);
                dp::zkml::Prover<dp::DynTranscript> prover(h->ctx, t);
                if (e2e) {   // from the host input vector: inference, prove, serialised proof in host memory
                    dp::zkml::Proof p = prover.prove(h->trace_input);
                    std::vector<uint64_t> bytes = p.flatten(h->model.nodes.size());
                    if (bytes.empty()) throw dp::Error(DP_ERR_STATE, "empty proof");
                    if (last_job) keep_last(p);
                } else { dp::zkml::Proof p = prover.prove(h->trace); if (last_job) keep_last(p); }
                const double sec = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
                if (getenv("DP_HOST_PROF") && idx == 0) { struct timespec cts1; clock_gettime(CLOCK_THREAD_CPUTIME_ID, &cts1);
                    fprintf(stderr, "[worker0] proof wall %.2f ms, thread CPU %.2f ms, transcript permutations %llu\n", sec * 1e3, (cts1.tv_sec - cts0.tv_sec) * 1e3 + (cts1.tv_nsec - cts0.tv_nsec) * 1e-6, (unsigned long long)t.permutations()); }
                if (!first_ever) { std::lock_guard<std::mutex> lk(mu); n_timed++; avg_proof_s += (sec - avg_proof_s) / (double)std::min<uint64_t>(n_timed, 64); }
            } catch (const std::exception &e) { std::lock_guard<std::mutex> lk(mu); failed = true; err = e.what(); }
            dp_profile_flush();   // per-kernel timing of the concurrent region (no-op unless dp_profile_enable(1))
            { std::lock_guard<std::mutex> lk(mu); inflight--; if (pending == 0 && inflight == 0) done_cv.notify_all(); }
        }
        if (inited) { dp_synchronize(); if (getenv("DP_HOST_PROF")) { static std::atomic<int> once{0}; if (!once.exchange(1)) dp_hostprof_dump(); } dp_shutdown(); }
    }
    ~ZkPool() { { std::lock_guard<std::mutex> lk(mu); stop = true; } cv.notify_all(); for (auto &t : th) t.join(); }
};
std::mutex g_pools_mu; std::map<void *, std::unique_ptr<ZkPool>> g_pools;
}
extern "C" void dph_zkml_pool_free(void *handle) { std::lock_guard<std::mutex> lk(g_pools_mu); g_pools.erase(handle); }
extern "C" int dph_zkml_prove_concurrent(void *handle, int device, uint32_t n_workers, uint32_t n_proofs, int e2e, const char *label, double *out_seconds) {
    DPH_TRY
    ZkHandle *h = (ZkHandle *)handle;
    if (!h->trace.valid()) throw dp::Error(DP_ERR_STATE, "dph_zkml_prove_concurrent: run inference first (mode 1)");
    ZkPool *pool;
    { std::lock_guard<std::mutex> lk(g_pools_mu); auto &pp = g_pools[handle]; if (!pp) { pp = std::make_unique<ZkPool>(); pp->h = h; pp->device = device; } pool = pp.get(); }
    while (pool->th.size() < n_workers) { const uint32_t idx = (uint32_t)pool->th.size(); pool->th.emplace_back([pool, idx] { pool->worker(idx); }); }
    static const bool no_stagger = getenv("DP_NO_STAGGER") != nullptr;
    auto t0 = std::chrono::steady_clock::now();
    {
        std::lock_guard<std::mutex> lk(pool->mu);
        pool->label = label; pool->failed = false; pool->has_last = false; pool->e2e = e2e != 0; pool->pending = n_proofs; pool->active = n_workers; pool->call_gen++;
        // stagger only when every worker gets several proofs (otherwise the ramps cost more than the overlap gains)
        pool->stagger_s = (!no_stagger && n_workers > 1 && n_proofs >= 3 * n_workers && pool->n_timed > 0) ? pool->avg_proof_s / n_workers : 0.0;
    }
    // only the first n_workers threads are woken usefully: notify_all, extra threads just compete for the same jobs
    pool->cv.notify_all();
    { std::unique_lock<std::mutex> lk(pool->mu); pool->done_cv.wait(lk, [&] { return pool->pending == 0 && pool->inflight == 0; }); }
    if (out_seconds) *out_seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    if (pool->failed) { g_herr = pool->err; return 1; }
    return 0;
    DPH_CATCH
}
// flat proof (the dph_zkml_prove image) of the job claimed last in the most recent dph_zkml_prove_concurrent call on `handle`
extern "C" int dph_zkml_last_concurrent_proof(void *handle, uint64_t *out, uint64_t cap, uint64_t *out_len) {
    DPH_TRY
    ZkHandle *h = (ZkHandle *)handle;
    ZkPool *pool = nullptr;
    { std::lock_guard<std::mutex> lk(g_pools_mu); auto it = g_pools.find(handle); if (it != g_pools.end()) pool = it->second.get(); }
    const char *none = "dph_zkml_last_concurrent_proof: no completed dph_zkml_prove_concurrent call";
    if (!pool) throw dp::Error(DP_ERR_STATE, none);
    std::vector<uint64_t> f;
    {
        std::lock_guard<std::mutex> lk(pool->mu);
        if (!pool->has_last) throw dp::Error(DP_ERR_STATE, none);
        f = pool->last.flatten(h->model.nodes.size());
    }
    *out_len = f.size();
    if (f.size() > cap) { g_herr = "dph_zkml_last_concurrent_proof: output buffer too small"; return 2; }
    memcpy(out, f.data(), 8 * f.size());
    return 0;
    DPH_CATCH
}

// One proof sharded over `world` ranks: `mles` are THIS rank's slices (nv_total - log2(world) variables each).
// Exchange: shm_region != NULL -> same-node shared-memory mailbox (sizeof = dph_shm_mailbox_bytes(), zero-initialised,
// mapped by every rank; `*shm_seq` carries the mailbox sequence number across calls); else `cb(user, send, n, recv)`.
extern "C" uint64_t dph_shm_mailbox_bytes() { return sizeof(ShmMailbox); }
// one raw all-gather through the mailbox (host-only; used by the CPU tests of the exchange itself)
extern "C" int dph_shm_allgather(void *shm_region, uint32_t world, uint32_t rank, uint64_t *shm_seq, const uint64_t *send, uint64_t n_words, uint64_t *recv) {
    DPH_TRY
    ShmExchange ex(shm_region, world, rank); ex.seq = *shm_seq;
    ex.allgather((const u64 *)send, n_words, (u64 *)recv);
    *shm_seq = ex.seq;
    return 0;
    DPH_CATCH
}
extern "C" int dph_sumcheck_prove_sharded(uint32_t world, uint32_t rank, dp_mle *const *mles, uint32_t n_mles, const dp_sc_product *products, uint32_t n_products,
                                          uint32_t nv_total, const char *label, void *shm_region, uint64_t *shm_seq, CallbackExchange::Fn cb, void *user,
                                          uint64_t *out_point, uint64_t *out_msgs, uint64_t *out_final) {
    DPH_TRY
    uint32_t logG = 0; while ((1u << logG) < world) logG++;
    VirtualPolynomial vp(nv_total - logG);
    std::vector<DeviceMle> views;
    for (uint32_t i = 0; i < n_mles; i++) {
        uint64_t len; int ext; check(dp_mle_info(mles[i], &len, &ext, nullptr));
        views.push_back(DeviceMle::wrap_device(dp_mle_device_ptr(mles[i]), len, ext));
    }
    for (uint32_t p = 0; p < n_products; p++) { std::vector<DeviceMle> l; for (uint32_t j = 0; j < products[p].n_idx; j++) l.push_back(views.at(products[p].idx[j])); vp.add_mle_list(l, Ext(products[p].coef[0], products[p].coef[1])); }
    DynTranscript tr(label);
    std::pair<IOPProof, IOPProverState> res;
    if (shm_region) {
        ShmExchange ex(shm_region, world, rank); if (shm_seq) ex.seq = *shm_seq;
        try { res = IOPProverState::prove_sharded(std::move(vp), nv_total, ex, tr); }
        catch (...) { ex.poison(); if (shm_seq) *shm_seq = ex.seq; throw; }   // peers fail fast instead of spinning on this rank's slot
        if (shm_seq) *shm_seq = ex.seq;
    }
    else { if (!cb && world > 1) throw Error(DP_ERR_INVALID, "prove_sharded: no exchange given"); CallbackExchange ex(cb, user, world, rank); res = IOPProverState::prove_sharded(std::move(vp), nv_total, ex, tr); }
    for (size_t i = 0; i < res.first.point.size(); i++) { out_point[2 * i] = res.first.point[i].c0; out_point[2 * i + 1] = res.first.point[i].c1; }
    size_t k = 0;
    for (auto &m : res.first.proofs) for (auto &e : m.evaluations) { out_msgs[2 * k] = e.c0; out_msgs[2 * k + 1] = e.c1; k++; }
    const ExtVec &fin = res.second.get_mle_final_evaluations();
    write_finals(fin, first_use_remap(products, n_products, n_mles), out_final);
    return 0;
    DPH_CATCH
}

// Basefold commit + open of ONE polynomial sharded over `world` ranks (every rank passes the whole polynomial, resident on its
// GPU).  Exchange as in dph_sumcheck_prove_sharded.  out = the flat proof image of dph_pcs_open (identical on every rank and
// identical to the unsharded proof), out_root = the commitment root.  `times_ms` (optional, 2 doubles): commit / open wall time.
extern "C" int dph_pcs_open_sharded(uint32_t world, uint32_t rank, dp_mle *poly, uint32_t full_log, const uint64_t *point, const char *label,
                                    void *shm_region, uint64_t *shm_seq, CallbackExchange::Fn cb, void *user,
                                    uint64_t *out, uint64_t cap, uint64_t *out_len, uint64_t *out_root, double *times_ms) {
    DPH_TRY
    uint64_t len; int ext; uint32_t nv; check(dp_mle_info(poly, &len, &ext, &nv));
    DeviceMle m = DeviceMle::wrap_device(dp_mle_device_ptr(poly), len, ext);
    BasefoldProverParams pp; pp.full_message_size_log = full_log;
    ExtVec pt; for (uint32_t i = 0; i < nv; i++) pt.push_back(Ext(point[2 * i], point[2 * i + 1]));
    DynTranscript t(label);
    auto run = [&](Exchange &ex) {
        auto t0 = std::chrono::steady_clock::now();
        auto comm = Basefold::commit_sharded(pp, m, ex);
        auto t1 = std::chrono::steady_clock::now();
        if (out_root) memcpy(out_root, comm.root.v, 32);
        BasefoldProof pr = Basefold::open_sharded(pp, comm, pt, t, ex);
        auto t2 = std::chrono::steady_clock::now();
        if (times_ms) { times_ms[0] = std::chrono::duration<double, std::milli>(t1 - t0).count(); times_ms[1] = std::chrono::duration<double, std::milli>(t2 - t1).count(); }
        return pr.flatten();
    };
    std::vector<uint64_t> f;
    if (shm_region) {
        ShmExchange ex(shm_region, world, rank); if (shm_seq) ex.seq = *shm_seq;
        try { f = run(ex); } catch (...) { ex.poison(); if (shm_seq) *shm_seq = ex.seq; throw; }
        if (shm_seq) *shm_seq = ex.seq;
    } else { if (!cb && world > 1) throw Error(DP_ERR_INVALID, "dph_pcs_open_sharded: no exchange given"); CallbackExchange ex(cb, user, world, rank); f = run(ex); }
    *out_len = f.size();
    if (f.size() > cap) { g_herr = "dph_pcs_open_sharded: output buffer too small"; return 2; }
    memcpy(out, f.data(), 8 * f.size());
    return 0;
    DPH_CATCH
}

// prove_batch_polys over T contiguous slices of the caller's device MLEs (views, no copies)
extern "C" int dph_sumcheck_prove_batch_polys(uint32_t T, dp_mle *const *mles, uint32_t n_mles, const dp_sc_product *products, uint32_t n_products,
                                              uint32_t max_nv, const char *label, uint64_t *out_point, uint64_t *out_msgs, uint64_t *out_final) {
    DPH_TRY
    uint32_t logT = 0; while ((1u << logT) < T) logT++;
    std::vector<VirtualPolynomial> polys;
    for (uint32_t t = 0; t < T; t++) {
        VirtualPolynomial vp(max_nv - logT);
        std::vector<DeviceMle> views;
        for (uint32_t i = 0; i < n_mles; i++) {
            uint64_t len; int ext; check(dp_mle_info(mles[i], &len, &ext, nullptr));
            uint64_t sl = len / T;
            views.push_back(DeviceMle::wrap_device((char *)dp_mle_device_ptr(mles[i]) + (size_t)t * sl * (ext ? 16 : 8), sl, ext));
        }
        for (uint32_t p = 0; p < n_products; p++) { std::vector<DeviceMle> l; for (uint32_t j = 0; j < products[p].n_idx; j++) l.push_back(views.at(products[p].idx[j])); vp.add_mle_list(l, Ext(products[p].coef[0], products[p].coef[1])); }
        polys.push_back(std::move(vp));
    }
    DynTranscript tr(label);
    auto res = IOPProverState::prove_batch_polys(T, std::move(polys), tr);
    for (size_t i = 0; i < res.first.point.size(); i++) { out_point[2 * i] = res.first.point[i].c0; out_point[2 * i + 1] = res.first.point[i].c1; }
    size_t k = 0;
    for (auto &m : res.first.proofs) for (auto &e : m.evaluations) { out_msgs[2 * k] = e.c0; out_msgs[2 * k + 1] = e.c1; k++; }
    const ExtVec &fin = res.second.get_mle_final_evaluations();
    write_finals(fin, first_use_remap(products, n_products, n_mles), out_final);
    return 0;
    DPH_CATCH
}

// ---- FFT-convolution layer in isolation (host/conv.hpp): inference + layer proof ----------------------------------
// The output claim is drawn as Prover::prove draws the model-output claim (iop/prover.rs:423-436): point from the
// transcript, eval = MLE(cleared output)(point).  Flat layout: host/conv.hpp flatten_conv_proof.
extern "C" int dph_conv_prove(uint32_t kw, uint32_t kx, uint32_t n_x, uint32_t real_nw, const int64_t *filter, const int64_t *bias, const uint32_t *unpadded_out,
                              const int64_t *input, const char *label, int64_t *out_after_bias, int64_t *out_cleared, uint64_t *out, uint64_t cap, uint64_t *out_len) {
    DPH_TRY
    using namespace dp::zkml;
    Convolution c; c.kw = kw; c.kx = kx; c.nw = n_x; c.real_nw = real_nw;
    c.filter.assign(filter, filter + (size_t)kw * kx * real_nw * real_nw); c.bias.assign(bias, bias + kw);
    for (int i = 0; i < 3; i++) c.unpadded_out[i] = unpadded_out[i];
    c.load();
    std::vector<Element> x(input, input + (size_t)kx * n_x * n_x);
    ConvData pd;
    std::vector<Element> cleared = c.op(x, pd);
    if (out_after_bias) memcpy(out_after_bias, pd.output_as_element.data(), 8 * pd.output_as_element.size());
    if (out_cleared) memcpy(out_cleared, cleared.data(), 8 * cleared.size());
    if (!out_len) return 0;
    DynTranscript t(label);
    Claim cl; for (size_t i = 0; i < ceil_log2(cleared.size()); i++) cl.point.push_back(t.read_challenge());
    cl.eval = DeviceMle::from_evaluations_vec(to_base(cleared)).evaluate(cl.point);
    ConvProof pr; Claim in_claim = c.prove_convolution_step(t, cl, pd, pr);
    std::vector<u64> fl = flatten_conv_proof(pr, in_claim);
    *out_len = fl.size();
    if (out) { if (fl.size() > cap) throw Error(DP_ERR_INVALID, "dph_conv_prove: output buffer too small"); memcpy(out, fl.data(), 8 * fl.size()); }
    return 0;
    DPH_CATCH
}

// General model builder: `desc` holds 9 int64 per node {kind, 8 shape words} and `data` the weights in node order
// (kind 5 MatMul {rows, inner, cols, transposed, has_bias}: the constant right matrix then the bias; kind 0 Dense {nrows, ncols}: weights then bias; 1 Requant {right_shift, fp_scale, multiplier, intermediate_bits};
//  2 ReLU; 3 Conv {kw, kx, nw, real_nw, unpadded_out[3]}: filter then bias; 4 Maxpool {C, H, W}).  Same handle type as
// dph_zkml_context_new: dph_zkml_prove / dph_zkml_prove_concurrent / dph_zkml_context_free apply.
extern "C" int dph_model_context_new(const int64_t *desc, uint32_t n_nodes, const int64_t *data, uint64_t input_len, void **out) {
    DPH_TRY
    using namespace dp::zkml;
    auto *h = new ZkHandle();
    h->model.input_len = input_len;
    const int64_t *w = data;
    for (uint32_t i = 0; i < n_nodes; i++) {
        const int64_t *d = desc + 9 * (size_t)i; Node n;
        switch (d[0]) {
        case 0: n.op = Op::Dense; n.nrows = d[1]; n.ncols = d[2]; n.weights.assign(w, w + n.nrows * n.ncols); w += n.nrows * n.ncols; n.bias.assign(w, w + n.nrows); w += n.nrows; break;
        case 1: n.op = Op::Requant; n.rq.right_shift = d[1]; n.rq.fp_scale = d[2]; n.rq.fixed_point_multiplier = d[3]; n.rq.intermediate_bit_size = d[4]; break;
        case 2: n.op = Op::Relu; break;
        case 3: { n.op = Op::Conv; n.kw = d[1]; n.kx = d[2]; n.nw = d[3]; n.real_nw = d[4]; for (int k = 0; k < 3; k++) n.unpadded_out[k] = d[5 + k];
                  size_t fl = n.kw * n.kx * n.real_nw * n.real_nw; n.weights.assign(w, w + fl); w += fl; n.bias.assign(w, w + n.kw); w += n.kw; break; }
        case 4: n.op = Op::Pool; n.pool_c = d[1]; n.pool_h = d[2]; n.pool_w = d[3]; break;
        case 5: n.op = Op::MatMul; n.mm_r = d[1]; n.mm_k = d[2]; n.mm_c = d[3]; n.mm_t = d[4] != 0; n.mm_bias = d[5] != 0; n.weights.assign(w, w + n.mm_k * n.mm_c); w += n.mm_k * n.mm_c;
                if (n.mm_bias) { n.bias.assign(w, w + n.mm_c); w += n.mm_c; } break;
        default: delete h; throw Error(DP_ERR_INVALID, "dph_model_context_new: unknown node kind");
        }
        h->model.nodes.push_back(std::move(n));
    }
    h->ctx = Context::generate(h->model);
    check(dp_synchronize());
    *out = h;
    return 0;
    DPH_CATCH
}

// batch_commit (+ simple_batch_open at `point` when given): polys are caller-owned device MLEs of equal size / field
extern "C" int dph_pcs_simple_batch(dp_mle *const *polys, uint32_t n, uint32_t full_log, const uint64_t *point, uint32_t nv, const uint64_t *evals, const char *label,
                                    uint64_t *out_root, uint64_t *out, uint64_t cap, uint64_t *out_len) {
    DPH_TRY
    BasefoldProverParams pp; pp.full_message_size_log = full_log;
    std::vector<DeviceMle> ps;
    for (uint32_t i = 0; i < n; i++) { uint64_t len; int ext; check(dp_mle_info(polys[i], &len, &ext, nullptr)); ps.push_back(DeviceMle::wrap_device(dp_mle_device_ptr(polys[i]), len, ext)); }
    BasefoldCommitmentWithWitness comm = Basefold::batch_commit(pp, ps);
    memcpy(out_root, comm.root.v, 32);
    if (!point) return 0;
    ExtVec pt, ev; for (uint32_t i = 0; i < nv; i++) pt.push_back(Ext(point[2 * i], point[2 * i + 1]));
    for (uint32_t i = 0; i < n; i++) ev.push_back(Ext(evals[2 * i], evals[2 * i + 1]));
    DynTranscript t(label);
    SimpleBatchProof sp = Basefold::simple_batch_open(pp, comm, pt, ev, t);
    std::vector<uint64_t> f = sp.flatten();
    *out_len = f.size();
    if (f.size() > cap) throw Error(DP_ERR_INVALID, "dph_pcs_simple_batch: output buffer too small");
    memcpy(out, f.data(), 8 * f.size());
    return 0;
    DPH_CATCH
}

// batch_open with an explicit evaluation list: `points` = n_points points concatenated (point k has point_nv[k] elements),
// evaluation j claims polys[eval_poly[j]] at points[eval_point[j]] (the value is computed here)
extern "C" int dph_pcs_batch_open_evals(dp_mle *const *polys, uint32_t n, uint32_t full_log, const uint64_t *points, const uint32_t *point_nv, uint32_t n_points,
                                        const uint32_t *eval_poly, const uint32_t *eval_point, uint32_t n_evals, const char *label, uint64_t *out, uint64_t cap, uint64_t *out_len) {
    DPH_TRY
    BasefoldProverParams pp; pp.full_message_size_log = full_log;
    std::vector<DeviceMle> ms; std::vector<BasefoldCommitmentWithWitness> comms; std::vector<ExtVec> pts; std::vector<Evaluation> evals;
    for (uint32_t i = 0; i < n; i++) { uint64_t len; int ext; check(dp_mle_info(polys[i], &len, &ext, nullptr)); ms.push_back(DeviceMle::wrap_device(dp_mle_device_ptr(polys[i]), len, ext)); comms.push_back(Basefold::commit(pp, ms.back())); }
    size_t o = 0;
    for (uint32_t k = 0; k < n_points; k++) { ExtVec pt; for (uint32_t j = 0; j < point_nv[k]; j++) pt.push_back(Ext(points[2 * (o + j)], points[2 * (o + j) + 1])); o += point_nv[k]; pts.push_back(pt); }
    for (uint32_t j = 0; j < n_evals; j++) { Evaluation ev; ev.poly = eval_poly[j]; ev.point = eval_point[j]; ev.value = ms.at(ev.poly).evaluate(pts.at(ev.point)); evals.push_back(ev); }
    DynTranscript t(label);
    BasefoldProof pr = Basefold::batch_open(pp, ms, comms, pts, evals, t);
    std::vector<uint64_t> f = pr.flatten();
    *out_len = f.size();
    if (f.size() > cap) throw Error(DP_ERR_INVALID, "dph_pcs_batch_open_evals: output buffer too small");
    memcpy(out, f.data(), 8 * f.size());
    return 0;
    DPH_CATCH
}
