// bis_context.cu -- context, vectors, device scalars, timers.
// C-ABI: include/bis_b200.h ("context", "vectors", "device scalars").
#include "bis_internal.cuh"

#include <cstdlib>
#include <cstring>

static thread_local char g_err[1024] = "";

void bis_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}

extern "C" const char *bis_last_error(void) { return g_err; }
extern "C" int bis_version(void) { return BIS_VERSION; }

extern "C" int bis_device_count(int *count) {
    BIS_REQUIRE(count, "bis_device_count: null output");
    BIS_CUDA(cudaGetDeviceCount(count));
    return 0;
}

// every live context, for bis_cuda_malloc's out-of-memory retry
static std::vector<bis_context *> g_contexts;

static void vector_cache_release(bis_context *c) {
    if (c->vec_cache.empty()) return;
    int cur = 0;
    cudaGetDevice(&cur);
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    for (auto &e : c->vec_cache) cudaFree(e.second);
    c->vec_cache.clear();
    c->vec_cache_bytes = 0;
    cudaSetDevice(cur);
}

// called where a matrix is about to be built (thrust scratch does not go through bis_cuda_malloc)
void bis_vector_cache_trim(bis_context *c) {
    size_t fr = 0, tot = 0;
    if (c->vec_cache.empty() || cudaMemGetInfo(&fr, &tot) != cudaSuccess) return;
    if (fr < tot / 3) vector_cache_release(c);
}

void bis_vector_cache_release_all() {
    for (bis_context *c : g_contexts) vector_cache_release(c);
}

static int context_init(bis_context *c, int device) {
    int ndev = 0;
    BIS_CUDA(cudaGetDeviceCount(&ndev));
    BIS_REQUIRE(ndev > 0, "no CUDA device: this library has no CPU fallback");
    BIS_REQUIRE(device >= 0 && device < ndev, "device %d out of range (%d devices)", device, ndev);
    c->device = device;
    BIS_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    BIS_CUDA(cudaGetDeviceProperties(&prop, device));
    BIS_REQUIRE(prop.major >= 10,
                "device %d is sm_%d%d; this library is built for sm_100a only", device,
                prop.major, prop.minor);
    c->sm_count = prop.multiProcessorCount;
    c->l2_bytes = (size_t)prop.l2CacheSize;
    BIS_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    BIS_CUDA(cudaStreamCreateWithFlags(&c->comm_stream, cudaStreamNonBlocking));
    BIS_CUDA(cudaEventCreate(&c->ev_timer0));
    BIS_CUDA(cudaEventCreate(&c->ev_timer1));
    BIS_CUDA(cudaEventCreateWithFlags(&c->ev_main, cudaEventDisableTiming));
    BIS_CUDA(cudaEventCreateWithFlags(&c->ev_comm, cudaEventDisableTiming));
    BIS_CUDA(cudaEventCreateWithFlags(&c->ev_scalar, cudaEventDisableTiming));
    BIS_CUDA(bis_cuda_malloc(&c->d_scalars, sizeof(double) * BIS_NUM_SCALARS));
    BIS_CUDA(cudaMemset(c->d_scalars, 0, sizeof(double) * BIS_NUM_SCALARS));
    BIS_CUDA(cudaMallocHost(&c->h_scalars, sizeof(double) * BIS_NUM_SCALARS));
    BIS_CUDA(bis_cuda_malloc(&c->d_partials, sizeof(double) * BIS_MAX_RED * BIS_MAX_RED_BLOCKS));
    BIS_CUDA(bis_cuda_malloc(&c->d_counter, sizeof(unsigned int)));
    BIS_CUDA(cudaMemset(c->d_counter, 0, sizeof(unsigned int)));
    BIS_CUDA(bis_cuda_malloc(&c->d_errflag, sizeof(int)));
    BIS_CUDA(cudaMemset(c->d_errflag, 0, sizeof(int)));
    BIS_CUDA(cudaDeviceSynchronize());
    // experiment switches (must be set alike on every rank)
    if (const char *e = getenv("BIS_SPMV_FUSED")) c->opt_spmv_fused = atoi(e);
    if (const char *e = getenv("BIS_TRSV_VARIANT")) c->opt_trsv_variant = atoi(e);
    if (const char *e = getenv("BIS_GRAPH")) c->opt_graph = atoi(e);
    if (const char *e = getenv("BIS_WIN_ROWS")) c->opt_win_rows = atoi(e);
    if (const char *e = getenv("BIS_WAVE_CLUSTER")) c->opt_wave_cluster = atoi(e);
    if (const char *e = getenv("BIS_SPMV_VDICT")) c->opt_spmv_vdict = atoi(e) ? 1 : 0;
    if (const char *e = getenv("BIS_WAVE_BACKOFF_NS")) c->opt_wave_backoff_ns = atoi(e) < 0 ? 0 : atoi(e);
    if (const char *e = getenv("BIS_PRECOND_INNER_ITERS")) c->opt_precond_inner_iters = atoi(e);
    if (const char *e = getenv("BIS_PERM_MODE"))     // NONE / C (colouring) / BFS / RCM / CM, or the option's number
        c->opt_perm_mode = (e[0] == 'C' || e[0] == 'c') ? ((e[1] == 'M' || e[1] == 'm') ? 4 : 1)
                         : (e[0] == 'B' || e[0] == 'b') ? 2 : (e[0] == 'R' || e[0] == 'r') ? 3 : (e[0] >= '1' && e[0] <= '4') ? e[0] - '0' : 0;
    return 0;
}

extern "C" int bis_context_create(int device, bis_context **ctx) {
    BIS_REQUIRE(ctx, "bis_context_create: null output");
    bis_context *c = new bis_context;
    if (context_init(c, device) != 0) {
        delete c;
        return 1;
    }
    g_contexts.push_back(c);
    *ctx = c;
    return 0;
}

extern "C" int bis_nccl_unique_id(void *out, size_t bytes) {
    BIS_REQUIRE(out && bytes >= sizeof(ncclUniqueId), "bis_nccl_unique_id: need %zu bytes",
                sizeof(ncclUniqueId));
    ncclUniqueId id;
    BIS_NCCL(ncclGetUniqueId(&id));
    memcpy(out, &id, sizeof id);
    return 0;
}

extern "C" int bis_context_create_distributed(int device, int rank, int nranks,
                                              const void *nccl_id, size_t nccl_id_bytes,
                                              bis_context **ctx) {
    BIS_REQUIRE(ctx, "bis_context_create_distributed: null output");
    BIS_REQUIRE(nranks >= 1 && rank >= 0 && rank < nranks, "bad rank %d / nranks %d", rank, nranks);
    bis_context *c = new bis_context;
    if (context_init(c, device) != 0) {
        delete c;
        return 1;
    }
    c->rank = rank;
    c->nranks = nranks;
    if (nranks > 1) {
        if (!nccl_id || nccl_id_bytes < sizeof(ncclUniqueId)) {
            bis_set_error("bis_context_create_distributed: nccl_id must hold %zu bytes",
                          sizeof(ncclUniqueId));
            delete c;
            return 2;
        }
        ncclUniqueId id;
        memcpy(&id, nccl_id, sizeof id);
        ncclResult_t r = ncclCommInitRank(&c->comm, nranks, id, rank);
        if (r != ncclSuccess) {
            bis_set_error("ncclCommInitRank failed: %s", ncclGetErrorString(r));
            delete c;
            return 1;
        }
        // a second communicator for the halo exchange so that send/recv on the
        // comm stream never interleaves with the reductions on the main stream
        r = ncclCommSplit(c->comm, 0, rank, &c->comm_halo, nullptr);
        if (r != ncclSuccess) {
            bis_set_error("ncclCommSplit failed: %s", ncclGetErrorString(r));
            ncclCommDestroy(c->comm);
            delete c;
            return 1;
        }
        if (bis_peer_link_setup(c) != 0) {
            ncclCommDestroy(c->comm_halo);
            ncclCommDestroy(c->comm);
            delete c;
            return 1;
        }
    }
    g_contexts.push_back(c);
    *ctx = c;
    return 0;
}

extern "C" int bis_context_destroy(bis_context *c) {
    if (!c) return 0;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    vector_cache_release(c);
    for (size_t i = 0; i < g_contexts.size(); ++i)
        if (g_contexts[i] == c) {
            g_contexts.erase(g_contexts.begin() + (long)i);
            break;
        }
    bis_peer_link_teardown(c);
    if (c->comm_halo) ncclCommDestroy(c->comm_halo);
    if (c->comm) ncclCommDestroy(c->comm);
    cudaFree(c->d_scalars);
    cudaFreeHost(c->h_scalars);
    cudaFree(c->d_partials);
    cudaFree(c->d_block_partials);
    cudaFree(c->d_counter);
    cudaFree(c->d_errflag);
    cudaFree(c->d_barrier_word);
    cudaFree(c->d_flush);
    for (int i = 0; i < BIS_PROF_NTAGS; ++i)
        for (cudaEvent_t e : c->prof[i].ev) cudaEventDestroy(e);
    cudaEventDestroy(c->ev_timer0);
    cudaEventDestroy(c->ev_timer1);
    cudaEventDestroy(c->ev_main);
    cudaEventDestroy(c->ev_comm);
    cudaEventDestroy(c->ev_scalar);
    cudaStreamDestroy(c->stream);
    cudaStreamDestroy(c->comm_stream);
    delete c;
    return 0;
}

extern "C" int bis_context_synchronize(bis_context *c) {
    BIS_REQUIRE(c, "null context");
    BIS_CUDA(cudaStreamSynchronize(c->stream));
    int flag = 0;
    BIS_CUDA(cudaMemcpy(&flag, c->d_errflag, sizeof(int), cudaMemcpyDeviceToHost));
    if (flag) {
        cudaMemset(c->d_errflag, 0, sizeof(int));
        bis_set_error("device watchdog fired (code %d): %s", flag,
                      flag >= 20 ? "a peer rank did not deliver its part of a reduction or halo exchange"
                                 : "a level-scheduled triangular solve did not make progress");
        return 3;
    }
    return 0;
}

extern "C" int bis_context_rank(const bis_context *c, int *rank, int *nranks) {
    BIS_REQUIRE(c, "null context");
    if (rank) *rank = c->rank;
    if (nranks) *nranks = c->nranks;
    return 0;
}

extern "C" int bis_context_info(bis_context *c, int64_t info[8]) {
    BIS_REQUIRE(c && info, "null argument");
    size_t fr = 0, tot = 0;
    BIS_CUDA(cudaSetDevice(c->device));
    BIS_CUDA(cudaMemGetInfo(&fr, &tot));
    for (int i = 0; i < 8; ++i) info[i] = 0;
    info[0] = c->sm_count;
    info[1] = (int64_t)fr;
    info[2] = (int64_t)tot;
    info[3] = c->launches;
    info[4] = (int64_t)c->l2_bytes;
    info[6] = c->chain_solves;
    info[7] = c->wave_solves;
    info[5] = (c->peer_on && c->opt_dist_p2p) ? 1 : 0;   // 1: collectives run over peer memory, 0: NCCL
    return 0;
}

extern "C" int bis_timer_start(bis_context *c) {
    BIS_REQUIRE(c, "null context");
    BIS_CUDA(cudaEventRecord(c->ev_timer0, c->stream));
    return 0;
}

extern "C" int bis_timer_stop(bis_context *c, double *elapsed_ms) {
    BIS_REQUIRE(c && elapsed_ms, "null argument");
    BIS_CUDA(cudaEventRecord(c->ev_timer1, c->stream));
    BIS_CUDA(cudaEventSynchronize(c->ev_timer1));
    float ms = 0.f;
    BIS_CUDA(cudaEventElapsedTime(&ms, c->ev_timer0, c->ev_timer1));
    *elapsed_ms = (double)ms;
    return 0;
}

int bis_ensure_dynamic_smem(bis_context *c, const void *func, size_t bytes) {
    auto it = c->smem_configured.find(func);
    if (it != c->smem_configured.end() && it->second >= bytes) return 0;
    BIS_CUDA(cudaSetDevice(c->device));
    BIS_CUDA(cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    c->smem_configured[func] = bytes;
    return 0;
}

// ---- per-family kernel timing ---------------------------------------------------
static int prof_flush(bis_context *c, ProfTag &t) {
    if (t.used == 0) return 0;
    BIS_CUDA(cudaEventSynchronize(t.ev[t.used - 1]));
    for (size_t i = 0; i + 1 < t.used; i += 2) {
        float ms = 0.f;
        BIS_CUDA(cudaEventElapsedTime(&ms, t.ev[i], t.ev[i + 1]));
        t.acc_ms += (double)ms;
        t.count++;
    }
    t.used = 0;
    (void)c;
    return 0;
}

int bis_prof_begin(bis_context *c, int tag) {
    if (!c->profile) return 0;
    ProfTag &t = c->prof[tag];
    if (t.used >= 16384) BIS_CHECK(prof_flush(c, t));   // bounded pool; a flush waits for the stream
    while (t.ev.size() < t.used + 2) {
        cudaEvent_t e;
        BIS_CUDA(cudaEventCreate(&e));
        t.ev.push_back(e);
    }
    BIS_CUDA(cudaEventRecord(t.ev[t.used], c->stream));
    return 0;
}

int bis_prof_end(bis_context *c, int tag) {
    if (!c->profile) return 0;
    ProfTag &t = c->prof[tag];
    BIS_CUDA(cudaEventRecord(t.ev[t.used + 1], c->stream));
    t.used += 2;
    return 0;
}

extern "C" int bis_profile_enable(bis_context *c, int on) {
    BIS_REQUIRE(c, "null context");
    BIS_CUDA(cudaStreamSynchronize(c->stream));
    for (int i = 0; i < BIS_PROF_NTAGS; ++i) {
        BIS_CHECK(prof_flush(c, c->prof[i]));
        c->prof[i].acc_ms = 0.0;
        c->prof[i].count = 0;
    }
    c->profile = on ? 1 : 0;
    return 0;
}

extern "C" int bis_profile_read(bis_context *c, const char *family, double *total_ms, int64_t *launches) {
    BIS_REQUIRE(c && family && total_ms && launches, "null argument");
    std::string f(family);
    int tag = f == "spmv" ? BIS_PROF_SPMV : f == "sptrsv" ? BIS_PROF_SPTRSV : f == "vector" ? BIS_PROF_VECTOR : -1;
    BIS_REQUIRE(tag >= 0, "bis_profile_read: unknown kernel family '%s' (spmv, sptrsv, vector)", family);
    BIS_CHECK(prof_flush(c, c->prof[tag]));
    *total_ms = c->prof[tag].acc_ms;
    *launches = c->prof[tag].count;
    return 0;
}

// ---- CUDA graphs ----------------------------------------------------------------------------------
// An iteration body is a fixed sequence of launches whose arguments (device addresses, scalar slots)
// repeat with the period of the method's pointer exchange; alpha, beta, ... are formed on the device,
// so nothing in it depends on the host.  begin/end record that sequence once from the ordinary C-ABI
// calls (nothing executes while recording), launch replays it: one submission instead of 3..30.
struct bis_graph {
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    int64_t kernel_nodes = 0;
};

extern "C" int bis_graph_begin(bis_context *c) {
    BIS_REQUIRE(c, "null context");
    BIS_REQUIRE(!c->capturing, "bis_graph_begin: already recording");
    BIS_REQUIRE(c->nranks == 1, "bis_graph_begin: the halo / reduction epochs of a distributed context are launch arguments");
    BIS_REQUIRE(!c->profile, "bis_graph_begin: per-launch profiling is on");
    BIS_CUDA(cudaSetDevice(c->device));
    BIS_CUDA(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
    c->capturing = 1;
    return 0;
}

extern "C" int bis_graph_end(bis_context *c, bis_graph **out) {
    BIS_REQUIRE(c && out, "null argument");
    BIS_REQUIRE(c->capturing, "bis_graph_end: not recording");
    c->capturing = 0;
    c->graph_epoch++;
    *out = nullptr;
    cudaGraph_t g = nullptr;
    cudaError_t e = cudaStreamEndCapture(c->stream, &g);
    if (e != cudaSuccess || !g) {
        cudaGetLastError();
        bis_set_error("bis_graph_end: the recorded sequence cannot be a graph: %s", cudaGetErrorString(e));
        return 1;
    }
    bis_graph *bg = new bis_graph;
    bg->graph = g;
    e = cudaGraphInstantiate(&bg->exec, g, 0);
    if (e != cudaSuccess) {
        cudaGetLastError();
        cudaGraphDestroy(g);
        delete bg;
        bis_set_error("bis_graph_end: cudaGraphInstantiate failed: %s", cudaGetErrorString(e));
        return 1;
    }
    size_t n_nodes = 0;
    if (cudaGraphGetNodes(g, nullptr, &n_nodes) == cudaSuccess && n_nodes) {
        std::vector<cudaGraphNode_t> nodes(n_nodes);
        if (cudaGraphGetNodes(g, nodes.data(), &n_nodes) == cudaSuccess)
            for (size_t i = 0; i < n_nodes; ++i) {
                cudaGraphNodeType t;
                if (cudaGraphNodeGetType(nodes[i], &t) == cudaSuccess && t == cudaGraphNodeTypeKernel) bg->kernel_nodes++;
            }
    }
    *out = bg;
    return 0;
}

// Abandons a recording (the caller then issues the same calls again, eagerly).
extern "C" int bis_graph_abort(bis_context *c) {
    BIS_REQUIRE(c, "null context");
    if (!c->capturing) return 0;
    c->capturing = 0;
    c->graph_epoch++;
    cudaGraph_t g = nullptr;
    cudaStreamEndCapture(c->stream, &g);
    if (g) cudaGraphDestroy(g);
    cudaGetLastError();
    return 0;
}

extern "C" int bis_graph_launch(bis_context *c, bis_graph *g) {
    BIS_REQUIRE(c && g && g->exec, "bis_graph_launch: null argument");
    BIS_REQUIRE(!c->capturing, "bis_graph_launch: recording");
    BIS_CUDA(cudaSetDevice(c->device));
    BIS_CUDA(cudaGraphLaunch(g->exec, c->stream));
    c->launches += g->kernel_nodes;   // the kernels a replay runs count like the launches they replace
    c->graph_epoch++;
    return 0;
}

extern "C" int bis_graph_free(bis_context *c, bis_graph *g) {
    if (!g) return 0;
    if (c) {
        cudaSetDevice(c->device);
        cudaStreamSynchronize(c->stream);
    }
    if (g->exec) cudaGraphExecDestroy(g->exec);
    if (g->graph) cudaGraphDestroy(g->graph);
    delete g;
    return 0;
}

extern "C" int bis_context_get_option(bis_context *c, const char *key, int *value) {
    BIS_REQUIRE(c && key && value, "null argument");
    std::string k(key);
    if (k == "graph") *value = (c->opt_graph && c->nranks == 1) ? 1 : 0;
    else if (k == "precond_inner_iters") *value = c->opt_precond_inner_iters;
    else if (k == "perm_mode") *value = c->opt_perm_mode;
    else if (k == "spmv_vdict") *value = c->opt_spmv_vdict;
    else if (k == "spmv_value_bytes") *value = c->last_spmv_value_bytes;   // read-only: what the last windowed SpMV streamed per nonzero
    else if (k == "factor_keep_crs") *value = c->opt_factor_keep_crs;
    else if (k == "spmv_variant") *value = c->opt_spmv_variant;
    else if (k == "trsv_variant") *value = c->opt_trsv_variant;
    else if (k == "spmv_fused") *value = c->opt_spmv_fused;
    else if (k == "dist_p2p") *value = c->opt_dist_p2p;
    else {
        bis_set_error("bis_context_get_option: unknown option '%s'", key);
        return 2;
    }
    return 0;
}

extern "C" int bis_flush_l2(bis_context *c) {
    BIS_REQUIRE(c, "null context");
    if (!c->d_flush) {
        c->flush_bytes = c->l2_bytes ? 2 * c->l2_bytes : ((size_t)256 << 20);
        BIS_CUDA(bis_cuda_malloc(&c->d_flush, c->flush_bytes));
    }
    BIS_CUDA(cudaMemsetAsync(c->d_flush, 1, c->flush_bytes, c->stream));
    return 0;
}

extern "C" int bis_context_set_option(bis_context *c, const char *key, int value) {
    BIS_REQUIRE(c && key, "null argument");
    std::string k(key);
    if (k == "spmv_variant") c->opt_spmv_variant = value;
    else if (k == "spmv_fused") c->opt_spmv_fused = value;
    else if (k == "dist_p2p") {
        // the transport must change on all ranks at the same point of the stream
        BIS_CUDA(cudaStreamSynchronize(c->stream));
        c->opt_dist_p2p = value;
    }
    else if (k == "spmv_lanes") c->opt_spmv_lanes = value;
    else if (k == "graph") c->opt_graph = value;
    else if (k == "perm_mode") {
        BIS_REQUIRE(value >= 0 && value <= 4, "perm_mode: 0 (NONE), 1 (C, multicolouring), 2 (BFS levels), 3 (reverse Cuthill-McKee) or 4 (Cuthill-McKee)");
        c->opt_perm_mode = value;
    }
    else if (k == "precond_inner_iters") {
        BIS_REQUIRE(value >= 0 && value <= 64, "precond_inner_iters outside [0, 64]");
        c->opt_precond_inner_iters = value;
    }
    else if (k == "trsv_variant") c->opt_trsv_variant = value;
    else if (k == "trsv_debug") c->opt_trsv_debug = value;
    else if (k == "vector_cache") {
        c->opt_vector_cache = value;
        if (!value) vector_cache_release(c);
    }
    else if (k == "trsv_gates") c->opt_trsv_gates = value;
    else if (k == "trsv_block") c->opt_trsv_block = value;
    else if (k == "trsv_sleep1") c->opt_trsv_sleep[0] = value;
    else if (k == "trsv_sleep2") c->opt_trsv_sleep[1] = value;
    else if (k == "trsv_sleep3") c->opt_trsv_sleep[2] = value;
    else if (k == "trsv_sleep4") c->opt_trsv_sleep[3] = value;
    else if (k == "trsv_poll_ns") c->opt_trsv_poll_ns = value;
    else if (k == "spmv_rows") c->opt_spmv_rows = value;
    else if (k == "spmv_stages") c->opt_spmv_stages = value;
    else if (k == "factor_keep_crs") c->opt_factor_keep_crs = value ? 1 : 0;
    else if (k == "spmv_smem_kb") c->opt_spmv_smem_kb = value;
    else if (k == "spmv_l2_mb") c->opt_spmv_l2_mb = value;
    else if (k == "spmv_blocked") c->opt_spmv_blocked = value;
    else if (k == "spmv_mult") c->opt_spmv_mult = value;
    else if (k == "win_rows") c->opt_win_rows = value;
    else if (k == "wave_cluster") c->opt_wave_cluster = value;
    else if (k == "spmv_vdict") c->opt_spmv_vdict = value ? 1 : 0;
    else if (k == "wave_backoff_ns") c->opt_wave_backoff_ns = value < 0 ? 0 : value;
#ifdef BIS_PERF_DEBUG
    else if (k == "wave_debug") c->opt_wave_debug = value;
    else if (k == "spmv_debug") c->opt_spmv_debug = value;
#endif
    else {
        bis_set_error("unknown option '%s'", key);
        return 2;
    }
    return 0;
}

// ---- vectors ----------------------------------------------------------------
extern "C" int bis_vector_alloc(bis_context *c, int64_t n, double **v) {
    BIS_REQUIRE(c && v && n >= 0, "bis_vector_alloc: bad argument");
    BIS_CUDA(cudaSetDevice(c->device));
    // +2: the x windows of SpMV variant 3 are copied in 16-byte units and may overrun an odd length
    size_t bytes = sizeof(double) * ((size_t)(n > 0 ? n : 1) + 2);
    *v = nullptr;
    for (size_t i = c->vec_cache.size(); i-- > 0;)
        if (c->vec_cache[i].first == bytes) {
            *v = static_cast<double *>(c->vec_cache[i].second);
            c->vec_cache.erase(c->vec_cache.begin() + (long)i);
            c->vec_cache_bytes -= bytes;
            break;
        }
    if (!*v) BIS_CUDA(bis_cuda_malloc(v, bytes));
    c->vec_bytes[*v] = bytes;
    BIS_CUDA(cudaMemsetAsync(*v, 0, bytes, c->stream));
    return 0;
}

extern "C" int bis_vector_free(bis_context *c, double *v) {
    BIS_REQUIRE(c, "null context");
    if (!v) return 0;
    BIS_CUDA(cudaStreamSynchronize(c->stream));
    auto it = c->vec_bytes.find(v);
    if (it != c->vec_bytes.end()) {
        const size_t bytes = it->second;
        c->vec_bytes.erase(it);
        if (c->opt_vector_cache && c->vec_cache_bytes + bytes <= ((size_t)48 << 30) && c->vec_cache.size() < 256) {
            c->vec_cache.emplace_back(bytes, v);
            c->vec_cache_bytes += bytes;
            return 0;
        }
    }
    BIS_CUDA(cudaFree(v));
    return 0;
}

extern "C" int bis_vector_upload(bis_context *c, double *dst, const double *src, int64_t n) {
    BIS_REQUIRE(c && (n == 0 || (dst && src)), "bis_vector_upload: null pointer");
    if (n == 0) return 0;
    BIS_CUDA(cudaMemcpyAsync(dst, src, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
    BIS_CUDA(cudaStreamSynchronize(c->stream));   // src is never retained
    return 0;
}

extern "C" int bis_vector_download(bis_context *c, double *dst, const double *src, int64_t n) {
    BIS_REQUIRE(c && (n == 0 || (dst && src)), "bis_vector_download: null pointer");
    if (n == 0) return 0;
    BIS_CUDA(cudaMemcpyAsync(dst, src, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
    BIS_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
}

// ---- device scalars -----------------------------------------------------------
extern "C" int bis_scalar_set(bis_context *c, int slot, double value) {
    BIS_REQUIRE(c && slot >= 0 && slot < BIS_NUM_SCALARS, "bis_scalar_set: bad slot %d", slot);
    // stream-ordered 8-byte write from pageable memory is staged by the driver
    BIS_CUDA(cudaMemcpyAsync(c->d_scalars + slot, &value, sizeof(double), cudaMemcpyHostToDevice,
                             c->stream));
    BIS_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
}

extern "C" int bis_scalar_get(bis_context *c, int first_slot, int count, double *values) {
    BIS_REQUIRE(c && values && first_slot >= 0 && count >= 0 &&
                    first_slot + count <= BIS_NUM_SCALARS,
                "bis_scalar_get: bad range [%d,+%d)", first_slot, count);
    if (count == 0) return 0;
    BIS_CUDA(cudaMemcpyAsync(c->h_scalars + first_slot, c->d_scalars + first_slot,
                             sizeof(double) * count, cudaMemcpyDeviceToHost, c->stream));
    BIS_CUDA(cudaStreamSynchronize(c->stream));
    memcpy(values, c->h_scalars + first_slot, sizeof(double) * count);
    return 0;
}

// Split read: begin() enqueues the copy behind everything queued so far and returns at once, end()
// waits for THAT copy only -- work queued in between (the next iteration) keeps the device busy
// while the host looks at the value.  One read may be outstanding per context.
extern "C" int bis_scalar_read_begin(bis_context *c, int first_slot, int count) {
    BIS_REQUIRE(c && first_slot >= 0 && count > 0 && first_slot + count <= BIS_NUM_SCALARS,
                "bis_scalar_read_begin: bad range [%d,+%d)", first_slot, count);
    BIS_CUDA(cudaMemcpyAsync(c->h_scalars + first_slot, c->d_scalars + first_slot, sizeof(double) * count,
                             cudaMemcpyDeviceToHost, c->stream));
    BIS_CUDA(cudaEventRecord(c->ev_scalar, c->stream));
    return 0;
}

extern "C" int bis_scalar_read_end(bis_context *c, int first_slot, int count, double *values) {
    BIS_REQUIRE(c && values && first_slot >= 0 && count > 0 && first_slot + count <= BIS_NUM_SCALARS,
                "bis_scalar_read_end: bad range [%d,+%d)", first_slot, count);
    BIS_CUDA(cudaEventSynchronize(c->ev_scalar));
    memcpy(values, c->h_scalars + first_slot, sizeof(double) * count);
    return 0;
}

extern "C" int bis_scalar_copy(bis_context *c, int dst_slot, int src_slot) {
    BIS_REQUIRE(c && dst_slot >= 0 && dst_slot < BIS_NUM_SCALARS && src_slot >= 0 &&
                    src_slot < BIS_NUM_SCALARS,
                "bis_scalar_copy: bad slot");
    BIS_CUDA(cudaMemcpyAsync(c->d_scalars + dst_slot, c->d_scalars + src_slot, sizeof(double),
                             cudaMemcpyDeviceToDevice, c->stream));
    return 0;
}

// Called after a reduction kernel wrote its slot(s): sum over ranks.
int bis_reduce_finish(bis_context *c, int slot_a, int slot_b) {
    if (c->nranks <= 1) return 0;
    if (c->peer_on && c->opt_dist_p2p) return 0;   // the reducing kernel's last block already summed over ranks
    if (slot_a >= 0 && slot_b == slot_a + 1) {
        BIS_NCCL(ncclAllReduce(c->d_scalars + slot_a, c->d_scalars + slot_a, 2, ncclDouble, ncclSum,
                               c->comm, c->stream));
        return 0;
    }
    if (slot_a >= 0)
        BIS_NCCL(ncclAllReduce(c->d_scalars + slot_a, c->d_scalars + slot_a, 1, ncclDouble, ncclSum,
                               c->comm, c->stream));
    if (slot_b >= 0)
        BIS_NCCL(ncclAllReduce(c->d_scalars + slot_b, c->d_scalars + slot_b, 1, ncclDouble, ncclSum,
                               c->comm, c->stream));
    return 0;
}

// ---- row partition: 8 virtual slabs ------------------------------------------------------------------
static int64_t pow2_ceil(int64_t v) {
    int64_t p = 1;
    while (p < v) p <<= 1;
    return p;
}

void bis_partition_rule(int64_t n_global, int64_t plane, int64_t vb[BIS_NSLAB + 1], int *chunk) {
    // rows per block of a reducing streaming kernel: 8192..16384 blocks on a large problem
    int64_t ch = pow2_ceil((n_global + 16383) / 16384);
    if (ch < BIS_RED_CHUNK_MIN) ch = BIS_RED_CHUNK_MIN;
    if (ch > (1 << 20)) ch = 1 << 20;
    *chunk = (int)ch;
    // equal row blocks, rounded up to whole chunks (then streaming kernels AND the windowed SpMV reduce
    // partition-invariantly; an eighth of HPCG-128/256/512 is a whole number of chunks and of z-planes), on
    // small problems only to whole SpMV tiles of 128 rows, on tiny ones not at all -- never leaving a slab empty
    (void)plane;
    int64_t per = (n_global + BIS_NSLAB - 1) / BIS_NSLAB;
    for (int64_t unit : {ch, (int64_t)128}) {
        const int64_t r = (per + unit - 1) / unit * unit;
        if (r * (BIS_NSLAB - 1) < n_global) {
            per = r;
            break;
        }
    }
    for (int v = 0; v <= BIS_NSLAB; ++v) vb[v] = per * v < n_global ? per * v : n_global;
}

void bis_partition_rows(int64_t n_global, int64_t plane, int rank, int nranks, int64_t *begin, int64_t *end) {
    if (nranks >= 1 && BIS_NSLAB % nranks == 0) {
        int64_t vb[BIS_NSLAB + 1];
        int ch;
        bis_partition_rule(n_global, plane, vb, &ch);
        const int per = BIS_NSLAB / nranks;
        *begin = vb[rank * per];
        *end = vb[(rank + 1) * per];
        return;
    }
    // rank counts that do not divide 8: contiguous row blocks, whole planes when there are enough
    const int64_t planes = plane > 0 ? n_global / plane : 0;
    if (plane > 0 && planes >= nranks) {
        const int64_t q = planes / nranks, r = planes % nranks;
        const int64_t b = rank * q + (rank < r ? rank : r);
        *begin = b * plane;
        *end = (b + q + (rank < r ? 1 : 0)) * plane;
    } else {
        const int64_t q = n_global / nranks, r = n_global % nranks;
        *begin = rank * q + (rank < r ? rank : r);
        *end = *begin + q + (rank < r ? 1 : 0);
    }
}

static RowPartition make_partition(int nranks, int64_t n_global, int64_t plane, int64_t row_begin, int64_t n_local) {
    RowPartition p;
    p.n_global = n_global;
    p.row_begin = row_begin;
    p.n_local = n_local;
    int64_t vb[BIS_NSLAB + 1];
    bis_partition_rule(n_global, plane, vb, &p.chunk);
    p.n_slab = 1;
    p.slab_first = 0;
    p.slab_row[0] = 0;
    p.slab_row[1] = n_local;
    p.invariant = false;
    if (nranks >= 1 && BIS_NSLAB % nranks == 0) {
        // the row block must be a union of consecutive virtual slabs
        const int per = BIS_NSLAB / nranks;
        for (int v = 0; v + per <= BIS_NSLAB; v += per)
            if (vb[v] == row_begin && vb[v + per] == row_begin + n_local) {
                p.n_slab = per;
                p.slab_first = v;
                for (int i = 0; i <= per; ++i) p.slab_row[i] = vb[v + i] - row_begin;
                p.invariant = true;
                break;
            }
    }
    return p;
}

void bis_partition_set(bis_context *c, int64_t n_global, int64_t plane, int64_t row_begin, int64_t n_local) {
    c->part = make_partition(c->nranks, n_global, plane, row_begin, n_local);
}

RowPartition bis_partition_for(const bis_context *c, int64_t n) {
    if (c->part.n_local == n && c->part.n_global > 0) return c->part;
    // a vector of another length: on one GPU the default rule for that length (still the fixed tree);
    // in a distributed context its global layout is unknown: one record per rank
    if (c->nranks == 1) return make_partition(1, n, 0, 0, n);
    RowPartition p;
    p.n_global = p.n_local = n;
    p.chunk = BIS_RED_CHUNK_MIN;
    p.slab_row[1] = n;
    return p;
}

extern "C" int bis_partition_row_block(int64_t n_global, int64_t plane, int rank, int nranks, int64_t *begin,
                                       int64_t *end) {
    BIS_REQUIRE(begin && end && nranks >= 1 && rank >= 0 && rank < nranks && n_global >= 0, "bis_partition_row_block: bad argument");
    bis_partition_rows(n_global, plane, rank, nranks, begin, end);
    return 0;
}

// Reduction arguments without a slab layout (the launcher fills n_slab / slab_off / total_blocks).
RedArgs bis_red_args(bis_context *c, int slot_a, int slot_b) {
    RedArgs ra;
    ra.partials = c->d_partials;
    ra.counter = c->d_counter;
    ra.scalars = c->d_scalars;
    ra.slot[0] = slot_a;
    ra.slot[1] = slot_b;
    ra.block_offset = 0;
    ra.total_blocks = 0;
    ra.finalize = 1;
    ra.n_slab = 1;
    for (int i = 0; i <= BIS_NSLAB; ++i) ra.slab_off[i] = 0;
    ra.n_rec = 1;
    ra.rec_first = 0;
    ra.peer_n = 0;
    ra.peer_rank = c->rank;
    ra.peer_epoch = 0;
    for (int p = 0; p < BIS_MAX_PEERS; ++p) ra.peer_bank[p] = c->peer_bank[p];
    ra.errflag = c->d_errflag;
    ra.waitstat = c->d_waitstat;
    if (c->nranks > 1 && c->peer_on && c->opt_dist_p2p && (slot_a >= 0 || slot_b >= 0)) {
        ra.peer_n = c->nranks;
        ra.peer_epoch = ++c->red_epoch;
        ra.n_rec = c->nranks;       // one record per rank unless bis_red_set_slabs finds the invariant layout
        ra.rec_first = c->rank;
    }
    return ra;
}

// Slab layout of the partials: `off[i]` = first partial of local slab i (n_slab + 1 entries).  With an
// invariant partition the 8 slab records are exchanged; otherwise the rank contributes one record.
void bis_red_set_slabs(const bis_context *c, RedArgs &ra, const RowPartition &part, const int *off, int total) {
    ra.total_blocks = total;
    const bool inv = part.invariant && BIS_NSLAB % c->nranks == 0;
    if (inv) {
        ra.n_slab = part.n_slab;
        for (int i = 0; i <= part.n_slab; ++i) ra.slab_off[i] = off[i];
        for (int i = part.n_slab + 1; i <= BIS_NSLAB; ++i) ra.slab_off[i] = off[part.n_slab];
        if (ra.peer_n > 1) {
            ra.n_rec = BIS_NSLAB;
            ra.rec_first = part.slab_first;
        } else {
            ra.n_rec = part.n_slab;   // one GPU: all 8; NCCL transport: the local slabs, then ncclAllReduce
            ra.rec_first = 0;
        }
    } else {
        ra.n_slab = 1;
        ra.slab_off[0] = 0;
        for (int i = 1; i <= BIS_NSLAB; ++i) ra.slab_off[i] = total;
        if (ra.peer_n > 1) {
            ra.n_rec = c->nranks;
            ra.rec_first = c->rank;
        } else {
            ra.n_rec = 1;
            ra.rec_first = 0;
        }
    }
}
