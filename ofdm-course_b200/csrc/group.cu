// ofdm_group: the five ofdm_sweep_* calls run on several GPUs from ONE host call (C, MATLAB / MEX, Julia hosts).
//
// A group is one ofdm_ctx per member; member i is rank i of world n.  A call starts one host thread per member, which makes
// the member's device current, zeroes its device outputs, runs the single-context sweep for (rank i, world n) on the member's
// stream, copies the result back and synchronises.  The calling thread then assembles the host outputs: integer arrays are
// summed, per-stream cells are copied from the member whose ofdm_sweep_share range holds them (never summed, so -0.0 and NaN
// payloads survive).  The sweeps' outputs do not depend on the rank count, so the result is that of one context with world 1.
//
// Contexts are independent: libofdm_b200 keeps its mutable state in its ofdm_ctx (caches, scratch, streams, the error text)
// and has no __constant__ symbols.  Two things are process-wide: the driver entry point of the tensor-map encoder, set once
// under the C++ rule for function-local statics, and each kernel's dynamic shared-memory limit on a device, which two members
// on one GPU share -- func_smem_optin only ever raises it, under a lock, so no member's opt-in is undone before its launch.
// The CUDA runtime's error state and current device are per host thread.
#include <algorithm>
#include <thread>

#include "common.cuh"

namespace {

// Output arrays per sweep (part 2 has three); every cell is 8 bytes (int64 or double).
constexpr int GROUP_MAX_OUT = 3;

// One output array of a sweep.  `fields` == 0: an integer array, summed over the members.  Otherwise a per-stream array
// laid out [point][field][j], j < per_point, whose cells of work item point * per_point + j belong to one member.
struct GroupOut {
    void* host;
    int64_t cells;
    int64_t fields;
};

struct Member {
    int device = 0;
    ofdm_ctx* ctx = nullptr;
    int rc = OFDM_OK;
    int64_t first = 0, count = 0;                       // this member's share of the call's work items
    void* dev[GROUP_MAX_OUT] = {nullptr, nullptr, nullptr};
    size_t dev_bytes[GROUP_MAX_OUT] = {0, 0, 0};
    std::vector<int64_t> host[GROUP_MAX_OUT];           // the cells copied back, from cell host_first[k] on
    int64_t host_first[GROUP_MAX_OUT] = {0, 0, 0};
};

int64_t dim(int64_t v) { return v > 0 ? v : 0; }

}  // namespace

struct ofdm_group {
    std::vector<Member> m;
    std::string err;
};

// Runs f(member, index) on one host thread per member and joins them all.  A member whose thread cannot be started gets
// OFDM_ERR_CUDA (nothing throws across the ABI).
template <typename F> static void group_each(std::vector<Member>& members, F&& f) {
    std::vector<std::thread> th;
    th.reserve(members.size());
    for (size_t i = 0; i < members.size(); ++i) {
        try {
            th.emplace_back([&f, &members, i] {
                try {
                    f(members[i], (int)i);
                } catch (...) {   // std::bad_alloc of a host staging buffer
                    members[i].rc = ctx_fail(members[i].ctx, OFDM_ERR_CUDA, "out of host memory");
                }
            });
        } catch (...) {
            members[i].rc = ctx_fail(members[i].ctx, OFDM_ERR_CUDA, "could not start a host thread for this member");
        }
    }
    for (auto& t : th) t.join();
}

static int group_fail(ofdm_group* g, int code, const char* msg) {
    g->err = msg;
    return code;
}

// The status of the lowest-index failing member (OFDM_OK when none failed), with its text in g->err.
static int group_status(ofdm_group* g) {
    for (size_t i = 0; i < g->m.size(); ++i) {
        const Member& m = g->m[i];
        if (m.rc == OFDM_OK) continue;
        char buf[640];
        snprintf(buf, sizeof buf, "device %d (member %d): %s", m.device, (int)i, m.ctx ? ofdm_last_error(m.ctx) : "context not created");
        g->err = buf;
        return m.rc;
    }
    g->err.clear();
    return OFDM_OK;
}

static void group_free_members(std::vector<Member>& members) {
    group_each(members, [](Member& m, int) {
        if (!m.ctx) return;
        cudaSetDevice(m.device);
        for (int k = 0; k < GROUP_MAX_OUT; ++k) if (m.dev[k]) cudaFree(m.dev[k]);
        ofdm_ctx_destroy(m.ctx);
        m.ctx = nullptr;
    });
}

// One group call: `total` work items, `per_point` of them per point, the outputs `outs`, and
// call(ctx, rank, world, dev) the single-context sweep on the member's device buffers dev[k] (one per output).
template <typename Call>
static int group_run(ofdm_group* g, int64_t total, int64_t per_point, const std::vector<GroupOut>& outs, Call&& call) {
    const int world = (int)g->m.size();
    const int n_out = (int)outs.size();
    group_each(g->m, [&](Member& m, int rank) {
        ofdm_ctx* ctx = m.ctx;
        m.rc = OFDM_OK;
        m.first = m.count = 0;
        const cudaError_t e = cudaSetDevice(m.device);
        if (e != cudaSuccess) { m.rc = ctx_fail(ctx, OFDM_ERR_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e)); return; }
        ofdm_sweep_share(total, rank, world, &m.first, &m.count);
        int rc = OFDM_OK;
        for (int k = 0; k < n_out && rc == OFDM_OK; ++k) {         // grow-only device outputs, never NULL
            const size_t bytes = std::max<size_t>(sizeof(int64_t) * (size_t)outs[k].cells, 256);
            if (m.dev_bytes[k] >= bytes) continue;
            if (m.dev[k]) { cudaFree(m.dev[k]); m.dev[k] = nullptr; m.dev_bytes[k] = 0; }
            rc = ofdm_malloc(ctx, &m.dev[k], bytes);
            if (rc == OFDM_OK) m.dev_bytes[k] = bytes;
        }
        if (m.count > 0)
            for (int k = 0; k < n_out && rc == OFDM_OK; ++k) rc = ofdm_memset(ctx, m.dev[k], 0, sizeof(int64_t) * (size_t)outs[k].cells);
        if (rc == OFDM_OK) rc = call(ctx, rank, world, m.dev);     // validates the params even when the share is empty
        if (rc == OFDM_OK && m.count > 0) {
            for (int k = 0; k < n_out && rc == OFDM_OK; ++k) {
                int64_t lo = 0, hi = outs[k].cells;               // integer arrays: all of it
                if (outs[k].fields) {                              // per-stream arrays: the points this share touches
                    const int64_t row = outs[k].fields * per_point;
                    lo = m.first / per_point * row;
                    hi = ((m.first + m.count - 1) / per_point + 1) * row;
                }
                m.host_first[k] = lo;
                m.host[k].resize((size_t)(hi - lo));
                rc = ofdm_d2h(ctx, m.host[k].data(), (const int64_t*)m.dev[k] + lo, sizeof(int64_t) * (size_t)(hi - lo));
            }
        }
        const cudaError_t s = cudaStreamSynchronize(ctx->stream);   // nothing stays enqueued, also after a failure
        if (rc == OFDM_OK && s != cudaSuccess) rc = ctx_fail(ctx, OFDM_ERR_CUDA, "cudaStreamSynchronize: %s", cudaGetErrorString(s));
        m.rc = rc;
    });
    const int rc = group_status(g);
    if (rc != OFDM_OK) return rc;

    for (int k = 0; k < n_out; ++k) {
        const GroupOut& o = outs[k];
        if (!o.fields) {
            int64_t* out = (int64_t*)o.host;
            std::fill(out, out + o.cells, (int64_t)0);
            for (const Member& m : g->m)
                if (m.count > 0) for (int64_t c = 0; c < o.cells; ++c) out[c] += m.host[k][c];
            continue;
        }
        for (const Member& m : g->m) {
            for (int64_t w = m.first; w < m.first + m.count;) {      // one point's run of this member's work items at a time
                const int64_t p = w / per_point, j0 = w - p * per_point;
                const int64_t j1 = std::min(per_point, m.first + m.count - p * per_point);
                for (int64_t f = 0; f < o.fields; ++f) {
                    const int64_t c = (p * o.fields + f) * per_point + j0;
                    memcpy((int64_t*)o.host + c, m.host[k].data() + (c - m.host_first[k]), sizeof(int64_t) * (size_t)(j1 - j0));
                }
                w = p * per_point + j1;
            }
        }
    }
    return OFDM_OK;
}

extern "C" int ofdm_group_create(ofdm_group** out, const int* devices, int n_devices, int precision) {
    if (!out) return OFDM_ERR_INVALID;
    *out = nullptr;
    if (!devices || n_devices <= 0) return OFDM_ERR_INVALID;
    ofdm_group* g = nullptr;
    try {
        g = new ofdm_group();
        g->m.resize((size_t)n_devices);
    } catch (...) {
        delete g;
        return OFDM_ERR_INVALID;
    }
    for (int i = 0; i < n_devices; ++i) g->m[i].device = devices[i];
    // ofdm_ctx_create makes its device current: on the members' own threads, the caller's current device stays as it was
    group_each(g->m, [precision](Member& m, int) { m.rc = ofdm_ctx_create(&m.ctx, m.device, precision); });
    for (const Member& m : g->m) {
        if (m.rc == OFDM_OK) continue;
        const int rc = m.rc;
        group_free_members(g->m);
        delete g;
        return rc;
    }
    *out = g;
    return OFDM_OK;
}

extern "C" void ofdm_group_destroy(ofdm_group* g) {
    if (!g) return;
    group_free_members(g->m);
    delete g;
}

extern "C" const char* ofdm_group_last_error(const ofdm_group* g) { return g ? g->err.c_str() : "null group"; }
extern "C" int ofdm_group_size(const ofdm_group* g) { return g ? (int)g->m.size() : OFDM_ERR_INVALID; }

extern "C" int ofdm_group_sweep_ber(ofdm_group* g, const ofdm_link_params* lp, const ofdm_sweep_params* sp, int64_t* counts_host) {
    if (!g) return OFDM_ERR_INVALID;
    if (!lp || !sp || !counts_host) return group_fail(g, OFDM_ERR_INVALID, "ofdm_group_sweep_ber: bad argument");
    const int64_t n = dim(sp->n_snr), spp = dim(sp->streams_per_point);
    return group_run(g, n * spp, std::max<int64_t>(spp, 1), {{counts_host, n * 4, 0}}, [&](ofdm_ctx* ctx, int rank, int world, void* const* dev) {
        ofdm_sweep_params p = *sp;
        p.rank = rank;
        p.world = world;
        return ofdm_sweep_ber(ctx, lp, &p, (int64_t*)dev[0]);
    });
}

extern "C" int ofdm_group_sweep_mse(ofdm_group* g, const ofdm_link_params* lp, const ofdm_sweep_params* sp, int Ldict, double* mse_host,
                                    int64_t* counts_host) {
    if (!g) return OFDM_ERR_INVALID;
    if (!lp || !sp || !mse_host || !counts_host) return group_fail(g, OFDM_ERR_INVALID, "ofdm_group_sweep_mse: bad argument");
    const int64_t n = dim(sp->n_snr), spp = dim(sp->streams_per_point);
    return group_run(g, n * spp, std::max<int64_t>(spp, 1), {{mse_host, n * 4 * spp, 4}, {counts_host, n * 2, 0}},
                     [&](ofdm_ctx* ctx, int rank, int world, void* const* dev) {
                         ofdm_sweep_params p = *sp;
                         p.rank = rank;
                         p.world = world;
                         return ofdm_sweep_mse(ctx, lp, &p, Ldict, (double*)dev[0], (int64_t*)dev[1]);
                     });
}

extern "C" int ofdm_group_sweep_sync(ofdm_group* g, const ofdm_link_params* lp, const ofdm_sync_params* sp, double* rec_host, int64_t* counts_host) {
    if (!g) return OFDM_ERR_INVALID;
    if (!lp || !sp || !rec_host || !counts_host) return group_fail(g, OFDM_ERR_INVALID, "ofdm_group_sweep_sync: bad argument");
    const int64_t n = dim(sp->n_snr), spp = dim(sp->streams_per_point);
    return group_run(g, n * spp, std::max<int64_t>(spp, 1), {{rec_host, n * 9 * spp, 9}, {counts_host, n * 4, 0}},
                     [&](ofdm_ctx* ctx, int rank, int world, void* const* dev) {
                         ofdm_sync_params p = *sp;
                         p.rank = rank;
                         p.world = world;
                         return ofdm_sweep_sync(ctx, lp, &p, (double*)dev[0], (int64_t*)dev[1]);
                     });
}

extern "C" int ofdm_group_sweep_papr(ofdm_group* g, const ofdm_link_params* lp, const ofdm_papr_params* pp, double* papr_host, int64_t* hist_host) {
    if (!g) return OFDM_ERR_INVALID;
    if (!lp || !pp || !papr_host || !hist_host) return group_fail(g, OFDM_ERR_INVALID, "ofdm_group_sweep_papr: bad argument");
    const int64_t n = dim(pp->n_points), spp = dim(pp->streams_per_point);
    return group_run(g, n * spp, std::max<int64_t>(spp, 1), {{papr_host, n * spp, 1}, {hist_host, n * dim(pp->n_bins), 0}},
                     [&](ofdm_ctx* ctx, int rank, int world, void* const* dev) {
                         ofdm_papr_params p = *pp;
                         p.rank = rank;
                         p.world = world;
                         return ofdm_sweep_papr(ctx, lp, &p, (double*)dev[0], (int64_t*)dev[1]);
                     });
}

extern "C" int ofdm_group_sweep_mer(ofdm_group* g, const ofdm_link_params* lp, const ofdm_mer_params* mp, double* mer_host, int64_t* counts_host) {
    if (!g) return OFDM_ERR_INVALID;
    if (!lp || !mp || !mer_host || !counts_host) return group_fail(g, OFDM_ERR_INVALID, "ofdm_group_sweep_mer: bad argument");
    const int64_t n = dim(mp->n_points), spp = dim(mp->streams_per_point);
    return group_run(g, n * spp, std::max<int64_t>(spp, 1), {{mer_host, n * 2 * spp, 2}, {counts_host, n * 3, 0}},
                     [&](ofdm_ctx* ctx, int rank, int world, void* const* dev) {
                         ofdm_mer_params p = *mp;
                         p.rank = rank;
                         p.world = world;
                         return ofdm_sweep_mer(ctx, lp, &p, (double*)dev[0], (int64_t*)dev[1]);
                     });
}

extern "C" int ofdm_group_sweep_part2(ofdm_group* g, const ofdm_link_params* base, const ofdm_part2_params* pp, double* nmse_host,
                                      int64_t* counts_host, int64_t* runs_host) {
    if (!g) return OFDM_ERR_INVALID;
    if (!base || !pp || !nmse_host || !counts_host || !runs_host) return group_fail(g, OFDM_ERR_INVALID, "ofdm_group_sweep_part2: bad argument");
    const int64_t n = dim(pp->n_points), runs = dim(pp->mc_runs);
    return group_run(g, n * runs, std::max<int64_t>(runs, 1), {{nmse_host, n * 4 * runs, 4}, {counts_host, n * 12, 0}, {runs_host, n * 2, 0}},
                     [&](ofdm_ctx* ctx, int rank, int world, void* const* dev) {
                         ofdm_part2_params p = *pp;
                         p.rank = rank;
                         p.world = world;
                         return ofdm_sweep_part2(ctx, base, &p, (double*)dev[0], (int64_t*)dev[1], (int64_t*)dev[2]);
                     });
}
