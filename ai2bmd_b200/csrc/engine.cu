// Host side of the ViSNet sm_100a engine: workspace, launch sequence, CUDA-graph replay, C ABI.
// See include/visnet_b200.h for the boundary each entry point replaces in the reference.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/visnet_b200.h"
#include "k_edge.cuh"
#include "k_caph.cuh"
#include "k_comm.cuh"
#include "k_edge_tc.cuh"
#include "k_fused.cuh"
#include "k_graph_embed.cuh"
#include <nvtx3/nvToolsExt.h>
#include "k_head.cuh"
#include "k_md.cuh"
#include "k_nonbonded.cuh"
#include "k_pme.cuh"
#include "k_restraint.cuh"
#include "k_node.cuh"
#include "k_node2.cuh"
#include "k_node_tc.cuh"

using namespace vb;

namespace {
// NVTX range around every public entry that enqueues or captures work (header-only NVTX v3: a no-op unless a tool injects
// itself), so an Nsight Systems timeline shows evaluations, graph captures and MD blocks by name.
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
    NvtxRange(const NvtxRange&) = delete;
    NvtxRange& operator=(const NvtxRange&) = delete;
};

std::string g_create_error;

#define CUDA_TRY(h, expr)                                                                            \
    do {                                                                                             \
        cudaError_t _e = (expr);                                                                     \
        if (_e != cudaSuccess) {                                                                     \
            (h)->set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return VB_ERR_CUDA;                                                                      \
        }                                                                                            \
    } while (0)

// ---------------------------------------------------------------------------------------------------------
// Last launch of an evaluation: per-fragment energies and, when a protein map is set, the signed whole-protein
// reduction (combiner.py:11-41) as a gather over a CSR of the map sorted by destination atom -- no memset, no
// atomics, fixed summation order.  Block roles by index:
//   [0, fb)        warp per fragment:      energy[g] = float(sum_a eatom[a] + mean)         (visnet.py:146-149)
//   [fb, fb + pb)  thread per protein atom: ef[3p..] = sum_m sign[m] * forces[src[m]]       (combiner.py:38-39)
//   fb + pb        one block:               ef[3P]   = sum_g frag_sign[g] * energy[g]       (combiner.py:11-21)
// ---------------------------------------------------------------------------------------------------------
constexpr int FIN_THREADS = 256;
__device__ __forceinline__ float fragment_energy(const Workspace& ws, int g, float mean, int lane) {
    double s = 0.0;
    for (int a = ws.frag_start[g] + lane; a < ws.frag_start[g + 1]; a += 32) s += (double)ws.eatom[a];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    return (float)(s + (double)mean);
}
__global__ void __launch_bounds__(FIN_THREADS) finalize_kernel(Workspace ws, const float* __restrict__ scalars, int fb, int pb,
                                                               int n_protein, const int* __restrict__ map_rowptr,
                                                               const int* __restrict__ map_src, const float* __restrict__ map_sign,
                                                               const float* __restrict__ frag_sign,
                                                               const float* __restrict__ forces, float* __restrict__ energy,
                                                               float* __restrict__ ef) {
    pdl_entry();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float mean = __ldg(scalars + 1);
    const int b = blockIdx.x;
    if (b < fb) {
        const int g = b * (FIN_THREADS / 32) + warp;
        if (g < ws.G) {
            const float e = fragment_energy(ws, g, mean, lane);
            if (lane == 0) energy[g] = e;
        }
    } else if (b < fb + pb) {
        const int p = (b - fb) * FIN_THREADS + threadIdx.x;
        if (p < n_protein) {
            float fx = 0.f, fy = 0.f, fz = 0.f;
            for (int m = map_rowptr[p]; m < map_rowptr[p + 1]; m++) {
                const float s = map_sign[m];
                const int a = map_src[m];
                fx = fmaf(s, forces[3 * a], fx); fy = fmaf(s, forces[3 * a + 1], fy); fz = fmaf(s, forces[3 * a + 2], fz);
            }
            ef[3 * p] = fx; ef[3 * p + 1] = fy; ef[3 * p + 2] = fz;
        }
    } else {
        __shared__ double red[FIN_THREADS / 32];
        double acc = 0.0;
        for (int g = warp; g < ws.G; g += FIN_THREADS / 32) {
            const float e = fragment_energy(ws, g, mean, lane);
            acc += (double)frag_sign[g] * (double)e;
        }
        if (lane == 0) red[warp] = acc;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
            for (int w = 0; w < FIN_THREADS / 32; w++) t += red[w];
            ef[3 * (size_t)n_protein] = (float)t;
        }
    }
}

}  // namespace

// Buffers one evaluation reads and writes.  They are kernel arguments, so a captured graph is specific to them.
struct StepIO {
    const float* pos = nullptr;   // [N][3]
    float* energy = nullptr;      // [G]
    float* forces = nullptr;      // [N][3]
    float* ef = nullptr;          // [3*n_protein + 1] or nullptr (no whole-protein reduction)
    bool operator==(const StepIO& o) const { return pos == o.pos && energy == o.energy && forces == o.forces && ef == o.ef; }
};

struct vb_handle {
    int device = 0;
    int sm_count = 148;
    std::string err;
    std::mutex mu;
    // weights
    float* d_weights = nullptr;
    ModelW mw{};
    // topology / workspace
    bool has_topology = false;
    Workspace ws{};
    char* arena = nullptr;
    size_t arena_bytes = 0;
    float* d_pos = nullptr;      // [N][3]
    float* d_energy = nullptr;   // [G]
    unsigned long long* d_tl = nullptr;   // optional in-kernel timelines [4L+2][TC_TL_SLOTS]: edge fwd l, edge bwd L+l, node fwd 2L+k, node bwd 3L+1+k
    int timeline = 0;
    float* d_forces = nullptr;   // [N][3]
    float *h_pos = nullptr, *h_energy = nullptr, *h_forces = nullptr;   // pinned staging
    cudaStream_t own_stream = nullptr;
    // protein map, as a CSR over protein (destination) atoms: entries of atom p are map_rowptr[p]..map_rowptr[p+1]
    int n_protein = 0, n_map = 0;
    int *d_map_rowptr = nullptr, *d_map_src = nullptr;
    float *d_map_sign = nullptr, *d_frag_sign = nullptr;
    float* d_ef = nullptr;       // [3*n_protein + 1] internal whole-protein buffer (diagnostic runs)
    int* d_flags = nullptr;      // [0]: set by the neighbour stage when a step produced more edges than the workspace holds
    // cap-hydrogen refinement (k_caph.cuh): flat term arrays + scratch in one device allocation
    bool caph_ready = false;
    CaphDev caph{};
    void* caph_mem = nullptr;
    // NVLink peer-memory all-reduce (k_comm.cuh): window in this rank's HBM + IPC mappings of every peer's window
    bool comm_ready = false;
    int comm_auto = 1;           // append the all-reduce to every evaluation that produces the whole-protein buffer
    void* comm_base = nullptr;
    void* comm_peer[COMM_MAX_WORLD] = {};
    CommParams comm{};
    // options
    int use_graph = 1, npw = 0, te_fwd = 0, te_bwd = 32;
    int use_pdl = 0;   // programmatic dependent launch between the stages: measured neutral to slower (DESIGN.md section 5)
    int npw_opt = 0, te_fwd_opt = 0, edge_tc_opt = -1;   // user choices (0 / -1 = choose by problem size)
    int tc_rows_opt = 0, tc_rows = 128;                  // kernel variant: capacity of a tcgen05 tile (32 / 64 / 96 / 128; MMA M stays 128)
    int tile_rows = 128;                                 // edges per tile actually used (<= tc_rows): whole waves of CTAs
    long long edges_plan = 0;                            // edge count the tile length was planned for (estimate or calibrated)
    int krot = 1;      // rotate the K loops of the SIMT node GEMM units per CTA (L2 slice hot-spotting: all CTAs walk the same weights)
    int node_nb = 0;   // nodes per CTA of the CTA-cooperative SIMT node kernels (0 = automatic)
    int node_impl = 1; // 0: warp-per-node kernels (k_node.cuh), 1: CTA-cooperative kernels (k_node2.cuh)
    int fused = 0, fused_opt = -1;   // 1: one launch per layer and direction (k_fused.cuh); -1 = choose by problem size
    int node_tc = 0, node_tc_opt = -1;   // 1: node stage on tensor cores (k_node_tc.cuh); -1 = choose by problem size
    int embed_batch_opt = -1;            // embedding kernels: several nodes per CTA (1), one (0), by size (-1)
    int edge_tc = -1;  // bit 0: forward edge stage on tcgen05, bit 1: adjoint edge stage on tcgen05; -1 = by size
    // graph cache: one instantiated graph per (kind, I/O pointer set); pointers are baked into the captured launches
    struct GraphEntry { int kind; StepIO io; cudaGraphExec_t exec; };
    std::vector<GraphEntry> graphs;
    int launches = 0;
    bool accum_dirty = false;    // a truncated vb_debug_run left accumulators (XA, VA, GQKV, ...) un-consumed
    std::vector<std::string> stage_names;
    // device-resident MD state (k_md.cuh)
    bool md_ready = false;
    MdParams md{};
    double *d_mx = nullptr, *d_mv = nullptr, *d_mmass = nullptr, *d_ehist = nullptr;
    int *d_real = nullptr, *d_acc = nullptr, *d_rem = nullptr;
    float* d_blen = nullptr;
    long long* d_step = nullptr;
    long long ehist_cap = 1 << 16;
    float* md_ef = nullptr;              // caller-owned [3*n_protein + 1]
    // non-bonded MM term (k_nonbonded.cuh)
    bool nb_ready = false;
    NbParams nb{};
    float *d_nb_q = nullptr, *d_nb_sigma = nullptr, *d_nb_eps = nullptr;
    int *d_nb_rowptr = nullptr, *d_nb_col = nullptr;
    double* d_nb_eatom = nullptr;
    // PME non-bonded term (k_pme.cuh); at most one of nb_ready / pme_ready is set
    bool pme_ready = false;
    PmeParams pme{};
    void* pme_mem = nullptr;
    // Hookean restraints (k_restraint.cuh)
    bool rs_ready = false;
    RsParams rs{};
    void* rs_mem = nullptr;

    bool has_topology_sizes() const { return ws.N > 0; }
    void set_error(const char* fmt, ...) {
        char buf[1024];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof(buf), fmt, ap);
        va_end(ap);
        err = buf;
    }
    void drop_graph() {
        for (auto& g : graphs) cudaGraphExecDestroy(g.exec);
        graphs.clear();
    }
    void free_map() {
        cudaFree(d_map_rowptr); cudaFree(d_map_src); cudaFree(d_map_sign); cudaFree(d_frag_sign); cudaFree(d_ef);
        d_map_rowptr = d_map_src = nullptr; d_map_sign = d_frag_sign = d_ef = nullptr;
        n_protein = n_map = 0;
    }
    void free_caph() {
        cudaFree(caph_mem);
        caph_mem = nullptr; caph = CaphDev{}; caph_ready = false;
    }
    void free_comm() {
        for (int r = 0; r < COMM_MAX_WORLD; r++)
            if (comm_peer[r] && r != comm.rank) cudaIpcCloseMemHandle(comm_peer[r]);
        cudaFree(comm_base); cudaFree(comm.counters);
        comm_base = nullptr; comm = CommParams{}; comm_ready = false;
        for (auto& p : comm_peer) p = nullptr;
    }
    void free_nb() {
        cudaFree(d_nb_q); cudaFree(d_nb_sigma); cudaFree(d_nb_eps); cudaFree(d_nb_rowptr); cudaFree(d_nb_col); cudaFree(d_nb_eatom);
        d_nb_q = d_nb_sigma = d_nb_eps = nullptr; d_nb_rowptr = d_nb_col = nullptr; d_nb_eatom = nullptr;
        nb_ready = false;
    }
    void free_pme() {
        cudaFree(pme_mem);
        pme_mem = nullptr; pme = PmeParams{}; pme_ready = false;
    }
    void free_rs() {
        cudaFree(rs_mem);
        rs_mem = nullptr; rs = RsParams{}; rs_ready = false;
    }
    void free_md() {
        cudaFree(d_mx); cudaFree(d_mv); cudaFree(d_mmass); cudaFree(d_ehist);
        cudaFree(d_real); cudaFree(d_acc); cudaFree(d_rem); cudaFree(d_blen); cudaFree(d_step);
        d_mx = d_mv = d_mmass = d_ehist = nullptr; d_real = d_acc = d_rem = nullptr; d_blen = nullptr; d_step = nullptr;
        md_ready = false;
    }
};

namespace {

// ---- weight table ---------------------------------------------------------------------------------
size_t layer_floats() {
    size_t n = 0;
#define X(name, count) n += (size_t)(count);
    VB_LAYER_WEIGHTS(X)
#undef X
    return n;
}
size_t global_floats() {
    size_t n = 0;
#define X(name, count) n += (size_t)(count);
    VB_GLOBAL_WEIGHTS(X)
#undef X
    return n;
}
size_t total_floats() { return global_floats() + (size_t)L * layer_floats(); }

void bind_weights(ModelW& mw, const float* base) {
    const float* p = base;
#define X(name, count) mw.name = p; p += (size_t)(count);
    VB_GLOBAL_WEIGHTS(X)
#undef X
    for (int l = 0; l < L; l++) {
#define X(name, count) mw.layer[l].name = p; p += (size_t)(count);
        VB_LAYER_WEIGHTS(X)
#undef X
    }
}

std::string build_manifest() {
    std::string s;
    char buf[128];
#define X(name, count) snprintf(buf, sizeof(buf), "%s:%zu;", #name, (size_t)(count)); s += buf;
    VB_GLOBAL_WEIGHTS(X)
#undef X
    for (int l = 0; l < L; l++) {
#define X(name, count) snprintf(buf, sizeof(buf), "layer%d.%s:%zu;", l, #name, (size_t)(count)); s += buf;
        VB_LAYER_WEIGHTS(X)
#undef X
    }
    return s;
}

// ---- arena ------------------------------------------------------------------------------------------
struct ArenaPlan {
    size_t off = 0;
    size_t take(size_t bytes) {
        const size_t o = off;
        off += (bytes + 255) & ~(size_t)255;
        return o;
    }
};

template <typename T>
void carve(ArenaPlan& plan, char* base, T*& ptr, size_t count) {
    const size_t o = plan.take(count * sizeof(T));
    ptr = base ? reinterpret_cast<T*>(base + o) : nullptr;
}

void layout_workspace(vb_handle* h, char* base, ArenaPlan& plan, int*& z, int*& frag_of, int*& frag_start) {
    Workspace& ws = h->ws;
    const size_t N = ws.N, G = ws.G, E = ws.Ecap;
    carve(plan, base, z, N);
    carve(plan, base, frag_of, N);
    carve(plan, base, frag_start, G + 1);
    carve(plan, base, ws.deg, N);
    carve(plan, base, ws.slots, N * KNB);
    carve(plan, base, ws.rowptr, N + 1);
    carve(plan, base, ws.esrc, E);
    carve(plan, base, ws.edst, E);
    carve(plan, base, ws.geom, E * 8);
    carve(plan, base, ws.rbf, E * NR);
    carve(plan, base, ws.eacc, E * 4);
    carve(plan, base, ws.grbf, E * NR);
    for (int l = 0; l <= L; l++) { carve(plan, base, ws.X[l], N * D); carve(plan, base, ws.V[l], N * 3 * D); }
    for (int l = 0; l < L; l++) {
        carve(plan, base, ws.F[l], E * D);
        carve(plan, base, ws.VN[l], N * 3 * D);
        carve(plan, base, ws.QKV[l], N * 3 * D);
        carve(plan, base, ws.V123[l], N * 9 * D);
        carve(plan, base, ws.VDOT[l], N * D);
        carve(plan, base, ws.TU[l], N * 6 * D);
        carve(plan, base, ws.O[l], N * 3 * D);
        carve(plan, base, ws.P1[l], E * 3 * D);
        carve(plan, base, ws.SP[l], E * 2 * D);
        carve(plan, base, ws.ATT[l], E * H);
    }
    carve(plan, base, ws.XA, N * D);
    carve(plan, base, ws.VA, N * 3 * D);
    carve(plan, base, ws.GX, N * D);
    carve(plan, base, ws.GVEC, N * 3 * D);
    carve(plan, base, ws.GF, E * D);
    carve(plan, base, ws.GXA, 3 * N * D);
    carve(plan, base, ws.XN, N * D);
    carve(plan, base, ws.PX, 3 * N * D);
    carve(plan, base, ws.PV, 5 * 3 * N * D);
    carve(plan, base, ws.GO, N * 3 * D);
    carve(plan, base, ws.GQKV, N * 3 * D);
    carve(plan, base, ws.GVNMSG, N * 3 * D);
    carve(plan, base, ws.GTU, N * 6 * D);
    carve(plan, base, ws.GQKV2, N * 3 * D);
    carve(plan, base, ws.GVNMSG2, N * 3 * D);
    carve(plan, base, ws.GTU2, N * 6 * D);
    carve(plan, base, ws.eatom, N);
    carve(plan, base, h->d_pos, N * 3);
    carve(plan, base, h->d_forces, N * 3 + G);          // forces, then the fragment energies: one D2H copy brings both back
    h->d_energy = h->d_forces ? h->d_forces + N * 3 : nullptr;
}

// ---- launch sequence --------------------------------------------------------------------------------
struct Launcher {
    vb_handle* h;
    cudaStream_t st;
    int limit;          // stop after this many stages (debug); <0 = all
    int count = 0;
    bool record_names;
    cudaError_t status = cudaSuccess;
    std::vector<cudaEvent_t>* events = nullptr;   // optional: one event recorded before every stage

    bool next(const char* name) {
        if (record_names) h->stage_names.push_back(name);
        if (limit >= 0 && count >= limit) return false;
        if (events && count < (int)events->size()) cudaEventRecord((*events)[count], st);
        count++;
        return true;
    }
    void check() {
        if (status == cudaSuccess) status = cudaGetLastError();
    }
    // Optionally ("use_pdl") launch with the programmatic-dependent-launch attribute: the next grid may start launching
    // as soon as the last CTA of this one exits and waits at griddepcontrol.wait (pdl_entry() at the top of every
    // kernel) for its completion.  Off by default: measured neutral (exit-time trigger) to slower (entry-time trigger).
    template <typename... KArgs, typename... Args>
    void launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, Args&&... args) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = h->use_pdl ? 1 : 0;
        cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, KArgs(std::forward<Args>(args))...);
        if (status == cudaSuccess && e != cudaSuccess) status = e;
    }
};

template <int NPW>
void launch_node_fwd(Launcher& Lc, int k) {
    vb_handle* h = Lc.h;
    NodeArgs a{k, h->mw, h->ws};
    const int blocks = (h->ws.N + NODE_WARPS * NPW - 1) / (NODE_WARPS * NPW);
    Lc.launch(node_fwd_kernel<NPW>, dim3(blocks), dim3(NODE_WARPS * 32), 0, a);
    Lc.check();
}
template <int NPW>
void launch_node_bwd(Launcher& Lc, int k) {
    vb_handle* h = Lc.h;
    NodeArgs a{k, h->mw, h->ws};
    const int blocks = (h->ws.N + NODE_WARPS * NPW - 1) / (NODE_WARPS * NPW);
    Lc.launch(node_bwd_kernel<NPW>, dim3(blocks), dim3(NODE_WARPS * 32), node_bwd_smem_bytes<NPW>(), a);
    Lc.check();
}
template <int NPW>
void launch_head(Launcher& Lc) {
    vb_handle* h = Lc.h;
    const int blocks = (h->ws.N + NODE_WARPS * NPW - 1) / (NODE_WARPS * NPW);
    Lc.launch(head_kernel<NPW>, dim3(blocks), dim3(NODE_WARPS * 32), HeadSmem<NPW>::BYTES, h->mw, h->ws);
    Lc.check();
}
template <int TE, int NW>
void launch_edge_fwd(Launcher& Lc, int l, int occ) {
    vb_handle* h = Lc.h;
    EdgeArgs a{l, h->mw, h->ws};
    const int tiles = (h->ws.Ecap + TE - 1) / TE;
    const int blocks = std::max(1, std::min(tiles, h->sm_count * occ));
    Lc.launch(edge_fwd_kernel<TE, NW>, dim3(blocks), dim3(NW * 32), edge_fwd_smem_bytes<TE>(), a);
    Lc.check();
}
template <int TE, int NW>
void launch_edge_bwd(Launcher& Lc, int l, int occ) {
    vb_handle* h = Lc.h;
    EdgeArgs a{l, h->mw, h->ws};
    const int tiles = (h->ws.Ecap + TE - 1) / TE;
    const int blocks = std::max(1, std::min(tiles, h->sm_count * occ));
    Lc.launch(edge_bwd_kernel<TE, NW>, dim3(blocks), dim3(NW * 32), edge_bwd_smem_bytes<TE>(), a);
    Lc.check();
}

template <int NB>
void launch_node_fwd2(Launcher& Lc, int k) {
    vb_handle* h = Lc.h;
    NodeArgs a{k, h->mw, h->ws, h->timeline ? h->d_tl + (size_t)2 * L * TC_TL_SLOTS + (size_t)k * N2_TL_SLOTS : nullptr, h->krot};
    Lc.launch(node_fwd2_kernel<NB>, dim3((h->ws.N + NB - 1) / NB), dim3(N2Cfg<NB>::THREADS), sizeof(NodeFwd2SmemK<NB>), a);
    Lc.check();
}
template <int NB>
void launch_node_bwd2(Launcher& Lc, int k) {
    vb_handle* h = Lc.h;
    NodeArgs a{k, h->mw, h->ws, h->timeline ? h->d_tl + (size_t)2 * L * TC_TL_SLOTS + (size_t)(L + 1 + k) * N2_TL_SLOTS : nullptr, h->krot};
    Lc.launch(node_bwd2_kernel<NB>, dim3((h->ws.N + NB - 1) / NB), dim3(N2Cfg<NB>::THREADS), sizeof(NodeBwd2SmemK<NB>), a);
    Lc.check();
}
// nodes per CTA of the CTA-cooperative SIMT node kernels: the fewest (1..4) that still fit one wave, else 8
int node_nb(const vb_handle* h) {
    if (h->node_nb > 0) return h->node_nb;
    for (int nb = 1; nb <= 4; nb++)
        if ((h->ws.N + nb - 1) / nb <= h->sm_count) return nb;
    return 8;
}
void node_fwd(Launcher& Lc, int k) {
    if (Lc.h->node_impl == 1) {
        if (Lc.h->npw == 2) launch_node_fwd2<16>(Lc, k);
        else switch (node_nb(Lc.h)) {           // one wave of 16-warp CTAs with as few nodes each as that allows
            case 1: launch_node_fwd2<1>(Lc, k); break;
            case 2: launch_node_fwd2<2>(Lc, k); break;
            case 3: launch_node_fwd2<3>(Lc, k); break;
            case 4: launch_node_fwd2<4>(Lc, k); break;
            default: launch_node_fwd2<8>(Lc, k);
        }
        return;
    }
    Lc.h->npw == 2 ? launch_node_fwd<2>(Lc, k) : launch_node_fwd<1>(Lc, k);
}
void node_bwd(Launcher& Lc, int k) {
    if (Lc.h->node_impl == 1) {
        switch (node_nb(Lc.h)) {
            case 1: launch_node_bwd2<1>(Lc, k); break;
            case 2: launch_node_bwd2<2>(Lc, k); break;
            case 3: launch_node_bwd2<3>(Lc, k); break;
            case 4: launch_node_bwd2<4>(Lc, k); break;
            default: launch_node_bwd2<8>(Lc, k);
        }
        return;
    }
    Lc.h->npw == 2 ? launch_node_bwd<2>(Lc, k) : launch_node_bwd<1>(Lc, k);
}
void head(Launcher& Lc) {
    vb_handle* h = Lc.h;
    if (h->ws.N <= 4096) {            // small systems: K-split head, one node per CTA
        Lc.launch(head2_kernel, dim3(h->ws.N), dim3(128), 0, h->mw, h->ws);
        Lc.check();
        return;
    }
    h->npw == 2 ? launch_head<2>(Lc) : launch_head<1>(Lc);
}
void launch_edge_fwd_tc(Launcher& Lc, int l) {
    vb_handle* h = Lc.h;
    EdgeTcArgs a{};
    a.layer = l; a.mw = h->mw; a.ws = h->ws;
    const LayerW& lw = h->mw.layer[l];
    const size_t chunk = 4 * 8192;
    int n = 0;
    a.jobs[n++] = TcJob{lw.tcW1, (int)TC_COL_D0, 0};                       // dk
    a.jobs[n++] = TcJob{lw.tcW1 + chunk, (int)TC_COL_D1, 0};               // dv
    if (l < L - 1) a.jobs[n++] = TcJob{lw.tcW1 + 2 * chunk, (int)TC_COL_D0, 0};   // f
    a.jobs[n++] = TcJob{lw.tcWs, (int)TC_COL_D1, 0};                       // s1
    a.jobs[n++] = TcJob{lw.tcWs + chunk, (int)TC_COL_D0, 0};               // s2
    a.njobs = n;
    a.tl = h->timeline ? h->d_tl + (size_t)l * TC_TL_SLOTS : nullptr;
    a.tile_rows = h->tile_rows;
    const int rows = h->tc_rows;
    const int tiles = (h->ws.Ecap + h->tile_rows - 1) / h->tile_rows;
    const int blocks = std::max(1, std::min(tiles, h->sm_count));
    if (rows == 32) Lc.launch(edge_fwd_tc_kernel<32>, dim3(blocks), dim3(TC2_THREADS), TC_SMEM_BYTES, a);
    else if (rows == 64) Lc.launch(edge_fwd_tc_kernel<64>, dim3(blocks), dim3(TC2_THREADS), TC_SMEM_BYTES, a);
    else if (rows == 96) Lc.launch(edge_fwd_tc_kernel<96>, dim3(blocks), dim3(TC2_THREADS), TC_SMEM_BYTES, a);
    else Lc.launch(edge_fwd_tc_kernel<128>, dim3(blocks), dim3(TC2_THREADS), TC_SMEM_BYTES, a);
    Lc.check();
}

void edge_fwd(Launcher& Lc, int l) {
    if (Lc.h->edge_tc & 1) { launch_edge_fwd_tc(Lc, l); return; }
    if (Lc.h->te_fwd == 64) launch_edge_fwd<64, 8>(Lc, l, 2);
    else launch_edge_fwd<32, 8>(Lc, l, 4);
}
void launch_edge_bwd_tc(Launcher& Lc, int l) {
    vb_handle* h = Lc.h;
    EdgeTcArgs a{};
    a.layer = l; a.mw = h->mw; a.ws = h->ws;
    const LayerW& lw = h->mw.layer[l];
    const size_t chunk = 4 * 8192;
    const bool upd = l < L - 1;
    int n = 0;
    a.jobs[n++] = TcJob{lw.tcWsN, (int)TC_COL_D1, 0};                        // g_m  = g_s1' Ws[0:128]
    a.jobs[n++] = TcJob{lw.tcWsN + chunk, (int)TC_COL_D1, 1};                //      + g_s2' Ws[128:256]
    a.jobs[n++] = TcJob{lw.tcW1N + chunk, (int)TC_COL_D0, 0};                // g_f  = g_Pdv Wdv
    a.jobs[n++] = TcJob{lw.tcW1N, (int)TC_COL_D0, 1};                        //      + g_Pdk Wdk
    if (upd) a.jobs[n++] = TcJob{lw.tcW1N + 2 * chunk, (int)TC_COL_D0, 1};   //      + g_Pf  Wf
    a.njobs = n;
    a.tl = h->timeline ? h->d_tl + (size_t)(L + l) * TC_TL_SLOTS : nullptr;
    a.tile_rows = h->tile_rows;
    const int rows = h->tc_rows;
    const int tiles = (h->ws.Ecap + h->tile_rows - 1) / h->tile_rows;
    const int blocks = std::max(1, std::min(tiles, h->sm_count));
    if (rows == 32) Lc.launch(edge_bwd_tc_kernel<32>, dim3(blocks), dim3(TC2_THREADS), TC_SMEM_BYTES, a);
    else if (rows == 64) Lc.launch(edge_bwd_tc_kernel<64>, dim3(blocks), dim3(TC2_THREADS), TC_SMEM_BYTES, a);
    else if (rows == 96) Lc.launch(edge_bwd_tc_kernel<96>, dim3(blocks), dim3(TC2_THREADS), TC_SMEM_BYTES, a);
    else Lc.launch(edge_bwd_tc_kernel<128>, dim3(blocks), dim3(TC2_THREADS), TC_SMEM_BYTES, a);
    Lc.check();
}

void edge_bwd(Launcher& Lc, int l) {
    if (Lc.h->edge_tc & 2) { launch_edge_bwd_tc(Lc, l); return; }
    if (Lc.h->te_bwd == 64) launch_edge_bwd<64, 8>(Lc, l, 1);
    else launch_edge_bwd<32, 8>(Lc, l, 2);
}

void fill_fwd_jobs(const LayerW& lw, int l, TcJob* jobs, int& n) {
    const size_t chunk = 4 * 8192;
    n = 0;
    jobs[n++] = TcJob{lw.tcW1, (int)TC_COL_D0, 0};                       // dk
    jobs[n++] = TcJob{lw.tcW1 + chunk, (int)TC_COL_D1, 0};               // dv
    if (l < L - 1) jobs[n++] = TcJob{lw.tcW1 + 2 * chunk, (int)TC_COL_D0, 0};   // f
    jobs[n++] = TcJob{lw.tcWs, (int)TC_COL_D1, 0};                       // s1
    jobs[n++] = TcJob{lw.tcWs + chunk, (int)TC_COL_D0, 0};               // s2
}
void fill_bwd_jobs(const LayerW& lw, int l, TcJob* jobs, int& n) {
    const size_t chunk = 4 * 8192;
    n = 0;
    jobs[n++] = TcJob{lw.tcWsN, (int)TC_COL_D1, 0};                        // g_m  = g_s1' Ws[0:128]
    jobs[n++] = TcJob{lw.tcWsN + chunk, (int)TC_COL_D1, 1};                //      + g_s2' Ws[128:256]
    jobs[n++] = TcJob{lw.tcW1N + chunk, (int)TC_COL_D0, 0};                // g_f  = g_Pdv Wdv
    jobs[n++] = TcJob{lw.tcW1N, (int)TC_COL_D0, 1};                        //      + g_Pdk Wdk
    if (l < L - 1) jobs[n++] = TcJob{lw.tcW1N + 2 * chunk, (int)TC_COL_D0, 1};   //      + g_Pf  Wf
}
int fused_grid(const vb_handle* h) {
    const int nblocks = (h->ws.N + FU_NB - 1) / FU_NB;
    return std::max(1, std::min(nblocks, h->sm_count));
}
// edge stage l + node stage l+1 (forward) / node adjoint l+1 + edge adjoint l (backward), one launch each
void launch_fused_fwd(Launcher& Lc, int l) {
    vb_handle* h = Lc.h;
    FusedArgs a{};
    a.layer = l; a.mw = h->mw; a.ws = h->ws;
    fill_fwd_jobs(h->mw.layer[l], l, a.jobs, a.njobs);
    Lc.launch(fused_fwd_kernel, dim3(fused_grid(h)), dim3(TC2_THREADS), TC_SMEM_BYTES, a);
    Lc.check();
}
void launch_fused_bwd(Launcher& Lc, int l) {
    vb_handle* h = Lc.h;
    const Workspace& ws = h->ws;
    FusedArgs a{};
    a.layer = l; a.mw = h->mw; a.ws = ws;
    fill_bwd_jobs(h->mw.layer[l], l, a.jobs, a.njobs);
    float* set[2][3] = {{ws.GQKV, ws.GVNMSG, ws.GTU}, {ws.GQKV2, ws.GVNMSG2, ws.GTU2}};
    const int pa = l & 1, pc = (l + 1) & 1;
    a.acc_qkv = set[pa][0]; a.acc_vn = set[pa][1]; a.acc_tu = set[pa][2];
    a.con_qkv = set[pc][0]; a.con_vn = set[pc][1]; a.con_tu = set[pc][2];
    Lc.launch(fused_bwd_kernel, dim3(fused_grid(h)), dim3(TC2_THREADS), TC_SMEM_BYTES, a);
    Lc.check();
}

// ---- node stage on tensor cores (k_node_tc.cuh) --------------------------------------------------------------
void node_tc_common(const vb_handle* h, NodeTcArgs& a, int k) {
    a.layer = k; a.mw = h->mw; a.ws = h->ws;
    a.tx = (h->ws.N + TC_TE - 1) / TC_TE;
    a.tv = (3 * h->ws.N + TC_TE - 1) / TC_TE;
    a.njx = 3; a.njv = 5; a.jx = 1; a.jv = 1;
}
void node_tc_jobs(TcJob* jobs, const float* img, int n) {
    for (int c = 0; c < n; c++) jobs[c] = TcJob{img + (size_t)c * 4 * 8192, 0, 0};
}
int node_tc_grid(const NodeTcArgs& a) { return a.tx * (a.njx / a.jx) + a.tv * (a.njv / a.jv); }
// one job per CTA while that still fits ~2 waves (each CTA then streams a single weight image); otherwise a CTA runs all
// chunks of its row tile on one staged A operand
bool node_tc_split(const vb_handle* h, const NodeTcArgs&) { return h->ws.gxa_parts == 3; }   // one decision per topology (set_gxa_parts)

void launch_node_oproj_tc(Launcher& Lc, int k) {           // O[k-1] = xa Wo[k-1]^T + bo
    vb_handle* h = Lc.h;
    NodeTcArgs a{};
    node_tc_common(h, a, k);
    a.tv = 0;
    node_tc_jobs(a.jobs_x, h->mw.layer[k - 1].tcWo, 3);
    if (!node_tc_split(h, a)) a.jx = 3;
    Lc.launch(node_tc_kernel<NT_OPROJ>, dim3(node_tc_grid(a)), dim3(TC2_THREADS), TC_SMEM_BYTES, a);
    Lc.check();
}
void launch_node_norm_fwd(Launcher& Lc, int k) {
    vb_handle* h = Lc.h;
    Lc.launch(node_norm_fwd_kernel, dim3((h->ws.N + NN_WARPS - 1) / NN_WARPS), dim3(NN_WARPS * 32), 0, k, h->mw, h->ws);
    Lc.check();
}
void launch_node_proj_tc(Launcher& Lc, int k) {            // [q|k|v], [v1|v2|v3|t|u] of stage k
    vb_handle* h = Lc.h;
    NodeTcArgs a{};
    node_tc_common(h, a, k);
    node_tc_jobs(a.jobs_x, h->mw.layer[k].tcWqkv, 3);
    node_tc_jobs(a.jobs_v, h->mw.layer[k].tcWvt, 5);
    if (k == 0) a.tv = 0;                                   // vec = 0 at the first layer: V123 / TU / VN stay zero
    if (k == L - 1) a.njv = 3;                              // no edge update in the last layer: t, u unused
    if (!node_tc_split(h, a)) { a.jx = a.njx; a.jv = a.njv; }
    Lc.launch(node_tc_kernel<NT_PROJ>, dim3(node_tc_grid(a)), dim3(TC2_THREADS), TC_SMEM_BYTES, a);
    Lc.check();
}
void launch_node_bwdA_tc(Launcher& Lc, int k) {            // K-chunk partials of the stage-k adjoint contractions
    vb_handle* h = Lc.h;
    NodeTcArgs a{};
    node_tc_common(h, a, k);
    node_tc_jobs(a.jobs_x, h->mw.layer[k].tcWqkvN, 3);
    node_tc_jobs(a.jobs_v, h->mw.layer[k].tcWvtN, 5);
    if (k == L - 1) a.njv = 3;
    a.acc_qkv = h->ws.GQKV; a.acc_tu = h->ws.GTU;
    if (!node_tc_split(h, a)) { a.jx = a.njx; a.jv = a.njv; }   // all K chunks in one CTA, accumulated in TMEM
    Lc.launch(node_tc_kernel<NT_BWDA>, dim3(node_tc_grid(a)), dim3(TC2_THREADS), TC_SMEM_BYTES, a);
    Lc.check();
}
void launch_node_norm_bwd(Launcher& Lc, int k) {
    vb_handle* h = Lc.h;
    NodeTcArgs a{};
    node_tc_common(h, a, k);
    if (k == L - 1) a.njv = 3;
    Lc.launch(node_norm_bwd_kernel, dim3((h->ws.N + NN_WARPS - 1) / NN_WARPS), dim3(NN_WARPS * 32), 0, k, h->mw, h->ws,
              h->ws.GQKV, h->ws.GVNMSG, h->ws.GTU, node_tc_split(h, a) ? 1 : 0);
    Lc.check();
}
void launch_node_bwdB_tc(Launcher& Lc, int k) {            // dE/dxa partials = [g_o1 | g_x vdot | g_x] Wo[k-1]
    vb_handle* h = Lc.h;
    NodeTcArgs a{};
    node_tc_common(h, a, k);
    a.tv = 0;
    node_tc_jobs(a.jobs_x, h->mw.layer[k - 1].tcWoN, 3);
    if (h->ws.gxa_parts == 1) a.jx = 3;                        // accumulate the three K chunks in TMEM: one complete dE/dxa
    Lc.launch(node_tc_kernel<NT_BWDB>, dim3(node_tc_grid(a)), dim3(TC2_THREADS), TC_SMEM_BYTES, a);
    Lc.check();
}
// stage k of the node forward / adjoint as launches named for the stage checks
void node_fwd_tc(Launcher& Lc, int k) {
    char name[64];
    if (k >= 1) { snprintf(name, sizeof(name), "oproj%d", k); if (Lc.next(name)) launch_node_oproj_tc(Lc, k); }
    snprintf(name, sizeof(name), "norm%d", k);
    if (Lc.next(name)) launch_node_norm_fwd(Lc, k);
    if (k < L) { snprintf(name, sizeof(name), "proj%d", k); if (Lc.next(name)) launch_node_proj_tc(Lc, k); }
}
void node_bwd_tc(Launcher& Lc, int k) {
    char name[64];
    if (k <= L - 1) { snprintf(name, sizeof(name), "bwdA%d", k); if (Lc.next(name)) launch_node_bwdA_tc(Lc, k); }
    snprintf(name, sizeof(name), "bnorm%d", k);
    if (Lc.next(name)) launch_node_norm_bwd(Lc, k);
    if (k >= 1) { snprintf(name, sizeof(name), "bwdB%d", k); if (Lc.next(name)) launch_node_bwdB_tc(Lc, k); }
}

void enqueue_finalize(Launcher& Lc, const StepIO& io) {
    vb_handle* h = Lc.h;
    const Workspace& ws = h->ws;
    const bool prot = io.ef != nullptr;
    const int fb = (ws.G + FIN_THREADS / 32 - 1) / (FIN_THREADS / 32);
    const int pb = prot ? (h->n_protein + FIN_THREADS - 1) / FIN_THREADS : 0;
    Lc.launch(finalize_kernel, dim3(fb + pb + (prot ? 1 : 0)), dim3(FIN_THREADS), 0, ws, h->mw.scalars, fb, pb, h->n_protein,
              h->d_map_rowptr, h->d_map_src, h->d_map_sign, h->d_frag_sign, io.forces, io.energy, io.ef);
    Lc.check();
}

// Enqueue one full evaluation (energy + forces [+ whole-protein reduction]) on Lc.st with the given I/O buffers.
void enqueue_all(Launcher& Lc, const StepIO& io) {
    vb_handle* h = Lc.h;
    Workspace& ws = h->ws;
    const int N = ws.N;
    char name[64];
    if (Lc.next("nbr_build")) {
        Lc.launch(nbr_build_kernel, dim3((N + 127) / 128), dim3(128), 0, N, io.pos, ws.frag_of, ws.frag_start, h->mw.cutoff,
                  ws.slots, ws.deg, io.forces);
        Lc.check();
    }
    if (Lc.next("rowptr_scan")) { Lc.launch(rowptr_scan_kernel, dim3(1), dim3(1024), 0, N, ws.deg, ws.rowptr, ws.Ecap, h->d_flags); Lc.check(); }
    if (Lc.next("edge_geom")) { Lc.launch(edge_geom_kernel, dim3((N + 3) / 4), dim3(128), 0, N, io.pos, h->mw, ws); Lc.check(); }
    // batches: several nodes per CTA share the embedding weights ("embed_batch": bit 0 forward kernel, bit 1 adjoint kernel)
    const bool batch = h->embed_batch_opt >= 0 ? (h->embed_batch_opt & 1) : N > 8 * h->sm_count;
    const bool batch_bwd = h->embed_batch_opt >= 0 ? (h->embed_batch_opt & 2) != 0 : N > 8 * h->sm_count;
    if (Lc.next("embed_node")) {
        if (batch) Lc.launch(embed_node_kernel<8>, dim3((N + 7) / 8), dim3(EMB_THREADS), 0, h->mw, ws);
        else Lc.launch(embed_node_small_kernel, dim3((N + EMS_NB - 1) / EMS_NB), dim3(EMS_THREADS), 0, h->mw, ws,
                       h->timeline ? h->d_tl + (size_t)2 * L * TC_TL_SLOTS + (size_t)(2 * L + 2) * N2_TL_SLOTS : (unsigned long long*)nullptr);
        Lc.check();
    }
    const int eblocks = std::max(1, std::min((ws.Ecap + 3) / 4, h->sm_count * 16));     // four edges per block and pass
    if (Lc.next("embed_edge")) { Lc.launch(embed_edge_kernel, dim3(eblocks), dim3(128), 0, h->mw, ws); Lc.check(); }
    if (h->fused) {
        // one launch per layer and direction: "fwdL" = edge stage L + node stage L+1, "bwdL" = node adjoint L+1 + edge adjoint L
        if (Lc.next("node_fwd0")) launch_node_fwd2<4>(Lc, 0);
        for (int l = 0; l < L; l++) {
            snprintf(name, sizeof(name), "fwd%d", l);
            if (Lc.next(name)) launch_fused_fwd(Lc, l);
        }
        if (Lc.next("head")) head(Lc);
        for (int l = L - 1; l >= 0; l--) {
            snprintf(name, sizeof(name), "bwd%d", l);
            if (Lc.next(name)) launch_fused_bwd(Lc, l);
        }
        if (Lc.next("node_bwd0")) launch_node_bwd2<4>(Lc, 0);
    } else if (h->node_tc) {
        // node stage on tensor cores: three launches per stage (GEMM tiles / warp-per-node glue / GEMM tiles)
        for (int l = 0; l < L; l++) {
            node_fwd_tc(Lc, l);
            snprintf(name, sizeof(name), "edge_fwd%d", l);
            if (Lc.next(name)) edge_fwd(Lc, l);
        }
        node_fwd_tc(Lc, L);
        if (Lc.next("head")) head(Lc);
        for (int l = L - 1; l >= 0; l--) {
            node_bwd_tc(Lc, l + 1);
            snprintf(name, sizeof(name), "edge_bwd%d", l);
            if (Lc.next(name)) edge_bwd(Lc, l);
        }
        node_bwd_tc(Lc, 0);
    } else {
        for (int l = 0; l < L; l++) {
            snprintf(name, sizeof(name), "node_fwd%d", l);
            if (Lc.next(name)) node_fwd(Lc, l);
            snprintf(name, sizeof(name), "edge_fwd%d", l);
            if (Lc.next(name)) edge_fwd(Lc, l);
        }
        if (Lc.next("node_fwd6")) node_fwd(Lc, L);
        if (Lc.next("head")) head(Lc);
        for (int l = L - 1; l >= 0; l--) {
            snprintf(name, sizeof(name), "node_bwd%d", l + 1);
            if (Lc.next(name)) node_bwd(Lc, l + 1);
            snprintf(name, sizeof(name), "edge_bwd%d", l);
            if (Lc.next(name)) edge_bwd(Lc, l);
        }
        if (Lc.next("node_bwd0")) node_bwd(Lc, 0);
    }
    if (Lc.next("embed_edge_bwd")) {
        const int bb = std::max(1, std::min((ws.Ecap + EEB_WARPS - 1) / EEB_WARPS, h->sm_count * 4));
        Lc.launch(embed_edge_bwd_kernel, dim3(bb), dim3(EEB_WARPS * 32), 0, h->mw, ws);
        Lc.check();
    }
    if (Lc.next("embed_node_bwd")) {
        Lc.launch(embed_node_bwd_kernel, dim3(batch_bwd ? std::min(N, 5 * h->sm_count) : N), dim3(ENB_WARPS * 32), 0, h->mw, ws, io.forces);
        Lc.check();
    }
    if (Lc.next("finalize")) enqueue_finalize(Lc, io);
}

template <typename K>
cudaError_t opt_in_smem(K kernel, size_t bytes) {
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

int configure_kernels(vb_handle* h) {
    CUDA_TRY(h, opt_in_smem(edge_fwd_kernel<32, 8>, edge_fwd_smem_bytes<32>()));
    CUDA_TRY(h, opt_in_smem(edge_fwd_kernel<64, 8>, edge_fwd_smem_bytes<64>()));
    CUDA_TRY(h, opt_in_smem(edge_bwd_kernel<32, 8>, edge_bwd_smem_bytes<32>()));
    CUDA_TRY(h, opt_in_smem(edge_bwd_kernel<64, 8>, edge_bwd_smem_bytes<64>()));
    CUDA_TRY(h, opt_in_smem(node_bwd_kernel<1>, node_bwd_smem_bytes<1>()));
    CUDA_TRY(h, opt_in_smem(node_bwd_kernel<2>, node_bwd_smem_bytes<2>()));
    CUDA_TRY(h, opt_in_smem(head_kernel<1>, HeadSmem<1>::BYTES));
    CUDA_TRY(h, opt_in_smem(head_kernel<2>, HeadSmem<2>::BYTES));
    CUDA_TRY(h, opt_in_smem(edge_fwd_tc_kernel<32>, TC_SMEM_BYTES));
    CUDA_TRY(h, opt_in_smem(edge_fwd_tc_kernel<64>, TC_SMEM_BYTES));
    CUDA_TRY(h, opt_in_smem(edge_fwd_tc_kernel<96>, TC_SMEM_BYTES));
    CUDA_TRY(h, opt_in_smem(edge_fwd_tc_kernel<128>, TC_SMEM_BYTES));
    CUDA_TRY(h, opt_in_smem(edge_bwd_tc_kernel<32>, TC_SMEM_BYTES));
    CUDA_TRY(h, opt_in_smem(edge_bwd_tc_kernel<64>, TC_SMEM_BYTES));
    CUDA_TRY(h, opt_in_smem(edge_bwd_tc_kernel<96>, TC_SMEM_BYTES));
    CUDA_TRY(h, opt_in_smem(edge_bwd_tc_kernel<128>, TC_SMEM_BYTES));
    CUDA_TRY(h, opt_in_smem(fused_fwd_kernel, TC_SMEM_BYTES));
    CUDA_TRY(h, opt_in_smem(fused_bwd_kernel, TC_SMEM_BYTES));
    CUDA_TRY(h, opt_in_smem(node_tc_kernel<NT_OPROJ>, TC_SMEM_BYTES));
    CUDA_TRY(h, opt_in_smem(node_tc_kernel<NT_PROJ>, TC_SMEM_BYTES));
    CUDA_TRY(h, opt_in_smem(node_tc_kernel<NT_BWDA>, TC_SMEM_BYTES));
    CUDA_TRY(h, opt_in_smem(node_tc_kernel<NT_BWDB>, TC_SMEM_BYTES));

    CUDA_TRY(h, opt_in_smem(node_fwd2_kernel<1>, sizeof(NodeFwd2SmemK<1>)));
    CUDA_TRY(h, opt_in_smem(node_bwd2_kernel<1>, sizeof(NodeBwd2SmemK<1>)));
    CUDA_TRY(h, opt_in_smem(node_fwd2_kernel<2>, sizeof(NodeFwd2SmemK<2>)));
    CUDA_TRY(h, opt_in_smem(node_bwd2_kernel<2>, sizeof(NodeBwd2SmemK<2>)));
    CUDA_TRY(h, opt_in_smem(node_fwd2_kernel<3>, sizeof(NodeFwd2SmemK<3>)));
    CUDA_TRY(h, opt_in_smem(node_bwd2_kernel<3>, sizeof(NodeBwd2SmemK<3>)));
    CUDA_TRY(h, opt_in_smem(node_fwd2_kernel<4>, sizeof(NodeFwd2SmemK<4>)));
    CUDA_TRY(h, opt_in_smem(node_bwd2_kernel<4>, sizeof(NodeBwd2SmemK<4>)));
    CUDA_TRY(h, opt_in_smem(node_fwd2_kernel<8>, sizeof(NodeFwd2SmemK<8>)));
    CUDA_TRY(h, opt_in_smem(node_fwd2_kernel<16>, sizeof(NodeFwd2SmemK<16>)));
    CUDA_TRY(h, opt_in_smem(node_bwd2_kernel<8>, sizeof(NodeBwd2SmemK<8>)));
    return VB_OK;
}

// Accumulators that a producer stage adds into and the consuming stage re-zeroes: clean after a truncated diagnostic run.
int clean_accumulators(vb_handle* h, cudaStream_t st) {
    const Workspace& ws = h->ws;
    const size_t N = ws.N;
    CUDA_TRY(h, cudaMemsetAsync(ws.XA, 0, N * D * 4, st));
    CUDA_TRY(h, cudaMemsetAsync(ws.VA, 0, N * 3 * D * 4, st));
    CUDA_TRY(h, cudaMemsetAsync(ws.GQKV, 0, N * 3 * D * 4, st));
    CUDA_TRY(h, cudaMemsetAsync(ws.GVNMSG, 0, N * 3 * D * 4, st));
    CUDA_TRY(h, cudaMemsetAsync(ws.GTU, 0, N * 6 * D * 4, st));
    CUDA_TRY(h, cudaMemsetAsync(ws.GQKV2, 0, N * 3 * D * 4, st));
    CUDA_TRY(h, cudaMemsetAsync(ws.GVNMSG2, 0, N * 3 * D * 4, st));
    CUDA_TRY(h, cudaMemsetAsync(ws.GTU2, 0, N * 6 * D * 4, st));
    CUDA_TRY(h, cudaMemsetAsync(ws.GX, 0, N * D * 4, st));
    CUDA_TRY(h, cudaMemsetAsync(ws.GXA, 0, 3 * N * D * 4, st));
    h->accum_dirty = false;
    return VB_OK;
}

enum { K_EVAL = 0, K_HOST = 1, K_MD_EVAL = 2, K_MD_STEP = 3 };

// Run `enqueue(stream)` -- a sequence of launches / async copies that depends only on (kind, io) and the handle's
// configuration -- either directly or as a replay of its cached CUDA graph.  A failed capture always ends the capture
// (the stream stays usable) and is retried once without programmatic-dependent-launch edges.
template <typename F>
int run_cached(vb_handle* h, cudaStream_t st, int kind, const StepIO& io, F&& enqueue) {
    if (h->accum_dirty) { if (int rc = clean_accumulators(h, st)) return rc; }
    if (!h->use_graph) return enqueue(st);
    for (auto& g : h->graphs)
        if (g.kind == kind && g.io == io) { CUDA_TRY(h, cudaGraphLaunch(g.exec, st)); return VB_OK; }
    cudaGraphExec_t exec = nullptr;
    for (int attempt = 0; attempt < 2 && !exec; attempt++) {
        cudaGraph_t graph = nullptr;
        CUDA_TRY(h, cudaStreamBeginCapture(h->own_stream, cudaStreamCaptureModeThreadLocal));
        const int rc = enqueue(h->own_stream);
        const cudaError_t e_end = cudaStreamEndCapture(h->own_stream, &graph);
        cudaError_t e_inst = cudaSuccess;
        if (rc == VB_OK && e_end == cudaSuccess) e_inst = cudaGraphInstantiate(&exec, graph, 0);
        if (graph) cudaGraphDestroy(graph);
        if (rc == VB_OK && e_end == cudaSuccess && e_inst == cudaSuccess) break;
        exec = nullptr;
        (void)cudaGetLastError();
        if (h->use_pdl && attempt == 0) { h->use_pdl = 0; continue; }
        if (rc == VB_OK) h->set_error("graph capture failed: %s / %s", cudaGetErrorString(e_end), cudaGetErrorString(e_inst));
        return VB_ERR_CUDA;
    }
    if (h->graphs.size() >= 8) { cudaGraphExecDestroy(h->graphs.front().exec); h->graphs.erase(h->graphs.begin()); }
    h->graphs.push_back({kind, io, exec});
    CUDA_TRY(h, cudaGraphLaunch(exec, st));
    return VB_OK;
}

// all-reduce of buf[n] over the connected ranks (k_comm.cuh), one launch on st
int enqueue_allreduce(vb_handle* h, cudaStream_t st, float* buf, long long n) {
    if (n > h->comm.max_floats) { h->set_error("all-reduce of %lld floats exceeds the window (%lld)", n, h->comm.max_floats); return VB_ERR_ARG; }
    const int ctas = (int)std::max<long long>(1, std::min<long long>((n + COMM_THREADS - 1) / COMM_THREADS, COMM_MAX_CTAS));
    comm_allreduce_kernel<<<ctas, COMM_THREADS, 0, st>>>(h->comm, buf, n);
    CUDA_TRY(h, cudaGetLastError());
    return VB_OK;
}

// every launch of one evaluation; with `reduce` the whole-protein buffer is all-reduced over the connected ranks last
int enqueue_eval(vb_handle* h, cudaStream_t st, const StepIO& io, bool reduce = false) {
    Launcher Lc{h, st, -1, 0, false};
    enqueue_all(Lc, io);
    if (Lc.status != cudaSuccess) { h->set_error("kernel launch failed: %s", cudaGetErrorString(Lc.status)); return VB_ERR_CUDA; }
    if (reduce && io.ef && h->comm_ready && h->comm_auto) return enqueue_allreduce(h, st, io.ef, 3LL * h->n_protein + 1);
    return VB_OK;
}

// one evaluation on the given buffers, asynchronous on st
int run_eval(vb_handle* h, cudaStream_t st, const StepIO& io) {
    return run_cached(h, st, K_EVAL, io, [&](cudaStream_t s) -> int { return enqueue_eval(h, s, io, true); });
}

StepIO internal_io(vb_handle* h, bool protein) {
    StepIO io;
    io.pos = h->d_pos; io.energy = h->d_energy; io.forces = h->d_forces;
    io.ef = protein ? h->d_ef : nullptr;
    return io;
}

// dE/dxa arrives as three K-chunk partials only when the tensor-core node stage runs one chunk per CTA (small systems)
void set_gxa_parts(vb_handle* h) {
    h->ws.gxa_parts = 1;
    if (h->node_tc && h->has_topology_sizes()) {
        const int tx = (h->ws.N + TC_TE - 1) / TC_TE, tv = (3 * h->ws.N + TC_TE - 1) / TC_TE;
        if (tx * 3 + tv * 5 <= 2 * h->sm_count) h->ws.gxa_parts = 3;
    }
}

// stage names / launch count of one evaluation under the current options (nothing is launched)
void record_stages(vb_handle* h) {
    h->stage_names.clear();
    Launcher Lc{h, nullptr, 0, 0, true};
    enqueue_all(Lc, internal_io(h, false));
    h->launches = (int)h->stage_names.size();
}

// Tile length of the tcgen05 edge kernels.  A tile's latency is a fixed part (every CTA streams the layer's weights
// L2 -> shared memory, barriers, TMEM round trips) plus per-row SIMT phases in which each of the 16 compute warps owns
// ceil(rows / 16) rows.  So the edges are cut into the fewest whole waves of tiles <= 128 edges, and the tile length is
// the smallest MULTIPLE OF 16 that still fits those waves: Chignolin (6.7k edges) 141 tiles of 48 instead of 105 of 64,
// WW (19.7k) 247 tiles of 80 in two even waves instead of 154 of 128 (one full wave + 6 tiles).  Lengths between
// multiples of 16 were measured slower (more CTAs, same rows per warp: Trp-cage 88 vs 96 +3 %), and so was 112 instead
// of 128 (ABD +2 %, 512 fragments +2.5 %): from 7 rows per warp on the full tile is kept.  `edges` is an estimate (17 per
// atom, +3 % margin) until vb_set_option("calibrate") replaces it by the count of the last evaluation.
void plan_tiles(vb_handle* h, long long edges) {
    const long long sm = h->sm_count;
    const long long padded = edges + edges * 3 / 100 + 1;
    const long long waves = std::max<long long>(1, (padded + sm * 128 - 1) / (sm * 128));
    long long rpw = (padded + sm * waves * 16 - 1) / (sm * waves * 16);
    if (rpw >= 7) rpw = 8;
    const long long rows = 16 * std::min<long long>(8, std::max<long long>(1, rpw));
    if (h->tc_rows_opt > 0) {                      // user-fixed tile capacity: full tiles of that length (round-1 behaviour)
        h->tc_rows = h->tc_rows_opt;
        h->tile_rows = h->tc_rows_opt;
    } else {
        h->tc_rows = rows <= 32 ? 32 : rows <= 64 ? 64 : rows <= 96 ? 96 : 128;
        h->tile_rows = (int)rows;
    }
    h->edges_plan = edges;
}

void choose_defaults(vb_handle* h) {
    const int N = h->ws.N;
    h->npw = h->npw_opt; h->te_fwd = h->te_fwd_opt; h->edge_tc = h->edge_tc_opt;
    // fused per-layer launches (k_fused.cuh) are opt-in: inside a graph a launch boundary costs ~1-2 us, less than what the
    // fused kernels lose to the 96-register budget of a 576-thread CTA running the node GEMMs (profiles/README.md)
    h->fused = h->fused_opt >= 0 ? h->fused_opt : 0;
    // node stage on tensor cores from ~600 atoms on (measured, graph replay: Chignolin 391 atoms 0.78 -> 0.82 ms slower,
    // Trp-cage 737 atoms 1.08 -> 0.97 ms, WW 2.07 -> 1.81, ABD 2.22 -> 1.98, 512 fragments 13.8 -> 12.3: the three-launch
    // stage has a higher fixed latency than the single SIMT kernel, profiles/README.md)
    h->node_tc = h->node_tc_opt >= 0 ? h->node_tc_opt : (N >= 600 ? 1 : 0);
    if (h->fused) h->node_tc = 0;
    set_gxa_parts(h);
    if (h->npw == 0) h->npw = (N > 4096) ? 2 : 1;
    if (h->te_fwd == 0) h->te_fwd = ((long long)N * 17 / 64 >= 2LL * h->sm_count) ? 64 : 32;
    // tcgen05 edge kernels (one tile per CTA, 16 compute warps): with the tile length chosen below both stages beat
    // the fp32 SIMT kernels at every size measured, down to a single 26-atom fragment (tools/tc_crossover.py,
    // profiles/README.md); the SIMT kernels stay selectable ("edge_tc" 0..2) as the independent implementation
    if (h->edge_tc < 0) h->edge_tc = 3;
    plan_tiles(h, h->edges_plan > 0 ? h->edges_plan : (long long)N * 17);
}

}  // namespace

// =====================================================================================================
// C ABI
// =====================================================================================================
extern "C" {

const char* vb_weight_manifest(void) {
    static const std::string m = build_manifest();
    return m.c_str();
}

const char* vb_last_error(const vb_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int vb_create(const float* weights_host, size_t n_floats, const vb_hparams* hp, int device, vb_handle** out) {
    if (!weights_host || !hp || !out) { g_create_error = "vb_create: null argument"; return VB_ERR_ARG; }
    *out = nullptr;
    if (hp->hidden_channels != D || hp->num_layers != L || hp->num_heads != H || hp->num_rbf != NR ||
        hp->max_num_neighbors != KNB || !(hp->cutoff > 0.f)) {
        g_create_error = "vb_create: hyper-parameters differ from the compiled specialisation (128/6/8/32/32)";
        return VB_ERR_ARG;
    }
    if (n_floats != total_floats()) {
        char buf[160];
        snprintf(buf, sizeof(buf), "vb_create: weight blob has %zu floats, manifest needs %zu", n_floats, total_floats());
        g_create_error = buf;
        return VB_ERR_ARG;
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || device < 0 || device >= ndev) {
        g_create_error = std::string("vb_create: no usable CUDA device (") + cudaGetErrorString(e) +
                         "); this engine has no CPU fallback";
        return VB_ERR_CUDA;
    }
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    if (prop.major < 10) {
        g_create_error = "vb_create: device is not sm_100 class; the kernels are built for sm_100a only";
        return VB_ERR_CUDA;
    }
    vb_handle* h = new vb_handle();
    h->device = device;
    h->sm_count = prop.multiProcessorCount;
    auto fail = [&](int rc) { g_create_error = h->err; vb_destroy(h); return rc; };
    if (cudaSetDevice(device) != cudaSuccess) { h->set_error("cudaSetDevice failed"); return fail(VB_ERR_CUDA); }
    if (cudaMalloc(&h->d_weights, n_floats * sizeof(float)) != cudaSuccess) { h->set_error("weights alloc failed"); return fail(VB_ERR_ALLOC); }
    if (cudaMemcpy(h->d_weights, weights_host, n_floats * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess) {
        h->set_error("weights upload failed");
        return fail(VB_ERR_CUDA);
    }
    bind_weights(h->mw, h->d_weights);
    h->mw.cutoff = hp->cutoff;
    if (cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking) != cudaSuccess) { h->set_error("stream create failed"); return fail(VB_ERR_CUDA); }
    if (configure_kernels(h) != VB_OK) return fail(VB_ERR_CUDA);
    if (const char* s = getenv("VB_USE_GRAPH")) h->use_graph = atoi(s);
    if (const char* s = getenv("VB_NPW")) h->npw_opt = atoi(s);
    if (const char* s = getenv("VB_TE_FWD")) h->te_fwd_opt = atoi(s);
    if (const char* s = getenv("VB_TE_BWD")) h->te_bwd = atoi(s);
    if (const char* s = getenv("VB_EDGE_TC")) h->edge_tc_opt = atoi(s);
    if (const char* s = getenv("VB_USE_PDL")) h->use_pdl = atoi(s) ? 1 : 0;
    if (const char* s = getenv("VB_TC_ROWS")) { const int v = atoi(s); if (v == 32 || v == 64 || v == 96 || v == 128) h->tc_rows_opt = v; }
    if (const char* s = getenv("VB_NODE_IMPL")) h->node_impl = atoi(s);
    if (const char* s = getenv("VB_FUSED")) h->fused_opt = atoi(s) ? 1 : 0;
    if (const char* s = getenv("VB_NODE_TC")) h->node_tc_opt = atoi(s) ? 1 : 0;
    *out = h;
    return VB_OK;
}

void vb_destroy(vb_handle* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    h->drop_graph();
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    cudaFree(h->d_weights);
    cudaFree(h->d_tl);
    h->free_md();
    h->free_nb();
    h->free_pme();
    h->free_rs();
    h->free_comm();
    h->free_caph();
    cudaFree(h->arena);
    h->free_map();
    cudaFree(h->d_flags);
    cudaFreeHost(h->h_pos); cudaFreeHost(h->h_forces);
    delete h;
}

int vb_set_topology(vb_handle* h, int64_t n_atoms, int64_t n_graphs, const int64_t* z_host,
                    const int64_t* batch_host, int64_t max_edges) {
    NvtxRange nvtx_("vb_set_topology");
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (n_atoms <= 0 || n_graphs <= 0 || !z_host || !batch_host || n_atoms > (1 << 26)) {
        h->set_error("vb_set_topology: bad sizes/pointers");
        return VB_ERR_ARG;
    }
    std::vector<int> z(n_atoms), frag_of(n_atoms), frag_start(n_graphs + 1, 0);
    for (int64_t i = 0; i < n_atoms; i++) {
        if (z_host[i] < 0 || z_host[i] >= 100) { h->set_error("vb_set_topology: atomic number out of range [0,100)"); return VB_ERR_ARG; }
        const int64_t g = batch_host[i];
        if (g < 0 || g >= n_graphs || (i > 0 && g < batch_host[i - 1])) {
            h->set_error("vb_set_topology: batch must be sorted with values in [0,G)");
            return VB_ERR_ARG;
        }
        z[i] = (int)z_host[i];
        frag_of[i] = (int)g;
        frag_start[g + 1]++;
    }
    for (int64_t g = 0; g < n_graphs; g++) frag_start[g + 1] += frag_start[g];
    CUDA_TRY(h, cudaSetDevice(h->device));
    h->drop_graph();
    h->free_md();                 // the MD recipe indexes the fragment atoms of the old topology
    h->free_map();                // ... and so does the protein map: it must be set again
    h->free_caph();               // ... and the hydrogen-refinement terms
    h->has_topology = false;
    cudaFree(h->arena); h->arena = nullptr;
    cudaFreeHost(h->h_pos); cudaFreeHost(h->h_forces);
    h->h_pos = h->h_energy = h->h_forces = nullptr;
    h->ws = Workspace{};
    h->edges_plan = 0;
    h->ws.N = (int)n_atoms;
    h->ws.G = (int)n_graphs;
    const int64_t worst = n_atoms * KNB;
    h->ws.Ecap = (int)((max_edges > 0 && max_edges < worst) ? max_edges : worst);
    int *dz = nullptr, *dfo = nullptr, *dfs = nullptr;
    ArenaPlan dry;
    layout_workspace(h, nullptr, dry, dz, dfo, dfs);
    h->arena_bytes = dry.off;
    if (cudaMalloc(&h->arena, h->arena_bytes) != cudaSuccess) {
        cudaGetLastError();
        h->set_error("vb_set_topology: workspace allocation of %zu bytes failed", h->arena_bytes);
        h->arena = nullptr;
        return VB_ERR_ALLOC;
    }
    ArenaPlan real;
    layout_workspace(h, h->arena, real, dz, dfo, dfs);
    h->ws.z = dz; h->ws.frag_of = dfo; h->ws.frag_start = dfs;
    CUDA_TRY(h, cudaMemset(h->arena, 0, h->arena_bytes));
    if (!h->d_flags) CUDA_TRY(h, cudaMalloc(&h->d_flags, sizeof(int) * 4));
    CUDA_TRY(h, cudaMemset(h->d_flags, 0, sizeof(int) * 4));
    CUDA_TRY(h, cudaMemcpy(dz, z.data(), sizeof(int) * n_atoms, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(dfo, frag_of.data(), sizeof(int) * n_atoms, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(dfs, frag_start.data(), sizeof(int) * (n_graphs + 1), cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMallocHost(&h->h_pos, sizeof(float) * 3 * n_atoms));
    CUDA_TRY(h, cudaMallocHost(&h->h_forces, sizeof(float) * (3 * n_atoms + n_graphs)));   // forces, then energies (one copy)
    h->h_energy = h->h_forces + 3 * n_atoms;
    choose_defaults(h);
    record_stages(h);
    h->has_topology = true;
    return VB_OK;
}

int vb_forward(vb_handle* h, const float* pos_dev, float* energy_dev, float* forces_dev, void* stream) {
    NvtxRange nvtx_("vb_forward");
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (!h->has_topology) { h->set_error("vb_forward: call vb_set_topology first"); return VB_ERR_STATE; }
    if (!pos_dev || !energy_dev || !forces_dev) { h->set_error("vb_forward: null buffer"); return VB_ERR_ARG; }
    CUDA_TRY(h, cudaSetDevice(h->device));
    StepIO io;
    io.pos = pos_dev; io.energy = energy_dev; io.forces = forces_dev;
    return run_eval(h, (cudaStream_t)stream, io);     // the kernels read / write the caller's buffers directly
}

namespace {
int check_edge_overflow(vb_handle* h, const char* who) {
    if ((int64_t)h->ws.Ecap >= (int64_t)h->ws.N * KNB) return VB_OK;      // worst-case capacity: cannot overflow
    int flag = 0;
    CUDA_TRY(h, cudaMemcpy(&flag, h->d_flags, sizeof(int), cudaMemcpyDeviceToHost));
    if (flag) {
        h->set_error("%s: a step produced more edges than the max_edges = %d given to vb_set_topology (results invalid)", who, h->ws.Ecap);
        return VB_ERR_STATE;
    }
    return VB_OK;
}
}  // namespace

int vb_forward_host(vb_handle* h, const float* pos_host, float* energy_host, float* forces_host) {
    NvtxRange nvtx_("vb_forward_host");
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (!h->has_topology) { h->set_error("vb_forward_host: call vb_set_topology first"); return VB_ERR_STATE; }
    if (!pos_host || !energy_host || !forces_host) { h->set_error("vb_forward_host: null buffer"); return VB_ERR_ARG; }
    const int N = h->ws.N, G = h->ws.G;
    cudaStream_t st = h->own_stream;
    CUDA_TRY(h, cudaSetDevice(h->device));
    memcpy(h->h_pos, pos_host, sizeof(float) * 3 * N);
    // H2D of the positions, every kernel, D2H of energies and forces: one graph replay (pinned staging buffers are fixed)
    const StepIO io = internal_io(h, false);
    int rc = run_cached(h, st, K_HOST, io, [&](cudaStream_t s) -> int {
        CUDA_TRY(h, cudaMemcpyAsync(h->d_pos, h->h_pos, sizeof(float) * 3 * N, cudaMemcpyHostToDevice, s));
        if (int r = enqueue_eval(h, s, io)) return r;
        CUDA_TRY(h, cudaMemcpyAsync(h->h_forces, h->d_forces, sizeof(float) * (3 * N + G), cudaMemcpyDeviceToHost, s));   // forces + energies
        return (int)VB_OK;
    });
    if (rc != VB_OK) return rc;
    CUDA_TRY(h, cudaStreamSynchronize(st));
    if (int r = check_edge_overflow(h, "vb_forward_host")) return r;
    memcpy(energy_host, h->h_energy, sizeof(float) * G);
    memcpy(forces_host, h->h_forces, sizeof(float) * 3 * N);
    return VB_OK;
}

int vb_set_protein_map(vb_handle* h, int64_t n_protein_atoms, int64_t n_map, const int32_t* src_atom_host,
                       const int32_t* dst_atom_host, const float* sign_host, const float* frag_sign_host) {
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (!h->has_topology) { h->set_error("vb_set_protein_map: call vb_set_topology first"); return VB_ERR_STATE; }
    if (n_protein_atoms <= 0 || n_protein_atoms > (1 << 28) || n_map < 0 || !frag_sign_host ||
        (n_map > 0 && (!src_atom_host || !dst_atom_host || !sign_host))) {
        h->set_error("vb_set_protein_map: bad arguments");
        return VB_ERR_ARG;
    }
    for (int64_t m = 0; m < n_map; m++) {
        if (src_atom_host[m] < 0 || src_atom_host[m] >= h->ws.N || dst_atom_host[m] < 0 || dst_atom_host[m] >= n_protein_atoms) {
            h->set_error("vb_set_protein_map: index out of range at entry %lld", (long long)m);
            return VB_ERR_ARG;
        }
    }
    // CSR over destination atoms (entries of one atom keep their order in the map): the reduction is a gather
    const int P = (int)n_protein_atoms;
    std::vector<int> rowptr(P + 1, 0), src(std::max<int64_t>(n_map, 1));
    std::vector<float> sgn(std::max<int64_t>(n_map, 1));
    for (int64_t m = 0; m < n_map; m++) rowptr[dst_atom_host[m] + 1]++;
    for (int p = 0; p < P; p++) rowptr[p + 1] += rowptr[p];
    {
        std::vector<int> fill(rowptr.begin(), rowptr.end() - 1);
        for (int64_t m = 0; m < n_map; m++) {
            const int k = fill[dst_atom_host[m]]++;
            src[k] = src_atom_host[m];
            sgn[k] = sign_host[m];
        }
    }
    CUDA_TRY(h, cudaSetDevice(h->device));
    CUDA_TRY(h, cudaDeviceSynchronize());
    h->drop_graph();              // captured launches hold the old map pointers / n_protein
    h->free_md();                 // the MD state is sized by n_protein
    h->free_rs();                 // ... and so are the restraints
    h->free_map();
    CUDA_TRY(h, cudaMalloc(&h->d_map_rowptr, sizeof(int) * (P + 1)));
    CUDA_TRY(h, cudaMalloc(&h->d_map_src, sizeof(int) * src.size()));
    CUDA_TRY(h, cudaMalloc(&h->d_map_sign, sizeof(float) * sgn.size()));
    CUDA_TRY(h, cudaMalloc(&h->d_frag_sign, sizeof(float) * h->ws.G));
    CUDA_TRY(h, cudaMalloc(&h->d_ef, sizeof(float) * (3 * (size_t)P + 1)));
    CUDA_TRY(h, cudaMemcpy(h->d_map_rowptr, rowptr.data(), sizeof(int) * (P + 1), cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(h->d_map_src, src.data(), sizeof(int) * src.size(), cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(h->d_map_sign, sgn.data(), sizeof(float) * sgn.size(), cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(h->d_frag_sign, frag_sign_host, sizeof(float) * h->ws.G, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemset(h->d_ef, 0, sizeof(float) * (3 * (size_t)P + 1)));
    h->n_protein = P;
    h->n_map = (int)n_map;
    return VB_OK;
}

int vb_forward_protein(vb_handle* h, const float* pos_dev, float* ef_prot_dev, void* stream) {
    NvtxRange nvtx_("vb_forward_protein");
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (!h->has_topology || h->n_protein <= 0) { h->set_error("vb_forward_protein: topology / protein map not set"); return VB_ERR_STATE; }
    if (!pos_dev || !ef_prot_dev) { h->set_error("vb_forward_protein: null buffer"); return VB_ERR_ARG; }
    CUDA_TRY(h, cudaSetDevice(h->device));
    StepIO io = internal_io(h, false);
    io.pos = pos_dev; io.ef = ef_prot_dev;            // the signed reduction is the evaluation's last launch
    return run_eval(h, (cudaStream_t)stream, io);
}

// ---- device-resident MD (k_md.cuh) ---------------------------------------------------------------------
namespace {
StepIO md_io(vb_handle* h) {
    StepIO io = internal_io(h, false);
    io.ef = h->md_ef;
    return io;
}
// fragment placement -> evaluation + signed whole-protein reduction [-> MM or PME non-bonded term] [-> restraints], all on st
int md_eval_enqueue(vb_handle* h, cudaStream_t st) {
    const int N = h->ws.N;
    md_place_kernel<<<(N + 255) / 256, 256, 0, st>>>(N, h->d_real, h->d_acc, h->d_rem, h->d_blen, h->d_mx, h->d_pos);
    if (h->caph_ready) caph_relax_kernel<<<1, CAPH_THREADS, 0, st>>>(h->caph, h->d_pos);   // hydrogen refinement, in place
    if (int rc = enqueue_eval(h, st, md_io(h))) return rc;
    if (h->nb_ready && h->nb.hi > h->nb.lo) {      // non-bonded MM term on the same protein coordinates
        nonbonded_kernel<double><<<(h->nb.hi - h->nb.lo + 7) / 8, 256, 0, st>>>(h->nb, h->d_mx, h->md_ef, h->d_nb_eatom);
        nonbonded_energy_kernel<<<1, 256, 0, st>>>(h->nb, h->d_nb_eatom, h->md_ef);
    }
    if (h->pme_ready) pme_launch<double>(h->pme, h->d_mx, h->md_ef, st);   // PME non-bonded term instead
    if (h->rs_ready && h->rs.hi > h->rs.lo)         // Hookean restraints on the same protein coordinates
        restraint_kernel<<<1, RS_THREADS, 0, st>>>(h->rs, h->d_mx, h->md_ef);
    CUDA_TRY(h, cudaGetLastError());
    if (h->comm_ready && h->comm_auto) return enqueue_allreduce(h, st, h->md_ef, 3LL * h->n_protein + 1);
    return VB_OK;
}
void md_kick1_enqueue(vb_handle* h, cudaStream_t st) {
    md_kick1_kernel<<<1, MD_K1_THREADS, 0, st>>>(h->md, h->d_step, h->d_mmass, h->md_ef, h->d_mx, h->d_mv);
}
void md_kick2_enqueue(vb_handle* h, cudaStream_t st) {
    md_kick2_kernel<<<1, MD_K2_THREADS, 0, st>>>(h->md, h->d_step, h->d_mmass, h->md_ef, h->d_mv, h->d_ehist, h->ehist_cap);
}
int md_check(vb_handle* h, const char* who) {
    if (!h->md_ready) { h->set_error("%s: call vb_md_setup first", who); return VB_ERR_STATE; }
    return VB_OK;
}
}  // namespace

int vb_md_setup(vb_handle* h, int64_t n_protein_atoms, const double* masses_host, const int32_t* real_host,
                const int32_t* acc_host, const int32_t* rem_host, const float* blen_host, double dt, double kT,
                double friction, uint64_t seed, float* ef_prot_dev) {
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (!h->has_topology || h->n_protein <= 0) { h->set_error("vb_md_setup: topology / protein map not set"); return VB_ERR_STATE; }
    if (n_protein_atoms != h->n_protein || !masses_host || !real_host || !acc_host || !rem_host || !blen_host || !ef_prot_dev ||
        !(dt > 0.0) || kT < 0.0 || friction < 0.0) {
        h->set_error("vb_md_setup: bad arguments (n_protein must equal the protein map's)");
        return VB_ERR_ARG;
    }
    const int N = h->ws.N, P = h->n_protein;
    for (int a = 0; a < N; a++) {
        const bool cap = real_host[a] < 0;
        if ((!cap && real_host[a] >= P) || (cap && (acc_host[a] < 0 || acc_host[a] >= P || rem_host[a] < 0 || rem_host[a] >= P ||
                                                     acc_host[a] == rem_host[a]))) {
            h->set_error("vb_md_setup: recipe index out of range at fragment atom %d", a);
            return VB_ERR_ARG;
        }
    }
    for (int i = 0; i < P; i++)
        if (!(masses_host[i] > 0.0)) { h->set_error("vb_md_setup: non-positive mass at atom %d", i); return VB_ERR_ARG; }
    CUDA_TRY(h, cudaSetDevice(h->device));
    h->drop_graph();
    h->free_md();
    CUDA_TRY(h, cudaMalloc(&h->d_mx, sizeof(double) * 3 * P));
    CUDA_TRY(h, cudaMalloc(&h->d_mv, sizeof(double) * 3 * P));
    CUDA_TRY(h, cudaMalloc(&h->d_mmass, sizeof(double) * P));
    CUDA_TRY(h, cudaMalloc(&h->d_ehist, sizeof(double) * h->ehist_cap));
    CUDA_TRY(h, cudaMalloc(&h->d_real, sizeof(int) * N));
    CUDA_TRY(h, cudaMalloc(&h->d_acc, sizeof(int) * N));
    CUDA_TRY(h, cudaMalloc(&h->d_rem, sizeof(int) * N));
    CUDA_TRY(h, cudaMalloc(&h->d_blen, sizeof(float) * N));
    CUDA_TRY(h, cudaMalloc(&h->d_step, sizeof(long long)));
    CUDA_TRY(h, cudaMemcpy(h->d_mmass, masses_host, sizeof(double) * P, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(h->d_real, real_host, sizeof(int) * N, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(h->d_acc, acc_host, sizeof(int) * N, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(h->d_rem, rem_host, sizeof(int) * N, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(h->d_blen, blen_host, sizeof(float) * N, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemset(h->d_mx, 0, sizeof(double) * 3 * P));
    CUDA_TRY(h, cudaMemset(h->d_mv, 0, sizeof(double) * 3 * P));
    CUDA_TRY(h, cudaMemset(h->d_ehist, 0, sizeof(double) * h->ehist_cap));
    CUDA_TRY(h, cudaMemset(h->d_step, 0, sizeof(long long)));
    h->md = MdParams{P, dt, kT, friction, (unsigned long long)seed, nullptr, 0};
    h->md_ef = ef_prot_dev;
    h->md_ready = true;
    return VB_OK;
}

int vb_md_set_normals(vb_handle* h, const double* pool_dev, int64_t pool_steps) {
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (int rc = md_check(h, "vb_md_set_normals")) return rc;
    if ((pool_dev == nullptr) != (pool_steps == 0) || pool_steps < 0) { h->set_error("vb_md_set_normals: bad arguments"); return VB_ERR_ARG; }
    h->md.pool = pool_dev;
    h->md.pool_steps = pool_steps;
    h->drop_graph();              // kernel arguments are baked into the captured step
    return VB_OK;
}

int vb_md_set_state(vb_handle* h, const double* x_host, const double* v_host, int64_t step) {
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (int rc = md_check(h, "vb_md_set_state")) return rc;
    if (!x_host || !v_host || step < 0) { h->set_error("vb_md_set_state: bad arguments"); return VB_ERR_ARG; }
    CUDA_TRY(h, cudaSetDevice(h->device));
    CUDA_TRY(h, cudaDeviceSynchronize());
    const long long s = step;
    CUDA_TRY(h, cudaMemcpy(h->d_mx, x_host, sizeof(double) * 3 * h->n_protein, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(h->d_mv, v_host, sizeof(double) * 3 * h->n_protein, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(h->d_step, &s, sizeof(long long), cudaMemcpyHostToDevice));
    return VB_OK;
}

int vb_md_eval(vb_handle* h, void* stream) {
    NvtxRange nvtx_("vb_md_eval");
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (int rc = md_check(h, "vb_md_eval")) return rc;
    CUDA_TRY(h, cudaSetDevice(h->device));
    return run_cached(h, (cudaStream_t)stream, K_MD_EVAL, md_io(h), [&](cudaStream_t s) -> int { return md_eval_enqueue(h, s); });
}

int vb_md_kick1(vb_handle* h, void* stream) {
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (int rc = md_check(h, "vb_md_kick1")) return rc;
    CUDA_TRY(h, cudaSetDevice(h->device));
    md_kick1_enqueue(h, (cudaStream_t)stream);
    CUDA_TRY(h, cudaGetLastError());
    return VB_OK;
}

int vb_md_kick2(vb_handle* h, void* stream) {
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (int rc = md_check(h, "vb_md_kick2")) return rc;
    CUDA_TRY(h, cudaSetDevice(h->device));
    md_kick2_enqueue(h, (cudaStream_t)stream);
    CUDA_TRY(h, cudaGetLastError());
    return VB_OK;
}

int vb_md_run(vb_handle* h, int64_t n_steps, void* stream) {
    NvtxRange nvtx_("vb_md_run");
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (int rc = md_check(h, "vb_md_run")) return rc;
    if (n_steps < 0) { h->set_error("vb_md_run: negative step count"); return VB_ERR_ARG; }
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(h, cudaSetDevice(h->device));
    for (int64_t s = 0; s < n_steps; s++) {          // one graph replay per step
        int rc = run_cached(h, st, K_MD_STEP, md_io(h), [&](cudaStream_t cs) -> int {
            md_kick1_enqueue(h, cs);
            if (int r = md_eval_enqueue(h, cs)) return r;
            md_kick2_enqueue(h, cs);
            CUDA_TRY(h, cudaGetLastError());
            return (int)VB_OK;
        });
        if (rc != VB_OK) return rc;
    }
    return VB_OK;
}

int vb_md_get_state(vb_handle* h, double* x_host, double* v_host, int64_t* step_out, double* epot_hist_host, int64_t n_hist) {
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (int rc = md_check(h, "vb_md_get_state")) return rc;
    if (n_hist < 0 || n_hist > h->ehist_cap || (n_hist > 0 && !epot_hist_host)) { h->set_error("vb_md_get_state: bad history request"); return VB_ERR_ARG; }
    CUDA_TRY(h, cudaSetDevice(h->device));
    CUDA_TRY(h, cudaDeviceSynchronize());
    long long step = 0;
    CUDA_TRY(h, cudaMemcpy(&step, h->d_step, sizeof(long long), cudaMemcpyDeviceToHost));
    if (x_host) CUDA_TRY(h, cudaMemcpy(x_host, h->d_mx, sizeof(double) * 3 * h->n_protein, cudaMemcpyDeviceToHost));
    if (v_host) CUDA_TRY(h, cudaMemcpy(v_host, h->d_mv, sizeof(double) * 3 * h->n_protein, cudaMemcpyDeviceToHost));
    if (step_out) *step_out = step;
    if (n_hist > 0) {       // potential energies recorded at the end of the last n_hist steps, oldest first
        std::vector<double> ring(h->ehist_cap);
        CUDA_TRY(h, cudaMemcpy(ring.data(), h->d_ehist, sizeof(double) * h->ehist_cap, cudaMemcpyDeviceToHost));
        for (int64_t i = 0; i < n_hist; i++) {
            const long long sidx = step - n_hist + i;
            epot_hist_host[i] = sidx >= 0 ? ring[sidx % h->ehist_cap] : 0.0;
        }
    }
    return VB_OK;
}


// ---- non-bonded MM term (k_nonbonded.cuh) ----------------------------------------------------------------
namespace {
// CSR exclusion table over P atoms: rowptr[0] = 0, monotone, every row strictly ascending indices in [0, P)
int check_exclusions(vb_handle* h, const char* who, int P, const int32_t* rowptr, const int32_t* col) {
    const int64_t nx = rowptr[P];
    if (rowptr[0] != 0 || nx < 0 || (nx > 0 && !col)) { h->set_error("%s: bad exclusion table", who); return VB_ERR_ARG; }
    for (int i = 0; i < P; i++) {
        if (rowptr[i + 1] < rowptr[i]) { h->set_error("%s: exclusion row pointer not monotone", who); return VB_ERR_ARG; }
        for (int k = rowptr[i]; k < rowptr[i + 1]; k++) {
            const int c = col[k];
            if (c < 0 || c >= P || (k > rowptr[i] && c <= col[k - 1])) {
                h->set_error("%s: exclusion row %d must be strictly ascending atom indices", who, i);
                return VB_ERR_ARG;
            }
        }
    }
    return VB_OK;
}
// ASE 3.22 unit system (CODATA 2014): nonbonded.py:18 / pme.py:120 k = 1/(4 pi eps0) * 10e6 * mol * C^-2 ; kJ/mol in eV
void coulomb_units(double* k, double* kj_mol) {
    const double c = 299792458.0, mu0 = 4.0e-7 * 3.14159265358979323846, eps0 = 1.0 / mu0 / (c * c);
    const double e_ch = 1.6021766208e-19, nav = 6.022140857e23, coul = 1.0 / e_ch, kj = 1000.0 / e_ch;
    *k = 1.0 / (4.0 * 3.14159265358979323846 * eps0) * 10e6 * nav / (coul * coul);
    *kj_mol = kj / nav;
}
}  // namespace

int vb_set_nonbonded(vb_handle* h, int64_t n_protein_atoms, const float* charges_host, const float* sigmas_nm_host,
                     const float* epsilons_kj_host, const int32_t* excl_rowptr_host, const int32_t* excl_col_host,
                     int64_t atom_lo, int64_t atom_hi) {
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (n_protein_atoms <= 0 || !charges_host || !sigmas_nm_host || !epsilons_kj_host || !excl_rowptr_host ||
        atom_lo < 0 || atom_hi < atom_lo || atom_hi > n_protein_atoms) {
        h->set_error("vb_set_nonbonded: bad arguments");
        return VB_ERR_ARG;
    }
    if (h->n_protein > 0 && h->n_protein != n_protein_atoms) {
        h->set_error("vb_set_nonbonded: n_protein_atoms differs from the protein map's");
        return VB_ERR_ARG;
    }
    const int P = (int)n_protein_atoms;
    const int64_t nx = excl_rowptr_host[P];
    if (int rc = check_exclusions(h, "vb_set_nonbonded", P, excl_rowptr_host, excl_col_host)) return rc;
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (h->pme_ready) {                 // one non-bonded term at a time; MD graph replays may still read the PME arrays
        CUDA_TRY(h, cudaDeviceSynchronize());
        h->free_pme();
    }
    h->drop_graph();
    h->free_nb();
    CUDA_TRY(h, cudaMalloc(&h->d_nb_q, sizeof(float) * P));
    CUDA_TRY(h, cudaMalloc(&h->d_nb_sigma, sizeof(float) * P));
    CUDA_TRY(h, cudaMalloc(&h->d_nb_eps, sizeof(float) * P));
    CUDA_TRY(h, cudaMalloc(&h->d_nb_rowptr, sizeof(int) * (P + 1)));
    CUDA_TRY(h, cudaMalloc(&h->d_nb_col, sizeof(int) * std::max<int64_t>(nx, 1)));
    CUDA_TRY(h, cudaMalloc(&h->d_nb_eatom, sizeof(double) * P));
    CUDA_TRY(h, cudaMemcpy(h->d_nb_q, charges_host, sizeof(float) * P, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(h->d_nb_sigma, sigmas_nm_host, sizeof(float) * P, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(h->d_nb_eps, epsilons_kj_host, sizeof(float) * P, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemcpy(h->d_nb_rowptr, excl_rowptr_host, sizeof(int) * (P + 1), cudaMemcpyHostToDevice));
    if (nx > 0) CUDA_TRY(h, cudaMemcpy(h->d_nb_col, excl_col_host, sizeof(int) * nx, cudaMemcpyHostToDevice));
    CUDA_TRY(h, cudaMemset(h->d_nb_eatom, 0, sizeof(double) * P));
    double k, kj_mol;
    coulomb_units(&k, &kj_mol);
    h->nb = NbParams{P, (int)atom_lo, (int)atom_hi, h->d_nb_q, h->d_nb_sigma, h->d_nb_eps, h->d_nb_rowptr, h->d_nb_col,
                     (float)k, (float)kj_mol};
    h->nb_ready = true;
    return VB_OK;
}

int vb_nonbonded(vb_handle* h, const float* prot_pos_dev, float* ef_prot_dev, void* stream) {
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (!h->nb_ready) { h->set_error("vb_nonbonded: call vb_set_nonbonded first"); return VB_ERR_STATE; }
    if (!prot_pos_dev || !ef_prot_dev) { h->set_error("vb_nonbonded: null buffer"); return VB_ERR_ARG; }
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (h->nb.hi > h->nb.lo) {
        nonbonded_kernel<float><<<(h->nb.hi - h->nb.lo + 7) / 8, 256, 0, st>>>(h->nb, prot_pos_dev, ef_prot_dev, h->d_nb_eatom);
        nonbonded_energy_kernel<<<1, 256, 0, st>>>(h->nb, h->d_nb_eatom, ef_prot_dev);
    }
    CUDA_TRY(h, cudaGetLastError());
    return VB_OK;
}


// ---- PME non-bonded term (k_pme.cuh) -------------------------------------------------------------------------------
int vb_set_pme(vb_handle* h, const vb_pme_params* pp) {
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    auto bad = [&](const char* what) { h->set_error("vb_set_pme: %s", what); return VB_ERR_ARG; };
    if (!pp) return bad("null parameters");
    const int64_t n = pp->n_protein_atoms;
    if (n <= 0 || n > (1 << 24) || !pp->charges || !pp->sigmas_nm || !pp->epsilons_kj || !pp->excl_rowptr)
        return bad("bad arguments");
    if (pp->atom_lo < 0 || pp->atom_hi < pp->atom_lo || pp->atom_hi > n) return bad("bad slice: [atom_lo, atom_hi) must lie in [0, n)");
    if (h->n_protein > 0 && h->n_protein != n) return bad("n_protein_atoms differs from the protein map's");
    for (int a = 0; a < 3; a++) {
        if (!std::isfinite(pp->cell[a]) || !(pp->cell[a] > 0.0)) return bad("cell lengths must be finite and positive");
        if (pp->grid[a] < 4) return bad("grid dimensions must be at least 4 (spline order)");
        if (pp->grid[a] > 4096) return bad("grid dimensions must be at most 4096");
    }
    if ((int64_t)pp->grid[0] * pp->grid[1] * pp->grid[2] > (1LL << 27)) return bad("grid has more than 2^27 points");
    if (!std::isfinite(pp->beta) || !(pp->beta > 0.0)) return bad("beta must be finite and positive");
    if (!std::isfinite(pp->cutoff) || !(pp->cutoff > 0.0)) return bad("cutoff must be finite and positive");
    const int P = (int)n;
    if (int rc = check_exclusions(h, "vb_set_pme", P, pp->excl_rowptr, pp->excl_col)) return rc;
    const int64_t nx = pp->excl_rowptr[P];
    const int K1 = pp->grid[0], K2 = pp->grid[1], K3 = pp->grid[2], H3 = K3 / 2 + 1;
    // host tables: per-axis twiddles cos / sin(2 pi j / K) and B-spline moduli 36 / (4 + 2 cos(2 pi m / K))^2
    std::vector<double> tw, bmod;
    for (int K : {K1, K2, K3})
        for (int j = 0; j < K; j++) {
            const double th = 2.0 * 3.14159265358979323846 * j / K;
            tw.push_back(cos(th)); tw.push_back(sin(th));
            bmod.push_back(36.0 / ((4.0 + 2.0 * cos(th)) * (4.0 + 2.0 * cos(th))));
        }
    double qsum = 0.0, q2 = 0.0;
    for (int i = 0; i < P; i++) { qsum += pp->charges[i]; q2 += (double)pp->charges[i] * pp->charges[i]; }
    const float qtot = (float)qsum, zero_pos[3] = {0.f, 0.f, 0.f};
    // MD graph replays enqueued before this call may still read the old arrays
    CUDA_TRY(h, cudaSetDevice(h->device));
    CUDA_TRY(h, cudaDeviceSynchronize());
    h->drop_graph();
    h->free_nb();                       // one non-bonded term at a time (FragmentCalculator's nonbonded_calcs[type])
    h->free_pme();
    struct Piece { const void* src; size_t bytes; size_t off; };
    std::vector<Piece> pieces;
    size_t total = 0;
    auto add = [&](const void* src, size_t bytes) {
        pieces.push_back({src, bytes, total});
        total += (std::max<size_t>(bytes, 8) + 255) & ~(size_t)255;
        return pieces.size() - 1;
    };
    const size_t nh = (size_t)K1 * K2 * H3, ngrid = (size_t)K1 * K2 * K3;
    const int n_partial = (int)((nh + PME_THREADS - 1) / PME_THREADS);
    const size_t i_q = add(pp->charges, 4 * (size_t)P), i_s = add(pp->sigmas_nm, 4 * (size_t)P), i_e = add(pp->epsilons_kj, 4 * (size_t)P);
    const size_t i_rp = add(pp->excl_rowptr, 4 * (size_t)(P + 1)), i_cl = add(nx > 0 ? pp->excl_col : nullptr, 4 * (size_t)nx);
    const size_t i_tw = add(tw.data(), 8 * tw.size()), i_bm = add(bmod.data(), 8 * bmod.size());
    const size_t i_base = add(nullptr, 12 * (size_t)P), i_w = add(nullptr, 96 * (size_t)P);
    const size_t i_bp = add(nullptr, 4 * (size_t)(K1 + 1)), i_ba = add(nullptr, 4 * (size_t)P);
    const size_t i_Q = add(nullptr, 8 * ngrid), i_A = add(nullptr, 16 * nh), i_B = add(nullptr, 16 * nh);
    const size_t i_pa = add(nullptr, 8 * (size_t)n_partial), i_ea = add(nullptr, 8 * (size_t)PME_NATOM * P);
    const size_t i_t = add(nullptr, 8 * PT_N);
    const size_t i_zp = add(zero_pos, sizeof(zero_pos)), i_qt = add(&qtot, 4), i_ef1 = add(nullptr, 16);
    CUDA_TRY(h, cudaMalloc(&h->pme_mem, total));
    char* base = static_cast<char*>(h->pme_mem);
    CUDA_TRY(h, cudaMemset(base, 0, total));
    for (const Piece& pc : pieces)
        if (pc.src && pc.bytes) CUDA_TRY(h, cudaMemcpy(base + pc.off, pc.src, pc.bytes, cudaMemcpyHostToDevice));
    auto at = [&](size_t i) { return static_cast<void*>(base + pieces[i].off); };
    double k, kj_mol;
    coulomb_units(&k, &kj_mol);
    PmeParams& m = h->pme;
    m = PmeParams{};
    m.n = P; m.lo = (int)pp->atom_lo; m.hi = (int)pp->atom_hi; m.recip = pp->atom_lo == 0;
    m.q = (const float*)at(i_q); m.sigma = (const float*)at(i_s); m.eps = (const float*)at(i_e);
    m.excl_rowptr = (const int*)at(i_rp); m.excl_col = (const int*)at(i_cl);
    m.coulomb_k = (float)k; m.kj_mol = (float)kj_mol;
    m.beta = (float)pp->beta; m.rc2 = (float)pp->cutoff * (float)pp->cutoff;
    m.beta64 = pp->beta; m.k64 = k; m.kj64 = kj_mol;
    m.K1 = K1; m.K2 = K2; m.K3 = K3; m.H3 = H3;
    m.L1 = pp->cell[0]; m.L2 = pp->cell[1]; m.L3 = pp->cell[2];
    m.tw = (const double*)at(i_tw); m.bmod = (const double*)at(i_bm);
    m.base = (int*)at(i_base); m.w = (double*)at(i_w); m.bin_ptr = (int*)at(i_bp); m.bin_atom = (int*)at(i_ba);
    m.Q = (double*)at(i_Q); m.A = (double2*)at(i_A); m.B = (double2*)at(i_B);
    m.partial = (double*)at(i_pa); m.eatom = (double*)at(i_ea); m.terms = (double*)at(i_t);
    // electro_neutral (pme.py:99-110): the same kernels on one particle of charge q_tot at the origin give its E_rec
    PmeParams one = m;
    one.n = 1; one.lo = one.hi = 0; one.recip = true; one.q = (const float*)at(i_qt);
    pme_launch<float>(one, (const float*)at(i_zp), (float*)at(i_ef1), h->own_stream);
    double rec1 = 0.0;
    CUDA_TRY(h, cudaGetLastError());
    CUDA_TRY(h, cudaStreamSynchronize(h->own_stream));
    CUDA_TRY(h, cudaMemcpy(&rec1, m.terms + PT_REC, sizeof(double), cudaMemcpyDeviceToHost));
    const double sqpi = sqrt(3.14159265358979323846);
    m.slf = -pp->beta / sqpi * q2;                                          // electro_slf, pme.py:86-87
    m.neutral = -rec1 + pp->beta * qsum * qsum / sqpi;                     // E_rec of fp32 q_tot (helpmelib.MatrixF)
    h->pme_ready = true;
    return VB_OK;
}

int vb_pme(vb_handle* h, const float* prot_pos_dev, float* ef_prot_dev, void* stream) {
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (!h->pme_ready) { h->set_error("vb_pme: call vb_set_pme first"); return VB_ERR_STATE; }
    if (!prot_pos_dev || !ef_prot_dev) { h->set_error("vb_pme: null buffer"); return VB_ERR_ARG; }
    CUDA_TRY(h, cudaSetDevice(h->device));
    pme_launch<float>(h->pme, prot_pos_dev, ef_prot_dev, (cudaStream_t)stream);
    CUDA_TRY(h, cudaGetLastError());
    return VB_OK;
}

// ---- Hookean restraints (k_restraint.cuh) ------------------------------------------------------------------------
int vb_set_restraints(vb_handle* h, const vb_restraint_set* rs) {
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (h->n_protein <= 0) { h->set_error("vb_set_restraints: call vb_set_protein_map first"); return VB_ERR_STATE; }
    if (!rs) { h->set_error("vb_set_restraints: null restraint set"); return VB_ERR_ARG; }
    const int P = h->n_protein;
    const int64_t np_ = rs->n_point, nq = rs->n_pair;
    auto bad = [&](const char* fmt, long long i) { h->set_error(fmt, i); return VB_ERR_ARG; };
    if (np_ < 0 || nq < 0 || np_ + nq > (1 << 29)) return bad("vb_set_restraints: bad restraint count (%lld)", (long long)(np_ + nq));
    if (rs->atom_lo < 0 || rs->atom_hi < rs->atom_lo || rs->atom_hi > P)
        return bad("vb_set_restraints: bad slice: [atom_lo, atom_hi) must lie in [0, %lld)", (long long)P);
    if ((np_ > 0 && (!rs->point_atom || !rs->point_anchor || !rs->point_k || !rs->point_rt)) ||
        (nq > 0 && (!rs->pair_ij || !rs->pair_k || !rs->pair_rt)))
        return bad("vb_set_restraints: null array for %lld restraints", (long long)(np_ + nq));
    auto finite_nonneg = [](double v) { return std::isfinite(v) && v >= 0.0; };
    for (int64_t i = 0; i < np_; i++) {
        if (rs->point_atom[i] < 0 || rs->point_atom[i] >= P) return bad("vb_set_restraints: point restraint %lld: atom index out of range", (long long)i);
        if (!finite_nonneg(rs->point_k[i]) || !finite_nonneg(rs->point_rt[i]))
            return bad("vb_set_restraints: point restraint %lld: k and rt must be finite and non-negative", (long long)i);
        for (int c = 0; c < 3; c++)
            if (!std::isfinite(rs->point_anchor[3 * i + c])) return bad("vb_set_restraints: point restraint %lld: non-finite anchor", (long long)i);
    }
    for (int64_t q = 0; q < nq; q++) {
        const int i = rs->pair_ij[2 * q], j = rs->pair_ij[2 * q + 1];
        if (i < 0 || i >= P || j < 0 || j >= P) return bad("vb_set_restraints: pair restraint %lld: atom index out of range", (long long)q);
        if (i == j) return bad("vb_set_restraints: pair restraint %lld: i == j", (long long)q);
        if (!finite_nonneg(rs->pair_k[q]) || !finite_nonneg(rs->pair_rt[q]))
            return bad("vb_set_restraints: pair restraint %lld: k and rt must be finite and non-negative", (long long)q);
    }
    // CSR over destination atoms, entries in restraint-id order within a row
    std::vector<int> row(P + 1, 0);
    for (int64_t i = 0; i < np_; i++) row[rs->point_atom[i] + 1]++;
    for (int64_t q = 0; q < 2 * nq; q++) row[rs->pair_ij[q] + 1]++;
    for (int a = 0; a < P; a++) row[a + 1] += row[a];
    std::vector<int> ent(std::max<int64_t>(row[P], 1)), fill(row.begin(), row.end() - 1);
    for (int64_t i = 0; i < np_; i++) ent[fill[rs->point_atom[i]]++] = (int)(2 * i);
    for (int64_t q = 0; q < nq; q++) {
        const int id = (int)(np_ + q);
        ent[fill[rs->pair_ij[2 * q]]++] = 2 * id;
        ent[fill[rs->pair_ij[2 * q + 1]]++] = 2 * id + 1;
    }
    // MD graph replays enqueued before this call may still read the old arrays
    CUDA_TRY(h, cudaSetDevice(h->device));
    CUDA_TRY(h, cudaDeviceSynchronize());
    h->drop_graph();
    h->free_rs();
    if (np_ == 0 && nq == 0) return VB_OK;            // empty set: the term is removed
    struct Piece { const void* src; size_t bytes; size_t off; };
    std::vector<Piece> pieces;
    size_t total = 0;
    auto add = [&](const void* src, size_t bytes) {
        pieces.push_back({src, bytes, total});
        total += (std::max<size_t>(bytes, 8) + 255) & ~(size_t)255;
        return pieces.size() - 1;
    };
    const size_t i_row = add(row.data(), sizeof(int) * row.size()), i_ent = add(ent.data(), sizeof(int) * ent.size());
    const size_t i_pa = add(rs->point_anchor, 24 * (size_t)np_), i_pk = add(rs->point_k, 8 * (size_t)np_), i_pr = add(rs->point_rt, 8 * (size_t)np_);
    const size_t i_qij = add(rs->pair_ij, 8 * (size_t)nq), i_qk = add(rs->pair_k, 8 * (size_t)nq), i_qr = add(rs->pair_rt, 8 * (size_t)nq);
    CUDA_TRY(h, cudaMalloc(&h->rs_mem, total));
    char* base = static_cast<char*>(h->rs_mem);
    for (const Piece& pc : pieces)
        if (pc.bytes) CUDA_TRY(h, cudaMemcpy(base + pc.off, pc.src, pc.bytes, cudaMemcpyHostToDevice));
    auto ip = [&](size_t i) { return reinterpret_cast<const int*>(base + pieces[i].off); };
    auto dp = [&](size_t i) { return reinterpret_cast<const double*>(base + pieces[i].off); };
    h->rs = RsParams{P, (int)rs->atom_lo, (int)rs->atom_hi, (int)np_, ip(i_row), ip(i_ent), dp(i_pa), dp(i_pk), dp(i_pr),
                     ip(i_qij), dp(i_qk), dp(i_qr)};
    h->rs_ready = true;
    return VB_OK;
}

int vb_restraints(vb_handle* h, const double* prot_pos_dev, float* ef_prot_dev, void* stream) {
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (h->n_protein <= 0) { h->set_error("vb_restraints: call vb_set_protein_map first"); return VB_ERR_STATE; }
    if (!prot_pos_dev || !ef_prot_dev) { h->set_error("vb_restraints: null buffer"); return VB_ERR_ARG; }
    CUDA_TRY(h, cudaSetDevice(h->device));
    if (h->rs_ready && h->rs.hi > h->rs.lo)
        restraint_kernel<<<1, RS_THREADS, 0, (cudaStream_t)stream>>>(h->rs, prot_pos_dev, ef_prot_dev);
    CUDA_TRY(h, cudaGetLastError());
    return VB_OK;
}


// ---- cap-hydrogen refinement (k_caph.cuh) --------------------------------------------------------------------------
int vb_set_caph(vb_handle* h, const vb_caph_problem* pr) {
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (!h->has_topology) { h->set_error("vb_set_caph: call vb_set_topology first"); return VB_ERR_STATE; }
    if (!pr) { h->set_error("vb_set_caph: null problem"); return VB_ERR_ARG; }
    const int64_t N = h->ws.N;
    auto bad = [&](const char* what) { h->set_error("vb_set_caph: %s", what); return VB_ERR_ARG; };
    if (pr->n_h < 0 || pr->n_bonds < 0 || pr->n_angles < 0 || pr->n_dih < 0 || pr->n_pairs < 0 || pr->n_mirror < 0) return bad("negative count");
    if (pr->max_iter < 1 || pr->max_iter > 64) return bad("max_iter must be in [1, 64]");
    if (!(pr->scnb > 0.f) || !(pr->scee > 0.f) || !(pr->lr > 0.f)) return bad("scnb, scee and lr must be positive");
    const int64_t n_terms = pr->n_bonds + pr->n_angles + pr->n_dih + pr->n_pairs;
    if (n_terms > (1 << 27) || pr->n_h > (1 << 26)) return bad("problem too large");
    auto check_idx = [&](const int32_t* a, int64_t count, const char* what) {
        if (count > 0 && !a) { h->set_error("vb_set_caph: %s is null", what); return false; }
        for (int64_t i = 0; i < count; i++)
            if (a[i] < 0 || a[i] >= N) { h->set_error("vb_set_caph: %s[%lld] = %d is not a fragment atom", what, (long long)i, a[i]); return false; }
        return true;
    };
    if (!check_idx(pr->h_idx, pr->n_h, "h_idx") || !check_idx(pr->bond_ij, 2 * pr->n_bonds, "bond_ij") ||
        !check_idx(pr->angle_ijk, 3 * pr->n_angles, "angle_ijk") || !check_idx(pr->dih_ijkl, 4 * pr->n_dih, "dih_ijkl") ||
        !check_idx(pr->pair_ij, 2 * pr->n_pairs, "pair_ij") || !check_idx(pr->mirror_dst, pr->n_mirror, "mirror_dst") ||
        !check_idx(pr->mirror_src, pr->n_mirror, "mirror_src"))
        return VB_ERR_ARG;
    if ((pr->n_bonds && (!pr->bond_k || !pr->bond_r0)) || (pr->n_angles && (!pr->angle_k || !pr->angle_t0)) ||
        (pr->n_dih && (!pr->dih_k || !pr->dih_n || !pr->dih_p)) || (pr->n_pairs && (!pr->pair_a || !pr->pair_b || !pr->pair_qq)))
        return bad("null parameter array");
    // gather table: for every optimised hydrogen the scratch rows (term * 4 + slot) that carry a gradient on it
    std::vector<int> slot_of(N, -1);
    for (int64_t i = 0; i < pr->n_h; i++) {
        if (slot_of[pr->h_idx[i]] >= 0) return bad("h_idx lists an atom twice");
        slot_of[pr->h_idx[i]] = (int)i;
    }
    std::vector<std::vector<int>> rows(pr->n_h);
    int64_t term = 0;
    auto scan = [&](const int32_t* idx, int64_t count, int width) {
        for (int64_t t = 0; t < count; t++, term++)
            for (int k = 0; k < width; k++) {
                const int hs = slot_of[idx[t * width + k]];
                if (hs >= 0) rows[hs].push_back((int)(term * 4 + k));
            }
    };
    scan(pr->bond_ij, pr->n_bonds, 2);
    scan(pr->angle_ijk, pr->n_angles, 3);
    scan(pr->dih_ijkl, pr->n_dih, 4);
    scan(pr->pair_ij, pr->n_pairs, 2);
    std::vector<int> gat_rowptr(pr->n_h + 1, 0), gat_entry;
    for (int64_t i = 0; i < pr->n_h; i++) {
        gat_rowptr[i + 1] = gat_rowptr[i] + (int)rows[i].size();
        gat_entry.insert(gat_entry.end(), rows[i].begin(), rows[i].end());
    }
    CUDA_TRY(h, cudaSetDevice(h->device));
    CUDA_TRY(h, cudaDeviceSynchronize());
    h->drop_graph();
    h->free_caph();
    // one allocation, carved in 256-byte steps
    struct Piece { const void* src; size_t bytes; size_t off; };
    std::vector<Piece> pieces;
    size_t total = 0;
    auto add = [&](const void* src, size_t bytes) {
        pieces.push_back({src, bytes, total});
        total += (std::max<size_t>(bytes, 4) + 255) & ~(size_t)255;
        return pieces.size() - 1;
    };
    const size_t nh = (size_t)pr->n_h, n3 = 3 * nh;
    const size_t i_h = add(pr->h_idx, 4 * nh);
    const size_t i_bij = add(pr->bond_ij, 8 * (size_t)pr->n_bonds), i_bk = add(pr->bond_k, 4 * (size_t)pr->n_bonds), i_br = add(pr->bond_r0, 4 * (size_t)pr->n_bonds);
    const size_t i_aijk = add(pr->angle_ijk, 12 * (size_t)pr->n_angles), i_ak = add(pr->angle_k, 4 * (size_t)pr->n_angles), i_at = add(pr->angle_t0, 4 * (size_t)pr->n_angles);
    const size_t i_dijkl = add(pr->dih_ijkl, 16 * (size_t)pr->n_dih), i_dk = add(pr->dih_k, 4 * (size_t)pr->n_dih), i_dn = add(pr->dih_n, 4 * (size_t)pr->n_dih), i_dp = add(pr->dih_p, 4 * (size_t)pr->n_dih);
    const size_t i_pij = add(pr->pair_ij, 8 * (size_t)pr->n_pairs), i_pa = add(pr->pair_a, 4 * (size_t)pr->n_pairs), i_pb = add(pr->pair_b, 4 * (size_t)pr->n_pairs), i_pq = add(pr->pair_qq, 4 * (size_t)pr->n_pairs);
    const size_t i_md = add(pr->mirror_dst, 4 * (size_t)pr->n_mirror), i_ms = add(pr->mirror_src, 4 * (size_t)pr->n_mirror);
    const size_t i_gr = add(gat_rowptr.data(), 4 * gat_rowptr.size()), i_ge = add(gat_entry.data(), 4 * gat_entry.size());
    const size_t i_tg = add(nullptr, 4 * 12 * (size_t)n_terms);
    const size_t i_vec = add(nullptr, 4 * (2 * (size_t)pr->max_iter + 4) * n3);
    const size_t i_ev = add(nullptr, 4);
    CUDA_TRY(h, cudaMalloc(&h->caph_mem, total));
    CUDA_TRY(h, cudaMemset(h->caph_mem, 0, total));
    char* base = static_cast<char*>(h->caph_mem);
    for (const Piece& pc : pieces)
        if (pc.src && pc.bytes) CUDA_TRY(h, cudaMemcpy(base + pc.off, pc.src, pc.bytes, cudaMemcpyHostToDevice));
    auto ip = [&](size_t i) { return reinterpret_cast<const int*>(base + pieces[i].off); };
    auto fp = [&](size_t i) { return reinterpret_cast<const float*>(base + pieces[i].off); };
    CaphDev& c = h->caph;
    c.n_h = (int)pr->n_h; c.h_idx = ip(i_h);
    c.n_bonds = (int)pr->n_bonds; c.bond_ij = ip(i_bij); c.bond_k = fp(i_bk); c.bond_r0 = fp(i_br);
    c.n_angles = (int)pr->n_angles; c.angle_ijk = ip(i_aijk); c.angle_k = fp(i_ak); c.angle_t0 = fp(i_at);
    c.n_dih = (int)pr->n_dih; c.dih_ijkl = ip(i_dijkl); c.dih_k = fp(i_dk); c.dih_n = fp(i_dn); c.dih_p = fp(i_dp);
    c.n_pairs = (int)pr->n_pairs; c.pair_ij = ip(i_pij); c.pair_a = fp(i_pa); c.pair_b = fp(i_pb); c.pair_qq = fp(i_pq);
    c.n_mirror = (int)pr->n_mirror; c.mirror_dst = ip(i_md); c.mirror_src = ip(i_ms);
    c.gat_rowptr = ip(i_gr); c.gat_entry = ip(i_ge);
    c.scnb = pr->scnb; c.scee = pr->scee; c.max_iter = pr->max_iter; c.lr = pr->lr; c.tol_grad = pr->tol_grad; c.tol_change = pr->tol_change;
    c.tg = reinterpret_cast<float*>(base + pieces[i_tg].off);
    c.vec = reinterpret_cast<float*>(base + pieces[i_vec].off);
    c.evals_out = reinterpret_cast<int*>(base + pieces[i_ev].off);
    h->caph_ready = true;
    return VB_OK;
}

int vb_caph_relax(vb_handle* h, float* pos_dev, void* stream) {
    NvtxRange nvtx_("vb_caph_relax");
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (!h->caph_ready) { h->set_error("vb_caph_relax: call vb_set_caph first"); return VB_ERR_STATE; }
    if (!pos_dev) { h->set_error("vb_caph_relax: null buffer"); return VB_ERR_ARG; }
    CUDA_TRY(h, cudaSetDevice(h->device));
    caph_relax_kernel<<<1, CAPH_THREADS, 0, (cudaStream_t)stream>>>(h->caph, pos_dev);
    CUDA_TRY(h, cudaGetLastError());
    return VB_OK;
}

// ---- NVLink peer-memory all-reduce (k_comm.cuh) ------------------------------------------------------------------
int vb_comm_init(vb_handle* h, int rank, int world, int64_t max_floats, void* ipc_handle_out) {
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (world < 1 || world > COMM_MAX_WORLD || rank < 0 || rank >= world || max_floats <= 0 || !ipc_handle_out) {
        h->set_error("vb_comm_init: bad arguments (world <= %d)", COMM_MAX_WORLD);
        return VB_ERR_ARG;
    }
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    CUDA_TRY(h, cudaSetDevice(h->device));
    CUDA_TRY(h, cudaDeviceSynchronize());
    h->drop_graph();
    h->free_comm();
    const size_t flag_bytes = ((size_t)2 * world * sizeof(int) + 255) & ~(size_t)255;
    const size_t bytes = flag_bytes + (size_t)2 * world * (size_t)max_floats * sizeof(float);
    CUDA_TRY(h, cudaMalloc(&h->comm_base, bytes));
    CUDA_TRY(h, cudaMemset(h->comm_base, 0, bytes));
    CUDA_TRY(h, cudaMalloc(&h->comm.counters, 4 * sizeof(unsigned int)));
    CUDA_TRY(h, cudaMemset(h->comm.counters, 0, 4 * sizeof(unsigned int)));
    h->comm.rank = rank; h->comm.world = world; h->comm.max_floats = max_floats;
    cudaIpcMemHandle_t hd;
    CUDA_TRY(h, cudaIpcGetMemHandle(&hd, h->comm_base));
    memcpy(ipc_handle_out, &hd, sizeof(hd));
    return VB_OK;
}

int vb_comm_connect(vb_handle* h, const void* all_handles) {
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (!h->comm_base || !all_handles) { h->set_error("vb_comm_connect: call vb_comm_init first"); return VB_ERR_STATE; }
    CUDA_TRY(h, cudaSetDevice(h->device));
    const int world = h->comm.world;
    const size_t flag_bytes = ((size_t)2 * world * sizeof(int) + 255) & ~(size_t)255;
    for (int r = 0; r < world; r++) {
        void* base = h->comm_base;
        if (r != h->comm.rank) {
            cudaIpcMemHandle_t hd;
            memcpy(&hd, static_cast<const char*>(all_handles) + (size_t)r * sizeof(hd), sizeof(hd));
            cudaError_t e = cudaIpcOpenMemHandle(&base, hd, cudaIpcMemLazyEnablePeerAccess);
            if (e != cudaSuccess) {
                h->set_error("vb_comm_connect: cudaIpcOpenMemHandle for rank %d failed: %s (GPUs without peer access?)", r, cudaGetErrorString(e));
                (void)cudaGetLastError();
                return VB_ERR_CUDA;
            }
        }
        h->comm_peer[r] = base;
        h->comm.flags[r] = reinterpret_cast<int*>(base);
        h->comm.slots[r] = reinterpret_cast<float*>(static_cast<char*>(base) + flag_bytes);
    }
    h->comm_ready = true;
    h->drop_graph();
    return VB_OK;
}

int vb_comm_allreduce(vb_handle* h, float* buf_dev, int64_t n, void* stream) {
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (!h->comm_ready) { h->set_error("vb_comm_allreduce: call vb_comm_init / vb_comm_connect first"); return VB_ERR_STATE; }
    if (!buf_dev || n <= 0) { h->set_error("vb_comm_allreduce: bad arguments"); return VB_ERR_ARG; }
    CUDA_TRY(h, cudaSetDevice(h->device));
    return enqueue_allreduce(h, (cudaStream_t)stream, buf_dev, n);
}

int vb_get_edges(vb_handle* h, int32_t* slots_host, int32_t* deg_host) {
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (!h->has_topology || !slots_host || !deg_host) { h->set_error("vb_get_edges: bad state/arguments"); return VB_ERR_STATE; }
    CUDA_TRY(h, cudaSetDevice(h->device));
    CUDA_TRY(h, cudaDeviceSynchronize());
    CUDA_TRY(h, cudaMemcpy(slots_host, h->ws.slots, sizeof(int) * (size_t)h->ws.N * KNB, cudaMemcpyDeviceToHost));
    CUDA_TRY(h, cudaMemcpy(deg_host, h->ws.deg, sizeof(int) * (size_t)h->ws.N, cudaMemcpyDeviceToHost));
    return VB_OK;
}

int vb_launches_per_forward(const vb_handle* h) { return h ? h->launches : 0; }

int vb_set_option(vb_handle* h, const char* key, int64_t value) {
    if (!h || !key) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    const std::string k(key);
    if (k == "use_graph") h->use_graph = (int)value;
    else if (k == "use_pdl" && (value == 0 || value == 1)) h->use_pdl = (int)value;
    else if (k == "npw" && (value == 1 || value == 2)) h->npw = h->npw_opt = (int)value;
    else if (k == "te_fwd" && (value == 32 || value == 64)) h->te_fwd = h->te_fwd_opt = (int)value;
    else if (k == "te_bwd" && (value == 32 || value == 64)) h->te_bwd = (int)value;
    else if (k == "edge_tc" && value >= 0 && value <= 3) h->edge_tc = h->edge_tc_opt = (int)value;
    else if (k == "tc_rows" && (value == 0 || value == 32 || value == 64 || value == 96 || value == 128)) {
        h->tc_rows_opt = (int)value;
        if (h->has_topology) plan_tiles(h, h->edges_plan > 0 ? h->edges_plan : (long long)h->ws.N * 17);
    }
    else if (k == "calibrate" && value == 1) {
        // re-plan the tile length from the edge count of the last evaluation (synchronises)
        if (!h->has_topology) { h->set_error("vb_set_option: calibrate needs a topology"); return VB_ERR_STATE; }
        int e = 0;
        if (cudaSetDevice(h->device) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess ||
            cudaMemcpy(&e, h->ws.rowptr + h->ws.N, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) {
            h->set_error("vb_set_option: calibrate failed: %s", cudaGetErrorString(cudaGetLastError()));
            return VB_ERR_CUDA;
        }
        if (e > 0) plan_tiles(h, e);
    }
    else if (k == "node_impl" && (value == 0 || value == 1)) h->node_impl = (int)value;
    else if (k == "node_nb" && (value == 0 || value == 1 || value == 2 || value == 3 || value == 4 || value == 8)) h->node_nb = (int)value;
    else if (k == "krot" && (value == 0 || value == 1)) h->krot = (int)value;
    else if (k == "fused" && (value == 0 || value == 1)) { h->fused = h->fused_opt = (int)value; if (value) h->node_tc = 0; set_gxa_parts(h); }
    else if (k == "node_tc" && (value == 0 || value == 1)) { h->node_tc = h->node_tc_opt = (int)value; if (value) h->fused = 0; set_gxa_parts(h); }
    else if (k == "comm_auto" && (value == 0 || value == 1)) h->comm_auto = (int)value;
    else if (k == "embed_batch" && value >= -1 && value <= 3) h->embed_batch_opt = (int)value;
    else if (k == "timeline" && (value == 0 || value == 1)) {
        if (value && !h->d_tl) {
            if (cudaSetDevice(h->device) != cudaSuccess || cudaMalloc(&h->d_tl, sizeof(unsigned long long) * (2 * L * TC_TL_SLOTS + (2 * L + 3) * N2_TL_SLOTS)) != cudaSuccess) {
                h->set_error("vb_set_option: timeline buffer allocation failed"); return VB_ERR_CUDA;
            }
            cudaMemset(h->d_tl, 0, sizeof(unsigned long long) * (2 * L * TC_TL_SLOTS + (2 * L + 3) * N2_TL_SLOTS));
        }
        h->timeline = (int)value;
    }
    else { h->set_error("vb_set_option: unknown key or bad value: %s", key); return VB_ERR_ARG; }
    h->drop_graph();
    if (h->has_topology) record_stages(h);
    return VB_OK;
}

int64_t vb_get_option(const vb_handle* h, const char* key) {
    if (!h || !key) return VB_ERR_ARG;
    const std::string k(key);
    if (k == "use_graph") return h->use_graph;
    if (k == "use_pdl") return h->use_pdl;
    if (k == "npw") return h->npw;
    if (k == "te_fwd") return h->te_fwd;
    if (k == "te_bwd") return h->te_bwd;
    if (k == "edge_tc") return h->edge_tc;
    if (k == "node_impl") return h->node_impl;
    if (k == "node_nb") return h->has_topology ? node_nb(h) : h->node_nb;
    if (k == "krot") return h->krot;
    if (k == "fused") return h->fused;
    if (k == "node_tc") return h->node_tc;
    if (k == "comm_auto") return h->comm_auto;
    if (k == "caph_ready") return h->caph_ready ? 1 : 0;
    if (k == "caph_evals") {           // energy evaluations of the last refinement (synchronises)
        int v = 0;
        if (!h->caph_ready || cudaDeviceSynchronize() != cudaSuccess ||
            cudaMemcpy(&v, h->caph.evals_out, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) return VB_ERR_STATE;
        return v;
    }
    if (k == "comm_ready") return h->comm_ready ? 1 : 0;
    if (k == "restraints_ready") return h->rs_ready ? 1 : 0;
    if (k == "pme_ready") return h->pme_ready ? 1 : 0;
    if (k == "edge_overflow") {
        int flag = 0;
        if (h->d_flags && cudaMemcpy(&flag, h->d_flags, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) return VB_ERR_CUDA;
        return flag;
    }
    if (k == "timeline") return h->timeline;
    if (k == "tc_rows") return h->tc_rows;
    if (k == "tile_rows") return h->tile_rows;
    if (k == "n_edges_capacity") return h->ws.Ecap;
    return VB_ERR_ARG;
}

int vb_num_stages(const vb_handle* h) { return h ? (int)h->stage_names.size() : 0; }
const char* vb_stage_name(const vb_handle* h, int stage) {
    if (!h || stage < 0 || stage >= (int)h->stage_names.size()) return "";
    return h->stage_names[stage].c_str();
}

int vb_debug_run(vb_handle* h, const float* pos_dev, int n_stages) {
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (!h->has_topology || !pos_dev) { h->set_error("vb_debug_run: bad state/arguments"); return VB_ERR_STATE; }
    CUDA_TRY(h, cudaSetDevice(h->device));
    CUDA_TRY(h, cudaMemcpy(h->d_pos, pos_dev, sizeof(float) * 3 * h->ws.N, cudaMemcpyDeviceToDevice));
    if (h->accum_dirty) { if (int rc = clean_accumulators(h, h->own_stream)) return rc; }
    Launcher Lc{h, h->own_stream, n_stages, 0, false};
    enqueue_all(Lc, internal_io(h, h->n_protein > 0));
    if (Lc.status != cudaSuccess) { h->set_error("debug launch failed: %s", cudaGetErrorString(Lc.status)); return VB_ERR_CUDA; }
    CUDA_TRY(h, cudaStreamSynchronize(h->own_stream));
    h->accum_dirty = n_stages >= 0 && n_stages < (int)h->stage_names.size();   // a consumer stage may not have re-zeroed its accumulators
    return VB_OK;
}

int vb_profile_stages(vb_handle* h, const float* pos_dev, int n_iter, float* ms_per_stage_host) {
    if (!h) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (!h->has_topology || !pos_dev || !ms_per_stage_host || n_iter <= 0) { h->set_error("vb_profile_stages: bad state/arguments"); return VB_ERR_STATE; }
    CUDA_TRY(h, cudaSetDevice(h->device));
    const int ns = (int)h->stage_names.size();
    std::vector<cudaEvent_t> ev(ns + 1);
    for (auto& e : ev) CUDA_TRY(h, cudaEventCreate(&e));
    std::vector<double> acc(ns, 0.0);
    CUDA_TRY(h, cudaMemcpy(h->d_pos, pos_dev, sizeof(float) * 3 * h->ws.N, cudaMemcpyDeviceToDevice));
    int rc = VB_OK;
    for (int it = 0; it < n_iter + 1 && rc == VB_OK; it++) {      // iteration 0 is an untimed warm-up
        Launcher Lc{h, h->own_stream, -1, 0, false};
        Lc.events = &ev;
        enqueue_all(Lc, internal_io(h, h->n_protein > 0));
        cudaEventRecord(ev[ns], h->own_stream);
        if (Lc.status != cudaSuccess || cudaStreamSynchronize(h->own_stream) != cudaSuccess) {
            h->set_error("vb_profile_stages: launch failed: %s", cudaGetErrorString(cudaGetLastError()));
            rc = VB_ERR_CUDA;
            break;
        }
        if (it == 0) continue;
        for (int s = 0; s < ns; s++) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, ev[s], ev[s + 1]);
            acc[s] += ms;
        }
    }
    for (auto& e : ev) cudaEventDestroy(e);
    if (rc == VB_OK)
        for (int s = 0; s < ns; s++) ms_per_stage_host[s] = (float)(acc[s] / n_iter);
    return rc;
}

int vb_tc_selftest(int device, const float* a_host, const float* img_host, float* d_host, int reps, float* ms_out) {
    // D[128][128] = A[128][128] * W^T through the tcgen05/TMEM/TMA pipeline of the tensor-core edge kernels.
    if (!a_host || !img_host || !d_host || reps <= 0) return VB_ERR_ARG;
    if (cudaSetDevice(device) != cudaSuccess) { g_create_error = "vb_tc_selftest: cudaSetDevice failed"; return VB_ERR_CUDA; }
    float *dA = nullptr, *dI = nullptr, *dD = nullptr;
    const size_t nA = (size_t)TC_TE * D * sizeof(float), nI = (size_t)(D / tc::SLAB_K) * tc::STAGE_BYTES;
    cudaMalloc(&dA, nA); cudaMalloc(&dI, nI); cudaMalloc(&dD, nA);
    cudaMemcpy(dA, a_host, nA, cudaMemcpyHostToDevice);
    cudaMemcpy(dI, img_host, nI, cudaMemcpyHostToDevice);
    cudaMemset(dD, 0, nA);
    cudaFuncSetAttribute(tc_selftest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TC_SMEM_BYTES);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    cudaEventRecord(e0);
    tc_selftest_kernel<<<1, TC_THREADS, TC_SMEM_BYTES>>>(dA, dI, dD, reps);
    cudaEventRecord(e1);
    cudaError_t err = cudaDeviceSynchronize();
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    if (ms_out) *ms_out = ms;
    if (err == cudaSuccess) err = cudaMemcpy(d_host, dD, nA, cudaMemcpyDeviceToHost);
    cudaFree(dA); cudaFree(dI); cudaFree(dD);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (err != cudaSuccess) { g_create_error = std::string("vb_tc_selftest: ") + cudaGetErrorString(err); return VB_ERR_CUDA; }
    return VB_OK;
}

int64_t vb_debug_read(vb_handle* h, const char* name, int layer, void* host_dst, int64_t cap_bytes) {
    if (!h || !name || !host_dst) return VB_ERR_ARG;
    std::lock_guard<std::mutex> lk(h->mu);
    if (std::string(name) == "pme_terms") {              // needs no topology: the PME term stands on its own
        if (!h->pme_ready) { h->set_error("vb_debug_read: pme_terms: no PME term set"); return VB_ERR_STATE; }
        const int64_t bytes = std::min<int64_t>(cap_bytes, sizeof(double) * PT_N);
        if (cudaSetDevice(h->device) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess ||
            cudaMemcpy(host_dst, h->pme.terms, bytes, cudaMemcpyDeviceToHost) != cudaSuccess) {
            h->set_error("vb_debug_read: copy failed: %s", cudaGetErrorString(cudaGetLastError()));
            return VB_ERR_CUDA;
        }
        return bytes;
    }
    if (!h->has_topology) return VB_ERR_STATE;
    const Workspace& ws = h->ws;
    const size_t N = ws.N, E = ws.Ecap, G = ws.G;
    const void* src = nullptr;
    size_t bytes = 0;
    const std::string k(name);
    auto lay = [&](int hi) { return layer >= 0 && layer < hi; };
#define BUF(key, ptr, count, elt) if (k == key) { src = (ptr); bytes = (size_t)(count) * (elt); }
    if (k == "X" && lay(L + 1)) { src = ws.X[layer]; bytes = N * D * 4; }
    else if (k == "V" && lay(L + 1)) { src = ws.V[layer]; bytes = N * 3 * D * 4; }
    else if (k == "F" && lay(L)) { src = ws.F[layer]; bytes = E * D * 4; }
    else if (k == "VN" && lay(L)) { src = ws.VN[layer]; bytes = N * 3 * D * 4; }
    else if (k == "QKV" && lay(L)) { src = ws.QKV[layer]; bytes = N * 3 * D * 4; }
    else if (k == "V123" && lay(L)) { src = ws.V123[layer]; bytes = N * 9 * D * 4; }
    else if (k == "VDOT" && lay(L)) { src = ws.VDOT[layer]; bytes = N * D * 4; }
    else if (k == "TU" && lay(L)) { src = ws.TU[layer]; bytes = N * 6 * D * 4; }
    else if (k == "O" && lay(L)) { src = ws.O[layer]; bytes = N * 3 * D * 4; }
    else if (k == "P1" && lay(L)) { src = ws.P1[layer]; bytes = E * 3 * D * 4; }
    else if (k == "SP" && lay(L)) { src = ws.SP[layer]; bytes = E * 2 * D * 4; }
    else if (k == "ATT" && lay(L)) { src = ws.ATT[layer]; bytes = E * H * 4; }
    else if (k == "TL" && lay(2 * L) && h->d_tl) { src = h->d_tl + (size_t)layer * TC_TL_SLOTS; bytes = TC_TL_SLOTS * 8; }
    else if (k == "TLN" && lay(2 * L + 3) && h->d_tl) { src = h->d_tl + (size_t)2 * L * TC_TL_SLOTS + (size_t)layer * N2_TL_SLOTS; bytes = N2_TL_SLOTS * 8; }
    else BUF("XA", ws.XA, N * D, 4)
    else BUF("VA", ws.VA, N * 3 * D, 4)
    else BUF("GX", ws.GX, N * D, 4)
    else BUF("GVEC", ws.GVEC, N * 3 * D, 4)
    else BUF("GF", ws.GF, E * D, 4)
    else BUF("GXA", ws.GXA, N * D, 4)
    else BUF("GXA3", ws.GXA, 3 * N * D, 4)
    else BUF("GQKV", ws.GQKV, N * 3 * D, 4)
    else BUF("GVNMSG", ws.GVNMSG, N * 3 * D, 4)
    else BUF("GTU", ws.GTU, N * 6 * D, 4)
    else BUF("GQKV2", ws.GQKV2, N * 3 * D, 4)
    else BUF("GVNMSG2", ws.GVNMSG2, N * 3 * D, 4)
    else BUF("GTU2", ws.GTU2, N * 6 * D, 4)
    else BUF("geom", ws.geom, E * 8, 4)
    else BUF("rbf", ws.rbf, E * NR, 4)
    else BUF("eacc", ws.eacc, E * 4, 4)
    else BUF("grbf", ws.grbf, E * NR, 4)
    else BUF("esrc", ws.esrc, E, 4)
    else BUF("edst", ws.edst, E, 4)
    else BUF("rowptr", ws.rowptr, N + 1, 4)
    else BUF("eatom", ws.eatom, N, 4)
    else BUF("energy", h->d_energy, G, 4)
    else BUF("forces", h->d_forces, N * 3, 4)
#undef BUF
    if (!src) { h->set_error("vb_debug_read: unknown buffer %s[%d]", name, layer); return VB_ERR_ARG; }
    if ((int64_t)bytes > cap_bytes) bytes = (size_t)cap_bytes;
    if (cudaSetDevice(h->device) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess ||
        cudaMemcpy(host_dst, src, bytes, cudaMemcpyDeviceToHost) != cudaSuccess) {
        h->set_error("vb_debug_read: copy failed: %s", cudaGetErrorString(cudaGetLastError()));
        return VB_ERR_CUDA;
    }
    return (int64_t)bytes;
}

}  // extern "C"
