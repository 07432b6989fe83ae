// state.cu -- sampler state save / load (mq_state_size, mq_state_save, mq_state_load): checkpoint and resume bit for bit.
//
// What mq_step needs to continue a chain is in device memory only; a blob saved here holds all of it for the current
// buffer of every chain (DESIGN.md section 4c lists every member of Handle, SamplerDev, Ring and Posterior and where it
// goes).  pack_state_kernel gathers the current-buffer slices selected by mcur / ecur into one chain-major staging buffer;
// unpack_state_kernel scatters them into buffer 0.  The travel-time tables are not saved: they are a pure function of the
// current model, mq_state_load rebuilds them and compares a 64-bit hash of every (chain, phase) table with the hash the
// save stored (table_hash_kernel), so that a resumed chain is the same chain, not a statistically equivalent one.
// Host <-> device traffic is one copy per direction of the whole payload.
#include <stdio.h>
#include <string.h>

#include <vector>

#include "../../include/mcmceq_b200.h"
#include "chain.cuh"
#include "errors.h"
#include "forward.cuh"
#include "launch_count.h"
#include "sampler.cuh"
#include "state.h"

namespace mq {

// Scalars of one chain, at the start of its record; the float arrays follow (chain_floats).
struct ChainHead {
    double ll, rms, misfit, best_rms, best_snap_rms;
    int64_t acce, reject, best_number;
    uint64_t draws;
    int64_t counts[20];
    int32_t dim, best_dim, best_code, best_flag;
    float inv_control, pad;
    float mf[8], noise[8], best_noise[8];
};
static_assert(sizeof(ChainHead) % 8 == 0, "ChainHead");

// float arrays after the head: current state z vp vpvs [md], the same of the proposal buffer, eq [3ne], origin [ne],
// pres sres [ns], evsum [8ne], then the best-model snapshot z vp vpvs [md], eq [3ne], origin [ne], pres sres [ns].
// The proposal buffer of the model is not read by the sampler beyond what a proposal writes into it first, but a proposal
// writes only the nuclei of its model: the entries after them stay, and mq_get_models shows them.  With both buffers in
// the state a resumed handle shows the same arrays as the saved one, not only the same models.
__host__ __device__ inline size_t chain_floats(int md, int ne, int ns) { return 9 * (size_t)md + 16 * (size_t)ne + 4 * (size_t)ns; }
__host__ __device__ inline size_t chain_bytes(int md, int ne, int ns)
{
    return (sizeof(ChainHead) + chain_floats(md, ne, ns) * sizeof(float) + 7) / 8 * 8;
}

template <bool kPack>
__device__ __forceinline__ void move(float* rec, float* dev, int count)
{
    for (int i = threadIdx.x; i < count; i += blockDim.x) {
        if (kPack) rec[i] = dev[i];
        else dev[i] = rec[i];
    }
}

// One block per chain.  Pack: current buffers -> record.  Unpack: record -> buffer 0 (model proposal buffer -> 1), buffer
// indices 0, the evaluation view
// of the current state pointed at buffer 0 (what sync_cur_view writes), the chain's ring emptied.
template <bool kPack>
__device__ void state_chain(Handle& hd, SamplerDev& s, char* out, size_t rec_bytes)
{
    const int c = blockIdx.x, n = hd.n, md = hd.md, ne = hd.ne, ns = hd.ns;
    char* rec = out + (size_t)c * rec_bytes;
    ChainHead* H = (ChainHead*)rec;
    const int mc = kPack ? hd.mcur[c] : 0, ec = kPack ? hd.ecur[c] : 0;
    if (threadIdx.x == 0) {
        if (kPack) {
            H->ll = hd.ll[c]; H->rms = hd.rms[c]; H->misfit = hd.misfit[c];
            H->best_rms = s.best_rms[c]; H->best_snap_rms = s.best.rms[c];
            H->acce = s.acce[c]; H->reject = s.reject[c]; H->best_number = s.best.number[c]; H->draws = s.draws[c];
            H->dim = hd.dim[mc * n + c]; H->best_dim = s.best.dim[c]; H->best_code = s.best.code[c]; H->best_flag = s.best.flag[c];
            H->inv_control = s.inv_control[c]; H->pad = 0.f;
        } else {
            hd.ll[c] = H->ll; hd.rms[c] = H->rms; hd.misfit[c] = H->misfit;
            s.best_rms[c] = H->best_rms; s.best.rms[c] = H->best_snap_rms;
            s.acce[c] = H->acce; s.reject[c] = H->reject; s.best.number[c] = H->best_number; s.draws[c] = H->draws;
            hd.dim[c] = H->dim; s.best.dim[c] = H->best_dim; s.best.code[c] = H->best_code; s.best.flag[c] = H->best_flag;
            s.inv_control[c] = H->inv_control;
            hd.mcur[c] = 0; hd.tcur[2 * c] = 0; hd.tcur[2 * c + 1] = 0; hd.ecur[c] = 0;
            const EvalView& v = hd.cur_view;
            v.mbuf[c] = 0; v.tbuf[2 * c] = 0; v.tbuf[2 * c + 1] = 0; v.ebuf[c] = 0;
            v.q_idx[c] = -1; v.r_idx[c] = -1; v.ev_only[c] = -1;
            s.ring.wr[c] = 0; s.ring.rd[c] = 0; s.ring.lost[c] = 0; s.ring.pend[c] = 0;
        }
    }
    if (threadIdx.x < 20) {
        if (kPack) H->counts[threadIdx.x] = s.counts[20 * (size_t)c + threadIdx.x];
        else s.counts[20 * (size_t)c + threadIdx.x] = H->counts[threadIdx.x];
    }
    if (threadIdx.x < 8) {
        const size_t k = 8 * (size_t)c + threadIdx.x;
        if (kPack) { H->mf[threadIdx.x] = hd.mf[k]; H->noise[threadIdx.x] = hd.noise[k]; H->best_noise[threadIdx.x] = s.best.noise[k]; }
        else { hd.mf[k] = H->mf[threadIdx.x]; hd.noise[k] = H->noise[threadIdx.x]; s.best.noise[k] = H->best_noise[threadIdx.x]; }
    }
    float* f = (float*)(rec + sizeof(ChainHead));
    const size_t mo = ((size_t)mc * n + c) * md, eo = ((size_t)ec * n + c) * ne;
    move<kPack>(f, hd.z + mo, md); f += md;
    move<kPack>(f, hd.vp + mo, md); f += md;
    move<kPack>(f, hd.vpvs + mo, md); f += md;
    const size_t po = ((size_t)(1 - mc) * n + c) * md;
    move<kPack>(f, hd.z + po, md); f += md;
    move<kPack>(f, hd.vp + po, md); f += md;
    move<kPack>(f, hd.vpvs + po, md); f += md;
    move<kPack>(f, hd.eq + (size_t)c * ne * 3, 3 * ne); f += 3 * ne;
    move<kPack>(f, hd.origin + eo, ne); f += ne;
    move<kPack>(f, hd.pres + (size_t)c * ns, ns); f += ns;
    move<kPack>(f, hd.sres + (size_t)c * ns, ns); f += ns;
    move<kPack>(f, hd.evsum + eo * 8, 8 * ne); f += 8 * ne;
    const Snapshot& b = s.best;
    move<kPack>(f, b.z + (size_t)c * md, md); f += md;
    move<kPack>(f, b.vp + (size_t)c * md, md); f += md;
    move<kPack>(f, b.vpvs + (size_t)c * md, md); f += md;
    move<kPack>(f, b.eq + (size_t)c * ne * 3, 3 * ne); f += 3 * ne;
    move<kPack>(f, b.origin + (size_t)c * ne, ne); f += ne;
    move<kPack>(f, b.pres + (size_t)c * ns, ns); f += ns;
    move<kPack>(f, b.sres + (size_t)c * ns, ns);
}

__global__ void __launch_bounds__(128) pack_state_kernel(Handle hd, SamplerDev s, char* out, size_t rec_bytes)
{
    state_chain<true>(hd, s, out, rec_bytes);
}
__global__ void __launch_bounds__(128) unpack_state_kernel(Handle hd, SamplerDev s, char* in, size_t rec_bytes)
{
    state_chain<false>(hd, s, in, rec_bytes);
}

__host__ __device__ inline uint64_t splitmix64(uint64_t x)
{
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

// One block per (chain, phase): sum over the stored receiver rows (valid columns only, not the pitch padding) of
// splitmix64(position << 32 | float bits), position = (row * nz + source depth) * nxmod + column.  Order-independent, so
// the sum needs no fixed reduction order; any single changed value changes it.  tcur == nullptr: buffer 0.
__global__ void __launch_bounds__(256) table_hash_kernel(const float* tab, const int32_t* tcur, int n, size_t tab_stride, int n_rows,
                                                          int nz, int nxmod, int xp, uint64_t* out)
{
    const int item = blockIdx.x, c = item >> 1, ph = item & 1;
    const int tb = tcur ? tcur[item] : 0;
    const float* base = tab + (((size_t)tb * n + c) * 2 + ph) * tab_stride;
    const uint32_t count = (uint32_t)n_rows * (uint32_t)nz * (uint32_t)nxmod;
    uint64_t acc = 0;
    for (uint32_t j = threadIdx.x; j < count; j += blockDim.x) {
        const uint32_t line = j / (uint32_t)nxmod, i = j - line * (uint32_t)nxmod;
        acc += splitmix64(((uint64_t)j << 32) | __float_as_uint(base[(size_t)line * xp + i]));
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    __shared__ unsigned long long sum;
    if (threadIdx.x == 0) sum = 0;
    __syncthreads();
    if ((threadIdx.x & 31) == 0) atomicAdd(&sum, (unsigned long long)acc);
    __syncthreads();
    if (threadIdx.x == 0) out[item] = sum;
}

// ---- host side ------------------------------------------------------------------------------------------------
// sum64 (include/mcmceq_b200.h): h = (h ^ w) * 0x100000001B3, h ^= h >> 32 over the little-endian 64-bit words of the data,
// the last word zero-padded.  Each step is a bijection of h, so changing any one word always changes the result.
static uint64_t sum64(const void* data, size_t bytes, uint64_t h = 0x9E3779B97F4A7C15ull)
{
    const unsigned char* p = (const unsigned char*)data;
    size_t i = 0;
    for (; i + 8 <= bytes; i += 8) {
        uint64_t w;
        memcpy(&w, p + i, 8);
        h = (h ^ w) * 0x100000001B3ull;
        h ^= h >> 32;
    }
    if (i < bytes) {
        uint64_t w = 0;
        memcpy(&w, p + i, bytes - i);
        h = (h ^ w) * 0x100000001B3ull;
        h ^= h >> 32;
    }
    return h;
}

uint64_t config_checksum(const mq_config* cfg)
{
    mq_config c = *cfg;
    // bytes after a string's NUL are whatever the caller's buffer held: they do not count
    char* strs[3] = {c.dstring_start, c.dstring_main, c.inp_model_switch};
    const size_t caps[3] = {sizeof c.dstring_start, sizeof c.dstring_main, sizeof c.inp_model_switch};
    for (int k = 0; k < 3; k++) {
        const size_t len = strnlen(strs[k], caps[k]);
        if (len < caps[k]) memset(strs[k] + len, 0, caps[k] - len);
    }
    return sum64(&c, sizeof c);
}

uint64_t picks_checksum(const mq_picks* pk)
{
    const size_t ne = pk->n_events, np = pk->n_picks;
    const int32_t sizes[3] = {pk->n_events, pk->n_picks, pk->n_stations};
    uint64_t h = sum64(sizes, sizeof sizes);
    h = sum64(pk->ev_off, (ne + 1) * sizeof(int32_t), h);
    h = sum64(pk->n_p, ne * sizeof(int32_t), h);
    h = sum64(pk->st_id, np * sizeof(int32_t), h);
    h = sum64(pk->x, np * sizeof(float), h);
    h = sum64(pk->y, np * sizeof(float), h);
    h = sum64(pk->z, np * sizeof(float), h);
    h = sum64(pk->t, np * sizeof(float), h);
    h = sum64(pk->cls, np * sizeof(int32_t), h);
    const int32_t present[2] = {pk->reftime != nullptr, pk->fix != nullptr};
    h = sum64(present, sizeof present, h);
    if (pk->reftime) h = sum64(pk->reftime, ne * sizeof(double), h);
    if (pk->fix) h = sum64(pk->fix, 3 * ne * sizeof(double), h);
    return h;
}

namespace {

struct Plan {   // sizes and places of everything in a blob of this handle
    mq_state_header head;
    int n_sections;
    mq_state_section sec[6];
    size_t payload_off, payload_bytes, total_bytes;
    size_t rec_bytes;
    size_t chains_off, hash_off, post_off, post_int_bytes, beta_off, diag_off, hypo_off;   // offsets inside the payload (= the staging buffer)
};

// The diagnostics section: DiagHead, then ref [n][Q], sum [n][K][Q], sumsq [n][K][Q] (double), n_models [n] (int64),
// batch_len [n], full_batches [n] (int32).
struct DiagHead {
    int64_t burn_in;
    int32_t n_batches, n_quantities;
};
inline size_t diag_section_bytes(size_t n, size_t K, size_t Q)
{
    return sizeof(DiagHead) + (n * Q * (2 * K + 1)) * sizeof(double) + n * (sizeof(int64_t) + 2 * sizeof(int32_t));
}

inline size_t up8(size_t x) { return (x + 7) / 8 * 8; }

// The hypocentre section: HypoHead, then hist [ne][nb0 + nb1 + nb2] and outside [ne][3] (int32), zero padding to 8 bytes,
// ref [n][4][ne], sum [n][4][ne], cross [n][10][ne] (double), n_models [n] (int64).
struct HypoHead {
    int64_t burn_in;
    float bin_km;
    int32_t n_bins[3];
};
inline size_t hypo_int_bytes(size_t ne, const int nb[3]) { return up8(ne * ((size_t)nb[0] + nb[1] + nb[2] + 3) * sizeof(int32_t)); }
inline size_t hypo_section_bytes(size_t n, size_t ne, const int nb[3])
{
    return sizeof(HypoHead) + hypo_int_bytes(ne, nb) + n * ne * 18 * sizeof(double) + n * sizeof(int64_t);
}

bool has_tables(const Handle* h) { return h->cfg.eikonal == 1 && h->cfg.aflag != 1; }

// reciprocal tables are part of a state's identity only where tables exist
bool reciprocal_tables(const Handle* h) { return has_tables(h) && h->tables_mode == MQ_TABLES_RECIPROCAL; }

// the sections of a blob with the given options; the header's identity fields from the handle
void make_plan(const Handle* h, bool post, bool beta, bool tables, bool diag, bool hypo, Plan* P)
{
    memset(P, 0, sizeof *P);
    mq_state_header& H = P->head;
    memcpy(H.magic, MQ_STATE_MAGIC, sizeof H.magic);
    H.format = MQ_STATE_FORMAT;
    H.header_bytes = sizeof(mq_state_header);
    snprintf(H.version, sizeof H.version, "%s", mq_version());
    H.n_chains = h->n; H.max_dim = h->md; H.n_events = h->ne; H.n_stations = h->ns; H.n_picks = h->np;
    H.nz = h->nz; H.nxmod = h->nxmod; H.n_rows = h->n_rows;
    H.config_sum = config_checksum(&h->cfg);
    H.picks_sum = h->picks_sum;
    H.flags = (post ? MQ_STATE_POSTERIOR : 0) | (beta ? MQ_STATE_BETA : 0) | (tables ? MQ_STATE_TABLES : 0) | (diag ? MQ_STATE_DIAG : 0) |
              (tables && reciprocal_tables(h) ? MQ_STATE_RECIPROCAL : 0) | (hypo ? MQ_STATE_HYPO : 0);
    const size_t n = h->n;
    P->rec_bytes = chain_bytes(h->md, h->ne, h->ns);
    size_t off = 0;
    auto add = [&](uint32_t id, size_t bytes) {
        mq_state_section& s = P->sec[P->n_sections++];
        s.id = id; s.offset = off; s.bytes = bytes;
        const size_t at = off;
        off += up8(bytes);
        return at;
    };
    P->chains_off = add(MQ_STATE_SEC_CHAINS, n * P->rec_bytes);
    if (tables) P->hash_off = add(MQ_STATE_SEC_TABLES, 2 * n * sizeof(uint64_t));
    if (post) {
        const Posterior& Q = h->post;
        P->post_int_bytes = up8(Q.n_int * sizeof(int32_t));
        P->post_off = add(MQ_STATE_SEC_POSTERIOR, P->post_int_bytes + Q.n_dbl * sizeof(double));
    }
    if (beta) P->beta_off = add(MQ_STATE_SEC_BETA, n * sizeof(float));
    if (diag) P->diag_off = add(MQ_STATE_SEC_DIAG, diag_section_bytes(n, h->diag.K, h->diag.Q));
    if (hypo) P->hypo_off = add(MQ_STATE_SEC_HYPO, hypo_section_bytes(n, h->ne, h->hypo.nb));
    H.n_sections = P->n_sections;
    P->payload_off = sizeof(mq_state_header) + P->n_sections * sizeof(mq_state_section);
    P->payload_bytes = off;
    P->total_bytes = P->payload_off + off + sizeof(uint64_t);
    // section offsets in the blob are absolute
    for (int k = 0; k < P->n_sections; k++) P->sec[k].offset += P->payload_off;
}

void plan_of_handle(const Handle* h, Plan* P)
{
    make_plan(h, h->post.on != 0, h->beta != nullptr, has_tables(h), h->diag.on != 0, h->hypo.on != 0, P);
    mq_state_header& H = P->head;
    H.seed = h->seed;
    H.chain_offset = h->chain_offset;
    if (h->post.on) {
        H.post_dv = h->post.dv; H.post_dvpvs = h->post.dvpvs; H.post_ndv = h->post.ndv; H.post_ndvpvs = h->post.ndvpvs;
        H.post_burn_in = h->post.burn_in;
    }
}

struct DevBuf {   // device staging, freed on every path out
    void* p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
};

// the posterior block sizes of mq_posterior_begin for the given bin widths
void posterior_sizes(const Handle* h, float dv, float dvpvs, int* ndv, int* ndvpvs, size_t* n_int, size_t* n_dbl)
{
    *ndv = (int)((h->cfg.vpmax - h->cfg.vpmin) / dv) + 1;            // src/analyse_eq.c:427-430
    *ndvpvs = (int)((h->cfg.vpvsmax - h->cfg.vpvsmin) / dvpvs) + 1;
    *n_int = (size_t)(*ndv + *ndvpvs + 1) * h->nz;
    *n_dbl = 4 * (size_t)h->nz + 8 * (size_t)h->ne + 4 * (size_t)h->ns + 17;
}

bool any_batch_in_flight(const Sampler* s) { return s && (s->batch[0].state != 0 || s->batch[1].state != 0); }

}  // namespace
}  // namespace mq

using namespace mq;

extern "C" int mq_state_size(mq_handle* hh, uint64_t* bytes)
{
    if (!hh || !bytes) { set_error("mq_state_size: null"); return MQ_ERR_ARG; }
    Plan P;
    plan_of_handle(&hh->h, &P);
    *bytes = P.total_bytes;
    return MQ_OK;
}

extern "C" int mq_state_save(mq_handle* hh, void* buf, uint64_t cap, uint64_t* bytes)
{
    if (!hh) { set_error("mq_state_save: null"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    MQ_CUDA(cudaSetDevice(h->device));
    int rc = flags_poll(h, true);     // an error of an earlier asynchronous call comes first
    if (rc != MQ_OK) return rc;
    Sampler* s = (Sampler*)h->sampler;
    if (!h->models_set || !s || !s->started || !h->forward_done) {
        set_error("mq_state_save: no sampler state yet (mq_init_chains, or mq_set_models and a first mq_step)");
        return MQ_ERR_STATE;
    }
    if (any_batch_in_flight(s)) { set_error("mq_state_save: a drain batch is in flight (mq_batch_release it first)"); return MQ_ERR_BUSY; }
    Plan P;
    plan_of_handle(h, &P);
    if (bytes) *bytes = P.total_bytes;
    if (!buf || cap < P.total_bytes) {
        set_error("mq_state_save: buffer of %llu bytes, the state needs %llu (mq_state_size)", (unsigned long long)cap,
                  (unsigned long long)P.total_bytes);
        return MQ_ERR_ARG;
    }
    cudaStream_t st = h->stream;
    const size_t n = h->n;
    {
        // records are not state: a resumed run must not deliver one twice, so the caller drains first
        std::vector<int32_t> wr(n), rd(n), lost(n);
        MQ_CUDA(cudaMemcpyAsync(wr.data(), s->ring.wr, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        MQ_CUDA(cudaMemcpyAsync(rd.data(), s->ring.rd, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        MQ_CUDA(cudaMemcpyAsync(lost.data(), s->ring.lost, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        MQ_CUDA(cudaStreamSynchronize(st));
        for (size_t c = 0; c < n; c++)
            if (wr[c] != rd[c] || lost[c] != 0) {
                set_error("mq_state_save: chain %zu has undrained records (mq_drain first)", c);
                return MQ_ERR_STATE;
            }
    }
    DevBuf stage;
    MQ_CUDA(cudaMalloc(&stage.p, P.payload_bytes));
    char* d = (char*)stage.p;
    // the padding of records and sections is zero: the blob is a function of the state alone
    MQ_CUDA(cudaMemsetAsync(d, 0, P.payload_bytes, st));
    pack_state_kernel<<<h->n, 128, 0, st>>>(*h, s->dev(), d + P.chains_off, P.rec_bytes);
    count_launch();
    MQ_CUDA(cudaGetLastError());
    if (P.head.flags & MQ_STATE_TABLES) {
        table_hash_kernel<<<2 * h->n, 256, 0, st>>>(h->tab, h->tcur, h->n, h->tab_stride, h->n_rows, h->nz, h->nxmod, h->xp,
                                                     (uint64_t*)(d + P.hash_off));
        count_launch();
        MQ_CUDA(cudaGetLastError());
    }
    if (P.head.flags & MQ_STATE_POSTERIOR) {
        MQ_CUDA(cudaMemcpyAsync(d + P.post_off, h->post.iblock, h->post.n_int * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
        MQ_CUDA(cudaMemcpyAsync(d + P.post_off + P.post_int_bytes, h->post.dblock, h->post.n_dbl * sizeof(double), cudaMemcpyDeviceToDevice, st));
    }
    if (P.head.flags & MQ_STATE_BETA) MQ_CUDA(cudaMemcpyAsync(d + P.beta_off, h->beta, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (P.head.flags & MQ_STATE_DIAG) {
        const Diag& D = h->diag;
        const DiagHead dh = {(int64_t)D.burn_in, D.K, D.Q};
        const size_t nq = n * D.Q, nkq = nq * D.K;
        char* o = d + P.diag_off;
        MQ_CUDA(cudaMemcpyAsync(o, &dh, sizeof dh, cudaMemcpyHostToDevice, st)); o += sizeof dh;
        MQ_CUDA(cudaMemcpyAsync(o, D.ref, nq * sizeof(double), cudaMemcpyDeviceToDevice, st)); o += nq * sizeof(double);
        MQ_CUDA(cudaMemcpyAsync(o, D.sum, nkq * sizeof(double), cudaMemcpyDeviceToDevice, st)); o += nkq * sizeof(double);
        MQ_CUDA(cudaMemcpyAsync(o, D.sumsq, nkq * sizeof(double), cudaMemcpyDeviceToDevice, st)); o += nkq * sizeof(double);
        MQ_CUDA(cudaMemcpyAsync(o, D.n_models, n * sizeof(int64_t), cudaMemcpyDeviceToDevice, st)); o += n * sizeof(int64_t);
        MQ_CUDA(cudaMemcpyAsync(o, D.batch_len, n * sizeof(int32_t), cudaMemcpyDeviceToDevice, st)); o += n * sizeof(int32_t);
        MQ_CUDA(cudaMemcpyAsync(o, D.full_batches, n * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
        MQ_CUDA(cudaStreamSynchronize(st));   // dh is on this stack frame
    }
    if (P.head.flags & MQ_STATE_HYPO) {
        const Hypo& Y = h->hypo;
        const HypoHead yh = {(int64_t)Y.burn_in, Y.bin, {Y.nb[0], Y.nb[1], Y.nb[2]}};
        const size_t ne = h->ne, nh = ne * ((size_t)Y.nb[0] + Y.nb[1] + Y.nb[2]), nd = n * ne;
        char* o = d + P.hypo_off;
        MQ_CUDA(cudaMemcpyAsync(o, &yh, sizeof yh, cudaMemcpyHostToDevice, st)); o += sizeof yh;
        MQ_CUDA(cudaMemcpyAsync(o, Y.hist, nh * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
        MQ_CUDA(cudaMemcpyAsync(o + nh * sizeof(int32_t), Y.outside, ne * 3 * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
        o += hypo_int_bytes(ne, Y.nb);
        MQ_CUDA(cudaMemcpyAsync(o, Y.ref, 4 * nd * sizeof(double), cudaMemcpyDeviceToDevice, st)); o += 4 * nd * sizeof(double);
        MQ_CUDA(cudaMemcpyAsync(o, Y.sum, 4 * nd * sizeof(double), cudaMemcpyDeviceToDevice, st)); o += 4 * nd * sizeof(double);
        MQ_CUDA(cudaMemcpyAsync(o, Y.cross, 10 * nd * sizeof(double), cudaMemcpyDeviceToDevice, st)); o += 10 * nd * sizeof(double);
        MQ_CUDA(cudaMemcpyAsync(o, Y.n_models, n * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
        MQ_CUDA(cudaStreamSynchronize(st));   // yh is on this stack frame
    }
    char* out = (char*)buf;
    memcpy(out, &P.head, sizeof P.head);
    memcpy(out + sizeof P.head, P.sec, P.n_sections * sizeof(mq_state_section));
    MQ_CUDA(cudaMemcpyAsync(out + P.payload_off, d, P.payload_bytes, cudaMemcpyDeviceToHost, st));
    MQ_CUDA(cudaStreamSynchronize(st));
    const uint64_t sum = sum64(out, P.total_bytes - sizeof(uint64_t));
    memcpy(out + P.total_bytes - sizeof(uint64_t), &sum, sizeof sum);
    return check_device_errors(h);
}

extern "C" int mq_state_load(mq_handle* hh, const void* buf, uint64_t bytes)
{
    if (!hh || !buf) { set_error("mq_state_load: null"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    const char* in = (const char*)buf;
    // ---- everything is checked on the host before the first device write: a refused blob leaves the handle as it was
    mq_state_header H;
    if (bytes < sizeof H + sizeof(uint64_t)) { set_error("mq_state_load: %llu bytes is too short for a state", (unsigned long long)bytes); return MQ_ERR_ARG; }
    memcpy(&H, in, sizeof H);
    if (memcmp(H.magic, MQ_STATE_MAGIC, sizeof H.magic) != 0) { set_error("mq_state_load: not a sampler state (bad magic)"); return MQ_ERR_ARG; }
    if (H.format != MQ_STATE_FORMAT || H.header_bytes != sizeof H) {
        set_error("mq_state_load: state format %u (header %u bytes); this library reads format %u", H.format, H.header_bytes, MQ_STATE_FORMAT);
        return MQ_ERR_ARG;
    }
    {
        uint64_t stored;
        memcpy(&stored, in + bytes - sizeof stored, sizeof stored);
        if (sum64(in, bytes - sizeof stored) != stored) { set_error("mq_state_load: bad checksum (truncated or damaged state)"); return MQ_ERR_ARG; }
    }
    if (H.n_chains != h->n || H.max_dim != h->md || H.n_events != h->ne || H.n_stations != h->ns || H.n_picks != h->np ||
        H.nz != h->nz || H.nxmod != h->nxmod || H.n_rows != h->n_rows) {
        set_error("mq_state_load: state of %d chains x %d nuclei, %d events, %d stations, %d picks, plane %d x %d; the handle has "
                  "%d x %d, %d, %d, %d, %d x %d", H.n_chains, H.max_dim, H.n_events, H.n_stations, H.n_picks, H.nxmod, H.nz,
                  h->n, h->md, h->ne, h->ns, h->np, h->nxmod, h->nz);
        return MQ_ERR_ARG;
    }
    if (H.config_sum != config_checksum(&h->cfg)) { set_error("mq_state_load: the state was saved with another configuration"); return MQ_ERR_ARG; }
    if (H.picks_sum != h->picks_sum) { set_error("mq_state_load: the state was saved with other picks"); return MQ_ERR_ARG; }
    const bool post = (H.flags & MQ_STATE_POSTERIOR) != 0, beta = (H.flags & MQ_STATE_BETA) != 0, tables = (H.flags & MQ_STATE_TABLES) != 0;
    const bool diag = (H.flags & MQ_STATE_DIAG) != 0, hypo = (H.flags & MQ_STATE_HYPO) != 0;
    if ((H.flags & ~(uint32_t)(MQ_STATE_POSTERIOR | MQ_STATE_BETA | MQ_STATE_TABLES | MQ_STATE_DIAG | MQ_STATE_RECIPROCAL | MQ_STATE_HYPO)) ||
        tables != has_tables(h)) {
        set_error("mq_state_load: flags 0x%x do not fit the handle", H.flags);
        return MQ_ERR_ARG;
    }
    if (((H.flags & MQ_STATE_RECIPROCAL) != 0) != reciprocal_tables(h)) {
        set_error("mq_state_load: the state was saved with %s tables, the handle builds %s tables (mq_set_tables)",
                  (H.flags & MQ_STATE_RECIPROCAL) ? "reciprocal" : "parity", reciprocal_tables(h) ? "reciprocal" : "parity");
        return MQ_ERR_ARG;
    }
    int ndv = 0, ndvpvs = 0;
    size_t n_int = 0, n_dbl = 0;
    if (post) {
        if (!(H.post_dv > 0.f) || !(H.post_dvpvs > 0.f)) { set_error("mq_state_load: bad posterior bin widths"); return MQ_ERR_ARG; }
        posterior_sizes(h, H.post_dv, H.post_dvpvs, &ndv, &ndvpvs, &n_int, &n_dbl);
        if (ndv != H.post_ndv || ndvpvs != H.post_ndvpvs) { set_error("mq_state_load: posterior histogram sizes do not fit"); return MQ_ERR_ARG; }
    }
    // the diagnostics and hypocentre sections start with their own parameters, which must fit the handle (make_plan below
    // checks the whole section table)
    auto find_section = [&](uint32_t id) -> const mq_state_section* {
        const mq_state_section* sec = nullptr;
        if (H.n_sections <= 6 && sizeof H + H.n_sections * sizeof(mq_state_section) <= bytes)
            for (uint32_t k = 0; k < H.n_sections; k++) {
                const mq_state_section* e = (const mq_state_section*)(in + sizeof H + k * sizeof(mq_state_section));
                if (e->id == id) sec = e;
            }
        return sec;
    };
    DiagHead dh = {0, 0, 0};
    if (diag) {
        const mq_state_section* sec = find_section(MQ_STATE_SEC_DIAG);
        if (!sec || sec->bytes < sizeof dh || sec->offset > bytes - sizeof(uint64_t) || sec->bytes > bytes - sizeof(uint64_t) - sec->offset) {
            set_error("mq_state_load: flags 0x%x without a diagnostics section", H.flags);
            return MQ_ERR_ARG;
        }
        memcpy(&dh, in + sec->offset, sizeof dh);
        if (dh.burn_in < 0 || dh.n_batches < 8 || dh.n_batches > 64 || (dh.n_batches & 1) ||
            dh.n_quantities != diag_quantities(h->nz, h->ne, h->ns)) {
            set_error("mq_state_load: diagnostics of %d quantities x %d batches (burn-in %lld) do not fit the handle (%d quantities)",
                      dh.n_quantities, dh.n_batches, (long long)dh.burn_in, diag_quantities(h->nz, h->ne, h->ns));
            return MQ_ERR_ARG;
        }
    }
    // the hypocentre bin counts must be what the bin width gives on this handle's box
    HypoHead yh = {0, 0.f, {0, 0, 0}};
    if (hypo) {
        const mq_state_section* sec = find_section(MQ_STATE_SEC_HYPO);
        if (!sec || sec->bytes < sizeof yh || sec->offset > bytes - sizeof(uint64_t) || sec->bytes > bytes - sizeof(uint64_t) - sec->offset) {
            set_error("mq_state_load: flags 0x%x without a hypocentre section", H.flags);
            return MQ_ERR_ARG;
        }
        memcpy(&yh, in + sec->offset, sizeof yh);
        int nb[3] = {0, 0, 0};
        if (yh.burn_in < 0 || !(yh.bin_km > 0.f) || hypo_bins(h, yh.bin_km, nb) != 0 || nb[0] != yh.n_bins[0] ||
            nb[1] != yh.n_bins[1] || nb[2] != yh.n_bins[2]) {
            set_error("mq_state_load: hypocentre accumulators of bin width %g km, %d x %d x %d bins (burn-in %lld) do not fit the handle",
                      (double)yh.bin_km, yh.n_bins[0], yh.n_bins[1], yh.n_bins[2], (long long)yh.burn_in);
            return MQ_ERR_ARG;
        }
    }
    // the layout these options give must be the blob's, section by section
    Plan P;
    {
        Handle tmp = *h;                  // sizes of the posterior, diagnostics and hypocentre blocks as the state has them
        tmp.post.n_int = n_int; tmp.post.n_dbl = n_dbl;
        tmp.diag.K = dh.n_batches; tmp.diag.Q = dh.n_quantities;
        for (int a = 0; a < 3; a++) tmp.hypo.nb[a] = yh.n_bins[a];
        make_plan(&tmp, post, beta, tables, diag, hypo, &P);
    }
    if (bytes != P.total_bytes || H.n_sections != (uint32_t)P.n_sections ||
        memcmp(in + sizeof H, P.sec, P.n_sections * sizeof(mq_state_section)) != 0) {
        set_error("mq_state_load: layout of %llu bytes does not fit the handle (%llu expected)", (unsigned long long)bytes,
                  (unsigned long long)P.total_bytes);
        return MQ_ERR_ARG;
    }
    MQ_CUDA(cudaSetDevice(h->device));
    Sampler* s = (Sampler*)h->sampler;
    if (any_batch_in_flight(s)) { set_error("mq_state_load: a drain batch is in flight (mq_batch_release it first)"); return MQ_ERR_BUSY; }
    int rc = flags_poll(h, true);
    if (rc != MQ_OK) return rc;
    // ---- device side
    rc = sampler_get(h, &s);
    if (rc != MQ_OK) return rc;
    cudaStream_t st = h->stream;
    const size_t n = h->n;
    DevBuf stage, hashes;
    MQ_CUDA(cudaMalloc(&stage.p, P.payload_bytes));
    char* d = (char*)stage.p;
    MQ_CUDA(cudaMemcpyAsync(d, in + P.payload_off, P.payload_bytes, cudaMemcpyHostToDevice, st));
    if (post) {
        Posterior& Q = h->post;
        if (!Q.on || Q.n_int != n_int || Q.n_dbl != n_dbl) {
            cudaFree(Q.iblock); cudaFree(Q.dblock);
            Q.iblock = nullptr; Q.dblock = nullptr; Q.on = 0;
            MQ_CUDA(cudaMalloc((void**)&Q.iblock, n_int * sizeof(int32_t)));
            MQ_CUDA(cudaMalloc((void**)&Q.dblock, n_dbl * sizeof(double)));
        }
        Q.dv = H.post_dv; Q.dvpvs = H.post_dvpvs; Q.ndv = ndv; Q.ndvpvs = ndvpvs; Q.burn_in = H.post_burn_in;
        Q.n_int = n_int; Q.n_dbl = n_dbl;
        MQ_CUDA(cudaMemcpyAsync(Q.iblock, d + P.post_off, n_int * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
        MQ_CUDA(cudaMemcpyAsync(Q.dblock, d + P.post_off + P.post_int_bytes, n_dbl * sizeof(double), cudaMemcpyDeviceToDevice, st));
        Q.on = 1;
    } else if (h->post.on) {
        cudaStreamSynchronize(st);
        cudaFree(h->post.iblock); cudaFree(h->post.dblock);
        memset(&h->post, 0, sizeof h->post);
    }
    if (beta) {
        if (!h->beta) MQ_CUDA(cudaMalloc((void**)&h->beta, n * sizeof(float)));
        MQ_CUDA(cudaMemcpyAsync(h->beta, d + P.beta_off, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
    } else if (h->beta) {
        cudaStreamSynchronize(st);
        cudaFree(h->beta);
        h->beta = nullptr;
    }
    if (diag) {
        Diag& D = h->diag;
        if (!D.on || D.K != dh.n_batches) {
            MQ_CUDA(cudaStreamSynchronize(st));
            rc = diag_alloc(h, dh.n_batches, dh.burn_in);
            if (rc != MQ_OK) return rc;
        }
        D.burn_in = dh.burn_in;
        const size_t nq = n * D.Q, nkq = nq * D.K;
        const char* o = d + P.diag_off + sizeof dh;
        MQ_CUDA(cudaMemcpyAsync(D.ref, o, nq * sizeof(double), cudaMemcpyDeviceToDevice, st)); o += nq * sizeof(double);
        MQ_CUDA(cudaMemcpyAsync(D.sum, o, nkq * sizeof(double), cudaMemcpyDeviceToDevice, st)); o += nkq * sizeof(double);
        MQ_CUDA(cudaMemcpyAsync(D.sumsq, o, nkq * sizeof(double), cudaMemcpyDeviceToDevice, st)); o += nkq * sizeof(double);
        MQ_CUDA(cudaMemcpyAsync(D.n_models, o, n * sizeof(int64_t), cudaMemcpyDeviceToDevice, st)); o += n * sizeof(int64_t);
        MQ_CUDA(cudaMemcpyAsync(D.batch_len, o, n * sizeof(int32_t), cudaMemcpyDeviceToDevice, st)); o += n * sizeof(int32_t);
        MQ_CUDA(cudaMemcpyAsync(D.full_batches, o, n * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
    } else if (h->diag.on) {
        diag_destroy(h);
    }
    if (hypo) {
        Hypo& Y = h->hypo;
        if (!Y.on || Y.bin != yh.bin_km) {
            MQ_CUDA(cudaStreamSynchronize(st));
            rc = hypo_alloc(h, yh.bin_km, yh.burn_in);
            if (rc != MQ_OK) return rc;
        }
        Y.burn_in = yh.burn_in;
        const size_t ne = h->ne, nh = ne * ((size_t)Y.nb[0] + Y.nb[1] + Y.nb[2]), nd = n * ne;
        const char* o = d + P.hypo_off + sizeof yh;
        MQ_CUDA(cudaMemcpyAsync(Y.hist, o, nh * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
        MQ_CUDA(cudaMemcpyAsync(Y.outside, o + nh * sizeof(int32_t), ne * 3 * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
        o += hypo_int_bytes(ne, Y.nb);
        MQ_CUDA(cudaMemcpyAsync(Y.ref, o, 4 * nd * sizeof(double), cudaMemcpyDeviceToDevice, st)); o += 4 * nd * sizeof(double);
        MQ_CUDA(cudaMemcpyAsync(Y.sum, o, 4 * nd * sizeof(double), cudaMemcpyDeviceToDevice, st)); o += 4 * nd * sizeof(double);
        MQ_CUDA(cudaMemcpyAsync(Y.cross, o, 10 * nd * sizeof(double), cudaMemcpyDeviceToDevice, st)); o += 10 * nd * sizeof(double);
        MQ_CUDA(cudaMemcpyAsync(Y.n_models, o, n * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
    } else if (h->hypo.on) {
        hypo_destroy(h);
    }
    h->seed = H.seed;
    h->chain_offset = H.chain_offset;
    unpack_state_kernel<<<h->n, 128, 0, st>>>(*h, s->dev(), d + P.chains_off, P.rec_bytes);
    count_launch();
    MQ_CUDA(cudaGetLastError());
    h->models_set = true;
    h->forward_done = true;
    s->started = true;      // mq_step must not score the chains again nor reset the best models (start_sampler_state)
    if (!tables) { MQ_CUDA(cudaStreamSynchronize(st)); return check_device_errors(h); }
    // ---- the tables of every chain into buffer 0, as mq_forward builds them, and their hashes against the stored ones
    MQ_CUDA(launch_build_items_all(h, h->cur_view, 3));
    MQ_CUDA(launch_rasterise(h, h->cur_view, 2 * h->n));
    MQ_CUDA(launch_tables(h, 2 * h->n));
    MQ_CUDA(cudaMalloc(&hashes.p, 2 * n * sizeof(uint64_t)));
    table_hash_kernel<<<2 * h->n, 256, 0, st>>>(h->tab, nullptr, h->n, h->tab_stride, h->n_rows, h->nz, h->nxmod, h->xp,
                                                 (uint64_t*)hashes.p);
    count_launch();
    MQ_CUDA(cudaGetLastError());
    std::vector<uint64_t> got(2 * n), want(2 * n);
    MQ_CUDA(cudaMemcpyAsync(got.data(), hashes.p, 2 * n * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    MQ_CUDA(cudaStreamSynchronize(st));
    rc = check_device_errors(h);
    if (rc != MQ_OK) return rc;
    memcpy(want.data(), in + P.payload_off + P.hash_off, 2 * n * sizeof(uint64_t));
    for (size_t k = 0; k < 2 * n; k++)
        if (got[k] != want[k]) {
            // the handle holds the state but not its tables: it must not step on them
            h->models_set = false;
            h->forward_done = false;
            s->started = false;
            set_error("mq_state_load: the rebuilt %s table of chain %zu differs from the saved one (hash %016llx, saved %016llx)",
                      (k & 1) ? "S" : "P", k >> 1, (unsigned long long)got[k], (unsigned long long)want[k]);
            return MQ_ERR_STATE;
        }
    return MQ_OK;
}
