// host_pipeline.cu -- nvb_pipeline: host buffers in, host buffers out, `depth` batches in flight.
//
// The reference hands batches from an input thread to one compute thread per device and synchronises the device after every
// stage (nvBowtie/bowtie2/cuda/compute_thread.cu:213-243, defs.h:64 optional_device_synchronize, aligner_best_approx.h:219-241).
// Here a batch is three stream-ordered steps -- H2D copy, nvb_seed_extend[_paired], D2H copy -- on a copy-in stream, the
// slot's own compute stream and a copy-out stream, chained by events; nothing blocks the host until wait().  Consecutive
// batches use different compute streams, so their kernels may share the SMs (the seed search leaves the integer pipes
// half idle, the extension leaves DRAM idle).
#include "pipeline_core.cuh"
#include <cstdlib>
#include <new>
#include <vector>

using namespace nvb;

struct nvb_pipeline {
    int device;
    nvb_fm_index fmi; const uint32_t* d_genome; nvb_seed_extend_params params; nvb_pair_params pair; bool paired;
    uint32_t n_reads, read_len, wpr, bits, hit_capacity, depth;
    uint32_t n_compute;                 // compute streams shared round-robin by the slots (NVB_PIPELINE_COMPUTE_STREAMS, default 1)
    cudaStream_t compute[16];
    cudaStream_t h2d, d2h;
    struct Slot {
        cudaStream_t compute;
        uint32_t* d_in; void* d_temp; size_t temp_bytes;
        // device results (one allocation) and their pinned host mirror, same layout
        char *d_out, *h_out; size_t out_bytes;
        cudaEvent_t ev_in, ev_start, ev_done, ev_out;
        bool busy;
    };
    std::vector<Slot> slots;
    uint64_t next;
    // offsets into the out block
    size_t o_score, o_pos, o_nhits, o_pscore, o_pflags, o_mscore, o_mpos, o_mstrand, o_nrescue;
};

static void layout(nvb_pipeline* p, size_t* total)
{
    size_t off = 0;
    auto take = [&](size_t bytes) { off = align_up(off, 256); const size_t o = off; off += bytes; return o; };
    const size_t n = p->n_reads;
    p->o_nhits = take(4 * sizeof(uint32_t));
    if (!p->paired) { p->o_score = take(n * sizeof(int32_t)); p->o_pos = take(n * sizeof(uint32_t)); }
    else {
        p->o_pscore = take(n / 2 * sizeof(int32_t)); p->o_pflags = take(n / 2 * sizeof(uint32_t));
        p->o_mscore = take(n * sizeof(int32_t)); p->o_mpos = take(n * sizeof(uint32_t)); p->o_mstrand = take(n);
        p->o_nrescue = take(2 * sizeof(uint32_t));
    }
    *total = align_up(off, 256);
}

static nvb_string_set reads_view(const nvb_pipeline* p, const uint32_t* d_words)
{
    nvb_string_set r;
    r.d_words = d_words; r.bits = p->bits; r.big_endian = 1; r.d_offsets = nullptr; r.d_lengths = nullptr;
    r.stride = p->wpr * (32u / p->bits); r.length = p->read_len;
    return r;
}

// batches of one device may run at once: they record no stage events (the slot's ev_start / ev_done time the batch)
static int run_batch(nvb_pipeline* p, nvb_pipeline::Slot& s, size_t* temp_bytes, void* d_temp)
{
    const nvb_string_set rs = reads_view(p, s.d_in ? s.d_in : (const uint32_t*)16);
    char* o = s.d_out;
    if (!p->paired)
        return seed_extend_impl(&p->fmi, p->d_genome, &rs, p->n_reads, &p->params, p->hit_capacity,
                                o ? (int32_t*)(o + p->o_score) : (int32_t*)16, o ? (uint32_t*)(o + p->o_pos) : (uint32_t*)16,
                                o ? (uint32_t*)(o + p->o_nhits) : nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
                                d_temp, temp_bytes, s.compute, false);
    nvb_pair_out po;
    po.d_pair_score = (int32_t*)(o + p->o_pscore); po.d_pair_flags = (uint32_t*)(o + p->o_pflags);
    po.d_mate_score = (int32_t*)(o + p->o_mscore); po.d_mate_pos = (uint32_t*)(o + p->o_mpos); po.d_mate_strand = (uint8_t*)(o + p->o_mstrand);
    po.d_n_rescue = (uint32_t*)(o + p->o_nrescue);
    // as in nvb_seed_extend_paired: the single-end stage writes the per-read bests into the mate arrays
    return seed_extend_impl(&p->fmi, p->d_genome, &rs, p->n_reads, &p->params, p->hit_capacity, po.d_mate_score, po.d_mate_pos,
                            (uint32_t*)(o + p->o_nhits), nullptr, nullptr, nullptr, nullptr, nullptr, &p->pair, &po,
                            d_temp, temp_bytes, s.compute, false);
}

extern "C" void nvb_pipeline_destroy(nvb_pipeline* p)
{
    if (!p) return;
    int prev = 0; cudaGetDevice(&prev); cudaSetDevice(p->device);
    for (auto& s : p->slots) {
        if (s.compute) cudaStreamSynchronize(s.compute);
        if (s.d_in) cudaFree(s.d_in);
        if (s.d_temp) cudaFree(s.d_temp);
        if (s.d_out) cudaFree(s.d_out);
        if (s.h_out) cudaFreeHost(s.h_out);
        if (s.ev_in) cudaEventDestroy(s.ev_in);
        if (s.ev_start) cudaEventDestroy(s.ev_start);
        if (s.ev_done) cudaEventDestroy(s.ev_done);
        if (s.ev_out) cudaEventDestroy(s.ev_out);
    }
    for (uint32_t i = 0; i < p->n_compute; ++i) if (p->compute[i]) cudaStreamDestroy(p->compute[i]);
    if (p->h2d) cudaStreamDestroy(p->h2d);
    if (p->d2h) cudaStreamDestroy(p->d2h);
    cudaSetDevice(prev);
    delete p;
}

extern "C" int nvb_pipeline_create(const nvb_fm_index* fmi, const uint32_t* d_genome, const nvb_seed_extend_params* params,
                                   const nvb_pair_params* pair_params,
                                   uint32_t n_reads, uint32_t read_len, uint32_t words_per_read, uint32_t read_bits,
                                   uint32_t hit_capacity, uint32_t depth, nvb_pipeline** out)
{
    if (!fmi || !d_genome || !params || !out || n_reads == 0 || depth == 0 || depth > 16) return NVB_E_INVALID;
    if (!(read_bits == 2 || read_bits == 4) || (uint64_t)words_per_read * (32u / read_bits) < read_len) return NVB_E_INVALID;
    if (pair_params && (n_reads & 1u)) return NVB_E_INVALID;
    nvb_pipeline* p = new (std::nothrow) nvb_pipeline();
    if (!p) return (int)cudaErrorMemoryAllocation;
    *out = nullptr;
    p->fmi = *fmi; p->d_genome = d_genome; p->params = *params; p->paired = pair_params != nullptr;
    if (pair_params) p->pair = *pair_params;
    p->n_reads = n_reads; p->read_len = read_len; p->wpr = words_per_read; p->bits = read_bits; p->hit_capacity = hit_capacity; p->depth = depth;
    p->h2d = p->d2h = nullptr; p->next = 0;
    p->n_compute = 1;
    if (const char* e = getenv("NVB_PIPELINE_COMPUTE_STREAMS")) { const int v = atoi(e); if (v >= 1) p->n_compute = (uint32_t)v; }
    if (p->n_compute > depth) p->n_compute = depth;
    for (int i = 0; i < 16; ++i) p->compute[i] = nullptr;
    int rc = NVB_OK;
#define PIPE_TRY(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) { rc = (int)_e; goto fail; } } while (0)
    {
        PIPE_TRY(cudaGetDevice(&p->device));
        size_t out_bytes = 0; layout(p, &out_bytes);
        PIPE_TRY(cudaStreamCreateWithFlags(&p->h2d, cudaStreamNonBlocking));
        PIPE_TRY(cudaStreamCreateWithFlags(&p->d2h, cudaStreamNonBlocking));
        for (uint32_t i = 0; i < p->n_compute; ++i) PIPE_TRY(cudaStreamCreateWithFlags(&p->compute[i], cudaStreamNonBlocking));
        p->slots.resize(depth);
        for (auto& s : p->slots) { s = nvb_pipeline::Slot(); }
        uint32_t k = 0;
        for (auto& s : p->slots) {
            s.out_bytes = out_bytes; s.busy = false;
            s.compute = p->compute[k++ % p->n_compute];
            PIPE_TRY(cudaMalloc((void**)&s.d_in, (size_t)n_reads * words_per_read * sizeof(uint32_t) + 64));
            PIPE_TRY(cudaMalloc((void**)&s.d_out, out_bytes));
            PIPE_TRY(cudaHostAlloc((void**)&s.h_out, out_bytes, cudaHostAllocDefault));
            PIPE_TRY(cudaMemset(s.d_out, 0, out_bytes));
            PIPE_TRY(cudaEventCreateWithFlags(&s.ev_in, cudaEventDisableTiming));
            PIPE_TRY(cudaEventCreate(&s.ev_start));
            PIPE_TRY(cudaEventCreate(&s.ev_done));
            PIPE_TRY(cudaEventCreateWithFlags(&s.ev_out, cudaEventDisableTiming));
            size_t tb = 0;
            const int r = run_batch(p, s, &tb, nullptr);
            if (r != NVB_E_TEMP_SIZE) { rc = (r == NVB_OK) ? NVB_E_INVALID : r; goto fail; }
            s.temp_bytes = tb;
            PIPE_TRY(cudaMalloc(&s.d_temp, tb));
        }
    }
#undef PIPE_TRY
    *out = p;
    return NVB_OK;
fail:
    nvb_pipeline_destroy(p);
    return rc;
}

extern "C" int nvb_pipeline_submit(nvb_pipeline* p, const uint32_t* h_read_words, uint32_t* ticket)
{
    if (!p || !h_read_words || !ticket) return NVB_E_INVALID;
    const uint32_t k = (uint32_t)(p->next % p->depth);
    nvb_pipeline::Slot& s = p->slots[k];
    if (s.busy) NVB_CUDA_TRY(cudaEventSynchronize(s.ev_out));        // the slot's previous results must have left the device
    // copy-in must not overwrite reads that the slot's previous kernels may still be reading
    NVB_CUDA_TRY(cudaStreamWaitEvent(p->h2d, s.ev_done, 0));
    NVB_CUDA_TRY(cudaMemcpyAsync(s.d_in, h_read_words, (size_t)p->n_reads * p->wpr * sizeof(uint32_t), cudaMemcpyHostToDevice, p->h2d));
    NVB_CUDA_TRY(cudaEventRecord(s.ev_in, p->h2d));
    NVB_CUDA_TRY(cudaStreamWaitEvent(s.compute, s.ev_in, 0));
    NVB_CUDA_TRY(cudaStreamWaitEvent(s.compute, s.ev_out, 0));       // ... nor may the kernels overwrite results still being copied out
    NVB_CUDA_TRY(cudaEventRecord(s.ev_start, s.compute));
    size_t tb = s.temp_bytes;
    const int r = run_batch(p, s, &tb, s.d_temp);
    if (r != NVB_OK) return r;
    NVB_CUDA_TRY(cudaEventRecord(s.ev_done, s.compute));
    NVB_CUDA_TRY(cudaStreamWaitEvent(p->d2h, s.ev_done, 0));
    NVB_CUDA_TRY(cudaMemcpyAsync(s.h_out, s.d_out, s.out_bytes, cudaMemcpyDeviceToHost, p->d2h));
    NVB_CUDA_TRY(cudaEventRecord(s.ev_out, p->d2h));
    s.busy = true;
    *ticket = k;
    ++p->next;
    return NVB_OK;
}

extern "C" int nvb_pipeline_wait(nvb_pipeline* p, uint32_t ticket, nvb_pipeline_result* out)
{
    if (!p || ticket >= p->depth || !out) return NVB_E_INVALID;
    nvb_pipeline::Slot& s = p->slots[ticket];
    if (p->next == 0) return NVB_E_INVALID;                         // nothing was ever submitted
    if (s.busy) NVB_CUDA_TRY(cudaEventSynchronize(s.ev_out));       // (waiting twice for the same ticket returns the same buffers)
    s.busy = false;
    nvb_pipeline_result r = {};
    const char* h = s.h_out;
    r.n_hits = (const uint32_t*)(h + p->o_nhits);
    if (!p->paired) { r.best_score = (const int32_t*)(h + p->o_score); r.best_pos = (const uint32_t*)(h + p->o_pos); }
    else {
        r.pair_score = (const int32_t*)(h + p->o_pscore); r.pair_flags = (const uint32_t*)(h + p->o_pflags);
        r.mate_score = (const int32_t*)(h + p->o_mscore); r.mate_pos = (const uint32_t*)(h + p->o_mpos); r.mate_strand = (const uint8_t*)(h + p->o_mstrand);
        r.n_rescue = (const uint32_t*)(h + p->o_nrescue);
    }
    NVB_CUDA_TRY(cudaEventElapsedTime(&r.device_ms, s.ev_start, s.ev_done));
    *out = r;
    return NVB_OK;
}

extern "C" void nvb_pipeline_traffic(const nvb_pipeline* p, size_t* h2d_bytes, size_t* d2h_bytes)
{
    if (!p) return;
    if (h2d_bytes) *h2d_bytes = (size_t)p->n_reads * p->wpr * sizeof(uint32_t);
    if (d2h_bytes) *d2h_bytes = p->slots.empty() ? 0 : p->slots[0].out_bytes;
}
