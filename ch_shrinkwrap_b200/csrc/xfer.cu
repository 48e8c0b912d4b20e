// Host -> device staging for the large inputs of the C ABI (localisations, sigma, vertex records, faces).
//
// Callers hand over ordinary pageable numpy memory.  A plain cudaMemcpyAsync from pageable memory is staged by the
// driver on one thread (measured here: 6-7 GB/s, which made the uploads the largest part of an end-to-end block
// after the kernels).  nw_h2d splits the source over a few host threads; every thread copies its range through two
// pinned 4 MB buffers of its own and issues the DMA on its own stream, so the host memcpy of one piece overlaps the DMA of
// the previous one and the lanes add up to PCIe rate.  On return the source has been read completely (the caller may
// free it) and the handle's stream waits for every lane.
#include <thread>
#include <vector>
#include <cstring>
#include <algorithm>
#include "common.cuh"

struct UploadLane {
    cudaStream_t s = nullptr;
    char *buf[2] = {nullptr, nullptr};
    cudaEvent_t ev[2] = {nullptr, nullptr};
    bool used[2] = {false, false};
    cudaError_t err = cudaSuccess;
    int last = -1;
};
struct nw_uploader {
    std::vector<UploadLane> lanes;
    size_t chunk = (size_t)4 << 20;
    cudaEvent_t ev_start = nullptr;
};

static int uploader_init(nw_ctx *h) {
    if (h->uploader) return NW_OK;
    const int n = (int)std::min(8u, std::max(1u, std::thread::hardware_concurrency() / 2));
    nw_uploader *u = new nw_uploader;
    u->lanes.resize(n);
    h->uploader = u;                      // owned by the handle from here on (nw_uploader_destroy releases partial state)
    NW_CUDA(cudaEventCreateWithFlags(&u->ev_start, cudaEventDisableTiming));
    for (auto &l : u->lanes) {
        NW_CUDA(cudaStreamCreateWithFlags(&l.s, cudaStreamNonBlocking));
        for (int k = 0; k < 2; ++k) {
            NW_CUDA(cudaHostAlloc((void **)&l.buf[k], u->chunk, cudaHostAllocDefault));
            NW_CUDA(cudaEventCreateWithFlags(&l.ev[k], cudaEventDisableTiming));
        }
    }
    return NW_OK;
}

void nw_uploader_destroy(nw_ctx *h) {
    nw_uploader *u = h->uploader;
    if (!u) return;
    for (auto &l : u->lanes) {
        if (l.s) { cudaStreamSynchronize(l.s); cudaStreamDestroy(l.s); }
        for (int k = 0; k < 2; ++k) {
            if (l.buf[k]) cudaFreeHost(l.buf[k]);
            if (l.ev[k]) cudaEventDestroy(l.ev[k]);
        }
    }
    if (u->ev_start) cudaEventDestroy(u->ev_start);
    delete u;
    h->uploader = nullptr;
}

// stride == 4: plain copy; otherwise gather one int32 every `stride` bytes of the source (a field of packed records)
static inline void stage_piece(char *buf, const char *src, size_t off, size_t n, size_t stride) {
    if (stride == 4) { memcpy(buf, src + off, n); return; }
    int32_t *o = (int32_t *)buf;
    const char *p = src + (off / 4) * stride;
    const size_t cnt = n / 4, ahead = 24 * stride;            // one field per record: every element is its own cache line or nearly so
    for (size_t i = 0; i < cnt; ++i, p += stride) {
        __builtin_prefetch(p + ahead, 0, 0);
        memcpy(&o[i], p, 4);
    }
}

static void lane_copy(int device, nw_uploader *u, UploadLane *l, char *dst, const char *src, size_t off0, size_t bytes, size_t stride) {
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(l->s, u->ev_start, 0);
    int k = 0;
    for (size_t off = 0; off < bytes && e == cudaSuccess; off += u->chunk, k ^= 1) {
        const size_t n = std::min(u->chunk, bytes - off);
        if (l->used[k]) { e = cudaEventSynchronize(l->ev[k]); if (e != cudaSuccess) break; }   // DMA out of this buffer finished
        stage_piece(l->buf[k], src, off0 + off, n, stride);
        e = cudaMemcpyAsync(dst + off0 + off, l->buf[k], n, cudaMemcpyHostToDevice, l->s);
        if (e == cudaSuccess) e = cudaEventRecord(l->ev[k], l->s);
        l->used[k] = true;
        l->last = k;
    }
    l->err = e;
}

int nw_h2d(nw_ctx *h, void *dst, const void *src, size_t bytes) { return nw_h2d_strided32(h, dst, src, bytes, 4); }

// Several arrays in one go: their 4 MB pieces are dealt round-robin to the lanes, one thread team, one join -- a topology
// upload is three arrays (half-edge vertex field, faces, vertex records) and used to pay three spawn/join rounds with the
// lanes idle in between (measured at C3: 5.4 ms of host time for 80 MB).
struct Piece { char *dst; const char *src; size_t off, n, stride; };
static void lane_pieces(int device, nw_uploader *u, UploadLane *l, const std::vector<Piece> *pieces, int first, int step) {
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(l->s, u->ev_start, 0);
    int k = 0;
    for (size_t q = (size_t)first; q < pieces->size() && e == cudaSuccess; q += (size_t)step, k ^= 1) {
        const Piece &pc = (*pieces)[q];
        if (l->used[k]) { e = cudaEventSynchronize(l->ev[k]); if (e != cudaSuccess) break; }
        stage_piece(l->buf[k], pc.src, pc.off, pc.n, pc.stride);
        e = cudaMemcpyAsync(pc.dst + pc.off, l->buf[k], pc.n, cudaMemcpyHostToDevice, l->s);
        if (e == cudaSuccess) e = cudaEventRecord(l->ev[k], l->s);
        l->used[k] = true;
        l->last = k;
    }
    l->err = e;
}

int nw_h2d_many(nw_ctx *h, const nw_h2d_job *jobs, int n_jobs) {
    size_t total = 0;
    for (int j = 0; j < n_jobs; ++j) total += jobs[j].bytes;
    if (total == 0) return NW_OK;
    if (total < ((size_t)2 << 20)) {
        for (int j = 0; j < n_jobs; ++j) NW_CHECK(nw_h2d_strided32(h, jobs[j].dst, jobs[j].src, jobs[j].bytes, jobs[j].stride));
        return NW_OK;
    }
    NW_CHECK(uploader_init(h));
    nw_uploader *u = h->uploader;
    NW_CUDA(cudaEventRecord(u->ev_start, h->stream));
    std::vector<Piece> pieces;
    for (int j = 0; j < n_jobs; ++j)
        for (size_t off = 0; off < jobs[j].bytes; off += u->chunk)
            pieces.push_back({(char *)jobs[j].dst, (const char *)jobs[j].src, off, std::min(u->chunk, jobs[j].bytes - off), jobs[j].stride});
    const int n_lanes = (int)std::min<size_t>(u->lanes.size(), pieces.size());
    std::vector<std::thread> th;
    for (int t = 0; t < n_lanes; ++t) { u->lanes[t].err = cudaSuccess; u->lanes[t].last = -1; }
    for (int t = 0; t + 1 < n_lanes; ++t) th.emplace_back(lane_pieces, h->device, u, &u->lanes[t], &pieces, t, n_lanes);
    lane_pieces(h->device, u, &u->lanes[n_lanes - 1], &pieces, n_lanes - 1, n_lanes);       // the caller's thread takes a lane too
    for (auto &t : th) t.join();
    for (int t = 0; t < n_lanes; ++t) {
        UploadLane &l = u->lanes[t];
        if (l.err != cudaSuccess) { h->err = std::string("nw_h2d_many: ") + cudaGetErrorString(l.err); return NW_ERR_CUDA; }
        if (l.last >= 0) NW_CUDA(cudaStreamWaitEvent(h->stream, l.ev[l.last], 0));
    }
    return NW_OK;
}

// dst: device pointer; src: any host memory; `bytes` = bytes written to dst (a multiple of 4 when stride != 4).  Ordered
// after everything already enqueued on h->stream; h->stream waits for the copy.  Small packed transfers take the direct path.
int nw_h2d_strided32(nw_ctx *h, void *dst, const void *src, size_t bytes, size_t stride) {
    if (bytes == 0) return NW_OK;
    if (stride == 4 && bytes < ((size_t)2 << 20)) {
        NW_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, h->stream));
        return NW_OK;
    }
    NW_CHECK(uploader_init(h));
    nw_uploader *u = h->uploader;
    NW_CUDA(cudaEventRecord(u->ev_start, h->stream));
    const size_t n_chunks = (bytes + u->chunk - 1) / u->chunk;
    const int n_lanes = (int)std::min<size_t>(u->lanes.size(), n_chunks);
    const size_t per = ((n_chunks + n_lanes - 1) / n_lanes) * u->chunk;
    std::vector<std::thread> th;
    for (int t = 0; t < n_lanes; ++t) {
        const size_t a = std::min(bytes, (size_t)t * per), b = std::min(bytes, (size_t)(t + 1) * per);
        u->lanes[t].err = cudaSuccess;
        u->lanes[t].last = -1;
        if (b <= a) continue;
        if (t == n_lanes - 1) lane_copy(h->device, u, &u->lanes[t], (char *)dst, (const char *)src, a, b - a, stride);   // caller's thread takes the last range
        else th.emplace_back(lane_copy, h->device, u, &u->lanes[t], (char *)dst, (const char *)src, a, b - a, stride);
    }
    for (auto &t : th) t.join();
    for (int t = 0; t < n_lanes; ++t) {
        UploadLane &l = u->lanes[t];
        if (l.err != cudaSuccess) { h->err = std::string("nw_h2d: ") + cudaGetErrorString(l.err); return NW_ERR_CUDA; }
        if (l.last >= 0) NW_CUDA(cudaStreamWaitEvent(h->stream, l.ev[l.last], 0));
    }
    return NW_OK;
}
