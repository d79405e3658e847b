// group.cu -- device groups: one host thread drives N contexts (one per GPU, or several on one GPU) through one clustering
// stage and merges their tentative labels on the devices, without torch.distributed.
//
// A member keeps its own stream and its own slice of the query slots (chb_set_labels); the group only moves int32 label
// windows (and the feature matrix, once per stage) between members.  chb_group_all_max is the exchange of every round:
//   1. an event on every member's stream (its round has been enqueued before the call);
//   2. every member's stream waits for its peers' events (the waits may cross devices) and pulls the N - 1 peer windows
//      into a local gather area with cudaMemcpyPeerAsync -- a device-to-device copy between contexts on one GPU, over
//      NVLink (or staged by the driver) between GPUs: one code path;
//   3. a second event per member after its pulls, waited for by its peers: no member overwrites its window while a peer
//      may still be reading it;
//   4. group_max_kernel reduces the N windows into the member's own buffer in one pass (int4 loads).
// After step 4 every member holds the element-wise MAX, ordered before whatever is enqueued on its stream next
// (chb_round_commit).  Errors are reported through chb_last_error(NULL).
#include <algorithm>
#include <vector>

#include "common.cuh"

struct chb_group {
    std::vector<chb_ctx *> m;
    std::vector<int> dev;          // member devices: destroying the group touches no member (they may be gone already)
    std::vector<int32_t *> buf;    // per member: the group buffer (cap[i] entries, padded to a multiple of 4)
    std::vector<int32_t *> gather; // per member: N - 1 peer windows of cap[i] entries each
    std::vector<int64_t> cap;
    std::vector<cudaEvent_t> ev_ready, ev_read; // per member, created on its device
};

namespace {

inline int64_t pad4(int64_t n) { return (n + 3) & ~(int64_t)3; }

// buf[i] = max(buf[i], gather[j * stride + i] for j < npeer), i < count; stride is a multiple of 4 (16-byte aligned windows)
__global__ void __launch_bounds__(256) group_max_kernel(int32_t *__restrict__ buf, const int32_t *__restrict__ gather, int64_t stride,
                                                        int32_t npeer, int64_t count)
{
    chb_pdl_enter();
    const int64_t n4 = count >> 2;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
    int4 *b4 = reinterpret_cast<int4 *>(buf);
    for (int64_t i = tid; i < n4; i += nthreads) {
        int4 v = b4[i];
        for (int32_t j = 0; j < npeer; ++j) {
            const int4 w = __ldcs(reinterpret_cast<const int4 *>(gather + j * stride) + i); // read once: do not keep in L2
            v.x = max(v.x, w.x);
            v.y = max(v.y, w.y);
            v.z = max(v.z, w.z);
            v.w = max(v.w, w.w);
        }
        b4[i] = v;
    }
    const int64_t t = (n4 << 2) + tid; // the last count % 4 entries
    if (t < count) {
        int32_t v = buf[t];
        for (int32_t j = 0; j < npeer; ++j) v = max(v, gather[j * stride + t]);
        buf[t] = v;
    }
}

int group_sync(chb_group *g)
{
    for (chb_ctx *c : g->m) {
        CHB_CUDA(nullptr, cudaSetDevice(c->device));
        CHB_CUDA(nullptr, cudaStreamSynchronize(c->stream));
    }
    return CHB_OK;
}

void group_free(chb_group *g)
{
    for (size_t i = 0; i < g->dev.size(); ++i) {
        cudaSetDevice(g->dev[i]);
        if (g->buf[i]) cudaFree(g->buf[i]);
        if (g->gather[i]) cudaFree(g->gather[i]);
        if (g->ev_ready[i]) cudaEventDestroy(g->ev_ready[i]);
        if (g->ev_read[i]) cudaEventDestroy(g->ev_read[i]);
    }
    delete g;
}

} // namespace

extern "C" {

int chb_group_create(chb_group **out, chb_ctx *const *members, int32_t n)
{
    if (!out) return chb_fail(nullptr, CHB_EINVAL, "chb_group_create: out is NULL");
    *out = nullptr;
    if (!members || n < 1) return chb_fail(nullptr, CHB_EINVAL, "chb_group_create: needs at least one member");
    for (int32_t i = 0; i < n; ++i) {
        if (!members[i]) return chb_fail(nullptr, CHB_EINVAL, "chb_group_create: member %d is NULL", i);
        for (int32_t j = 0; j < i; ++j)
            if (members[j] == members[i])
                return chb_fail(nullptr, CHB_EINVAL, "chb_group_create: members %d and %d are the same context", j, i);
    }
    chb_group *g = new chb_group();
    g->m.assign(members, members + n);
    for (int32_t i = 0; i < n; ++i) g->dev.push_back(members[i]->device);
    g->buf.assign(n, nullptr);
    g->gather.assign(n, nullptr);
    g->cap.assign(n, 0);
    g->ev_ready.assign(n, nullptr);
    g->ev_read.assign(n, nullptr);
    for (int32_t i = 0; i < n; ++i) {
        const int dev = members[i]->device;
        if (cudaSetDevice(dev) != cudaSuccess || cudaEventCreateWithFlags(&g->ev_ready[i], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&g->ev_read[i], cudaEventDisableTiming) != cudaSuccess) {
            (void)cudaGetLastError();
            group_free(g);
            return chb_fail(nullptr, CHB_ECUDA, "chb_group_create: event creation on device %d failed", dev);
        }
        // direct peer copies where the pair supports them; without peer access the same copies still work (driver-staged)
        for (int32_t j = 0; j < n; ++j) {
            const int peer = members[j]->device;
            int can = 0;
            if (peer != dev && cudaDeviceCanAccessPeer(&can, dev, peer) == cudaSuccess && can) {
                if (cudaDeviceEnablePeerAccess(peer, 0) != cudaSuccess) (void)cudaGetLastError(); // already enabled is fine
            }
        }
    }
    *out = g;
    return CHB_OK;
}

int chb_group_destroy(chb_group *g)
{
    if (!g) return CHB_OK;
    int rc = CHB_OK;
    for (size_t i = 0; i < g->dev.size(); ++i) { // the buffers may still be in use on a member's stream
        if (cudaSetDevice(g->dev[i]) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess)
            rc = chb_fail(nullptr, CHB_ECUDA, "chb_group_destroy: %s", cudaGetErrorString(cudaGetLastError()));
    }
    group_free(g);
    return rc;
}

int chb_group_buffer(chb_group *g, int32_t m, int64_t count, int32_t **buf_dev)
{
    CHB_CHECK(nullptr, g && buf_dev, CHB_EINVAL, "chb_group_buffer: NULL argument");
    CHB_CHECK(nullptr, m >= 0 && m < (int32_t)g->m.size(), CHB_EINVAL, "chb_group_buffer: member %d out of range [0,%d)", m,
              (int)g->m.size());
    CHB_CHECK(nullptr, count >= 0, CHB_EINVAL, "chb_group_buffer: count %lld < 0", (long long)count);
    const int64_t want = pad4(std::max<int64_t>(count, 1));
    if (g->cap[m] < want) {
        const int rc = group_sync(g); // peers may still be pulling from the old buffer
        if (rc != CHB_OK) return rc;
        chb_ctx *c = g->m[m];
        CHB_CUDA(nullptr, cudaSetDevice(c->device));
        if (g->buf[m]) cudaFree(g->buf[m]);
        if (g->gather[m]) cudaFree(g->gather[m]);
        g->buf[m] = g->gather[m] = nullptr;
        g->cap[m] = 0;
        const int64_t npeer = (int64_t)g->m.size() - 1;
        CHB_CUDA(nullptr, cudaMalloc(&g->buf[m], sizeof(int32_t) * (size_t)want));
        if (npeer > 0) CHB_CUDA(nullptr, cudaMalloc(&g->gather[m], sizeof(int32_t) * (size_t)(want * npeer)));
        g->cap[m] = want;
    }
    *buf_dev = g->buf[m];
    return CHB_OK;
}

int chb_group_all_max(chb_group *g, int64_t count)
{
    CHB_CHECK(nullptr, g, CHB_EINVAL, "chb_group_all_max: group is NULL");
    const int32_t n = (int32_t)g->m.size();
    CHB_CHECK(nullptr, count >= 0, CHB_EINVAL, "chb_group_all_max: count %lld < 0", (long long)count);
    for (int32_t i = 0; i < n; ++i)
        CHB_CHECK(nullptr, g->buf[i] && g->cap[i] >= count, CHB_EINVAL,
                  "chb_group_all_max: member %d has no group buffer of %lld entries (chb_group_buffer)", i, (long long)count);
    if (n == 1 || count == 0) return CHB_OK;
    const size_t bytes = sizeof(int32_t) * (size_t)count;
    for (int32_t i = 0; i < n; ++i) { // 1. every member's round is enqueued
        CHB_CUDA(nullptr, cudaSetDevice(g->m[i]->device));
        CHB_CUDA(nullptr, cudaEventRecord(g->ev_ready[i], g->m[i]->stream));
    }
    for (int32_t i = 0; i < n; ++i) { // 2. pull the peers' windows
        chb_ctx *c = g->m[i];
        CHB_CUDA(nullptr, cudaSetDevice(c->device));
        const int64_t stride = g->cap[i];
        int32_t j = 0;
        for (int32_t p = 0; p < n; ++p) {
            if (p == i) continue;
            CHB_CUDA(nullptr, cudaStreamWaitEvent(c->stream, g->ev_ready[p], 0));
            CHB_CUDA(nullptr, cudaMemcpyPeerAsync(g->gather[i] + j * stride, c->device, g->buf[p], g->m[p]->device, bytes, c->stream));
            ++j;
        }
        CHB_CUDA(nullptr, cudaEventRecord(g->ev_read[i], c->stream));
    }
    for (int32_t i = 0; i < n; ++i) { // 3. + 4. nobody still reads this window: reduce into it
        chb_ctx *c = g->m[i];
        CHB_CUDA(nullptr, cudaSetDevice(c->device));
        for (int32_t p = 0; p < n; ++p)
            if (p != i) CHB_CUDA(nullptr, cudaStreamWaitEvent(c->stream, g->ev_read[p], 0));
        const int64_t n4 = std::max<int64_t>(count >> 2, 1);
        const unsigned grid = (unsigned)std::min<int64_t>((n4 + 255) / 256, (int64_t)c->sm_count * 4);
        CHB_CUDA(nullptr, chb_launch_pdl(group_max_kernel, dim3(grid), dim3(256), 0, c->stream, g->buf[i], g->gather[i], g->cap[i],
                                         n - 1, count));
        ++c->tm.launches_other;
    }
    return CHB_OK;
}

int chb_group_replicate_features(chb_group *g, int32_t root)
{
    CHB_CHECK(nullptr, g, CHB_EINVAL, "chb_group_replicate_features: group is NULL");
    const int32_t n = (int32_t)g->m.size();
    CHB_CHECK(nullptr, root >= 0 && root < n, CHB_EINVAL, "chb_group_replicate_features: root %d out of range [0,%d)", root, n);
    chb_ctx *r = g->m[root];
    CHB_CHECK(nullptr, r->X && r->n > 0 && r->d > 0, CHB_EINVAL,
              "chb_group_replicate_features: member %d has no features (call a chb_set_features* function first)", root);
    CHB_CUDA(nullptr, cudaSetDevice(r->device));
    CHB_CUDA(nullptr, cudaEventRecord(g->ev_ready[root], r->stream));
    for (int32_t i = 0; i < n; ++i) {
        if (i == root) continue;
        chb_ctx *c = g->m[i];
        double *x = nullptr;
        int64_t cnt = 0;
        int rc = chb_features_buffer(c, r->n, r->d, &x, &cnt);
        if (rc != CHB_OK) return chb_fail(nullptr, rc, "chb_group_replicate_features: member %d: %s", i, c->err.c_str());
        CHB_CUDA(nullptr, cudaStreamWaitEvent(c->stream, g->ev_ready[root], 0));
        CHB_CUDA(nullptr, cudaMemcpyPeerAsync(x, c->device, r->X, r->device, sizeof(double) * (size_t)cnt, c->stream));
        rc = chb_features_commit(c, 1); // the FP32 copy and norms, as on a receiver of the NCCL broadcast
        if (rc != CHB_OK) return chb_fail(nullptr, rc, "chb_group_replicate_features: member %d: %s", i, c->err.c_str());
        CHB_CUDA(nullptr, cudaEventRecord(g->ev_read[i], c->stream));
    }
    // the root's matrix is not overwritten (a later chb_set_features*) while a member may still be copying it
    CHB_CUDA(nullptr, cudaSetDevice(r->device));
    for (int32_t i = 0; i < n; ++i)
        if (i != root) CHB_CUDA(nullptr, cudaStreamWaitEvent(r->stream, g->ev_read[i], 0));
    return CHB_OK;
}

} // extern "C"
