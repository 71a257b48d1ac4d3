// positionbaseddynamics_b200/csrc/engine.cu
//
// Host side of the B200 PBD/XPBD engine behind the C ABI of include/pbd_b200.h:
//   * flattening of a constraint list + the reference's colour groups into (colour,type) buckets of SoA arrays,
//   * the step driver that replaces TimeStepController::step (Simulation/TimeStepController.cpp:75-241) for
//     particle constraints: per substep  integrate -> maxIterations x (colour by colour, bucket by bucket) -> velocity update,
//     executed as plain launches, as a replayed CUDA graph, or as one cluster launch with the positions resident in
//     distributed shared memory (resident.cuh).
// There is no CPU fallback: every path that computes needs the CUDA device.
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <numeric>
#include <string>
#include <vector>
#include "kernels.cuh"
#include "resident.cuh"
#include "colouring.cuh"
#include "contacts.cuh"
#include <cub/cub.cuh>
#include <omp.h>
#include <parallel/algorithm>  // libstdc++ parallel mode (OpenMP): the per-bucket sorts of flatten
#include "host/pbd_model.h"

using namespace pbdk;

// ------------------------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------------------------
// OpenMP team of the host-side flatten.  GPU hosts expose far more hardware threads (128 here) than a process may actually use
// (measured: a 128-thread team made flatten 9x slower than the serial code, 8-16 threads 3x faster), so the team is capped.
static int host_threads() {
    static const int n = [] { const char *g = getenv("PBD_B200_HOST_THREADS"); const int want = g ? atoi(g) : 8; return std::max(1, std::min(want, omp_get_max_threads())); }();
    return n;
}

static thread_local std::string g_err;
static int fail(const char *fmt, ...) {
    char buf[1024];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof(buf), fmt, ap); va_end(ap);
    g_err = buf;
    return 1;
}
#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); } while (0)
#define CKE(e) do { int r_ = (e); if (r_) return r_; } while (0)

extern "C" const char *pbd_last_error(void) { return g_err.c_str(); }

// ------------------------------------------------------------------------------------------------------------
// engine state
// ------------------------------------------------------------------------------------------------------------
using pbd_b200::PodVector;        // std::vector whose resize() does not zero (filled from all threads right after)
struct HostType {                 // constraints of one type as handed in through pbd_add_constraints
    PodVector<unsigned> ids;      // insertion index in the reference's m_constraints
    PodVector<unsigned> bodies;   // nBodies per constraint
    PodVector<float> params;      // nParams per constraint (reference layout)
};

struct DevBuf {
    void *p = nullptr; size_t bytes = 0;
    int alloc(size_t b) {
        if (b <= bytes && p) return 0;
        if (p) cudaFree(p);
        p = nullptr; bytes = 0;
        if (b == 0) return 0;
        cudaError_t e = cudaMalloc(&p, b);
        if (e != cudaSuccess) return fail("cudaMalloc(%zu) -> %s", b, cudaGetErrorString(e));
        bytes = b;
        return 0;
    }
    void release() { if (p) cudaFree(p); p = nullptr; bytes = 0; }
};

struct DevType {
    DevBuf idx[3], gv[kMaxGeoV], gs[kMaxGeoS], mat[kMaxMat], lambda;
    std::vector<unsigned> order;  // position in the device arrays -> insertion id
    unsigned count = 0;
    TypeArrays arrays{};
};

struct pbd_engine {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool ownsStream = false;
    int smCount = 148;
    // particles
    unsigned n = 0;
    DevBuf pos, vel, oldp, lastp, pos0, stage, stage2, massStage, jacobiDelta;
    // rigid bodies coupled through joints (SURVEY.md 8f-1): float4 arrays X(xyz,invMass) Q(x,y,z,w) V(xyz,mass) W(omega) + history + inertia
    unsigned nRb = 0;
    DevBuf rbX, rbQ, rbV, rbW, rbOldX, rbLastX, rbOldQ, rbLastQ, rbI, rbIinv;
    // constraints (host copy, insertion order) and groups
    HostType host[PBD_NUM_TYPES];
    unsigned numConstraints = 0;
    std::vector<unsigned> groupOff, groupIds;
    bool groupsSet = false;
    // device image
    DevType dev[PBD_NUM_TYPES];
    std::vector<Bucket> buckets;
    DevBuf dBuckets, dTrace;
    bool imageDirty = true;
    bool sortBuckets = true;
    // parameters
    float dt = 0.005f; unsigned subSteps = 5, maxIter = 1; int velMethod = 0; float g[3] = {0.f, -9.81f, 0.f};
    int mode = PBD_MODE_AUTO;             // requested (pbd_set_mode)
    int active = PBD_MODE_GRAPH;          // what the current image runs in: == mode, or the resolution of PBD_MODE_AUTO
    bool autoNoResident = false;          // PBD_MODE_AUTO: the resident mode was tried for this model and refused
    // graph cache
    cudaGraphExec_t graphExec = nullptr;
    bool graphValid = false;
    unsigned long long graphLaunches = 0;  // kernel nodes of the captured step
    // stats
    pbd_stats stats{};
    cudaEvent_t evStart = nullptr, evStop = nullptr;
    // pbd_step_host_async: two staging slots, one upload and one download stream next to the compute stream
    struct HostPipe {
        cudaStream_t up = nullptr, down = nullptr;
        DevBuf inX[2], inV[2], outX[2], outV[2];
        cudaEvent_t uploaded[2] = {nullptr, nullptr}, consumed[2] = {nullptr, nullptr}, produced[2] = {nullptr, nullptr}, downloaded[2] = {nullptr, nullptr};
        unsigned long long issued = 0;
        bool ready = false;
    } pipe;
    // contact path (contacts.cuh): colliders, parameters, optional record of the last step's contacts
    std::vector<float> rbMass;
    std::vector<int> scratchInt;
    std::vector<ParticleCollider> pColliders;
    std::vector<RigidCollider> rColliders;
    DevBuf dPColliders, dRColliders, dRangeStart, dContacts, dContactCount;
    unsigned contactTotal = 0, contactCap = 0;
    float contactTolerance = 0.01f, contactStiffness = 100.0f; unsigned maxIterV = 5;  // CollisionDetection.cpp:25, SimulationModel.cpp:34, TimeStepController.cpp:23
    bool timingPending = false;
    bool mergeColours = true;             // one launch per colour when it holds several types (PBD_B200_MERGE=0 disables)
    std::vector<unsigned> slot;           // host particle index -> device slot (formula layouts or the tile-major permutation)
    DevBuf dSlot, dSlotOld, relayoutTmp;
    bool slotIsTiled = false;
    // resident mode (resident.cuh): G clusters x C CTAs = nTiles tiles, block size and type mask of the instantiation
    unsigned resG = 0, resC = 0, nTiles = 0, resThreads = 0, resMask = 0, resColours = 0, resTileCap = 0, resXThreads = 0;
    bool resChecked = false;              // co-residency of the clusters verified for the current image
    DevBuf dColourStart, dTileOff, dTileStart, dTileSmem, dXArrive, dXCounter;
    unsigned long long xBase = 0, xPerStep = 0;  // arrival counter of the X items: value at the next launch, arrivals per substep-sweep unit
    int layout = 1;                       // particle placement (device_image.h particle_slot); PBD_B200_LAYOUT=linear selects 0
    bool usePDL = true;                   // programmatic dependent launch between the kernels of a step (PBD_B200_PDL=0 disables)
    bool gatherCA = true;                 // particle gathers through L1 (tuning knob: PBD_B200_GATHER=cg selects L2-only loads)
    std::vector<unsigned long long> xArriveInt, xArriveCol;  // per-launch bookkeeping of the X counter (host copy of dXArrive)
};

static int use(pbd_engine *e) { CK(cudaSetDevice(e->device)); return 0; }

extern "C" int pbd_device_count(int *count) {
    cudaError_t err = cudaGetDeviceCount(count);
    if (err != cudaSuccess) { *count = 0; return fail("cudaGetDeviceCount -> %s", cudaGetErrorString(err)); }
    return 0;
}
extern "C" int pbd_num_bodies(int type) { return type_shape(type).nBodies; }
extern "C" int pbd_num_params(int type) { return type_shape(type).nParams; }

extern "C" int pbd_create(int device, void *stream, pbd_engine **out) {
    if (!out) return fail("pbd_create: out == NULL");
    int count = 0;
    cudaError_t err = cudaGetDeviceCount(&count);
    if (err != cudaSuccess || count == 0)
        return fail("pbd_create: no CUDA device available (%s); this engine has no CPU fallback",
                    err != cudaSuccess ? cudaGetErrorString(err) : "device count 0");
    if (device < 0 || device >= count) return fail("pbd_create: device %d out of range [0,%d)", device, count);
    pbd_engine *e = new pbd_engine();
    e->device = device;
    if (use(e)) { delete e; return 1; }
    cudaDeviceProp prop;
    err = cudaGetDeviceProperties(&prop, device);
    if (err != cudaSuccess) { delete e; return fail("cudaGetDeviceProperties -> %s", cudaGetErrorString(err)); }
    e->smCount = prop.multiProcessorCount;
    if (stream) { e->stream = (cudaStream_t)stream; e->ownsStream = false; }
    else {
        err = cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking);
        if (err != cudaSuccess) { delete e; return fail("cudaStreamCreate -> %s", cudaGetErrorString(err)); }
        e->ownsStream = true;
    }
    cudaEventCreate(&e->evStart); cudaEventCreate(&e->evStop);
    if (const char *g = getenv("PBD_B200_GATHER")) e->gatherCA = (strcmp(g, "cg") != 0);
    if (const char *g = getenv("PBD_B200_PDL")) e->usePDL = (strcmp(g, "0") != 0);
    if (const char *g = getenv("PBD_B200_MERGE")) e->mergeColours = (strcmp(g, "0") != 0);
    if (const char *g = getenv("PBD_B200_LAYOUT")) e->layout = (strcmp(g, "linear") == 0) ? 0 : 1;
    *out = e;
    return 0;
}

static void drop_graph(pbd_engine *e) {
    if (e->graphExec) { cudaGraphExecDestroy(e->graphExec); e->graphExec = nullptr; }
    e->graphValid = false;
}

extern "C" int pbd_destroy(pbd_engine *e) {
    if (!e) return 0;
    cudaSetDevice(e->device);
    cudaStreamSynchronize(e->stream);
    drop_graph(e);
    for (auto *b : {&e->pos, &e->vel, &e->oldp, &e->lastp, &e->pos0, &e->stage, &e->stage2, &e->massStage, &e->jacobiDelta, &e->dSlot, &e->dSlotOld, &e->relayoutTmp,
                    &e->dPColliders, &e->dRColliders, &e->dRangeStart, &e->dContacts, &e->dContactCount, &e->dColourStart, &e->dTileOff, &e->dTileStart, &e->dTileSmem, &e->dXArrive, &e->dXCounter, &e->dBuckets, &e->dTrace,
                    &e->rbX, &e->rbQ, &e->rbV, &e->rbW, &e->rbOldX, &e->rbLastX, &e->rbOldQ, &e->rbLastQ, &e->rbI, &e->rbIinv}) b->release();
    for (auto &d : e->dev) {
        for (auto &b : d.idx) b.release();
        for (auto &b : d.gv) b.release();
        for (auto &b : d.gs) b.release();
        for (auto &b : d.mat) b.release();
        d.lambda.release();
    }
    if (e->evStart) cudaEventDestroy(e->evStart);
    if (e->evStop) cudaEventDestroy(e->evStop);
    if (e->pipe.ready) {
        cudaStreamSynchronize(e->pipe.up); cudaStreamSynchronize(e->pipe.down);
        for (int s = 0; s < 2; s++) {
            for (auto *b : {&e->pipe.inX[s], &e->pipe.inV[s], &e->pipe.outX[s], &e->pipe.outV[s]}) b->release();
            for (cudaEvent_t ev : {e->pipe.uploaded[s], e->pipe.consumed[s], e->pipe.produced[s], e->pipe.downloaded[s]}) cudaEventDestroy(ev);
        }
        cudaStreamDestroy(e->pipe.up); cudaStreamDestroy(e->pipe.down);
    }
    if (e->ownsStream) cudaStreamDestroy(e->stream);
    delete e;
    return 0;
}

// ------------------------------------------------------------------------------------------------------------
// particles
// ------------------------------------------------------------------------------------------------------------
static inline unsigned nblk(unsigned n, unsigned t) { return (n + t - 1) / t; }

static float4 *attr_buf(pbd_engine *e, int attr) {
    switch (attr) {
    case PBD_ATTR_X: return (float4 *)e->pos.p;
    case PBD_ATTR_V: return (float4 *)e->vel.p;
    case PBD_ATTR_X0: return (float4 *)e->pos0.p;
    case PBD_ATTR_OLDX: return (float4 *)e->oldp.p;
    case PBD_ATTR_LASTX: return (float4 *)e->lastp.p;
    default: return nullptr;
    }
}

static int upload_slot_map(pbd_engine *e) {
    if (e->n == 0) return 0;
    CKE(e->dSlot.alloc((size_t)e->n * sizeof(unsigned)));
    CK(cudaMemcpy(e->dSlot.p, e->slot.data(), (size_t)e->n * sizeof(unsigned), cudaMemcpyHostToDevice));
    return 0;
}
static void formula_slot_map(pbd_engine *e, std::vector<unsigned> &m) {
    m.resize(e->n);
    for (unsigned i = 0; i < e->n; i++) m[i] = particle_slot(i, e->n, e->layout);
}
// move every particle array from the current slot map to `newSlot`
static int relayout(pbd_engine *e, const std::vector<unsigned> &newSlot) {
    if (e->n == 0 || newSlot == e->slot) { e->slot = newSlot; return 0; }
    const size_t nb = (size_t)e->n * sizeof(unsigned);
    CKE(e->dSlotOld.alloc(nb));
    CK(cudaMemcpy(e->dSlotOld.p, e->slot.data(), nb, cudaMemcpyHostToDevice));
    e->slot = newSlot;
    CKE(upload_slot_map(e));
    CKE(e->relayoutTmp.alloc((size_t)e->n * sizeof(float4)));
    for (DevBuf *b : {&e->pos, &e->vel, &e->oldp, &e->lastp, &e->pos0}) {
        k_relayout<<<(e->n + 255) / 256, 256, 0, e->stream>>>((const float4 *)b->p, (float4 *)e->relayoutTmp.p, e->n, (const unsigned *)e->dSlotOld.p, (const unsigned *)e->dSlot.p);
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(e->stream));
        std::swap(b->p, e->relayoutTmp.p); std::swap(b->bytes, e->relayoutTmp.bytes);
    }
    return 0;
}

// host AoS-3 -> staging -> float4 (keeps .w)
static int upload3(pbd_engine *e, const float *src, float4 *dst, int keepW) {
    const size_t bytes = (size_t)e->n * 3 * sizeof(float);
    CK(cudaMemcpyAsync(e->stage.p, src, bytes, cudaMemcpyHostToDevice, e->stream));
    k_pack3<<<nblk(e->n, 256), 256, 0, e->stream>>>((const float *)e->stage.p, dst, e->n, keepW, (const unsigned *)e->dSlot.p);
    CK(cudaGetLastError());
    return 0;
}

extern "C" int pbd_set_masses(pbd_engine *e, const float *mass) {
    if (!e || !mass) return fail("pbd_set_masses: null argument");
    CKE(use(e));
    if (e->n == 0) return 0;
    CK(cudaMemcpyAsync(e->massStage.p, mass, (size_t)e->n * sizeof(float), cudaMemcpyHostToDevice, e->stream));
    k_set_w<<<nblk(e->n, 256), 256, 0, e->stream>>>((float4 *)e->pos.p, (float4 *)e->vel.p, (const float *)e->massStage.p, e->n, (const unsigned *)e->dSlot.p);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(e->stream));  // staging buffers are reused by the next call
    return 0;
}

extern "C" int pbd_set_particles(pbd_engine *e, unsigned n, const float *x, const float *x0, const float *v, const float *mass) {
    if (!e || (n && (!x || !mass))) return fail("pbd_set_particles: null argument");
    CKE(use(e));
    CK(cudaStreamSynchronize(e->stream));
    if (n != e->n) { e->imageDirty = true; drop_graph(e); }
    e->n = n;
    const size_t b4 = (size_t)n * sizeof(float4);
    for (auto *b : {&e->pos, &e->vel, &e->oldp, &e->lastp, &e->pos0}) CKE(b->alloc(b4));
    CKE(e->stage.alloc((size_t)n * 3 * sizeof(float)));
    CKE(e->massStage.alloc((size_t)n * sizeof(float)));
    drop_graph(e);  // buffers may have moved
    formula_slot_map(e, e->slot); e->slotIsTiled = false; e->imageDirty = true;
    if (n == 0) return 0;
    CKE(upload_slot_map(e));
    CK(cudaMemsetAsync(e->vel.p, 0, b4, e->stream));
    CKE(upload3(e, x, (float4 *)e->pos.p, 0)); CK(cudaStreamSynchronize(e->stream));
    if (v) { CKE(upload3(e, v, (float4 *)e->vel.p, 0)); CK(cudaStreamSynchronize(e->stream)); }
    CKE(pbd_set_masses(e, mass));
    // oldX = lastX = x, x0 = x unless given (ParticleData::addVertex, ParticleData.h:127-137)
    CK(cudaMemcpyAsync(e->oldp.p, e->pos.p, b4, cudaMemcpyDeviceToDevice, e->stream));
    CK(cudaMemcpyAsync(e->lastp.p, e->pos.p, b4, cudaMemcpyDeviceToDevice, e->stream));
    CK(cudaMemcpyAsync(e->pos0.p, e->pos.p, b4, cudaMemcpyDeviceToDevice, e->stream));
    if (x0) { CKE(upload3(e, x0, (float4 *)e->pos0.p, 1)); }
    CK(cudaStreamSynchronize(e->stream));
    e->stats.num_particles = n;
    return 0;
}

extern "C" int pbd_set_attr(pbd_engine *e, int attr, const float *src) {
    if (!e || !src) return fail("pbd_set_attr: null argument");
    CKE(use(e));
    float4 *dst = attr_buf(e, attr);
    if (!dst) return fail("pbd_set_attr: bad attribute %d", attr);
    if (e->n == 0) return 0;
    CKE(upload3(e, src, dst, 1));
    CK(cudaStreamSynchronize(e->stream));
    return 0;
}

extern "C" int pbd_get_attr(pbd_engine *e, int attr, float *dst) {
    if (!e || !dst) return fail("pbd_get_attr: null argument");
    CKE(use(e));
    const float4 *src = attr_buf(e, attr);
    if (!src) return fail("pbd_get_attr: bad attribute %d", attr);
    if (e->n == 0) return 0;
    k_unpack3<<<nblk(e->n, 256), 256, 0, e->stream>>>(src, (float *)e->stage.p, e->n, (const unsigned *)e->dSlot.p);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(dst, e->stage.p, (size_t)e->n * 3 * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return 0;
}

// ------------------------------------------------------------------------------------------------------------
// rigid bodies (host arrays are tiny: plain synchronous copies)
// ------------------------------------------------------------------------------------------------------------
extern "C" int pbd_set_rigid_bodies(pbd_engine *e, unsigned n, const float *mass, const float *x, const float *q, const float *inertia,
                                    const float *v, const float *omega) {
    if (!e || (n && (!mass || !x || !q || !inertia))) return fail("pbd_set_rigid_bodies: null argument");
    CKE(use(e));
    CK(cudaStreamSynchronize(e->stream));
    if (n != e->nRb) { e->imageDirty = true; e->groupsSet = e->groupsSet && n == e->nRb; }
    drop_graph(e);
    e->nRb = n;
    e->rbMass.assign(mass, mass + n);
    if (n == 0) return 0;
    std::vector<float4> X(n), Q(n), V(n), W(n), I(n), Ii(n);
    for (unsigned i = 0; i < n; i++) {
        const float m = mass[i];
        X[i] = make_float4(x[3 * i], x[3 * i + 1], x[3 * i + 2], (m != 0.0f) ? 1.0f / m : 0.0f);
        Q[i] = make_float4(q[4 * i + 1], q[4 * i + 2], q[4 * i + 3], q[4 * i]);  // (w,x,y,z) -> (x,y,z,w)
        V[i] = v ? make_float4(v[3 * i], v[3 * i + 1], v[3 * i + 2], m) : make_float4(0.f, 0.f, 0.f, m);
        W[i] = omega ? make_float4(omega[3 * i], omega[3 * i + 1], omega[3 * i + 2], 0.f) : make_float4(0.f, 0.f, 0.f, 0.f);
        I[i] = make_float4(inertia[3 * i], inertia[3 * i + 1], inertia[3 * i + 2], 0.f);
        Ii[i] = make_float4(1.0f / inertia[3 * i], 1.0f / inertia[3 * i + 1], 1.0f / inertia[3 * i + 2], 0.f);  // RigidBody::setInertiaTensor (RigidBody.h:416-420)
    }
    const size_t b = (size_t)n * sizeof(float4);
    struct { DevBuf *d; const std::vector<float4> *h; } up[] = {{&e->rbX, &X}, {&e->rbQ, &Q}, {&e->rbV, &V}, {&e->rbW, &W}, {&e->rbOldX, &X}, {&e->rbLastX, &X},
                                                              {&e->rbOldQ, &Q}, {&e->rbLastQ, &Q}, {&e->rbI, &I}, {&e->rbIinv, &Ii}};
    for (auto &u : up) { CKE(u.d->alloc(b)); CK(cudaMemcpy(u.d->p, u.h->data(), b, cudaMemcpyHostToDevice)); }
    e->imageDirty = true;  // joint type arrays hold the rigid-body pointers
    return 0;
}

extern "C" int pbd_get_rigid_bodies(pbd_engine *e, float *x, float *q, float *v, float *omega) {
    if (!e) return fail("null engine");
    CKE(use(e));
    CK(cudaStreamSynchronize(e->stream));
    const unsigned n = e->nRb;
    if (n == 0) return 0;
    std::vector<float4> t(n);
    const size_t b = (size_t)n * sizeof(float4);
    if (x) { CK(cudaMemcpy(t.data(), e->rbX.p, b, cudaMemcpyDeviceToHost)); for (unsigned i = 0; i < n; i++) { x[3 * i] = t[i].x; x[3 * i + 1] = t[i].y; x[3 * i + 2] = t[i].z; } }
    if (q) { CK(cudaMemcpy(t.data(), e->rbQ.p, b, cudaMemcpyDeviceToHost)); for (unsigned i = 0; i < n; i++) { q[4 * i] = t[i].w; q[4 * i + 1] = t[i].x; q[4 * i + 2] = t[i].y; q[4 * i + 3] = t[i].z; } }
    if (v) { CK(cudaMemcpy(t.data(), e->rbV.p, b, cudaMemcpyDeviceToHost)); for (unsigned i = 0; i < n; i++) { v[3 * i] = t[i].x; v[3 * i + 1] = t[i].y; v[3 * i + 2] = t[i].z; } }
    if (omega) { CK(cudaMemcpy(t.data(), e->rbW.p, b, cudaMemcpyDeviceToHost)); for (unsigned i = 0; i < n; i++) { omega[3 * i] = t[i].x; omega[3 * i + 1] = t[i].y; omega[3 * i + 2] = t[i].z; } }
    return 0;
}

template <class V> static int upload_vec(DevBuf &buf, const V &v, cudaStream_t s) {  // V: std::vector / PodVector of PODs
    typedef typename V::value_type T;
    if (v.empty()) return 0;
    if (buf.alloc(v.size() * sizeof(T) + 16)) return 1;
    cudaError_t e = cudaMemcpyAsync(buf.p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, s);
    if (e != cudaSuccess) return fail("upload -> %s", cudaGetErrorString(e));
    e = cudaStreamSynchronize(s);  // the host vector dies with the caller's scope
    if (e != cudaSuccess) return fail("upload sync -> %s", cudaGetErrorString(e));
    return 0;
}

// ------------------------------------------------------------------------------------------------------------
// constraints and groups
// ------------------------------------------------------------------------------------------------------------
extern "C" int pbd_clear_constraints(pbd_engine *e) {
    if (!e) return fail("null engine");
    for (auto &h : e->host) { h.ids.clear(); h.bodies.clear(); h.params.clear(); }
    e->numConstraints = 0;
    e->groupOff.clear(); e->groupIds.clear(); e->groupsSet = false;
    e->imageDirty = true; e->autoNoResident = false;
    return 0;
}

extern "C" int pbd_add_constraints(pbd_engine *e, int type, unsigned count, const unsigned *bodies, const float *params, const unsigned *ids) {
    if (!e) return fail("null engine");
    if (type < 0 || type >= PBD_NUM_TYPES) return fail("pbd_add_constraints: unknown constraint type %d", type);
    if (count && (!bodies || !params)) return fail("pbd_add_constraints: null arrays");
    const TypeShape s = type_shape(type);
    {   // index validation, all threads (millions of indices for a big cloth)
        const size_t nIdx = (size_t)count * s.nBodies;
        long long badAt = -1;
        #pragma omp parallel for schedule(static) num_threads(host_threads()) reduction(max : badAt) if (nIdx > 100000)
        for (long long i = 0; i < (long long)nIdx; i++) {
            const bool isRb = (type == PBD_BALLJOINT) || (type == PBD_RB_PARTICLE_BALLJOINT && (i % 2) == 0);
            if (bodies[i] >= (isRb ? e->nRb : e->n)) badAt = std::max(badAt, i);
        }
        if (badAt >= 0) {
            const bool isRb = (type == PBD_BALLJOINT) || (type == PBD_RB_PARTICLE_BALLJOINT && (badAt % 2) == 0);
            if (isRb) return fail("pbd_add_constraints: rigid-body index %u out of range (%u bodies; call pbd_set_rigid_bodies first)", bodies[badAt], e->nRb);
            return fail("pbd_add_constraints: particle index %u out of range (n=%u)", bodies[badAt], e->n);
        }
    }
    HostType &h = e->host[type];
    {
        const size_t b0 = h.ids.size();
        h.ids.resize(b0 + count); h.bodies.resize((b0 + count) * s.nBodies); h.params.resize((b0 + count) * s.nParams);  // uninitialised, filled below
        unsigned *idDst = h.ids.data() + b0, *bDst = h.bodies.data() + b0 * s.nBodies; float *pDst = h.params.data() + b0 * s.nParams;
        const unsigned firstId = e->numConstraints;
        #pragma omp parallel for schedule(static) num_threads(host_threads()) if (count > 50000)
        for (long long i = 0; i < (long long)count; i++) {
            idDst[i] = ids ? ids[i] : firstId + (unsigned)i;
            std::memcpy(bDst + (size_t)i * s.nBodies, bodies + (size_t)i * s.nBodies, sizeof(unsigned) * s.nBodies);
            std::memcpy(pDst + (size_t)i * s.nParams, params + (size_t)i * s.nParams, sizeof(float) * s.nParams);
        }
    }
    e->numConstraints += count;
    e->groupsSet = false;  // any add invalidates the groups (SimulationModel: m_groupsInitialized = false)
    e->imageDirty = true; e->autoNoResident = false;
    return 0;
}

// insertion id -> (type, local index); verifies that the ids form a permutation of 0..N-1
static int build_id_map(pbd_engine *e, std::vector<std::pair<int, unsigned>> &map) {
    const unsigned N = e->numConstraints;
    map.resize(N);
    std::vector<int> &seenType = e->scratchInt; seenType.resize(N);
    #pragma omp parallel for schedule(static) num_threads(host_threads())
    for (long long i = 0; i < (long long)N; i++) seenType[i] = -1;
    for (int t = 0; t < PBD_NUM_TYPES; t++) {
        const HostType &h = e->host[t];
        long long bad = -1; int dup = 0;
        #pragma omp parallel for schedule(static) num_threads(host_threads()) reduction(max : bad) reduction(| : dup) if (h.ids.size() > 50000)
        for (long long i = 0; i < (long long)h.ids.size(); i++) {
            const unsigned id = h.ids[i];
            if (id >= N) { bad = std::max(bad, (long long)id); continue; }
            if (__atomic_exchange_n(&seenType[id], t, __ATOMIC_RELAXED) != -1) { dup = 1; bad = std::max(bad, (long long)id); continue; }
            map[id] = std::make_pair(t, (unsigned)i);
        }
        if (bad >= 0 && !dup) return fail("constraint id %u out of range (N=%u)", (unsigned)bad, N);
        if (dup) return fail("constraint id %u used twice", (unsigned)bad);
    }
    return 0;  // N ids, all below N, none twice: a permutation
}

extern "C" int pbd_set_groups(pbd_engine *e, unsigned nGroups, const unsigned *offsets, const unsigned *ids) {
    if (!e || (nGroups && (!offsets || !ids))) return fail("pbd_set_groups: null argument");
    const unsigned N = e->numConstraints;
    if (nGroups == 0 && N != 0) return fail("pbd_set_groups: %u constraints but no groups", N);
    if (nGroups && offsets[nGroups] != N) return fail("pbd_set_groups: groups cover %u constraints, model has %u", offsets[nGroups], N);
    if (nGroups && offsets[0] != 0) return fail("pbd_set_groups: offsets[0] must be 0");
    for (unsigned g = 0; g < nGroups; g++)
        if (offsets[g] > offsets[g + 1]) return fail("pbd_set_groups: offsets must be non-decreasing (group %u)", g);
    std::vector<unsigned char> seen(N, 0);
    for (unsigned i = 0; i < N; i++) {
        if (ids[i] >= N || seen[ids[i]]) return fail("pbd_set_groups: ids are not a permutation of 0..%u", N);
        seen[ids[i]] = 1;
    }
    e->groupOff.assign(offsets, offsets + nGroups + 1);
    e->groupIds.assign(ids, ids + N);
    if (nGroups == 0) e->groupOff.assign(1, 0u);
    e->groupsSet = true;
    e->imageDirty = true;
    return 0;
}

// insertion-ordered CSR of the constraint bodies (the colouring's input)
static int build_id_csr(pbd_engine *e, std::vector<unsigned> &off, std::vector<unsigned> &bodies) {
    std::vector<std::pair<int, unsigned>> map;
    CKE(build_id_map(e, map));
    const unsigned N = e->numConstraints;
    off.resize((size_t)N + 1);
    // off = exclusive prefix sum of the body counts (chunked two-pass scan), then every constraint copies its bodies
    const int T = std::max(1, host_threads());
    std::vector<unsigned long long> chunk((size_t)T + 1, 0ull);
    #pragma omp parallel num_threads(T)
    {
        const int t = omp_get_thread_num(), nt = omp_get_num_threads();
        const size_t lo = (size_t)N * t / nt, hi = (size_t)N * (t + 1) / nt;
        unsigned long long sum = 0;
        for (size_t id = lo; id < hi; id++) sum += (unsigned)type_shape(map[id].first).nBodies;
        chunk[(size_t)t + 1] = sum;
        #pragma omp barrier
        #pragma omp single
        for (int k = 0; k < nt; k++) chunk[(size_t)k + 1] += chunk[k];
        unsigned long long run = chunk[t];
        for (size_t id = lo; id < hi; id++) { off[id] = (unsigned)run; run += (unsigned)type_shape(map[id].first).nBodies; }
        if (t == nt - 1) off[N] = (unsigned)run;
    }
    if (N == 0) off[0] = 0;
    bodies.resize(off[N]);
    #pragma omp parallel for schedule(static) num_threads(T)
    for (long long id = 0; id < (long long)N; id++) {
        const int t = map[id].first;
        const int nb = type_shape(t).nBodies;
        std::memcpy(&bodies[off[id]], &e->host[t].bodies[(size_t)map[id].second * nb], sizeof(unsigned) * nb);
    }
    return 0;
}
// colour per constraint -> groups in insertion order (what SimulationModel::getConstraintGroups holds)
static void groups_from_colours(pbd_engine *e, const std::vector<unsigned> &colour, unsigned nColours) {
    const unsigned N = e->numConstraints;
    // stable counting sort by colour: per-thread histograms over contiguous id ranges, then every thread scatters its range
    const int T = std::max(1, host_threads());
    std::vector<unsigned> hist((size_t)T * nColours, 0u), goff(nColours + 1, 0u);
    e->groupIds.resize(N);
    #pragma omp parallel num_threads(T)
    {
        const int t = omp_get_thread_num(), nt = omp_get_num_threads();
        const size_t lo = (size_t)N * t / nt, hi = (size_t)N * (t + 1) / nt;
        unsigned *h = &hist[(size_t)t * nColours];
        for (size_t id = lo; id < hi; id++) h[colour[id]]++;
        #pragma omp barrier
        #pragma omp single
        {
            unsigned run = 0;
            for (unsigned c = 0; c < nColours; c++) {
                goff[c] = run;
                for (int k = 0; k < nt; k++) { const unsigned cntk = hist[(size_t)k * nColours + c]; hist[(size_t)k * nColours + c] = run; run += cntk; }
            }
            goff[nColours] = run;
        }
        for (size_t id = lo; id < hi; id++) e->groupIds[h[colour[id]]++] = (unsigned)id;
    }
    e->groupOff = goff;
    e->groupsSet = true; e->imageDirty = true;
}

// Greedy first fit in insertion order == SimulationModel::initConstraintGroups (Simulation/SimulationModel.cpp:1033-1094);
// the colouring itself is host/pbd_model.cpp:firstFitColouring (shared with the host model mirror).
extern "C" int pbd_color_first_fit(pbd_engine *e) {
    if (!e) return fail("null engine");
    std::vector<unsigned> off, bodies, colour;
    CKE(build_id_csr(e, off, bodies));
    // rigid-body and particle indices share one index space without offset (SimulationModel.cpp:1041,1058,1070)
    const unsigned nColours = pbd_b200::firstFitColouring(e->n + e->nRb, e->numConstraints, off.data(), bodies.data(), colour);
    groups_from_colours(e, colour, nColours);
    return 0;
}

// The same colouring computed on the device (colouring.cuh): identical groups, SURVEY.md section 8 f-3.
extern "C" int pbd_color_first_fit_device(pbd_engine *e, float *ms, unsigned *wavefronts) {
    if (!e) return fail("null engine");
    CKE(use(e));
    const unsigned N = e->numConstraints, V = e->n + e->nRb;
    if (ms) *ms = 0.0f;
    if (wavefronts) *wavefronts = 0;
    if (N == 0) { e->groupOff.assign(1, 0u); e->groupIds.clear(); e->groupsSet = true; e->imageDirty = true; return 0; }
    std::vector<unsigned> off, bodies;
    CKE(build_id_csr(e, off, bodies));
    const unsigned M = (unsigned)bodies.size();
    cudaStream_t s = e->stream;
    // one device allocation for all the work arrays (a dozen cudaMalloc / cudaFree pairs cost more than the colouring kernels of a small scene)
    int endBit = 1; while (endBit < 32 && (1ull << endBit) < (unsigned long long)V) endBit++;
    size_t tmpBytes = 0;
    CK(cub::DeviceRadixSort::SortPairs(nullptr, tmpBytes, (const unsigned *)nullptr, (unsigned *)nullptr, (const unsigned *)nullptr, (unsigned *)nullptr, (int)M, 0, endBit, s));
    struct View { void *p = nullptr; };
    View dOff, dBody, dBody4, dNext4, dKeys, dVals, dKeysS, dValsS, dIndeg, dColour, dA, dB, dCnt, dTmp;
    DevBuf dAll, dUsed;
    struct Release { std::vector<DevBuf *> b; ~Release() { for (auto *x : b) x->release(); } } rel{{&dAll, &dUsed}};
    {
        struct Want { View *v; size_t bytes; } want[] = {{&dOff, ((size_t)N + 1) * sizeof(unsigned)}, {&dBody, (size_t)M * sizeof(unsigned)}, {&dKeys, (size_t)M * sizeof(unsigned)},
            {&dVals, (size_t)M * sizeof(unsigned)}, {&dKeysS, (size_t)M * sizeof(unsigned)}, {&dValsS, (size_t)M * sizeof(unsigned)}, {&dBody4, (size_t)N * sizeof(uint4)},
            {&dNext4, (size_t)N * sizeof(uint4)}, {&dIndeg, (size_t)N * sizeof(unsigned)}, {&dColour, (size_t)N * sizeof(unsigned)}, {&dA, (size_t)N * sizeof(unsigned)},
            {&dB, (size_t)N * sizeof(unsigned)}, {&dCnt, 4 * sizeof(unsigned)}, {&dTmp, tmpBytes}};
        size_t total = 0;
        for (auto &w : want) total += (w.bytes + 255) & ~(size_t)255;
        CKE(dAll.alloc(total));
        size_t at = 0;
        for (auto &w : want) { w.v->p = (char *)dAll.p + at; at += (w.bytes + 255) & ~(size_t)255; }
    }
    CK(cudaMemcpyAsync(dOff.p, off.data(), ((size_t)N + 1) * sizeof(unsigned), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(dBody.p, bodies.data(), (size_t)M * sizeof(unsigned), cudaMemcpyHostToDevice, s));
    cudaEvent_t ev0, ev1;
    CK(cudaEventCreate(&ev0)); CK(cudaEventCreate(&ev1));
    CK(cudaEventRecord(ev0, s));
    // incidence lists: stable sort of (body, incidence) by body, then successor / in-degree of every constraint
    k_colour_expand<<<nblk(N, 256), 256, 0, s>>>((const unsigned *)dOff.p, (const unsigned *)dBody.p, (uint4 *)dBody4.p, (unsigned *)dKeys.p, (unsigned *)dVals.p, N);
    CK(cub::DeviceRadixSort::SortPairs(dTmp.p, tmpBytes, (const unsigned *)dKeys.p, (unsigned *)dKeysS.p, (const unsigned *)dVals.p, (unsigned *)dValsS.p, (int)M, 0, endBit, s));
    CK(cudaMemsetAsync(dNext4.p, 0xff, (size_t)N * sizeof(uint4), s));
    std::vector<unsigned> colour(N);
    unsigned cnt[4] = {0, 0, 0, 0};
    for (unsigned words = 2;; words *= 2) {  // 128 colours to begin with; doubled when a constraint finds none free
        CKE(dUsed.alloc((size_t)V * words * sizeof(unsigned long long)));
        CK(cudaMemsetAsync(dUsed.p, 0, (size_t)V * words * sizeof(unsigned long long), s));
        CK(cudaMemsetAsync(dIndeg.p, 0, (size_t)N * sizeof(unsigned), s));
        CK(cudaMemsetAsync(dCnt.p, 0, 4 * sizeof(unsigned), s));
        k_colour_links<<<nblk(M, 256), 256, 0, s>>>((const unsigned *)dKeysS.p, (const unsigned *)dValsS.p, M, (unsigned *)dNext4.p, (unsigned *)dIndeg.p);
        ColourArgs a{N, V, words, (const uint4 *)dBody4.p, (const uint4 *)dNext4.p, (unsigned *)dIndeg.p, (unsigned long long *)dUsed.p,
                     (unsigned *)dColour.p, (unsigned *)dA.p, (unsigned *)dB.p, (unsigned *)dCnt.p};
        k_colour_seed<<<nblk(N, 256), 256, 0, s>>>(a);
        k_colour_wavefronts<<<1, kColourThreads, 0, s>>>(a);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(cnt, dCnt.p, sizeof(cnt), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        if (!cnt[1]) break;
        if (words >= 1024) return fail("device colouring: more than %u colours needed", words * 64);
    }
    CK(cudaEventRecord(ev1, s));
    CK(cudaMemcpyAsync(colour.data(), dColour.p, (size_t)N * sizeof(unsigned), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    float t = 0.0f; cudaEventElapsedTime(&t, ev0, ev1);
    cudaEventDestroy(ev0); cudaEventDestroy(ev1);
    if (cnt[2] != N) return fail("device colouring: coloured %u of %u constraints (dependency cycle?)", cnt[2], N);
    unsigned nColours = 0;
    #pragma omp parallel for schedule(static) num_threads(host_threads()) reduction(max : nColours)
    for (long long id = 0; id < (long long)N; id++) nColours = std::max(nColours, colour[id] + 1);
    groups_from_colours(e, colour, nColours);
    if (ms) *ms = t;
    if (wavefronts) *wavefronts = cnt[3];
    return 0;
}

extern "C" int pbd_get_num_groups(pbd_engine *e, unsigned *nGroups) {
    if (!e || !nGroups) return fail("null argument");
    if (!e->groupsSet) return fail("groups not initialised (call pbd_set_groups or pbd_color_first_fit)");
    *nGroups = (unsigned)e->groupOff.size() - 1;
    return 0;
}
extern "C" int pbd_get_groups(pbd_engine *e, unsigned *offsets, unsigned *ids) {
    if (!e || !offsets || !ids) return fail("null argument");
    if (!e->groupsSet) return fail("groups not initialised");
    memcpy(offsets, e->groupOff.data(), e->groupOff.size() * sizeof(unsigned));
    memcpy(ids, e->groupIds.data(), e->groupIds.size() * sizeof(unsigned));
    return 0;
}

extern "C" int pbd_set_params(pbd_engine *e, float dt, unsigned subSteps, unsigned maxIter, int velMethod, const float gravity[3]) {
    if (!e) return fail("null engine");
    if (subSteps < 1) return fail("subSteps must be >= 1 (TimeStepController.cpp:50)");
    if (maxIter < 1) return fail("maxIterations must be >= 1 (TimeStepController.cpp:55)");
    if (velMethod != 0 && velMethod != 1) return fail("velocityUpdateMethod must be 0 or 1");
    if (!(dt > 0.0f)) return fail("time step size must be positive");
    const bool same = e->dt == dt && e->subSteps == subSteps && e->maxIter == maxIter && e->velMethod == velMethod &&
                      (!gravity || (e->g[0] == gravity[0] && e->g[1] == gravity[1] && e->g[2] == gravity[2]));
    if (same) return 0;  // callers such as a TimeStep adapter set the parameters before every step: keep the captured graph
    e->dt = dt; e->subSteps = subSteps; e->maxIter = maxIter; e->velMethod = velMethod;
    if (gravity) { e->g[0] = gravity[0]; e->g[1] = gravity[1]; e->g[2] = gravity[2]; }
    drop_graph(e);
    return 0;
}
extern "C" int pbd_set_mode(pbd_engine *e, int mode) {
    if (!e) return fail("null engine");
    if (mode != PBD_MODE_GRAPH && mode != PBD_MODE_RESIDENT && mode != PBD_MODE_LAUNCH && mode != PBD_MODE_JACOBI && mode != PBD_MODE_AUTO) return fail("unknown solver mode %d", mode);
    if (mode == e->mode) return 0;
    // the resident image encodes indices differently; with AUTO on either side the resolution may change
    if (mode == PBD_MODE_AUTO || e->mode == PBD_MODE_AUTO || (mode == PBD_MODE_RESIDENT) != (e->active == PBD_MODE_RESIDENT)) e->imageDirty = true;
    e->mode = mode; e->autoNoResident = false;
    if (mode != PBD_MODE_AUTO) e->active = mode;
    drop_graph(e);
    return 0;
}
extern "C" int pbd_get_mode(pbd_engine *e, int *requested, int *active) {
    if (!e) return fail("null engine");
    if (requested) *requested = e->mode;
    if (active) *active = e->active;
    return 0;
}
extern "C" int pbd_set_bucket_sort(pbd_engine *e, int enable) {
    if (!e) return fail("null engine");
    e->sortBuckets = enable != 0; e->imageDirty = true;
    return 0;
}

// ------------------------------------------------------------------------------------------------------------
// flattening: constraints + colour groups -> per-type SoA arrays ordered bucket by bucket
// ------------------------------------------------------------------------------------------------------------
// Q (row-major 4x4, solver order) = -Kp Kp^T ?  Returns true and Kp when the rank-one negative-semidefinite form of
// init_IsometricBendingConstraint (PositionBasedDynamics.cpp:169-180) reproduces Q to fp32 accuracy.
static bool factor_rank1(const float *Q, float Kp[4]) {
    int piv = 0; float best = 0.0f, maxAbs = 0.0f;
    for (int j = 0; j < 4; j++) { if (-Q[5 * j] > best) { best = -Q[5 * j]; piv = j; } }
    for (int i = 0; i < 16; i++) maxAbs = std::max(maxAbs, std::fabs(Q[i]));
    if (maxAbs == 0.0f) { Kp[0] = Kp[1] = Kp[2] = Kp[3] = 0.0f; return true; }
    if (!(best > 0.0f)) return false;
    const double kp = std::sqrt((double)best);
    double K[4];
    for (int k = 0; k < 4; k++) K[k] = -(double)Q[4 * piv + k] / kp;
    for (int j = 0; j < 4; j++)
        for (int k = 0; k < 4; k++)
            if (std::fabs((double)Q[4 * j + k] + K[j] * K[k]) > 1e-5 * (double)maxAbs) return false;
    for (int k = 0; k < 4; k++) Kp[k] = (float)K[k];
    return true;
}


// Resident mode (resident.cuh): the particles are partitioned into G cluster regions x C tiles by recursive coordinate
// bisection of the rest positions; the device arrays are permuted to tile-major order.
static void bisect(std::vector<unsigned> &idx, size_t lo, size_t hi, unsigned t0, unsigned nt, const std::vector<float4> &x, std::vector<unsigned> &tileOf) {
    if (nt == 1) { for (size_t i = lo; i < hi; i++) tileOf[idx[i]] = t0; return; }
    float mn[3] = {3.4e38f, 3.4e38f, 3.4e38f}, mx[3] = {-3.4e38f, -3.4e38f, -3.4e38f};
    for (size_t i = lo; i < hi; i++) {
        const float4 &p = x[idx[i]];
        const float c[3] = {p.x, p.y, p.z};
        for (int k = 0; k < 3; k++) { mn[k] = std::min(mn[k], c[k]); mx[k] = std::max(mx[k], c[k]); }
    }
    int ax = 0;
    for (int k = 1; k < 3; k++) if (mx[k] - mn[k] > mx[ax] - mn[ax]) ax = k;
    const unsigned ntL = nt / 2;
    const size_t mid = lo + (size_t)((double)(hi - lo) * ntL / nt);
    auto key = [&](unsigned i) { const float4 &p = x[i]; return ax == 0 ? p.x : (ax == 1 ? p.y : p.z); };
    std::nth_element(idx.begin() + lo, idx.begin() + mid, idx.begin() + hi, [&](unsigned a, unsigned b) { const float ka = key(a), kb = key(b); return ka < kb || (ka == kb && a < b); });
    // the two halves are independent: run them as tasks while they are big enough to pay for it
    #pragma omp task shared(idx, x, tileOf) if (hi - lo > 65536)
    bisect(idx, lo, mid, t0, ntL, x, tileOf);
    bisect(idx, mid, hi, t0 + ntL, nt - ntL, x, tileOf);
    #pragma omp taskwait
}

struct ResidentPlan {
    std::vector<unsigned> tileOf;             // host particle -> tile (cluster = tile / C, rank = tile % C)
    std::vector<unsigned> tileStart, tileSmem;
    std::vector<unsigned char> homedGlobal;   // host particle lives in global memory (touched by a constraint that spans clusters)
};

static bool is_rb_body(int type, int k) { return type == PBD_BALLJOINT || (type == PBD_RB_PARTICLE_BALLJOINT && k == 0); }

// Executing tile of a constraint: the tile that holds most of its shared-memory particles (ties: the lowest tile); none -> the tile of
// its first particle (0 for a joint between rigid bodies).  *touchesGlobal: one of its particles is global-homed.
static inline unsigned exec_tile(int t, const unsigned *b, int nb, const std::vector<unsigned> &tileOf, const std::vector<unsigned char> &homedGlobal, bool *touchesGlobal) {
    bool x = false;
    unsigned best = 0xffffffffu, bestCnt = 0, first = 0xffffffffu;
    for (int k = 0; k < nb; k++) {
        if (is_rb_body(t, k)) continue;
        if (first == 0xffffffffu) first = tileOf[b[k]];
        if (homedGlobal[b[k]]) { x = true; continue; }
        unsigned cnt = 0;
        for (int j = 0; j < nb; j++) cnt += (!is_rb_body(t, j) && !homedGlobal[b[j]] && tileOf[b[j]] == tileOf[b[k]]);
        if (cnt > bestCnt || (cnt == bestCnt && tileOf[b[k]] < best)) { best = tileOf[b[k]]; bestCnt = cnt; }
    }
    *touchesGlobal = x;
    return (best != 0xffffffffu) ? best : (first != 0xffffffffu ? first : 0u);
}

// the compiled instantiations of k_step_resident: F(kernel pointer) for the engine's (mask, block size, one CTA per cluster?)
template <class F> static int with_resident_kernel(const pbd_engine *e, unsigned C, F &&f) {
    const unsigned th = e->resThreads;
    const bool single = (C == 1);
    if (e->resMask == kMaskClothXPBD) {
        if (th == 512) return single ? f(k_step_resident<kMaskClothXPBD, 512, true>) : f(k_step_resident<kMaskClothXPBD, 512, false>);
        if (th == 768) return single ? f(k_step_resident<kMaskClothXPBD, 768, true>) : f(k_step_resident<kMaskClothXPBD, 768, false>);
        return single ? f(k_step_resident<kMaskClothXPBD, 640, true>) : f(k_step_resident<kMaskClothXPBD, 640, false>);
    }
    if (e->resMask == kMaskCloth) return single ? f(k_step_resident<kMaskCloth, 512, true>) : f(k_step_resident<kMaskCloth, 512, false>);
    if (e->resMask == kMaskLight) return single ? f(k_step_resident<kMaskLight, 512, true>) : f(k_step_resident<kMaskLight, 512, false>);
    if (e->resMask == kMaskFem) {
        if (th == 256) return single ? f(k_step_resident<kMaskFem, 256, true>) : f(k_step_resident<kMaskFem, 256, false>);
        return single ? f(k_step_resident<kMaskFem, 512, true>) : f(k_step_resident<kMaskFem, 512, false>);
    }
    if (e->resMask == kMaskSolid) {
        if (th == 256) return single ? f(k_step_resident<kMaskSolid, 256, true>) : f(k_step_resident<kMaskSolid, 256, false>);
        return single ? f(k_step_resident<kMaskSolid, 512, true>) : f(k_step_resident<kMaskSolid, 512, false>);
    }
    if (th == 512) return single ? f(k_step_resident<kMaskAll, 512, true>) : f(k_step_resident<kMaskAll, 512, false>);
    return single ? f(k_step_resident<kMaskAll, 256, true>) : f(k_step_resident<kMaskAll, 256, false>);
}

static void resident_launch_config(const pbd_engine *e, unsigned C, unsigned grid, size_t smem, cudaStream_t s, cudaLaunchConfig_t &cfg, cudaLaunchAttribute *attr) {
    cfg = cudaLaunchConfig_t{};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(e->resThreads); cfg.dynamicSmemBytes = smem; cfg.stream = s;
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = C; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
}

// how many clusters of C CTAs (one CTA per SM, `smem` bytes each) the device keeps resident at the same time
static int resident_max_clusters(const pbd_engine *e, unsigned C, size_t smem, int *out) {
    return with_resident_kernel(e, C, [&](auto kernel) -> int {
        CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxDynamicSmem));
        CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
        cudaLaunchConfig_t cfg; cudaLaunchAttribute attr[1];
        resident_launch_config(e, C, C, smem, e->stream, cfg, attr);
        cudaError_t err = cudaOccupancyMaxActiveClusters(out, kernel, &cfg);
        if (err != cudaSuccess) { cudaGetLastError(); *out = 0; }
        return 0;
    });
}

// shape of the launch: type mask / block size of the instantiation, clusters x CTAs per cluster
static int choose_resident_shape(pbd_engine *e) {
    unsigned present = 0, nTypes = 0;
    for (int t = 0; t < PBD_NUM_TYPES; t++) if (!e->host[t].ids.empty()) { present |= 1u << t; nTypes++; }
    e->resMask = kMaskAll;
    for (unsigned m : {kMaskClothXPBD, kMaskCloth, kMaskFem, kMaskLight, kMaskSolid})  // the leanest instantiation that covers the model
        if ((present & ~m) == 0) { e->resMask = m; break; }
    // the block sizes the instantiations compile for without spilling (cloth 96 registers, light 128, everything 236)
    e->resThreads = (e->resMask == kMaskClothXPBD) ? 640u : ((e->resMask == kMaskAll) ? 256u : 512u);
    if (const char *g = getenv("PBD_B200_RTHREADS")) { const int k = atoi(g); if (k == 256 || k == 512 || k == 640 || k == 768) e->resThreads = (unsigned)k; }
    // clamp to a block size the mask is instantiated for (with_resident_kernel): the kernel's THREADS must equal the launch's block size.
    // cloth-XPBD 512 / 640 / 768, cloth and light 512, FEM / solid / everything 256 / 512
    if (e->resMask == kMaskLight || e->resMask == kMaskCloth) e->resThreads = 512u;
    else if (e->resMask == kMaskClothXPBD) { if (e->resThreads < 512u) e->resThreads = 512u; }
    else if (e->resThreads > 512u) e->resThreads = 512u;
    const unsigned nGroups = (unsigned)std::max<size_t>(e->groupOff.size(), 2) - 1;
    const unsigned perPhase = e->numConstraints / std::max(1u, nGroups);
    // particles a tile can hold: what is left of the CTA's shared memory after the phase tables (bound: one bucket per colour and type)
    const size_t tables = resident_smem_bytes(0u, nGroups * std::max(1u, nTypes), nGroups);
    if (tables + 1024 * sizeof(float4) > kMaxDynamicSmem) return fail("resident mode: %u colour groups need %zu bytes of phase tables (use PBD_MODE_GRAPH)", nGroups, tables);
    const unsigned cap = (unsigned)(0.97 * (double)((kMaxDynamicSmem - tables) / sizeof(float4)));  // bisection splits counts evenly; slack for rounding
    unsigned G = 1, C = 1;
    if (e->n <= (unsigned)kMaxClusterCtas * cap && perPhase <= (unsigned)kMaxClusterCtas * 1024u) {
        // one cluster: enough CTAs that a colour phase is about one item per thread, and that the tiles fit
        while (C < (unsigned)kMaxClusterCtas && (perPhase > C * 256u || e->n > C * cap)) C *= 2;
    } else {
        // Too big for one cluster: one independent CTA per SM (clusters of 1).  Measured on cfg2 (profiles/README.md): 148 x 1 beats
        // 74 x 2, 33 x 4, 15 x 8 and 7 x 16 -- larger clusters have fewer X items but idle SMs (a cluster must fit a GPC) and a
        // colour barrier that waits for the slowest of C CTAs; with C = 1 the colour barrier is a __syncthreads.
        int mc = 0;
        CKE(resident_max_clusters(e, 1u, kMaxDynamicSmem, &mc));
        if (mc < 1) return fail("resident mode: a CTA with %zu bytes of shared memory is not schedulable on this device", kMaxDynamicSmem);
        C = 1; G = (unsigned)std::min(mc, e->smCount);
    }
    if (const char *g = getenv("PBD_B200_CLUSTERS")) {  // development knob "GxC"
        unsigned gg = 0, cc = 0;
        if (sscanf(g, "%ux%u", &gg, &cc) == 2 && gg >= 1 && cc >= 1 && cc <= (unsigned)kMaxClusterCtas && (cc & (cc - 1)) == 0) { G = gg; C = cc; }
    }
    if ((unsigned long long)G * C * cap < e->n)
        return fail("resident mode: %u particles do not fit %u x %u tiles of %u (use PBD_MODE_GRAPH)", e->n, G, C, cap);
    // (bodies without joints -- e.g. the static colliders of the contact path -- are integrated by CTA 0 and touch no constraint)
    if (G > 1 && (!e->host[PBD_BALLJOINT].ids.empty() || !e->host[PBD_RB_PARTICLE_BALLJOINT].ids.empty()))
        return fail("resident mode: rigid-body coupling is supported for scenes that fit one cluster (use PBD_MODE_GRAPH)");
    e->resG = G; e->resC = C; e->nTiles = G * C;
    e->resXThreads = (G > 1) ? 128u : 0u;  // refined in prepare_resident once the share of X items is known
    return 0;
}

static int prepare_resident(pbd_engine *e, ResidentPlan &pl) {
    CKE(choose_resident_shape(e));
    const unsigned n = e->n, G = e->resG, C = e->resC, T = e->nTiles;
    pl.tileOf.assign(n, 0); pl.homedGlobal.assign(n, 0); pl.tileStart.assign(T + 1, 0); pl.tileSmem.assign(T, 0);
    if (n) {
        // rest positions by host index
        std::vector<float4> raw(n), x(n);
        CK(cudaStreamSynchronize(e->stream));
        CK(cudaMemcpy(raw.data(), e->pos0.p, (size_t)n * sizeof(float4), cudaMemcpyDeviceToHost));
        for (unsigned i = 0; i < n; i++) x[i] = raw[e->slot[i]];
        std::vector<unsigned> idx(n), region(n);
        for (unsigned i = 0; i < n; i++) idx[i] = i;
        #pragma omp parallel num_threads(host_threads())
        #pragma omp single
        bisect(idx, 0, n, 0, G, x, region);  // cluster regions; idx is now grouped region by region
        size_t lo = 0;
        for (unsigned g = 0; g < G; g++) {
            size_t hi = lo;
            while (hi < n && region[idx[hi]] == g) hi++;
            if (C == 1) { for (size_t i = lo; i < hi; i++) pl.tileOf[idx[i]] = g; }
            else {
                #pragma omp parallel num_threads(host_threads())
                #pragma omp single
                bisect(idx, lo, hi, g * C, C, x, pl.tileOf);
            }
            lo = hi;
        }
        // global-homed = touched by a constraint whose particles lie in more than one cluster
        if (G > 1)
            for (int t = 0; t < PBD_NUM_TYPES; t++) {
                const HostType &h = e->host[t];
                const int nb = type_shape(t).nBodies;
                unsigned char *hg = pl.homedGlobal.data();
                #pragma omp parallel for schedule(static) num_threads(host_threads())
                for (long long c = 0; c < (long long)h.ids.size(); c++) {
                    const unsigned *b = &h.bodies[(size_t)c * nb];
                    bool spans = false;
                    for (int k = 1; k < nb; k++) spans |= (pl.tileOf[b[k]] / C != pl.tileOf[b[0]] / C);
                    if (spans) for (int k = 0; k < nb; k++) hg[b[k]] = 1;  // every writer stores the same byte
                }
            }
        // threads of a CTA dedicated to the X items: in proportion to their share, times 3.1 because an X item waits for L2 where
        // the others read shared memory (measured on cfg2, 11 % X items, 640 threads, after the bank-group fill: 160 / 192 / 224 / 256 X
        // threads -> 2.07 / 1.93 / 1.90 / 1.93 ms)
        if (G > 1) {
            unsigned long long xItems = 0;
            for (int t = 0; t < PBD_NUM_TYPES; t++) {
                const HostType &h = e->host[t];
                const int nb = type_shape(t).nBodies;
                #pragma omp parallel for schedule(static) num_threads(host_threads()) reduction(+ : xItems)
                for (long long c = 0; c < (long long)h.ids.size(); c++) {
                    bool x = false;
                    for (int k = 0; k < nb; k++) x |= (!is_rb_body(t, k) && pl.homedGlobal[h.bodies[(size_t)c * nb + k]]);
                    xItems += x;
                }
            }
            const double share = (double)xItems / std::max(1u, e->numConstraints);
            unsigned xt = ((unsigned)(e->resThreads * share * 3.1) + 31u) & ~31u;
            xt = std::max(64u, std::min(xt, (e->resThreads / 2u) & ~31u));
            if (const char *g = getenv("PBD_B200_XTHREADS")) { const int k = atoi(g); if (k >= 32 && k % 32 == 0 && (unsigned)k < e->resThreads) xt = (unsigned)k; }
            e->resXThreads = xt;
        }
        // tile-major slots: shared-memory particles first (host order), global-homed behind them
        std::vector<unsigned> cntS(T, 0), cntG(T, 0);
        for (unsigned i = 0; i < n; i++) (pl.homedGlobal[i] ? cntG : cntS)[pl.tileOf[i]]++;
        for (unsigned t = 0; t < T; t++) {
            pl.tileStart[t + 1] = pl.tileStart[t] + cntS[t] + cntG[t];
            pl.tileSmem[t] = cntS[t];
        }
        std::vector<unsigned> curS(T), curG(T), newSlot(n);
        for (unsigned t = 0; t < T; t++) { curS[t] = pl.tileStart[t]; curG[t] = pl.tileStart[t] + cntS[t]; }
        for (unsigned i = 0; i < n; i++) newSlot[i] = pl.homedGlobal[i] ? curG[pl.tileOf[i]]++ : curS[pl.tileOf[i]]++;
        CKE(relayout(e, newSlot));
        if (getenv("PBD_B200_VERBOSE")) {
            unsigned long long nGl = 0;
            for (unsigned i = 0; i < n; i++) nGl += pl.homedGlobal[i];
            fprintf(stderr, "[pbd_b200] resident: %u clusters x %u CTAs, %u threads (%u for X items), %u particles, %.2f %% global-homed, max tile %u\n", G, C, e->resThreads, e->resXThreads, n,
                    100.0 * nGl / n, *std::max_element(cntS.begin(), cntS.end()));
        }
    }
    e->slotIsTiled = true;
    e->resTileCap = 64u;  // multiple of 64: the bank swizzle permutes inside aligned 64-slot blocks
    for (unsigned t = 0; t < T; t++) e->resTileCap = std::max(e->resTileCap, (pl.tileSmem[t] + 63u) & ~63u);
    e->resChecked = false;
    CKE(upload_vec(e->dTileStart, pl.tileStart, e->stream));
    CKE(upload_vec(e->dTileSmem, pl.tileSmem, e->stream));
    return 0;
}

static int flatten_image(pbd_engine *e);
// PBD_MODE_AUTO: the resident mode where it is the faster exact mode -- models made of cloth and FEM / volume constraints (measured:
// cfg1, cfg2, cfg3, cfg5; profiles/README.md R2.1); mixed models with rigid coupling and the heavy solver families stay in graph
// mode (cfg4) -- falling back to the graph mode when the resident mode refuses the model.
static bool auto_prefers_resident(const pbd_engine *e) {
    if (e->autoNoResident || e->numConstraints == 0 || e->n == 0) return false;
    unsigned present = 0;
    for (int t = 0; t < PBD_NUM_TYPES; t++) if (!e->host[t].ids.empty()) present |= 1u << t;
    return (present & ~(kMaskCloth | kMaskFem)) == 0 || (present & ~kMaskLight) == 0;
}
static int flatten(pbd_engine *e) {
    if (!e->imageDirty) return 0;
    if (e->mode != PBD_MODE_AUTO) { e->active = e->mode; return flatten_image(e); }
    e->active = auto_prefers_resident(e) ? PBD_MODE_RESIDENT : PBD_MODE_GRAPH;
    int rc = flatten_image(e);
    if (rc && e->active == PBD_MODE_RESIDENT) {  // refused (does not fit, user-modified bending Q, ...): the graph mode takes every model
        if (getenv("PBD_B200_VERBOSE")) fprintf(stderr, "[pbd_b200] auto mode: resident refused (%s), using the graph mode\n", g_err.c_str());
        e->autoNoResident = true; e->active = PBD_MODE_GRAPH; e->imageDirty = true;
        rc = flatten_image(e);
    }
    return rc;
}
static int flatten_image(pbd_engine *e) {
    if (!e->imageDirty) return 0;
    CKE(use(e));
    static const bool verbose = getenv("PBD_B200_VERBOSE") != nullptr;
    double tPrev = omp_get_wtime();
    auto lap = [&](const char *what) { if (verbose) { const double t = omp_get_wtime(); fprintf(stderr, "[pbd_b200] flatten: %-34s %.3f s\n", what, t - tPrev); tPrev = t; } };
    if (!e->groupsSet) {
        if (e->numConstraints == 0) { e->groupOff.assign(1, 0u); e->groupIds.clear(); e->groupsSet = true; }
        else {
            // the reference-order-preserving first fit on the GPU (colouring.cuh); the host version is the fallback and the
            // PBD_B200_HOST_COLOURING=1 choice
            static const bool hostColouring = [] { const char *g = getenv("PBD_B200_HOST_COLOURING"); return g && atoi(g) != 0; }();
            if (hostColouring || pbd_color_first_fit_device(e, nullptr, nullptr)) CKE(pbd_color_first_fit(e));
        }
    }
    drop_graph(e);
    // the particle / rigid-body counts may have shrunk since the constraints were added (pbd_set_particles, pbd_set_rigid_bodies)
    for (int t = 0; t < PBD_NUM_TYPES; t++) {
        const HostType &h = e->host[t];
        const int nb = type_shape(t).nBodies;
        long long badAt = -1;
        #pragma omp parallel for schedule(static) num_threads(host_threads()) reduction(max : badAt) if (h.bodies.size() > 100000)
        for (long long i = 0; i < (long long)h.bodies.size(); i++) {
            const bool isRb = (t == PBD_BALLJOINT) || (t == PBD_RB_PARTICLE_BALLJOINT && (i % nb) == 0);
            if (h.bodies[i] >= (isRb ? e->nRb : e->n)) badAt = std::max(badAt, i);
        }
        if (badAt >= 0) {
            const bool isRb = (t == PBD_BALLJOINT) || (t == PBD_RB_PARTICLE_BALLJOINT && (badAt % nb) == 0);
            return fail("constraint of type %d refers to %s %u, but the engine holds %u: re-add the constraints after shrinking the model", t,
                        isRb ? "rigid body" : "particle", h.bodies[badAt], isRb ? e->nRb : e->n);
        }
    }
    std::vector<std::pair<int, unsigned>> map;
    CKE(build_id_map(e, map));
    const unsigned nGroups = (unsigned)e->groupOff.size() - 1;

    // 0. particle placement: tile-major for the resident mode, the formula layout otherwise
    const bool tiled = (e->active == PBD_MODE_RESIDENT);
    ResidentPlan pl;
    std::vector<unsigned> tileOff;
    std::vector<unsigned> &tileOf = pl.tileOf;
    if (tiled) CKE(prepare_resident(e, pl));
    else if (e->slotIsTiled) {
        std::vector<unsigned> m;
        formula_slot_map(e, m);
        CKE(relayout(e, m));
        e->slotIsTiled = false;
    }

    lap("colouring + validation + placement");
    // 1. order every type's constraints bucket by bucket
    // order of the items inside a run by kind of element (see the sort key below): measured +2.8 % on the tet scenes (cfg3 7.69 -> 7.47 ms),
    // -3.6 % on the cloth scenes (cfg2 1.98 -> 2.05 ms), so it is on for the solid instantiations only; PBD_B200_SIGSORT=0/1 forces it
    static const int sigSortEnv = [] { const char *g = getenv("PBD_B200_SIGSORT"); return g ? (atoi(g) != 0 ? 1 : 0) : -1; }();
    const bool sigSort = tiled && (sigSortEnv >= 0 ? sigSortEnv != 0 : (e->resMask == kMaskFem || e->resMask == kMaskSolid));
    // bank-group fill of the shared-memory runs (below): cfg2 1.976 -> 1.914 ms, cfg5 1.379 -> 1.366 ms; PBD_B200_BANKSORT=0 switches it off
    static const bool bankSortEnv = [] { const char *g = getenv("PBD_B200_BANKSORT"); return !g || atoi(g) != 0; }();
    const bool bankSort = tiled && bankSortEnv;
    static const bool bankSortClusters = [] { const char *g = getenv("PBD_B200_BANKSORT_CLUSTERS"); return !g || atoi(g) != 0; }();  // cfg3 7.46 -> 7.28 ms (bank group taken inside the CTA that holds the particle)
    std::vector<unsigned> order[PBD_NUM_TYPES];  // device position -> local host index
    e->buckets.clear();
    std::vector<unsigned> tmp[PBD_NUM_TYPES];
    for (unsigned g = 0; g < nGroups; g++) {
        for (auto &v : tmp) v.clear();
        for (unsigned i = e->groupOff[g]; i < e->groupOff[g + 1]; i++) {
            const auto &m = map[e->groupIds[i]];
            tmp[m.first].push_back(m.second);
        }
        for (int t = 0; t < PBD_NUM_TYPES; t++) {
            if (tmp[t].empty()) continue;
            const bool joint = (t == PBD_BALLJOINT || t == PBD_RB_PARTICLE_BALLJOINT);
            if ((e->sortBuckets && !joint) || tiled) {  // order inside a colour is free: sort by lowest particle slot for gather locality
                const int nb = type_shape(t).nBodies;
                const unsigned *bod = e->host[t].bodies.data();
                std::vector<std::pair<unsigned long long, unsigned>> keyed(tmp[t].size());
                #pragma omp parallel for schedule(static) num_threads(host_threads())
                for (long long i = 0; i < (long long)tmp[t].size(); i++) {
                    const unsigned *b = bod + (size_t)tmp[t][i] * nb;
                    unsigned mn = 0xffffffffu;
                    for (int k = 0; k < nb; k++) if (!is_rb_body(t, k)) mn = std::min(mn, e->slot[b[k]]);
                    if (joint) mn = (unsigned)i;  // joints keep their order
                    // resident: major key = executing tile, then X items (touching a global-homed particle) before the others
                    unsigned long long major = 0;
                    if (tiled) {
                        bool x = false;
                        const unsigned exec = exec_tile(t, b, nb, tileOf, pl.homedGlobal, &x);
                        major = 2ull * exec + (x ? 0u : 1u);
                        // Inside a run, constraints that are translates of each other (same slot offsets between their particles: the same
                        // kind of element of a regular mesh) come first by kind, then by position: consecutive lanes then read addresses that
                        // advance by one constant stride in every operand, which the tile's XOR swizzle spreads over the bank groups -- a mixed
                        // order makes the eight lanes of a quarter-warp hit random bank groups (2 wavefronts per 128 bytes on cfg2).
                        if (sigSort && !joint) {
                            unsigned long long hsh = 1469598103934665603ull;
                            for (int k = 1; k < nb; k++) { hsh ^= (unsigned long long)(e->slot[b[k]] - e->slot[b[0]]); hsh *= 1099511628211ull; }
                            major = (major << 19) | ((hsh ^ (hsh >> 23) ^ (hsh >> 41)) & 0x7ffffull);
                        } else major <<= 19;
                    }
                    keyed[i] = std::make_pair((major << 32) | mn, tmp[t][i]);
                }
                __gnu_parallel::stable_sort(keyed.begin(), keyed.end(), [](const std::pair<unsigned long long, unsigned> &a, const std::pair<unsigned long long, unsigned> &b) { return a.first < b.first; },
                                            __gnu_parallel::default_parallel_tag(host_threads()));
                if (tiled && (e->resC == 1 || bankSortClusters) && !joint && bankSort) {
                    // Shared-memory bank groups.  The eight lanes of a quarter-warp (eight consecutive items of a tile's run) read operand k of
                    // their items with one LDS.128; it takes as many wavefronts as the fullest 16-byte bank group (slot & 7 after the swizzle).
                    // Greedy re-ordering inside every run: each group of eight is filled with the items, out of the next `kWindow` unused
                    // ones, that add the fewest collisions over all operands.  The order inside a colour is free; results are bit-identical.
                    constexpr int kWindow = 64;
                    std::vector<size_t> runStart;
                    for (size_t i = 0; i < keyed.size(); i++) if (i == 0 || (keyed[i].first >> 51) != (keyed[i - 1].first >> 51)) runStart.push_back(i);
                    runStart.push_back(keyed.size());
                    double wfBefore = 0, wfAfter = 0, requests = 0;
                    const long long nRuns = (long long)runStart.size() - 1;
                    #pragma omp parallel for schedule(dynamic, 1) num_threads(host_threads()) reduction(+ : wfBefore, wfAfter, requests)
                    for (long long r = 0; r < nRuns; r++) {
                        const size_t lo = runStart[r], hi = runStart[r + 1], cnt = hi - lo;
                        if (!((keyed[lo].first >> 51) & 1ull) || cnt < 16) continue;  // X runs gather from global memory: left alone
                        std::vector<unsigned char> bg(cnt * 4, 0);
                        for (size_t i = 0; i < cnt; i++) {
                            const unsigned *b = bod + (size_t)keyed[lo + i].second * nb;
                            for (int k = 0; k < nb && k < 4; k++) bg[i * 4 + k] = (unsigned char)(tile_swizzle(e->slot[b[k]] - pl.tileStart[tileOf[b[k]]]) & 7u);  // bank group inside the CTA that holds the particle
                        }
                        auto wavefronts = [&](const std::vector<unsigned> &ord) {
                            double w = 0;
                            for (size_t g8 = 0; g8 + 8 <= cnt; g8 += 8)
                                for (int k = 0; k < nb && k < 4; k++) {
                                    unsigned char c8[8] = {0, 0, 0, 0, 0, 0, 0, 0}; unsigned mx = 0;
                                    for (int j = 0; j < 8; j++) mx = std::max<unsigned>(mx, ++c8[bg[ord[g8 + j] * 4 + k]]);
                                    w += mx;
                                }
                            return w;
                        };
                        std::vector<unsigned> ord(cnt);
                        for (size_t i = 0; i < cnt; i++) ord[i] = (unsigned)i;
                        wfBefore += wavefronts(ord); requests += (double)(cnt / 8) * std::min(nb, 4);
                        // greedy fill from a sliding pool of the next kWindow unused items (kept in run order)
                        std::vector<unsigned> out; out.reserve(cnt);
                        unsigned pool[kWindow]; int nPool = 0; size_t head = 0;
                        while (out.size() < cnt) {
                            unsigned char load[4][8] = {};
                            for (int j = 0; j < 8 && out.size() < cnt; j++) {
                                while (nPool < kWindow && head < cnt) pool[nPool++] = (unsigned)head++;
                                int best = 0, bestCost = 1 << 30;
                                for (int c = 0; c < nPool; c++) {
                                    const unsigned char *g4 = &bg[(size_t)pool[c] * 4];
                                    int cost = 0;
                                    for (int k = 0; k < nb && k < 4; k++) cost += load[k][g4[k]];
                                    if (cost < bestCost) { bestCost = cost; best = c; if (!cost) break; }
                                }
                                const unsigned pick = pool[best];
                                for (int c = best; c + 1 < nPool; c++) pool[c] = pool[c + 1];
                                nPool--;
                                out.push_back(pick);
                                for (int k = 0; k < nb && k < 4; k++) load[k][bg[(size_t)pick * 4 + k]]++;
                            }
                        }
                        wfAfter += wavefronts(out);
                        if (bankSort) {
                            std::vector<std::pair<unsigned long long, unsigned>> tmpRun(cnt);
                            for (size_t i = 0; i < cnt; i++) tmpRun[i] = keyed[lo + out[i]];
                            for (size_t i = 0; i < cnt; i++) keyed[lo + i] = tmpRun[i];
                        }
                    }
                    if (verbose && requests > 0) fprintf(stderr, "[pbd_b200] flatten:   colour %u type %d: %.2f wavefronts per quarter-warp gather as sorted, %.2f after the bank-group fill%s\n", g, t,
                                                         wfBefore / requests, wfAfter / requests, bankSort ? " (applied)" : "");
                }
                #pragma omp parallel for schedule(static) num_threads(host_threads())
                for (long long i = 0; i < (long long)keyed.size(); i++) tmp[t][i] = keyed[i].second;
                if (tiled) {  // runs of every tile inside this bucket: [2 tile] X items, [2 tile + 1] the others
                    const size_t base = tileOff.size();
                    tileOff.resize(base + 2 * e->nTiles + 1, 0u);
                    for (size_t i = 0; i < keyed.size(); i++) tileOff[base + (keyed[i].first >> 51) + 1]++;
                    for (unsigned k = 0; k < 2 * e->nTiles; k++) tileOff[base + k + 1] += tileOff[base + k];
                }
            }
            Bucket b; b.type = t; b.first = (unsigned)order[t].size(); b.count = (unsigned)tmp[t].size(); b.colour = g;
            e->buckets.push_back(b);
            order[t].insert(order[t].end(), tmp[t].begin(), tmp[t].end());
        }
    }

    lap("bucket ordering");
    // debug-grade safety: inside a colour no particle may be used twice (race freedom by construction, SURVEY.md section 5)
    {
        // particles and rigid bodies are stamped in separate index spaces (the reference's colouring shares one, which only
        // ever over-separates; a body really used twice in a colour would be a race here)
        std::vector<unsigned> stamp((size_t)e->n + e->nRb, 0xffffffffu);
        size_t bi = 0;
        for (unsigned g = 0; g < nGroups; g++) {
            for (; bi < e->buckets.size() && e->buckets[bi].colour == g; bi++) {
                const Bucket &b = e->buckets[bi];
                const int nb = type_shape(b.type).nBodies;
                long long bad = -1;  // items of a bucket in parallel: the stamp of a slot is exchanged atomically
                #pragma omp parallel for schedule(static) num_threads(host_threads()) reduction(max : bad) if (b.count > 20000)
                for (long long i = 0; i < (long long)b.count; i++) {
                    const unsigned *bd = &e->host[b.type].bodies[(size_t)order[b.type][b.first + i] * nb];
                    for (int k = 0; k < nb; k++) {
                        const bool isRb = (b.type == PBD_BALLJOINT) || (b.type == PBD_RB_PARTICLE_BALLJOINT && k == 0);
                        const size_t slot = isRb ? (size_t)e->n + bd[k] : bd[k];
                        if (__atomic_exchange_n(&stamp[slot], g, __ATOMIC_RELAXED) == g) bad = std::max(bad, (long long)slot);
                    }
                }
                if (bad >= 0) {
                    const bool isRb = (size_t)bad >= e->n;
                    return fail("colour group %u uses %s %u twice: the groups are not a valid colouring", g, isRb ? "rigid body" : "particle", (unsigned)(isRb ? bad - e->n : bad));
                }
            }
        }
    }

    lap("colouring validity check");
    // 2. build and upload the SoA arrays of every type
    double bytesPerSweep = 0.0;
    for (int t = 0; t < PBD_NUM_TYPES; t++) {
        DevType &d = e->dev[t];
        const HostType &h = e->host[t];
        const TypeShape s = type_shape(t);
        const unsigned cnt = (unsigned)order[t].size();
        d.count = cnt;
        e->stats.constraints_per_type[t] = cnt;
        d.arrays = TypeArrays{};
        d.order.resize(cnt);
        if (cnt == 0) continue;
        #pragma omp parallel for schedule(static) num_threads(host_threads())
        for (long long i = 0; i < (long long)cnt; i++) d.order[i] = h.ids[order[t][i]];
        auto P = [&](unsigned i, int k) { return h.params[(size_t)order[t][i] * s.nParams + k]; };
        auto B = [&](unsigned i, int k) {
            const unsigned raw = h.bodies[(size_t)order[t][i] * s.nBodies + k];
            if (is_rb_body(t, k)) return raw;
            if (tiled && !pl.homedGlobal[raw]) {  // lives in the shared memory of CTA (tile % C) of the executing cluster
                const unsigned tl = tileOf[raw];
                return kSmemFlag | ((tl % e->resC) << kRankShift) | tile_swizzle(e->slot[raw] - pl.tileStart[tl]);
            }
            return e->slot[raw];
        };

        if (verbose) fprintf(stderr, "[pbd_b200] flatten:   type %d (%u constraints)\n", t, cnt);
        lap("  order ids");
        // indices
        if (s.nBodies == 2) {
            PodVector<uint2> v(cnt);
            #pragma omp parallel for schedule(static) num_threads(host_threads())
            for (long long i = 0; i < (long long)cnt; i++) v[i] = make_uint2(B(i, 0), B(i, 1));
            CKE(upload_vec(d.idx[0], v, e->stream)); d.arrays.idx2 = (const uint2 *)d.idx[0].p;
        } else if (s.nBodies == 4) {
            PodVector<uint4> v(cnt);
            #pragma omp parallel for schedule(static) num_threads(host_threads())
            for (long long i = 0; i < (long long)cnt; i++) v[i] = make_uint4(B(i, 0), B(i, 1), B(i, 2), B(i, 3));
            CKE(upload_vec(d.idx[0], v, e->stream)); d.arrays.idx4 = (const uint4 *)d.idx[0].p;
        } else {
            for (int k = 0; k < 3; k++) {
                PodVector<unsigned> v(cnt);
                #pragma omp parallel for schedule(static) num_threads(host_threads())
                for (long long i = 0; i < (long long)cnt; i++) v[i] = B(i, k);
                CKE(upload_vec(d.idx[k], v, e->stream)); d.arrays.idx3[k] = (const unsigned *)d.idx[k].p;
            }
        }

        lap("  indices (remap + upload)");
        // geometry + material slots: (param index of each material slot)
        int matSlot[kMaxMat] = {-1, -1, -1, -1, -1};
        PodVector<float4> gv[kMaxGeoV]; PodVector<float> gs[kMaxGeoS];
        int variant = 0;
        switch (t) {
        case PBD_DISTANCE: case PBD_DISTANCE_XPBD: case PBD_DIHEDRAL: case PBD_VOLUME: case PBD_VOLUME_XPBD:
            gs[0].resize(cnt);
            #pragma omp parallel for schedule(static) num_threads(host_threads())
            for (long long i = 0; i < (long long)cnt; i++) gs[0][i] = P(i, 0);
            matSlot[0] = 1;
            break;
        case PBD_ISOBENDING: case PBD_ISOBENDING_XPBD: {
            matSlot[0] = 0;
            gv[0].resize(cnt);
            int notRank1 = 0;
            #pragma omp parallel for schedule(static) num_threads(host_threads()) reduction(| : notRank1)
            for (long long i = 0; i < (long long)cnt; i++) {
                float Q[16], Kp[4] = {0.f, 0.f, 0.f, 0.f};
                for (int k = 0; k < 16; k++) Q[k] = P((unsigned)i, 1 + k);
                if (!factor_rank1(Q, Kp)) notRank1 |= 1;
                gv[0][i] = make_float4(Kp[0], Kp[1], Kp[2], Kp[3]);
            }
            const bool rank1 = !notRank1;
            if (!rank1 && tiled) return fail("resident mode: IsometricBending with a user-modified Q matrix (not of the rank-one form) is evaluated by the per-bucket kernels only (use PBD_MODE_GRAPH)");
            if (!rank1) {  // user-modified Q somewhere in this type: literal 4x4 evaluation for the whole type
                variant = 1;
                for (int r = 0; r < 4; r++) {
                    gv[r].resize(cnt);
                    #pragma omp parallel for schedule(static) num_threads(host_threads())
                    for (long long i = 0; i < (long long)cnt; i++) gv[r][i] = make_float4(P(i, 1 + 4 * r), P(i, 2 + 4 * r), P(i, 3 + 4 * r), P(i, 4 + 4 * r));
                }
            }
            break; }
        case PBD_FEMTRIANGLE:
            gv[0].resize(cnt); gs[0].resize(cnt);
            #pragma omp parallel for schedule(static) num_threads(host_threads())
            for (long long i = 0; i < (long long)cnt; i++) { gs[0][i] = P(i, 0); gv[0][i] = make_float4(P(i, 1), P(i, 2), P(i, 3), P(i, 4)); }
            for (int k = 0; k < 5; k++) matSlot[k] = 5 + k;
            break;
        case PBD_STRAINTRIANGLE:
            gv[0].resize(cnt);
            #pragma omp parallel for schedule(static) num_threads(host_threads())
            for (long long i = 0; i < (long long)cnt; i++) gv[0][i] = make_float4(P(i, 0), P(i, 1), P(i, 2), P(i, 3));
            for (int k = 0; k < 5; k++) matSlot[k] = 4 + k;
            break;
        case PBD_FEMTET: case PBD_FEMTET_XPBD:
            gv[0].resize(cnt); gv[1].resize(cnt); gs[0].resize(cnt); gs[1].resize(cnt);
            #pragma omp parallel for schedule(static) num_threads(host_threads())
            for (long long i = 0; i < (long long)cnt; i++) {
                gv[0][i] = make_float4(P(i, 1), P(i, 2), P(i, 3), P(i, 4));
                gv[1][i] = make_float4(P(i, 5), P(i, 6), P(i, 7), P(i, 8));
                gs[0][i] = P(i, 9); gs[1][i] = P(i, 0);
            }
            matSlot[0] = 10; matSlot[1] = 11;
            break;
        case PBD_STRAINTET:
            gv[0].resize(cnt); gv[1].resize(cnt); gs[0].resize(cnt);
            #pragma omp parallel for schedule(static) num_threads(host_threads())
            for (long long i = 0; i < (long long)cnt; i++) {
                gv[0][i] = make_float4(P(i, 0), P(i, 1), P(i, 2), P(i, 3));
                gv[1][i] = make_float4(P(i, 4), P(i, 5), P(i, 6), P(i, 7));
                gs[0][i] = P(i, 8);
            }
            for (int k = 0; k < 4; k++) matSlot[k] = 9 + k;
            break;
        case PBD_BALLJOINT: case PBD_RB_PARTICLE_BALLJOINT:  // local connectors (jointInfo columns 0 [and 1]); global columns are recomputed per solve
            gv[0].resize(cnt);
            #pragma omp parallel for schedule(static) num_threads(host_threads())
            for (long long i = 0; i < (long long)cnt; i++) gv[0][i] = make_float4(P(i, 0), P(i, 1), P(i, 2), 0.0f);
            if (t == PBD_BALLJOINT) { gv[1].resize(cnt); for (unsigned i = 0; i < cnt; i++) gv[1][i] = make_float4(P(i, 3), P(i, 4), P(i, 5), 0.0f); }
            break;
        case PBD_SHAPEMATCHING:  // restCm | x0[0..3] packed in 3 float4 | w | numClusters ; stiffness is the material slot
            for (int k = 0; k < 6; k++) gv[k].resize(cnt);
            for (unsigned i = 0; i < cnt; i++) {
                gv[0][i] = make_float4(P(i, 1), P(i, 2), P(i, 3), 0.0f);
                gv[1][i] = make_float4(P(i, 4), P(i, 5), P(i, 6), P(i, 7));
                gv[2][i] = make_float4(P(i, 8), P(i, 9), P(i, 10), P(i, 11));
                gv[3][i] = make_float4(P(i, 12), P(i, 13), P(i, 14), P(i, 15));
                gv[4][i] = make_float4(P(i, 16), P(i, 17), P(i, 18), P(i, 19));
                gv[5][i] = make_float4(P(i, 20), P(i, 21), P(i, 22), P(i, 23));
                for (int k = 20; k < 24; k++) if (!(P(i, k) >= 1.0f)) return fail("ShapeMatching constraint: numClusters must be >= 1");
            }
            matSlot[0] = 0;
            break;
        default: return fail("flatten: constraint type %d has no kernel", t);
        }
        d.arrays.variant = variant;
        if (t == PBD_BALLJOINT || t == PBD_RB_PARTICLE_BALLJOINT) {
            d.arrays.rbX = (float4 *)e->rbX.p; d.arrays.rbQ = (float4 *)e->rbQ.p; d.arrays.rbIinv = (const float4 *)e->rbIinv.p;
        }
        lap("  geometry (host fill)");
        for (int k = 0; k < kMaxGeoV; k++) if (!gv[k].empty()) { CKE(upload_vec(d.gv[k], gv[k], e->stream)); d.arrays.gv[k] = (const float4 *)d.gv[k].p; }
        for (int k = 0; k < kMaxGeoS; k++) if (!gs[k].empty()) { CKE(upload_vec(d.gs[k], gs[k], e->stream)); d.arrays.gs[k] = (const float *)d.gs[k].p; }
        lap("  geometry (upload)");
        // material parameters: one uniform per type when every constraint agrees, else a per-constraint array
        for (int k = 0; k < kMaxMat; k++) {
            if (matSlot[k] < 0) continue;
            const float first = P(0, matSlot[k]);
            int differs = 0;
            #pragma omp parallel for schedule(static) num_threads(host_threads()) reduction(| : differs) if (cnt > 100000)
            for (long long i = 1; i < (long long)cnt; i++) differs |= (P((unsigned)i, matSlot[k]) != first) ? 1 : 0;
            const bool uniform = !differs;
            d.arrays.matU[k] = first;
            if (!uniform) {
                PodVector<float> v(cnt);
                #pragma omp parallel for schedule(static) num_threads(host_threads())
                for (long long i = 0; i < (long long)cnt; i++) v[i] = P(i, matSlot[k]);
                CKE(upload_vec(d.mat[k], v, e->stream)); d.arrays.mat[k] = (const float *)d.mat[k].p;
            }
        }
        if (s.xpbd) {
            CKE(d.lambda.alloc((size_t)cnt * sizeof(float) + 16));  // + 16 like the other streamed arrays: the L2 prefetch of a run rounds its end up to 16 bytes
            CK(cudaMemsetAsync(d.lambda.p, 0, (size_t)cnt * sizeof(float), e->stream));
            d.arrays.lambda = (float *)d.lambda.p;
        }
        lap("  material + multipliers");
        bytesPerSweep += (double)cnt * algorithmic_bytes(t, variant);
    }

    lap("SoA arrays + upload");
    // 3. bucket table; resident mode: colour ranges, per-tile runs and the arrival counts of the X items
    CKE(upload_vec(e->dBuckets, e->buckets, e->stream));
    if (tiled) {
        const unsigned T = e->nTiles, warps = e->resXThreads / 32u;  // the dedicated X warps of a CTA
        std::vector<unsigned> colourStart;
        for (size_t i = 0; i < e->buckets.size(); i++)
            if (i == 0 || e->buckets[i].colour != e->buckets[i - 1].colour) colourStart.push_back((unsigned)i);
        e->resColours = (unsigned)colourStart.size();
        colourStart.push_back((unsigned)e->buckets.size());
        if (tileOff.size() != e->buckets.size() * (2 * (size_t)T + 1)) return fail("flatten: internal error (tile runs)");
        // arrivals on the X counter: one per CTA that owns X work in the phase -- integration phase (global-homed particles), then every colour
        std::vector<unsigned> xArrive(1 + e->resColours, 0u);
        (void)warps;
        for (unsigned t = 0; t < T; t++) xArrive[0] += (pl.tileStart[t + 1] - pl.tileStart[t] - pl.tileSmem[t]) ? 1u : 0u;
        for (unsigned c = 0; c < e->resColours; c++)
            for (unsigned t = 0; t < T; t++) {
                unsigned any = 0;
                for (unsigned bi = colourStart[c]; bi < colourStart[c + 1]; bi++) {
                    const unsigned *off = &tileOff[(size_t)bi * (2 * T + 1) + 2 * t];
                    any |= (off[1] - off[0]);
                }
                xArrive[1 + c] += any ? 1u : 0u;
            }
        unsigned long long perSweep = 0;
        for (unsigned c = 0; c < e->resColours; c++) perSweep += xArrive[1 + c];
        e->xArriveInt.assign(1, xArrive[0]); e->xArriveCol.assign(1, perSweep);
        CKE(upload_vec(e->dColourStart, colourStart, e->stream));
        CKE(upload_vec(e->dTileOff, tileOff, e->stream));
        CKE(upload_vec(e->dXArrive, xArrive, e->stream));
        CKE(e->dXCounter.alloc(256));
        CK(cudaMemsetAsync(e->dXCounter.p, 0, 256, e->stream));
        e->xBase = 0;
        if (getenv("PBD_B200_VERBOSE")) {
            unsigned long long xItems = 0, mxRun = 0;
            for (size_t bi = 0; bi < e->buckets.size(); bi++)
                for (unsigned t = 0; t < T; t++) {
                    const unsigned *off = &tileOff[bi * (2 * (size_t)T + 1) + 2 * t];
                    xItems += off[1] - off[0];
                    mxRun = std::max<unsigned long long>(mxRun, off[2] - off[0]);
                }
            fprintf(stderr, "[pbd_b200] resident: %u colours, %zu buckets, %.2f %% X items, largest run of a tile in a bucket %llu (mean %.0f), X arrivals per sweep %llu\n",
                    e->resColours, e->buckets.size(), 100.0 * xItems / std::max(1u, e->numConstraints), mxRun,
                    (double)e->numConstraints / std::max<size_t>(1, e->buckets.size()) / T, perSweep);
        }
    }
    CK(cudaStreamSynchronize(e->stream));

    lap("phase tables");
    e->stats.num_constraints = e->numConstraints;
    e->stats.num_groups = nGroups;
    e->stats.num_buckets = (unsigned)e->buckets.size();
    // algorithmic bytes of one step: sweeps + prologue/epilogue per particle per substep (integrate 48 read + 64 write
    // when lastX is tracked, velocity update 32 (+16 second order) read + 16 write)  -- SURVEY.md section 8d
    e->stats.bytes_per_step = bytesPerSweep;  // finalised in pbd_get_stats with the current parameters
    e->imageDirty = false;
    return 0;
}

// ------------------------------------------------------------------------------------------------------------
// step drivers
// ------------------------------------------------------------------------------------------------------------
// Block size of a projection launch (kProjectThreads is only the compiled upper bound).  Measured on B200 (profiles/README.md
// section 3): 128 threads beat 256 on every config (more, smaller CTAs: faster ramp-up and drain of each dependent launch); a
// launch that would not even give every SM one CTA is spread further, down to one warp per CTA, because such phases are pure
// latency chains (cfg1, cfg3).  PBD_B200_BLOCK=<n> pins the size (development knob).
static unsigned project_block(const pbd_engine *e, unsigned count) {
    static const int pinned = [] { const char *g = getenv("PBD_B200_BLOCK"); return g ? atoi(g) : 0; }();
    if (pinned >= 32 && pinned <= kProjectThreads) return (unsigned)pinned & ~31u;
    const unsigned perSM = (count + (unsigned)e->smCount - 1) / (unsigned)e->smCount;
    return std::max(32u, std::min(128u, (perSM + 31u) & ~31u));
}

static int launch_bucket(pbd_engine *e, const Bucket &b, float h, int iterZero, cudaStream_t s) {
    float4 *pos = (float4 *)e->pos.p;
    const TypeArrays &a = e->dev[b.type].arrays;
    const unsigned block = project_block(e, b.count);
    const unsigned grid = nblk(b.count, block);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(block); cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = e->usePDL ? 1 : 0;
    cudaError_t le = cudaSuccess;
#define LBV(T, V) (e->gatherCA ? cudaLaunchKernelEx(&cfg, k_project<T, true, V>, pos, a, b.first, b.count, h, iterZero) \
                                : cudaLaunchKernelEx(&cfg, k_project<T, false, V>, pos, a, b.first, b.count, h, iterZero))
#define LB(T) case T: le = LBV(T, 0); break;
    switch (b.type) {
    case PBD_ISOBENDING: le = a.variant ? LBV(PBD_ISOBENDING, 1) : LBV(PBD_ISOBENDING, 0); break;
    case PBD_ISOBENDING_XPBD: le = a.variant ? LBV(PBD_ISOBENDING_XPBD, 1) : LBV(PBD_ISOBENDING_XPBD, 0); break;
        LB(PBD_DISTANCE) LB(PBD_DISTANCE_XPBD) LB(PBD_DIHEDRAL)
        LB(PBD_FEMTRIANGLE) LB(PBD_STRAINTRIANGLE) LB(PBD_VOLUME) LB(PBD_VOLUME_XPBD) LB(PBD_FEMTET)
        LB(PBD_FEMTET_XPBD) LB(PBD_STRAINTET) LB(PBD_SHAPEMATCHING) LB(PBD_BALLJOINT) LB(PBD_RB_PARTICLE_BALLJOINT)
    default: return fail("no kernel for constraint type %d", b.type);
    }
#undef LB
#undef LBV
    CK(le);
    return 0;
}

// all buckets [b0, b1) belong to one colour: one launch for up to kMultiSegments of them
static int launch_colour(pbd_engine *e, size_t b0, size_t b1, float h, int iterZero, cudaStream_t s, unsigned long long *launches) {
    // One launch per colour pays off when the colour is small (latency-bound phases: cfg3 14.3 -> 10.65 ms); a large colour is
    // better served by the specialised single-type kernels (cfg2, 250k-constraint colours: 2.92 -> 2.85 ms without merging).
    constexpr unsigned kMergeMaxConstraints = 65536;
    unsigned colourTotal = 0;
    for (size_t i = b0; i < b1; i++) colourTotal += e->buckets[i].count;
    if (b1 - b0 == 1 || !e->mergeColours || colourTotal > kMergeMaxConstraints) {
        for (size_t i = b0; i < b1; i++) { CKE(launch_bucket(e, e->buckets[i], h, iterZero, s)); (*launches)++; }
        return 0;
    }
    for (size_t c0 = b0; c0 < b1; c0 += kMultiSegments) {
        const size_t c1 = std::min(b1, c0 + (size_t)kMultiSegments);
        MultiArgs m{};
        m.nSeg = (int)(c1 - c0);
        unsigned blocks = 0, total = 0;
        for (size_t i = c0; i < c1; i++) total += e->buckets[i].count;
        const unsigned block = project_block(e, total);
        for (size_t i = c0; i < c1; i++) {
            const Bucket &b = e->buckets[i];
            const int k = (int)(i - c0);
            m.type[k] = b.type; m.first[k] = b.first; m.count[k] = b.count; m.blockStart[k] = blocks;
            m.arrays[k] = e->dev[b.type].arrays;
            blocks += nblk(b.count, block);
        }
        for (int k = m.nSeg; k <= kMultiSegments; k++) m.blockStart[k] = blocks;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(blocks); cfg.blockDim = dim3(block); cfg.stream = s;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = e->usePDL ? 1 : 0;
        float4 *pos = (float4 *)e->pos.p;
        CK(e->gatherCA ? cudaLaunchKernelEx(&cfg, k_project_multi<true>, pos, m, h, iterZero)
                       : cudaLaunchKernelEx(&cfg, k_project_multi<false>, pos, m, h, iterZero));
        (*launches)++;
    }
    return 0;
}

// prologue / epilogue launches share the PDL attribute so that the whole step is one programmatic dependency chain
template <typename... KArgs, typename... Args>
static cudaError_t launch_particles(pbd_engine *e, cudaStream_t s, void (*kernel)(KArgs...), unsigned n, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((n + 255) / 256); cfg.blockDim = dim3(256); cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = e->usePDL ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, args...);
}

static inline int track_last(const pbd_engine *e) { return 1; }  // lastX is part of the reference's particle state

// one TimeStepController::step as individual launches on stream s; returns the number of kernels launched
static int enqueue_step_launches(pbd_engine *e, cudaStream_t s, unsigned long long *launches) {
    const float h = e->dt / (float)e->subSteps;  // TimeStepController.cpp:91
    const float invH = (float)(1.0 / (double)h);
    const unsigned n = e->n;
    unsigned long long L = 0;
    RbState rb{(float4 *)e->rbX.p, (float4 *)e->rbQ.p, (float4 *)e->rbV.p, (float4 *)e->rbW.p, (float4 *)e->rbOldX.p, (float4 *)e->rbLastX.p,
               (float4 *)e->rbOldQ.p, (float4 *)e->rbLastQ.p, (const float4 *)e->rbI.p, (const float4 *)e->rbIinv.p, e->nRb};
    for (unsigned sub = 0; sub < e->subSteps; sub++) {
        if (e->nRb) { CK(launch_particles(e, s, k_rb_integrate, e->nRb, rb, h, e->g[0], e->g[1], e->g[2])); L++; }
        if (n) {
            CK(launch_particles(e, s, k_integrate, n, (float4 *)e->pos.p, (float4 *)e->vel.p, (float4 *)e->oldp.p, (float4 *)e->lastp.p, n, h, e->g[0], e->g[1], e->g[2], track_last(e)));
            L++;
        }
        for (unsigned it = 0; it < e->maxIter; it++)
            for (size_t b0 = 0; b0 < e->buckets.size();) {
                size_t b1 = b0 + 1;
                while (b1 < e->buckets.size() && e->buckets[b1].colour == e->buckets[b0].colour) b1++;
                CKE(launch_colour(e, b0, b1, h, it == 0, s, &L));
                b0 = b1;
            }
        if (n) {
            CK(launch_particles(e, s, k_velocity, n, (const float4 *)e->pos.p, (float4 *)e->vel.p, (const float4 *)e->oldp.p, (const float4 *)e->lastp.p, n, invH, e->velMethod));
            L++;
        }
        if (e->nRb) { CK(launch_particles(e, s, k_rb_velocity, e->nRb, rb, invH, (float)(2.0 / (double)h), e->velMethod)); L++; }
    }
    *launches = L;
    return 0;
}

// One step as one launch of k_step_resident: grid = nTiles CTAs in clusters of resC, one CTA per SM, all co-resident
// (the X items of different clusters wait for each other).
static int launch_resident(pbd_engine *e, cudaStream_t s, ResidentArgs &ra) {
    const size_t smem = resident_smem_bytes(ra.tileCap, ra.nBuckets, ra.nColours);
    if (smem > kMaxDynamicSmem) return fail("resident mode: a CTA needs %zu bytes of shared memory (tile of %u particles + phase tables), %zu available", smem, ra.tileCap, kMaxDynamicSmem);
    if (e->resG > 1 && !e->resChecked) {
        int mc = 0;
        CKE(resident_max_clusters(e, e->resC, smem, &mc));
        if ((unsigned)mc < e->resG)
            return fail("resident mode: the device runs %d clusters of %u CTAs at a time, the scene needs %u co-resident", mc, e->resC, e->resG);
        e->resChecked = true;
    }
    return with_resident_kernel(e, e->resC, [&](auto kernel) -> int {
        CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxDynamicSmem));
        if (e->resC > 8) CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
        cudaLaunchConfig_t cfg; cudaLaunchAttribute attr[1];
        resident_launch_config(e, e->resC, e->nTiles, smem, s, cfg, attr);
        CK(cudaLaunchKernelEx(&cfg, kernel, ra));
        return 0;
    });
}

static int enqueue_step_resident(pbd_engine *e, cudaStream_t s, unsigned long long *launches) {
    const float h = e->dt / (float)e->subSteps;
    ResidentArgs ra;
    ra.pos = (float4 *)e->pos.p; ra.vel = (float4 *)e->vel.p; ra.oldp = (float4 *)e->oldp.p; ra.lastp = (float4 *)e->lastp.p;
    ra.buckets = (const Bucket *)e->dBuckets.p;
    ra.colourStart = (const unsigned *)e->dColourStart.p; ra.tileOff = (const unsigned *)e->dTileOff.p;
    ra.tileStart = (const unsigned *)e->dTileStart.p; ra.tileSmem = (const unsigned *)e->dTileSmem.p; ra.xArrive = (const unsigned *)e->dXArrive.p;
    ra.nBuckets = (unsigned)e->buckets.size(); ra.nColours = e->resColours; ra.nTiles = e->nTiles; ra.subSteps = e->subSteps; ra.maxIter = e->maxIter;
    ra.tileCap = e->resTileCap; ra.xThreads = e->resXThreads; ra.clusterSize = e->resC;
    {   // L2 prefetch of the operand runs pays when the constraint stream of a sweep does not stay in L2 (126 MB) anyway
        static const char *g = getenv("PBD_B200_L2PREFETCH");
        double streamBytes = 0.0;
        for (int t = 0; t < PBD_NUM_TYPES; t++) {
            const TypeShape sh = type_shape(t);
            streamBytes += (double)e->dev[t].count * (4.0 * sh.nBodies + 16.0 * sh.nGeoV + 4.0 * sh.nGeoS + (sh.xpbd ? 4.0 : 0.0));
        }
        ra.l2Prefetch = g ? atoi(g) : (streamBytes > 48.0e6 ? 1 : 0);
        static const char *pm = getenv("PBD_B200_POLL");
        ra.relaxedPoll = pm ? atoi(pm) : 0;
    }
    ra.h = h; ra.invH = (float)(1.0 / (double)h); ra.twoInvH = (float)(2.0 / (double)h); ra.gx = e->g[0]; ra.gy = e->g[1]; ra.gz = e->g[2];
    ra.secondOrder = e->velMethod;
    ra.xCounter = (unsigned long long *)e->dXCounter.p;
    ra.xBase = e->xBase;
    e->xBase += (unsigned long long)e->subSteps * (e->xArriveInt[0] + (unsigned long long)e->maxIter * e->xArriveCol[0]);
    ra.rb = RbState{(float4 *)e->rbX.p, (float4 *)e->rbQ.p, (float4 *)e->rbV.p, (float4 *)e->rbW.p, (float4 *)e->rbOldX.p, (float4 *)e->rbLastX.p,
                    (float4 *)e->rbOldQ.p, (float4 *)e->rbLastQ.p, (const float4 *)e->rbI.p, (const float4 *)e->rbIinv.p, e->nRb};
    for (int t = 0; t < PBD_NUM_TYPES; t++) ra.types[t] = e->dev[t].arrays;
    *launches = 1;
    ra.trace = nullptr; ra.tracePhases = 0;
    static const char *tracePath = getenv("PBD_B200_TRACE");  // development aid: dump per-phase timelines of one step (tools/trace_resident.py)
    const unsigned kTracePhases = 256;
    if (tracePath) {
        CKE(e->dTrace.alloc((size_t)kTracePhases * e->nTiles * 4 * sizeof(unsigned long long)));
        CK(cudaMemsetAsync(e->dTrace.p, 0, e->dTrace.bytes, s));
        ra.trace = (unsigned long long *)e->dTrace.p; ra.tracePhases = kTracePhases;
    }
    struct TraceDump {  // runs after the launch below has been enqueued (scope exit)
        pbd_engine *e; cudaStream_t s; const char *path; unsigned phases;
        ~TraceDump() {
            if (!path) return;
            cudaStreamSynchronize(s);
            std::vector<unsigned long long> h((size_t)phases * e->nTiles * 4);
            cudaMemcpy(h.data(), e->dTrace.p, h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
            if (FILE *f = fopen(path, "wb")) { fwrite(h.data(), sizeof(unsigned long long), h.size(), f); fclose(f); }
        }
    } dump{e, s, tracePath, kTracePhases};
    return launch_resident(e, s, ra);
}

// Jacobi comparison path (kernels.cuh): per sweep one launch per type over all its constraints + the averaging pass
static int enqueue_step_jacobi(pbd_engine *e, cudaStream_t s, unsigned long long *launches) {
    if (e->nRb || e->dev[PBD_BALLJOINT].count || e->dev[PBD_RB_PARTICLE_BALLJOINT].count)
        return fail("PBD_MODE_JACOBI does not cover rigid-body coupling (use PBD_MODE_GRAPH)");
    const float h = e->dt / (float)e->subSteps;
    const float invH = (float)(1.0 / (double)h);
    const unsigned n = e->n;
    if (n == 0) { *launches = 0; return 0; }
    if (!e->jacobiDelta.p || e->jacobiDelta.bytes < (size_t)n * sizeof(float4)) {
        CKE(e->jacobiDelta.alloc((size_t)n * sizeof(float4)));
        CK(cudaMemsetAsync(e->jacobiDelta.p, 0, (size_t)n * sizeof(float4), s));
    }
    const float4 *pos = (const float4 *)e->pos.p; float4 *delta = (float4 *)e->jacobiDelta.p;
    unsigned long long L = 0;
    for (unsigned sub = 0; sub < e->subSteps; sub++) {
        k_integrate<<<nblk(n, 256), 256, 0, s>>>((float4 *)e->pos.p, (float4 *)e->vel.p, (float4 *)e->oldp.p, (float4 *)e->lastp.p, n, h, e->g[0], e->g[1], e->g[2], 1); L++;
        for (unsigned it = 0; it < e->maxIter; it++) {
            for (int t = 0; t < PBD_BALLJOINT; t++) {
                const unsigned cnt = e->dev[t].count;
                if (!cnt) continue;
                const TypeArrays &a = e->dev[t].arrays;
                const unsigned grid = nblk(cnt, 128);
                const int iz = (it == 0);
#define JB(T, V) k_project_jacobi<T, V><<<grid, 128, 0, s>>>(pos, delta, a, cnt, h, iz)
                switch (t) {
                case PBD_DISTANCE: JB(PBD_DISTANCE, 0); break; case PBD_DISTANCE_XPBD: JB(PBD_DISTANCE_XPBD, 0); break;
                case PBD_DIHEDRAL: JB(PBD_DIHEDRAL, 0); break;
                case PBD_ISOBENDING: if (a.variant) JB(PBD_ISOBENDING, 1); else JB(PBD_ISOBENDING, 0); break;
                case PBD_ISOBENDING_XPBD: if (a.variant) JB(PBD_ISOBENDING_XPBD, 1); else JB(PBD_ISOBENDING_XPBD, 0); break;
                case PBD_FEMTRIANGLE: JB(PBD_FEMTRIANGLE, 0); break; case PBD_STRAINTRIANGLE: JB(PBD_STRAINTRIANGLE, 0); break;
                case PBD_VOLUME: JB(PBD_VOLUME, 0); break; case PBD_VOLUME_XPBD: JB(PBD_VOLUME_XPBD, 0); break;
                case PBD_FEMTET: JB(PBD_FEMTET, 0); break; case PBD_FEMTET_XPBD: JB(PBD_FEMTET_XPBD, 0); break;
                case PBD_STRAINTET: JB(PBD_STRAINTET, 0); break; case PBD_SHAPEMATCHING: JB(PBD_SHAPEMATCHING, 0); break;
                default: break;
                }
#undef JB
                L++;
            }
            k_jacobi_apply<<<nblk(n, 256), 256, 0, s>>>((float4 *)e->pos.p, delta, n); L++;
        }
        k_velocity<<<nblk(n, 256), 256, 0, s>>>((const float4 *)e->pos.p, (float4 *)e->vel.p, (const float4 *)e->oldp.p, (const float4 *)e->lastp.p, n, invH, e->velMethod); L++;
    }
    CK(cudaGetLastError());
    *launches = L;
    return 0;
}

// ------------------------------------------------------------------------------------------------------------
// contact path (contacts.cuh)
// ------------------------------------------------------------------------------------------------------------
extern "C" int pbd_set_colliders(pbd_engine *e, unsigned nP, const pbd_particle_collider *pc, unsigned nR, const pbd_rigid_collider *rc) {
    if (!e || (nP && !pc) || (nR && !rc)) return fail("pbd_set_colliders: null argument");
    CKE(use(e));
    if (nR > (unsigned)kMaxRigidColliders) return fail("pbd_set_colliders: %u rigid colliders (the contact kernel keeps up to %d contacts per particle)", nR, kMaxRigidColliders);
    std::vector<ParticleCollider> P(nP);
    std::vector<RigidCollider> R(nR);
    std::vector<unsigned> start(nP + 1, 0u);
    for (unsigned i = 0; i < nP; i++) {
        if ((unsigned long long)pc[i].offset + pc[i].count > e->n) return fail("pbd_set_colliders: particle collider %u covers [%u, %u), the engine holds %u particles", i, pc[i].offset, pc[i].offset + pc[i].count, e->n);
        P[i].offset = pc[i].offset; P[i].count = pc[i].count; P[i].restitution = pc[i].restitution; P[i].friction = pc[i].friction;
        start[i + 1] = start[i] + pc[i].count;
    }
    for (unsigned i = 0; i < nR; i++) {
        const pbd_rigid_collider &c = rc[i];
        if (c.shape < 0 || c.shape >= kNumShapes) return fail("pbd_set_colliders: rigid collider %u has unknown shape %d", i, c.shape);
        if (c.body >= e->nRb) return fail("pbd_set_colliders: rigid collider %u refers to rigid body %u, the engine holds %u (pbd_set_rigid_bodies first)", i, c.body, e->nRb);
        if (e->rbMass[c.body] != 0.0f)
            return fail("pbd_set_colliders: rigid body %u has mass %g; contacts with dynamic bodies couple through the body and stay on the CPU time step (static colliders only)", c.body, e->rbMass[c.body]);
        RigidCollider &d = R[i];
        d.shape = c.shape; d.body = c.body; d.thickness = c.thickness; d.invert = c.invert_sdf ? -1.0f : 1.0f; d.restitution = c.restitution; d.friction = c.friction;
        for (int k = 0; k < 3; k++) { d.dim[k] = c.dim[k]; d.v1[k] = c.v1[k]; d.v2[k] = c.v2[k]; d.aabbMin[k] = c.aabb_min[k]; d.aabbMax[k] = c.aabb_max[k]; }
        for (int k = 0; k < 9; k++) d.R[k] = c.R[k];
    }
    CK(cudaStreamSynchronize(e->stream));
    e->pColliders.swap(P); e->rColliders.swap(R);
    e->contactTotal = start[nP];
    if (nP) { CKE(upload_vec(e->dPColliders, e->pColliders, e->stream)); CKE(upload_vec(e->dRangeStart, start, e->stream)); }
    if (nR) CKE(upload_vec(e->dRColliders, e->rColliders, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    return 0;
}
extern "C" int pbd_set_contact_params(pbd_engine *e, float tolerance, float stiffness, unsigned maxIterationsV) {
    if (!e) return fail("null engine");
    e->contactTolerance = tolerance; e->contactStiffness = stiffness; e->maxIterV = maxIterationsV;
    return 0;
}
extern "C" int pbd_record_contacts(pbd_engine *e, unsigned capacity) {
    if (!e) return fail("null engine");
    CKE(use(e));
    CK(cudaStreamSynchronize(e->stream));
    e->contactCap = capacity;
    if (capacity) {
        CKE(e->dContacts.alloc((size_t)capacity * sizeof(ContactRecord)));
        CKE(e->dContactCount.alloc(sizeof(unsigned)));
        CK(cudaMemset(e->dContactCount.p, 0, sizeof(unsigned)));
    }
    return 0;
}
extern "C" int pbd_get_contacts(pbd_engine *e, pbd_contact *out, unsigned capacity, unsigned *count) {
    if (!e || !count) return fail("pbd_get_contacts: null argument");
    CKE(use(e));
    *count = 0;
    if (!e->contactCap) return fail("pbd_get_contacts: recording is off (pbd_record_contacts)");
    CK(cudaStreamSynchronize(e->stream));
    unsigned found = 0;
    CK(cudaMemcpy(&found, e->dContactCount.p, sizeof(unsigned), cudaMemcpyDeviceToHost));
    *count = found;
    const unsigned kept = std::min(found, e->contactCap);
    static_assert(sizeof(pbd_contact) == sizeof(ContactRecord), "pbd_contact mirrors ContactRecord");
    std::vector<pbd_contact> tmp(kept);
    if (kept) CK(cudaMemcpy(tmp.data(), e->dContacts.p, (size_t)kept * sizeof(pbd_contact), cudaMemcpyDeviceToHost));
    std::sort(tmp.begin(), tmp.end(), [](const pbd_contact &a, const pbd_contact &b) { return a.particle != b.particle ? a.particle < b.particle : a.body < b.body; });
    if (out) for (unsigned i = 0; i < std::min(kept, capacity); i++) out[i] = tmp[i];
    return 0;
}
// after the substeps of a step: collision detection + velocity-level contact solve (TimeStepController.cpp:189-196)
static int enqueue_contacts(pbd_engine *e, cudaStream_t s, unsigned long long *launches) {
    if (e->rColliders.empty() || e->contactTotal == 0) return 0;
    for (const RigidCollider &c : e->rColliders)  // the bodies may have been replaced since pbd_set_colliders
        if (c.body >= e->nRb || e->rbMass[c.body] != 0.0f) return fail("contact path: collider on rigid body %u, which is missing or not static any more (pbd_set_colliders again)", c.body);
    for (const ParticleCollider &c : e->pColliders)
        if ((unsigned long long)c.offset + c.count > e->n) return fail("contact path: a particle collider covers particles beyond the %u the engine holds", e->n);
    ContactArgs a;
    a.pos = (float4 *)e->pos.p; a.vel = (float4 *)e->vel.p; a.slot = (const unsigned *)e->dSlot.p;
    a.rbX = (const float4 *)e->rbX.p; a.rbV = (const float4 *)e->rbV.p; a.rbW = (const float4 *)e->rbW.p;
    a.rigid = (const RigidCollider *)e->dRColliders.p; a.nRigid = (unsigned)e->rColliders.size();
    a.ranges = (const ParticleCollider *)e->dPColliders.p; a.nRanges = (unsigned)e->pColliders.size();
    a.rangeStart = (const unsigned *)e->dRangeStart.p; a.total = e->contactTotal;
    a.tolerance = e->contactTolerance; a.stiffness = e->contactStiffness; a.maxIterV = e->maxIterV;
    a.record = e->contactCap ? (ContactRecord *)e->dContacts.p : nullptr; a.recordCount = (unsigned *)e->dContactCount.p; a.recordCap = e->contactCap;
    if (e->contactCap) CK(cudaMemsetAsync(e->dContactCount.p, 0, sizeof(unsigned), s));
    k_contacts<<<(a.total + 127u) / 128u, 128, 0, s>>>(a);
    CK(cudaGetLastError());
    *launches += 1;
    return 0;
}

static int ensure_graph(pbd_engine *e, unsigned long long *launchesPerStep) {
    if (e->graphValid) return 0;
    cudaGraph_t graph = nullptr;
    CK(cudaStreamBeginCapture(e->stream, cudaStreamCaptureModeThreadLocal));
    unsigned long long L = 0;
    int rc = enqueue_step_launches(e, e->stream, &L);
    cudaError_t err = cudaStreamEndCapture(e->stream, &graph);
    if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
    if (err != cudaSuccess) return fail("cudaStreamEndCapture -> %s", cudaGetErrorString(err));
    err = cudaGraphInstantiate(&e->graphExec, graph, 0);
    cudaGraphDestroy(graph);
    if (err != cudaSuccess) return fail("cudaGraphInstantiate -> %s", cudaGetErrorString(err));
    e->graphValid = true;
    *launchesPerStep = L;
    return 0;
}

extern "C" int pbd_step(pbd_engine *e, unsigned nSteps) {
    if (!e) return fail("null engine");
    CKE(use(e));
    CKE(flatten(e));
    CK(cudaEventRecord(e->evStart, e->stream));
    for (unsigned s = 0; s < nSteps; s++) {
        unsigned long long L = 0;
        if (e->active == PBD_MODE_LAUNCH) {
            CKE(enqueue_step_launches(e, e->stream, &L));
        } else if (e->active == PBD_MODE_RESIDENT) {
            int rc = enqueue_step_resident(e, e->stream, &L);
            if (rc && e->mode == PBD_MODE_AUTO) {  // e.g. the clusters cannot be co-resident on this device: run the step in graph mode instead
                e->autoNoResident = true; e->imageDirty = true;
                CKE(flatten(e));
                unsigned long long LL = 0;
                if (!e->graphValid) { CKE(ensure_graph(e, &LL)); e->graphLaunches = LL; }
                CK(cudaGraphLaunch(e->graphExec, e->stream));
                L = e->graphLaunches; rc = 0;
            }
            CKE(rc);
        } else if (e->active == PBD_MODE_JACOBI) {
            CKE(enqueue_step_jacobi(e, e->stream, &L));
        } else {
            unsigned long long LL = 0;
            if (!e->graphValid) { CKE(ensure_graph(e, &LL)); e->graphLaunches = LL; }
            CK(cudaGraphLaunch(e->graphExec, e->stream));
            L = e->graphLaunches;
        }
        CKE(enqueue_contacts(e, e->stream, &L));
        e->stats.kernel_launches += L;
        e->stats.steps++;
        e->stats.projections += (unsigned long long)e->numConstraints * e->subSteps * e->maxIter;
    }
    CK(cudaEventRecord(e->evStop, e->stream));
    e->timingPending = true;
    return 0;
}

extern "C" int pbd_sync(pbd_engine *e) {
    if (!e) return fail("null engine");
    CKE(use(e));
    CK(cudaStreamSynchronize(e->stream));
    if (e->timingPending) {
        float ms = 0.0f;
        if (cudaEventElapsedTime(&ms, e->evStart, e->evStop) == cudaSuccess) e->stats.last_step_ms = ms;
        e->timingPending = false;
    }
    return 0;
}

extern "C" int pbd_pin_host(void *ptr, size_t bytes) {
    if (!ptr || !bytes) return fail("pbd_pin_host: null argument");
    const cudaError_t err = cudaHostRegister(ptr, bytes, cudaHostRegisterPortable);
    if (err != cudaSuccess) { cudaGetLastError(); return fail("cudaHostRegister -> %s", cudaGetErrorString(err)); }  // clear the sticky per-thread error: a later CK(cudaGetLastError()) must not see it
    return 0;
}
extern "C" int pbd_unpin_host(void *ptr) {
    if (!ptr) return 0;
    const cudaError_t err = cudaHostUnregister(ptr);
    if (err != cudaSuccess) { cudaGetLastError(); return fail("cudaHostUnregister -> %s", cudaGetErrorString(err)); }
    return 0;
}

extern "C" int pbd_step_host(pbd_engine *e, unsigned nSteps, const float *x_in, const float *v_in, float *x_out, float *v_out) {
    if (!e) return fail("null engine");
    CKE(use(e));
    if (e->n == 0) return pbd_step(e, nSteps);
    const size_t bytes = (size_t)e->n * 3 * sizeof(float);
    // two staging areas so that x and v uploads do not serialise on a host sync
    CKE(e->stage.alloc(bytes));
    DevBuf &stage2 = e->stage2;
    CKE(stage2.alloc(bytes));
    if (x_in) {
        CK(cudaMemcpyAsync(e->stage.p, x_in, bytes, cudaMemcpyHostToDevice, e->stream));
        k_pack3<<<nblk(e->n, 256), 256, 0, e->stream>>>((const float *)e->stage.p, (float4 *)e->pos.p, e->n, 1, (const unsigned *)e->dSlot.p);
    }
    if (v_in) {
        CK(cudaMemcpyAsync(stage2.p, v_in, bytes, cudaMemcpyHostToDevice, e->stream));
        k_pack3<<<nblk(e->n, 256), 256, 0, e->stream>>>((const float *)stage2.p, (float4 *)e->vel.p, e->n, 1, (const unsigned *)e->dSlot.p);
    }
    CK(cudaGetLastError());
    CKE(pbd_step(e, nSteps));
    if (x_out) {
        k_unpack3<<<nblk(e->n, 256), 256, 0, e->stream>>>((const float4 *)e->pos.p, (float *)e->stage.p, e->n, (const unsigned *)e->dSlot.p);
        CK(cudaMemcpyAsync(x_out, e->stage.p, bytes, cudaMemcpyDeviceToHost, e->stream));
    }
    if (v_out) {
        k_unpack3<<<nblk(e->n, 256), 256, 0, e->stream>>>((const float4 *)e->vel.p, (float *)stage2.p, e->n, (const unsigned *)e->dSlot.p);
        CK(cudaMemcpyAsync(v_out, stage2.p, bytes, cudaMemcpyDeviceToHost, e->stream));
    }
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(e->stream));
    return 0;
}

// Pipelined form of pbd_step_host: the upload of call k+1 and the download of call k-1 overlap the projection kernels of call k
// (three streams, two staging slots, ordering by events only -- the host never blocks here).
extern "C" int pbd_step_host_async(pbd_engine *e, unsigned nSteps, const float *x_in, const float *v_in, float *x_out, float *v_out) {
    if (!e) return fail("null engine");
    CKE(use(e));
    if (e->n == 0) return pbd_step(e, nSteps);
    const size_t bytes = (size_t)e->n * 3 * sizeof(float);
    auto &P = e->pipe;
    if (!P.ready) {
        CK(cudaStreamCreateWithFlags(&P.up, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&P.down, cudaStreamNonBlocking));
        for (int s = 0; s < 2; s++)
            for (cudaEvent_t *ev : {&P.uploaded[s], &P.consumed[s], &P.produced[s], &P.downloaded[s]}) CK(cudaEventCreateWithFlags(ev, cudaEventDisableTiming));
        P.ready = true;
    }
    const int s = (int)(P.issued & 1);
    const bool reuse = P.issued >= 2;  // the slot was used by call k-2: its consumers are ordered before us by events
    const unsigned *slot = (const unsigned *)e->dSlot.p;
    if (x_in || v_in) {
        if (reuse) CK(cudaStreamWaitEvent(P.up, P.consumed[s], 0));
        if (x_in) { CKE(P.inX[s].alloc(bytes)); CK(cudaMemcpyAsync(P.inX[s].p, x_in, bytes, cudaMemcpyHostToDevice, P.up)); }
        if (v_in) { CKE(P.inV[s].alloc(bytes)); CK(cudaMemcpyAsync(P.inV[s].p, v_in, bytes, cudaMemcpyHostToDevice, P.up)); }
        CK(cudaEventRecord(P.uploaded[s], P.up));
        CK(cudaStreamWaitEvent(e->stream, P.uploaded[s], 0));
        if (x_in) k_pack3<<<nblk(e->n, 256), 256, 0, e->stream>>>((const float *)P.inX[s].p, (float4 *)e->pos.p, e->n, 1, slot);
        if (v_in) k_pack3<<<nblk(e->n, 256), 256, 0, e->stream>>>((const float *)P.inV[s].p, (float4 *)e->vel.p, e->n, 1, slot);
        CK(cudaGetLastError());
    }
    CK(cudaEventRecord(P.consumed[s], e->stream));
    CKE(pbd_step(e, nSteps));
    if (x_out || v_out) {
        if (reuse) CK(cudaStreamWaitEvent(e->stream, P.downloaded[s], 0));
        if (x_out) { CKE(P.outX[s].alloc(bytes)); k_unpack3<<<nblk(e->n, 256), 256, 0, e->stream>>>((const float4 *)e->pos.p, (float *)P.outX[s].p, e->n, slot); }
        if (v_out) { CKE(P.outV[s].alloc(bytes)); k_unpack3<<<nblk(e->n, 256), 256, 0, e->stream>>>((const float4 *)e->vel.p, (float *)P.outV[s].p, e->n, slot); }
        CK(cudaGetLastError());
        CK(cudaEventRecord(P.produced[s], e->stream));
        CK(cudaStreamWaitEvent(P.down, P.produced[s], 0));
        if (x_out) CK(cudaMemcpyAsync(x_out, P.outX[s].p, bytes, cudaMemcpyDeviceToHost, P.down));
        if (v_out) CK(cudaMemcpyAsync(v_out, P.outV[s].p, bytes, cudaMemcpyDeviceToHost, P.down));
    }
    CK(cudaEventRecord(P.downloaded[s], P.down));
    P.issued++;
    return 0;
}

extern "C" int pbd_step_host_wait(pbd_engine *e, unsigned lag) {
    if (!e) return fail("null engine");
    CKE(use(e));
    auto &P = e->pipe;
    if (!P.ready || P.issued == 0) return 0;
    if (lag > 1) return fail("pbd_step_host_wait: lag %u (the pipeline has two slots: 0 = everything, 1 = all but the newest call)", lag);
    if (lag == 0) {
        CK(cudaStreamSynchronize(e->stream));
        CK(cudaStreamSynchronize(P.down));
        return 0;
    }
    if (P.issued < 2) return 0;
    CK(cudaEventSynchronize(P.downloaded[(P.issued - 2) & 1]));
    return 0;
}

extern "C" int pbd_get_lambdas(pbd_engine *e, int type, float *dst, unsigned *ids) {
    if (!e || !dst) return fail("null argument");
    if (type < 0 || type >= PBD_NUM_TYPES || !type_shape(type).xpbd) return fail("type %d has no multipliers", type);
    CKE(use(e)); CKE(flatten(e));
    DevType &d = e->dev[type];
    if (d.count == 0) return 0;
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaMemcpy(dst, d.lambda.p, (size_t)d.count * sizeof(float), cudaMemcpyDeviceToHost));
    if (ids) memcpy(ids, d.order.data(), (size_t)d.count * sizeof(unsigned));
    return 0;
}

extern "C" int pbd_get_stats(pbd_engine *e, pbd_stats *out) {
    if (!e || !out) return fail("null argument");
    CKE(use(e)); CKE(flatten(e));
    double sweep = 0.0;
    for (int t = 0; t < PBD_NUM_TYPES; t++) sweep += (double)e->dev[t].count * algorithmic_bytes(t, e->dev[t].arrays.variant);
    // per particle per substep: integrate 48 read + 64 write = 112, velocity update 32 read + 16 write = 48 (SURVEY.md 8d)
    const double perParticle = 112.0 + 48.0 + (e->velMethod ? 16.0 : 0.0);
    e->stats.bytes_per_step = (sweep * e->maxIter + (double)e->n * perParticle) * e->subSteps;
    *out = e->stats;
    return 0;
}

extern "C" int pbd_profile_step(pbd_engine *e, float *msPerType, float *msIntegrate, float *msVelocity, unsigned *launchesPerType) {
    if (!e) return fail("null engine");
    if (e->active == PBD_MODE_RESIDENT || e->active == PBD_MODE_JACOBI || e->mode == PBD_MODE_AUTO) return fail("pbd_profile_step: per-bucket launches do not exist in this mode (select PBD_MODE_GRAPH or PBD_MODE_LAUNCH first)");
    CKE(use(e)); CKE(flatten(e));
    CK(cudaStreamSynchronize(e->stream));
    // One event between every pair of consecutive launches, all recorded in stream order without host synchronisation
    // (a host sync per launch would time the idle-launch latency, not the kernel); read back after one final sync.
    const size_t nLaunch = (size_t)e->subSteps * (4 + (size_t)e->maxIter * e->buckets.size());
    RbState rb{(float4 *)e->rbX.p, (float4 *)e->rbQ.p, (float4 *)e->rbV.p, (float4 *)e->rbW.p, (float4 *)e->rbOldX.p, (float4 *)e->rbLastX.p,
               (float4 *)e->rbOldQ.p, (float4 *)e->rbLastQ.p, (const float4 *)e->rbI.p, (const float4 *)e->rbIinv.p, e->nRb};
    std::vector<cudaEvent_t> ev(nLaunch + 1);
    for (auto &x : ev) CK(cudaEventCreate(&x));
    std::vector<int> what(nLaunch);  // >= 0: type, -1 integrate, -2 velocity
    const float h = e->dt / (float)e->subSteps;
    const float invH = (float)(1.0 / (double)h);
    const unsigned n = e->n;
    const bool pdl = e->usePDL;
    e->usePDL = false;  // serialise: each kernel's duration must be its own
    size_t k = 0;
    int rc = 0;
    CK(cudaEventRecord(ev[0], e->stream));
    for (unsigned sub = 0; sub < e->subSteps && !rc; sub++) {
        if (e->nRb) { k_rb_integrate<<<nblk(e->nRb, 32), 32, 0, e->stream>>>(rb, h, e->g[0], e->g[1], e->g[2]); what[k] = -1; cudaEventRecord(ev[++k], e->stream); }
        if (n) {
            k_integrate<<<nblk(n, 256), 256, 0, e->stream>>>((float4 *)e->pos.p, (float4 *)e->vel.p, (float4 *)e->oldp.p, (float4 *)e->lastp.p, n, h, e->g[0], e->g[1], e->g[2], track_last(e));
            what[k] = -1; cudaEventRecord(ev[++k], e->stream);
        }
        for (unsigned it = 0; it < e->maxIter && !rc; it++)
            for (const Bucket &bk : e->buckets) {
                rc = launch_bucket(e, bk, h, it == 0, e->stream);
                if (rc) break;
                what[k] = bk.type; cudaEventRecord(ev[++k], e->stream);
            }
        if (n && !rc) {
            k_velocity<<<nblk(n, 256), 256, 0, e->stream>>>((const float4 *)e->pos.p, (float4 *)e->vel.p, (const float4 *)e->oldp.p, (const float4 *)e->lastp.p, n, invH, e->velMethod);
            what[k] = -2; cudaEventRecord(ev[++k], e->stream);
        }
        if (e->nRb && !rc) { k_rb_velocity<<<nblk(e->nRb, 32), 32, 0, e->stream>>>(rb, invH, (float)(2.0 / (double)h), e->velMethod); what[k] = -2; cudaEventRecord(ev[++k], e->stream); }
    }
    e->usePDL = pdl;
    cudaError_t se = cudaStreamSynchronize(e->stream);
    if (msPerType) for (int t = 0; t < PBD_NUM_TYPES; t++) msPerType[t] = 0.0f;
    if (launchesPerType) for (int t = 0; t < PBD_NUM_TYPES; t++) launchesPerType[t] = 0;
    float mi = 0.0f, mv = 0.0f;
    if (!rc && se == cudaSuccess)
        for (size_t i = 0; i < k; i++) {
            float ms = 0.0f;
            cudaEventElapsedTime(&ms, ev[i], ev[i + 1]);
            if (what[i] == -1) mi += ms;
            else if (what[i] == -2) mv += ms;
            else { if (msPerType) msPerType[what[i]] += ms; if (launchesPerType) launchesPerType[what[i]]++; }
        }
    for (auto &x : ev) cudaEventDestroy(x);
    if (rc) return rc;
    if (se != cudaSuccess) return fail("pbd_profile_step: %s", cudaGetErrorString(se));
    if (msIntegrate) *msIntegrate = mi;
    if (msVelocity) *msVelocity = mv;
    e->stats.steps++;
    e->stats.projections += (unsigned long long)e->numConstraints * e->subSteps * e->maxIter;
    return 0;
}
