// js/SortWorkerB200.js -- drop-in for src/worker/SortWorker.js of GaussianSplats3D (not run here: no Node.js in the image).
// Same factory signature and the same message protocol (SortWorker.js:83-113, 114-197, 202-256); the wasm module and its
// WebAssembly.Memory are replaced by one gs_engine on a B200 through the N-API addon in this directory.
//
// In the reference:   import { createSortWorker } from './worker/SortWorker.js';          (src/Viewer.js:13)
// With this engine:   import { createSortWorker } from 'gsplat-b200/js/SortWorkerB200.js';
//
// Shared-memory mode (Viewer option sharedMemoryForWorkers, the default): the four views the reference's worker carves out of its
// WebAssembly.Memory -- indexesToSort, sortedIndexes, precomputedDistances, transforms (SortWorker.js:180-191) -- are page-locked host
// buffers from gs_host_alloc, so the main thread fills them in place and the engine reads them with asynchronous copies and no staging.
import { createRequire } from 'module';
const addon = createRequire(import.meta.url)('./build/Release/gsplat_b200.node');

const MaxScenes = 32;                       // Constants.MaxScenes (src/Constants.js:7)

class B200SortWorker {
    constructor() {
        this.onmessage = null;
        this.engine = null;
        this.uploadedSplatCount = 0;
        this.canceled = false;
    }

    _emit(msg) { if (this.onmessage) this.onmessage({ data: msg }); }

    postMessage(data) {
        if (data.centers) {                                       // SortWorker.js:84-98
            addon.uploadCenters(this.engine, data.centers, this.dynamicMode ? data.sceneIndexes : null, data.range.from, data.range.count);
            this.uploadedSplatCount = data.range.from + data.range.count;
        } else if (data.sort) {                                   // SortWorker.js:99-113 -> sort() :31-81
            const s = data.sort;
            const renderCount = Math.min(s.splatRenderCount || 0, this.uploadedSplatCount);
            const sortCount = Math.min(s.splatSortCount || 0, this.uploadedSplatCount);
            const usePrecomputedDistances = !!s.usePrecomputedDistances;
            if (this.canceled) { this.canceled = false; this._emit({ sortCanceled: true }); return; }
            const shared = this.useSharedMemory;
            const params = {
                modelViewProj: s.modelViewProj,
                sortCount, renderCount,
                indexesToSort: shared ? this.indexesToSort : s.indexesToSort,
                transforms: this.dynamicMode ? (shared ? this.transforms : s.transforms) : null,
                usePrecomputedDistances,
                precomputedDistances: usePrecomputedDistances ? (shared ? this.precomputedDistances : s.precomputedDistances) : null,
            };
            let out = this.sortedIndexes;
            if (!shared) {
                if (!this.sortedIndexesOut || this.sortedIndexesOut.length < renderCount) this.sortedIndexesOut = new Uint32Array(renderCount);
                out = this.sortedIndexesOut;
            }
            const t0 = performance.now();
            addon.sort(this.engine, params, out);
            const msg = { sortDone: true, splatSortCount: sortCount, splatRenderCount: renderCount, sortTime: performance.now() - t0 };
            if (!shared) msg.sortedIndexes = out;
            this._emit(msg);
        } else if (data.init) {                                   // SortWorker.js:114-197
            const i = data.init;
            this.useSharedMemory = i.useSharedMemory;
            this.integerBasedSort = i.integerBasedSort;
            this.dynamicMode = i.dynamicMode;
            this.engine = addon.create({ maxSplatCount: i.splatCount, distanceMapRange: i.distanceMapRange,
                                         integerBasedSort: i.integerBasedSort ? 1 : 0, dynamicMode: i.dynamicMode ? 1 : 0,
                                         maxWidth: i.maxWidth || 0, maxHeight: i.maxHeight || 0, device: i.device || 0,
                                         splatRenderMode: i.splatRenderMode || 0 });   // Viewer option splatRenderMode (Viewer.js:199-202)
            const msg = { sortSetupPhase1Complete: true };
            if (this.useSharedMemory) {
                const n = i.splatCount;
                const indexesBuf = addon.hostAlloc(4 * n), sortedBuf = addon.hostAlloc(4 * n);
                const distancesBuf = addon.hostAlloc(4 * n), transformsBuf = addon.hostAlloc(4 * 16 * MaxScenes);
                this.indexesToSort = new Uint32Array(indexesBuf, 0, n);
                this.sortedIndexes = new Uint32Array(sortedBuf, 0, n);
                this.precomputedDistances = i.integerBasedSort ? new Int32Array(distancesBuf, 0, n) : new Float32Array(distancesBuf, 0, n);
                this.transforms = new Float32Array(transformsBuf, 0, 16 * MaxScenes);
                Object.assign(msg, {
                    indexesToSortBuffer: indexesBuf, indexesToSortOffset: 0,
                    sortedIndexesBuffer: sortedBuf, sortedIndexesOffset: 0,
                    precomputedDistancesBuffer: distancesBuf, precomputedDistancesOffset: 0,
                    transformsBuffer: transformsBuf, transformsOffset: 0,
                });
            }
            queueMicrotask(() => this._emit(msg));
        }
    }

    // the reference's Worker has no cancel message; its Viewer only reacts to 'sortCanceled' (Viewer.js:1264-1265).  Offered for hosts that
    // want to drop a queued sort before it starts.
    cancelNextSort() { this.canceled = true; }

    // engine handle for a renderer that shares the device-resident order with this sorter (js/SplatMeshB200.js)
    getEngine() { return this.engine; }

    terminate() { this.engine = null; }                          // the addon's finalizer calls gs_destroy
}

export function createSortWorker(splatCount, useSharedMemory, enableSIMDInSort, integerBasedSort, dynamicMode,
                                 splatSortDistanceMapPrecision = 16, renderOptions = {}) {
    void enableSIMDInSort;                                        // wasm variant choice has no counterpart here
    const worker = new B200SortWorker();
    worker.postMessage({ init: { splatCount, useSharedMemory, integerBasedSort, dynamicMode, distanceMapRange: 1 << splatSortDistanceMapPrecision,
                                 maxWidth: renderOptions.maxWidth, maxHeight: renderOptions.maxHeight, device: renderOptions.device } });
    return worker;
}
