// js/SplatMeshB200.js -- the render half of the drop-in (not run here: no Node.js in the image): takes the arrays the reference's
// SplatMesh builds for its data textures and the uniforms it sets per frame, and renders through the engine instead of WebGL.
//
//   const renderer = new B200SplatRenderer(sortWorker.getEngine());
//   renderer.setSplatData(splatMesh);                 // after SplatMesh.build (SplatMesh.js:306-405): the data-texture source arrays
//   ...per frame, after Viewer.updateSplatMesh() (Viewer.js:651-677):
//   const rgba = renderer.render(splatMesh, camera, renderWidth, renderHeight, splatRenderCount);   // Uint8Array, row 0 = top
//
// Field sources: SplatMesh.splatDataTextures.baseData (SplatMesh.js:741-770: covariances, centers, colors, sphericalHarmonics, sceneIndexes),
// SplatMesh.material.uniforms (SplatMaterial.js:365-527), three.js camera matrices (what WebGLRenderer hands the shader as
// modelViewMatrix / projectionMatrix / cameraPosition / viewMatrix).
import { createRequire } from 'module';
const addon = createRequire(import.meta.url)('./build/Release/gsplat_b200.node');

const GS_COV_F32 = 0, GS_SH_NONE = 0, GS_SH_F16 = 1, GS_SH_U8 = 2, GS_SH_F32 = 3, GS_FRAME_RGBA8 = 1;

function floatBits(f32) { return new Uint32Array(f32.buffer, f32.byteOffset, f32.length); }

export class B200SplatRenderer {
    constructor(engine) { this.engine = engine; this.frame = null; this.frames = null; }

    // centres + colours -> the uvec4 texel of SplatMesh.updateCenterColorsPaddedData (SplatMesh.js:1143-1153)
    setSplatData(splatMesh) {
        const base = splatMesh.splatDataTextures.baseData;
        const n = splatMesh.getSplatCount();
        const centers = floatBits(base.centers), colors = base.colors;
        const cc = new Uint32Array(4 * n);
        for (let i = 0; i < n; i++) {
            cc[4 * i] = (colors[4 * i] | (colors[4 * i + 1] << 8) | (colors[4 * i + 2] << 16) | (colors[4 * i + 3] << 24)) >>> 0;
            cc[4 * i + 1] = centers[3 * i]; cc[4 * i + 2] = centers[3 * i + 1]; cc[4 * i + 3] = centers[3 * i + 2];
        }
        const sh = base.sphericalHarmonics;
        const shDegree = splatMesh.minSphericalHarmonicsDegree || 0;
        let shFormat = GS_SH_NONE;
        if (sh && shDegree > 0) shFormat = (sh instanceof Uint8Array) ? GS_SH_U8 : ((sh instanceof Uint16Array) ? GS_SH_F16 : GS_SH_F32);
        // SplatRenderMode.TwoD (the engine was created with splatRenderMode: 1): the scale/rotation texture of
        // SplatMesh.updateScaleRotationsPaddedData (SplatMesh.js:1150-1170), 6 floats per splat, instead of covariances
        let scaleRotations = null;
        if (splatMesh.splatRenderMode === 1) {
            scaleRotations = new Float32Array(6 * n);
            for (let i = 0; i < n; i++) {
                for (let k = 0; k < 3; k++) scaleRotations[6 * i + k] = base.scales[3 * i + k];
                for (let k = 0; k < 3; k++) scaleRotations[6 * i + 3 + k] = base.rotations[4 * i + k];
            }
        }
        addon.uploadSplatData(this.engine, {
            from: 0, count: n, centersColors: cc, scaleRotations,
            covariances: base.covariances || null, covFormat: (base.covariances instanceof Uint16Array) ? 1 : GS_COV_F32,
            sphericalHarmonics: shFormat === GS_SH_NONE ? null : sh, shFormat, shDegree,
            sceneIndexes: splatMesh.dynamicMode ? base.sceneIndexes : null,
        });
    }

    // a .ksplat file can skip all of the above: decoded on the GPU into splat data AND sorter centres (gs_upload_ksplat)
    setSplatDataFromKSplat(arrayBuffer, options = {}) { return addon.uploadKsplat(this.engine, arrayBuffer, options); }

    uniformsFor(splatMesh, camera, width, height) {
        const u = splatMesh.material.uniforms;
        const modelView = camera.matrixWorldInverse.clone().multiply(splatMesh.matrixWorld);
        const out = {
            modelView: modelView.elements, projection: camera.projectionMatrix.elements,
            cameraPosition: camera.position.toArray(), focal: [u.focal.value.x, u.focal.value.y], viewport: [u.viewport.value.x, u.viewport.value.y],
            inverseFocalAdjustment: u.inverseFocalAdjustment.value, orthoZoom: u.orthoZoom.value, orthographicMode: u.orthographicMode.value,
            splatScale: u.splatScale.value, pointCloudModeEnabled: u.pointCloudModeEnabled.value,
            sphericalHarmonicsDegree: u.sphericalHarmonicsDegree.value, antialiased: splatMesh.antialiased ? 1 : 0,
            kernel2DSize: splatMesh.kernel2DSize, maxScreenSpaceSplatSize: splatMesh.maxScreenSpaceSplatSize,
            sphericalHarmonics8BitCompressionRangeMin: u.sphericalHarmonics8BitCompressionRangeMin.value,
            sphericalHarmonics8BitCompressionRangeMax: u.sphericalHarmonics8BitCompressionRangeMax.value,
            sceneCount: u.sceneCount.value, fadeInComplete: u.fadeInComplete.value, sceneCenter: u.sceneCenter.value.toArray(),
            visibleRegionFadeStartRadius: u.visibleRegionFadeStartRadius.value,
            dynamicMode: splatMesh.dynamicMode ? 1 : 0, enableOptionalEffects: splatMesh.enableOptionalEffects ? 1 : 0,
        };
        if (splatMesh.dynamicMode) {
            const t = new Float32Array(16 * 32);
            for (let s = 0; s < splatMesh.scenes.length; s++) t.set(splatMesh.getScene(s).transform.elements, 16 * s);
            out.transforms = t;
            out.viewMatrix = camera.matrixWorldInverse.elements;
        }
        if (splatMesh.enableOptionalEffects) {
            out.sceneOpacity = u.sceneOpacity.value; out.sceneVisibility = u.sceneVisibility.value;
        }
        void width; void height;
        return out;
    }

    // renderer.render(splatMesh, camera) (Viewer.js:1616): draws `renderCount` splats in the order of the engine's last sort
    render(splatMesh, camera, width, height, renderCount, sortedIndexes = null) {
        if (!this.frame || this.frame.length !== 4 * width * height) this.frame = new Uint8Array(addon.hostAlloc(4 * width * height));
        addon.render(this.engine, this.uniformsFor(splatMesh, camera, width, height),
                     { width, height, renderCount, sortedIndexes, frameFormat: GS_FRAME_RGBA8, flipY: 1 }, this.frame);
        return this.frame;
    }

    // sort + render in one engine call, two frames in flight (gs_frame_begin / gs_frame_end): returns the PREVIOUS frame's pixels, or
    // null for the first call; call finish() to collect the last one
    renderPipelined(splatMesh, camera, mvp, width, height, renderCount) {
        if (!this.frames) { this.frames = [0, 1].map(() => new Uint8Array(addon.hostAlloc(4 * width * height))); this.inFlight = 0; this.next = 0; }
        addon.frameBegin(this.engine, { modelViewProj: mvp, sortCount: renderCount, renderCount },
                         this.uniformsFor(splatMesh, camera, width, height), { width, height, renderCount, frameFormat: GS_FRAME_RGBA8, flipY: 1 },
                         this.frames[this.next]);
        this.next ^= 1;
        if (++this.inFlight < 2) return null;
        addon.frameEnd(this.engine);
        --this.inFlight;
        return this.frames[this.next];
    }
    finish() { if (this.inFlight) { addon.frameEnd(this.engine); --this.inFlight; return this.frames[this.next ^ 1]; } return null; }
}
