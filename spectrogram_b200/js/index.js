'use strict';
/*
 * JavaScript facade of the B200 spectrogram engine: a drop-in for the AnalyserNode the reference
 * builds in src/javascripts/UI/player.js:7-11 and polls in src/javascripts/3D/visualizer.js:346-368,
 * plus the batched form of that loop.  Host code stays JavaScript; every number is produced by
 * hand-written sm_100a CUDA kernels behind the thin Node-API addon (napi_shim.c -> libsgcore.so).
 * There is no JavaScript or CPU fallback: if the addon or a B200 is missing, construction throws.
 *
 * Drop-in use in the reference (UI/player.js):
 *     const { createAnalyser } = require('spectrogram-b200');
 *     const analyser = createAnalyser();          // instead of context.createAnalyser()
 *     analyser.fftSize = 2048;                     // player.js:10
 *     analyser.smoothingTimeConstant = 0;          // player.js:11
 *     ...
 *     analyser.push(float32Samples);               // stands in for mix.connect(analyser), player.js:25
 *     analyser.getByteFrequencyData(freqByteData); // visualizer.js:352,358 -- unchanged
 */
const path = require('path');

let native;
try {
  native = require(path.join(__dirname, 'build', 'spectrogram.node'));
} catch (err) {
  const e = new Error('spectrogram-b200: native addon not built (run make in spectrogram_b200/js): ' + err.message);
  e.code = 'ERR_ADDON_MISSING';
  throw e;
}

// Web Audio raises DOMException(IndexSizeError); Node has no DOMException constructor for addons,
// so the shim throws RangeError with code 'IndexSizeError' and the facade sets the name.
function rethrow(err) {
  if (err && err.code === 'IndexSizeError') err.name = 'IndexSizeError';
  throw err;
}
function guard(fn) {
  return function guarded() {
    try {
      return fn.apply(this, arguments);
    } catch (err) {
      return rethrow(err);
    }
  };
}

const engines = new Map();
function engineFor(device) {
  const d = device | 0;
  if (!engines.has(d)) engines.set(d, native.engineCreate(d));
  return engines.get(d);
}
// Engines live as long as the process uses the module; closeAll() releases their device and pinned memory.
function closeAll() {
  for (const e of engines.values()) native.engineDestroy(e);
  engines.clear();
}
// Objects that were not close()d by hand release their native handle when they are collected.
const reaper = typeof FinalizationRegistry === 'function'
  ? new FinalizationRegistry(({ destroy, handle }) => { try { destroy(handle); } catch (err) { /* engine already gone */ } })
  : null;
function own(obj, destroy, handle) {
  if (reaper) reaper.register(obj, { destroy, handle }, obj);
}
function disown(obj) {
  if (reaper) reaper.unregister(obj);
}
function wholeNumber(v, what) {
  if (!Number.isInteger(v) || v < 0) throw new TypeError(what + ' must be a whole number');
  return v;
}

class AnalyserNode {
  constructor(options) {
    const o = options || {};
    this._engine = engineFor(o.device || 0);
    this._h = native.analyserCreate(this._engine);
    own(this, native.analyserDestroy, this._h);
    if (o.fftSize !== undefined) this.fftSize = o.fftSize;
    if (o.minDecibels !== undefined) this.minDecibels = o.minDecibels;
    if (o.maxDecibels !== undefined) this.maxDecibels = o.maxDecibels;
    if (o.smoothingTimeConstant !== undefined) this.smoothingTimeConstant = o.smoothingTimeConstant;
  }
  get fftSize() { return native.analyserGet(this._h, 'fftSize'); }
  set fftSize(v) { guard(native.analyserSet)(this._h, 'fftSize', Number(v)); }
  get frequencyBinCount() { return native.analyserGet(this._h, 'frequencyBinCount'); }
  get minDecibels() { return native.analyserGet(this._h, 'minDecibels'); }
  set minDecibels(v) { guard(native.analyserSet)(this._h, 'minDecibels', Number(v)); }
  get maxDecibels() { return native.analyserGet(this._h, 'maxDecibels'); }
  set maxDecibels(v) { guard(native.analyserSet)(this._h, 'maxDecibels', Number(v)); }
  get smoothingTimeConstant() { return native.analyserGet(this._h, 'smoothingTimeConstant'); }
  set smoothingTimeConstant(v) { guard(native.analyserSet)(this._h, 'smoothingTimeConstant', Number(v)); }

  // audio in: what the render thread does for a browser AnalyserNode
  push(samples) {
    if (!(samples instanceof Float32Array)) throw new TypeError('push() needs a Float32Array');
    native.analyserPush(this._h, samples);
  }
  // graph plumbing is not part of the frame path; kept so call sites like player.js:25-26 run
  connect(dest) { return dest; }
  disconnect() {}

  // getters write into the caller-owned typed array: min(array.length, frequencyBinCount) elements
  getByteFrequencyData(array) {
    if (!(array instanceof Uint8Array)) throw new TypeError('getByteFrequencyData needs a Uint8Array');
    guard(native.getByteFrequencyData)(this._h, array);
  }
  getFloatFrequencyData(array) {
    if (!(array instanceof Float32Array)) throw new TypeError('getFloatFrequencyData needs a Float32Array');
    guard(native.getFloatFrequencyData)(this._h, array);
  }
  getByteTimeDomainData(array) {
    if (!(array instanceof Uint8Array)) throw new TypeError('getByteTimeDomainData needs a Uint8Array');
    guard(native.getByteTimeDomainData)(this._h, array);
  }
  getFloatTimeDomainData(array) {
    if (!(array instanceof Float32Array)) throw new TypeError('getFloatTimeDomainData needs a Float32Array');
    guard(native.getFloatTimeDomainData)(this._h, array);
  }
  close() {
    if (this._h) { disown(this); native.analyserDestroy(this._h); }
    this._h = null;
  }
}

const OUT_CTOR = { u8: Uint8Array, byte: Uint8Array, db: Float32Array, float: Float32Array, mag: Float32Array, rgba: Uint32Array, rgba8: Uint32Array };

/**
 * Batched frame path: pcm (Float32Array, nClips * clipLen samples, clip-major) ->
 * { frames, bins, data } with data laid out [clip][frame][bin] (the row-per-frame layout the
 * reference appends to its texture, visualizer.js:399-416).
 * opts: { fftSize, hop, window, minDecibels, maxDecibels, smoothingTimeConstant, output, align,
 *         nClips, device | devices }
 * devices: [0, 1, ...] shards clips in contiguous blocks, one engine per GPU running concurrently (the library
 * starts a host thread per engine), results gathered by host copy into one typed array (no collective; shards are
 * independent).
 */
function spectrogram(pcm, opts) {
  if (!(pcm instanceof Float32Array)) throw new TypeError('pcm must be a Float32Array');
  const o = Object.assign({ fftSize: 2048, hop: 512, output: 'u8' }, opts || {});
  const nClips = o.nClips || 1;
  if (pcm.length % nClips) throw new TypeError('pcm length is not a multiple of nClips');
  const clipLen = pcm.length / nClips;
  const frames = guard(native.numFrames)(o, clipLen);
  const bins = o.fftSize / 2;
  const Ctor = OUT_CTOR[o.output];
  if (!Ctor) throw new TypeError('unknown output ' + o.output);
  const data = new Ctor(nClips * frames * bins);
  const devices = o.devices || [o.device || 0];
  if (devices.length === 1) guard(native.stftBatch)(engineFor(devices[0]), pcm, nClips, clipLen, o, data);
  else guard(native.stftBatchMulti)(devices.map(engineFor), pcm, nClips, clipLen, o, data);   // sg_stft_batch_multi: one host thread per GPU inside the library
  return { frames, bins, data };
}

// opts.historyRows keeps a sonogram history per channel on the device: what a SonogramRing(bins, historyRows) fed
// every push's byte rows would hold.  view() then draws every channel's picture in one launch (output 'u8' only).
// BiquadFilterNode (W3C Web Audio), the filter the reference's draw mode puts in front of its analyser
// (Player.setBandpassFrequency, UI/player.js): bandpass.type = 'bandpass'; bandpass.Q.value = 10;
// bandpass.frequency.value = f.  process() filters on the GPU and carries the float64 state between calls.
const BIQUAD_TYPES = ['lowpass', 'highpass', 'bandpass', 'lowshelf', 'highshelf', 'peaking', 'notch', 'allpass'];
class AudioParam {
  constructor(value) {
    this.defaultValue = value;
    this.value = value;
  }
}
class BiquadFilterNode {
  constructor(options) {
    const o = options || {};
    this.sampleRate = o.sampleRate || 48000;
    this.channels = o.channels || 1;
    this._device = o.device || 0;
    this._type = 'lowpass';
    this.frequency = new AudioParam(350);
    this.Q = new AudioParam(1);
    this.gain = new AudioParam(0);
    this.detune = new AudioParam(0);
    this._state = new Float64Array(4 * this.channels);   // [channel] {x1, x2, y1, y2}
  }
  get type() { return this._type; }
  // WebIDL enum attribute: assigning a string outside the enum is ignored, not thrown
  set type(value) { if (BIQUAD_TYPES.includes(value)) this._type = value; }
  params() {
    return { type: this._type, sampleRate: this.sampleRate, frequency: this.frequency.value, Q: this.Q.value,
             gain: this.gain.value, detune: this.detune.value };
  }
  // normalised Float64Array [b0, b1, b2, a1, a2]
  coefficients() {
    const out = new Float64Array(5);
    guard(native.biquadCoefficients)(this.params(), out);
    return out;
  }
  // samples: Float32Array [channel][n]; returns (or fills `out`) the filtered samples
  process(samples, out) {
    const len = wholeNumber(samples.length / this.channels, 'samples.length / channels');
    const dst = out || new Float32Array(samples.length);
    guard(native.biquadFilter)(engineFor(this._device), this.params(), samples, this.channels, len, this._state, dst);
    return dst;
  }
  reset() { this._state.fill(0); }
}

class StreamBank {
  constructor(nChannels, opts, maxChunk) {
    this.opts = Object.assign({ fftSize: 1024, hop: 128, output: 'u8' }, opts || {});
    this.nChannels = nChannels;
    this.maxChunk = maxChunk || this.opts.hop;
    this._h = guard(native.streamCreate)(engineFor(this.opts.device || 0), nChannels, this.opts, this.maxChunk);
    own(this, native.streamDestroy, this._h);
    if (this.opts.historyRows) this.setHistory(this.opts.historyRows);
    this._filter = null;
    if (this.opts.filter) this.setFilter(this.opts.filter);
  }
  // a BiquadFilterNode in front of every channel's analyser (the draw mode's bandpass), or null to detach it.  The bank
  // keeps the filter state on the device; the node's parameters are re-sent before a push when they have changed.
  setFilter(node) {
    const p = node ? node.params() : null;
    guard(native.streamSetFilter)(this._h, p);
    this._filter = node || null;
    this._filterSent = p && JSON.stringify(p);
  }
  _syncFilter() {
    if (!this._filter) return;
    const p = this._filter.params(), key = JSON.stringify(p);
    if (key !== this._filterSent) { guard(native.streamSetFilter)(this._h, p); this._filterSent = key; }
  }
  // chunk: Float32Array [channel][chunkLen]; out: typed array [channel][chunkLen/hop][bins], or undefined when a
  // history is attached and only the pictures are wanted (no rows come back to the host)
  push(chunk, out, outRgba) {
    const chunkLen = wholeNumber(chunk.length / this.nChannels, 'chunk.length / nChannels');
    this._syncFilter();
    guard(native.streamPush)(this._h, chunk, chunkLen, out, outRgba);
  }
  // attach an empty history of `rows` rows per channel (texture zero, yoffset 0); 0 detaches it
  setHistory(rows) {
    guard(native.streamSetHistory)(this._h, rows);
  }
  get historyRows() {
    return native.streamHistoryInfo(this._h).rows;
  }
  get historyYoffset() {
    return native.streamHistoryInfo(this._h).yoffset;
  }
  _range(o) {
    const first = o.first || 0;
    return [first, o.count === undefined ? this.nChannels - first : o.count];
  }
  // textures of channels [first, first+count): Uint8Array [count][rows][bins], texture row order
  history(options) {
    const o = options || {};
    const [first, count] = this._range(o);
    const out = o.out || new Uint8Array(Math.max(count * this.historyRows * (this.opts.fftSize / 2), 0) || 0);
    guard(native.streamHistoryRead)(this._h, first, count, out);
    return out;
  }
  // RGBA8 pictures of channels [first, first+count) in one launch: Uint32Array [count][height][width], each what
  // SonogramRing.view draws for that channel
  view(width, height, options) {
    const o = options || {};
    const [first, count] = this._range(o);
    const out = o.out || new Uint32Array(Math.max(count * width * height, 0) || 0);   // bad sizes are the native's to report
    guard(native.streamView)(this._h, first, count, width, height, out);
    return out;
  }
  close() {
    if (this._h) { disown(this); native.streamDestroy(this._h); }
    this._h = null;
  }
}

// The reference's spectrogram history (a bins x 256 byte texture written one row per frame at yoffset,
// src/javascripts/3D/visualizer.js:60,301-329,399-416) kept on the device, and its sonogram picture
// (src/bin/shaders/sonogram-fragment.shader:14-27, sonogram-vertex.shader:19-58) rendered headlessly.
class SonogramRing {
  constructor(bins, rows, device) {
    this.bins = bins;
    this.rows = rows || 256;
    this._h = guard(native.ringCreate)(engineFor(device || 0), this.bins, this.rows);
    own(this, native.ringDestroy, this._h);
  }
  // frames: Uint8Array holding one or more byte rows (what getByteFrequencyData filled)
  append(frames) {
    if (!(frames instanceof Uint8Array)) throw new TypeError('frames must be a Uint8Array');
    guard(native.ringAppend)(this._h, frames, wholeNumber(frames.length / this.bins, 'frames.length / bins'));
  }
  get yoffset() {
    return native.ringYoffset(this._h);
  }
  // RGBA8 picture, Uint32Array [height][width] (little-endian R | G<<8 | B<<16 | A<<24)
  view(width, height, out) {
    const img = out || new Uint32Array(width * height);
    guard(native.ringView)(this._h, width, height, img);
    return img;
  }
  close() {
    if (this._h) { disown(this); native.ringDestroy(this._h); }
    this._h = null;
  }
}

// What decodeAudioData hands the reference (src/javascripts/util/util.js:10-12, played at UI/player.js:154-170):
// planar float32 channels.  Produced on the GPU from uncompressed PCM; compressed formats are not decoded here.
class AudioBuffer {
  constructor(planes, numberOfChannels, length, sampleRate) {
    this._planes = planes;                       // Float32Array [channel][frame]
    this.numberOfChannels = numberOfChannels;
    this.length = length;
    this.sampleRate = sampleRate;
    this.duration = sampleRate ? length / sampleRate : 0;
  }
  getChannelData(channel) {
    if (!(channel >= 0 && channel < this.numberOfChannels)) {
      const e = new RangeError('channel index out of range');
      e.code = e.name = 'IndexSizeError';
      throw e;
    }
    return this._planes.subarray(channel * this.length, (channel + 1) * this.length);
  }
}

// context.decodeAudioData(arrayBuffer, onBuffer, onError) (util/util.js:9-17) for RIFF/WAVE files holding PCM.
// Keeps the callback form the reference uses and also returns a Promise, like the browser's.  options.sampleRate is
// the context's rate (new AudioContext({sampleRate})): a file at another rate is resampled to it on the GPU.
function decodeAudioData(arrayBuffer, onBuffer, onError, options) {
  const o = options || {};
  return new Promise((resolve, reject) => {
    try {
      const file = arrayBuffer instanceof Uint8Array ? arrayBuffer : new Uint8Array(arrayBuffer);
      const info = guard(native.wavParse)(file);
      const bytes = info.length * info.channels * { u8: 1, s16: 2, s24: 3, s32: 4, f32: 4 }[info.format];
      const samples = file.subarray(info.dataOffset, info.dataOffset + bytes);
      let buffer;
      if (o.sampleRate && o.sampleRate !== info.sampleRate) {
        const length = guard(native.resampleNumFrames)(info.length, info.sampleRate, o.sampleRate);
        const planes = new Float32Array(info.channels * length);
        guard(native.pcmDecodeResampled)(engineFor(o.device || 0), samples, info, 1, 0, o.sampleRate, planes);
        buffer = new AudioBuffer(planes, info.channels, length, o.sampleRate);
      } else {
        const planes = new Float32Array(info.channels * info.length);
        guard(native.pcmDecode)(engineFor(o.device || 0), samples, info, 1, 0, planes);
        buffer = new AudioBuffer(planes, info.channels, info.length, info.sampleRate);
      }
      if (onBuffer) onBuffer(buffer);
      resolve(buffer);
    } catch (err) {
      if (onError) onError(err);
      reject(err);
    }
  });
}

// The frame path fed with interleaved PCM (Uint8Array view of the samples): ingest and, by default, the
// AnalyserNode's mono down-mix run on the GPU in front of the batched path.
// pcm = {format: 'u8'|'s16'|'s24'|'s32'|'f32', channels, sampleRate}; returns {frames, bins, planes, data}.
// options.sampleRate (the context's rate) resamples from pcm.sampleRate before framing when the two differ.
function spectrogramPcm(samples, pcm, options) {
  const o = Object.assign({ fftSize: 2048, hop: 512, output: 'u8', mix: true, clips: 1 }, options || {});
  const bytesPerFrame = (pcm.channels || 1) * { u8: 1, s16: 2, s24: 3, s32: 4, f32: 4 }[pcm.format];
  const resample = !!o.sampleRate && o.sampleRate !== pcm.sampleRate;
  let length = Math.floor(samples.length / (bytesPerFrame * o.clips));
  if (resample) length = guard(native.resampleNumFrames)(length, pcm.sampleRate || 0, o.sampleRate);
  const frames = guard(native.numFrames)(o, length);
  const bins = o.fftSize / 2;
  const planes = o.mix ? 1 : (pcm.channels || 1);
  const n = o.clips * planes * frames * bins;
  const Ctor = OUT_CTOR[o.output];
  if (!Ctor) throw new TypeError('unknown output ' + o.output);
  const data = new Ctor(n);
  if (resample) guard(native.stftPcmResampled)(engineFor(o.device || 0), samples, pcm, o.clips, o.mix ? 1 : 0, o.sampleRate, o, data);
  else guard(native.stftPcm)(engineFor(o.device || 0), samples, pcm, o.clips, o.mix ? 1 : 0, o, data);
  return { frames, bins, planes, data };
}

module.exports = {
  AnalyserNode,
  createAnalyser: (options) => new AnalyserNode(options),
  spectrogram,
  StreamBank,
  BiquadFilterNode,
  AudioParam,
  createBiquadFilter: (options) => new BiquadFilterNode(options),
  SonogramRing,
  AudioBuffer,
  decodeAudioData,
  spectrogramPcm,
  colormapReference: () => native.colormapReference(),
  deviceCount: () => native.deviceCount(),
  closeAll,
};
