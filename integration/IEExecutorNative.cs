// IEExecutorNative.cs -- SURVEY.md §8f N4: the sample's inference runner on top of libxrseg.so (P/Invoke).
//
// Drop next to Assets/Scripts/InferenceEngine/IEExecutor.cs and put libxrseg.so under Assets/Plugins/x86_64.  It keeps
// the public surface the sample's triggers use (RunInference / IsRunning / IsModelLoaded / CurrentFrameBoxes) and the
// Update-driven state machine (Running -> RequestingOutputs -> Success / Error -> Cleanup, IEExecutor.cs:389-456), but
// every tensor operation -- ToTensor, the 499-layer graph, readback, ParseBoxes, the mask loop -- is one call into the
// CUDA library.  NOT compiled in the build container (no Unity / dotnet there); the same entry points, struct layouts
// and call order are exercised through ctypes by xr_image_segmentation_b200/executor.py and the GPU tests.
using System;
using System.Collections.Generic;
using System.Runtime.InteropServices;
using Unity.Collections;
using Unity.Collections.LowLevel.Unsafe;
using UnityEngine;

public class IEExecutorNative : MonoBehaviour
{
    const string Lib = "xrseg";

    [StructLayout(LayoutKind.Sequential)]
    struct Config
    {
        public uint structSize; public int device, maxBatch, modelScale;
        public IntPtr weights; public UIntPtr weightsBytes;
        public float iouThreshold, scoreThreshold, maskThreshold;
        public int maxDet, maxCandidates, resizeMode, convImpl, useCudaGraph, microBatch;
        public int numClasses;   // 0 = from the model; a custom-trained YOLO11-seg may have 1..1024 classes
        [MarshalAs(UnmanagedType.ByValArray, SizeConst = 7)] public int[] reserved;
    }
    [StructLayout(LayoutKind.Sequential)]
    struct NativeBox { public float centerX, centerY, width, height; public int labelId, frame; }
    [StructLayout(LayoutKind.Sequential)]
    struct MaskParams { public uint structSize; public int mode, boxConvention; public float screenW, screenH; public int imageW, imageH, first, count; public float threshold; }
    const int FmtRgba8 = 1, FmtBottomUp = 0x100;   // xrseg_pixel_format
    const int ErrCapacity = -7;

    [DllImport(Lib)] static extern int xrseg_create(ref Config cfg, out IntPtr runner);
    [DllImport(Lib)] static extern void xrseg_destroy(IntPtr runner);
    [DllImport(Lib)] static extern IntPtr xrseg_last_error(IntPtr runner);
    [DllImport(Lib)] static extern int xrseg_schedule(IntPtr runner, IntPtr pixels, int w, int h, int strideBytes, int fmt, int batch);
    [DllImport(Lib)] static extern int xrseg_poll(IntPtr runner);
    [DllImport(Lib)] static extern int xrseg_decode(IntPtr runner, float screenW, float screenH, int convention, [Out] NativeBox[] boxes, int cap, out int n);
    [DllImport(Lib)] static extern int xrseg_masks(IntPtr runner, ref MaskParams p, IntPtr dst, UIntPtr capBytes);

    public struct Box { public float CenterX, CenterY, Width, Height; public string ClassName; }

    [SerializeField] TextAsset _sentisBytes;        // yolo11n-seg-sentis.sentis imported as a bytes asset
    [SerializeField] TextAsset _labelsAsset;        // yolo11n-labels.txt
    [SerializeField] float _confidenceThreshold = 0.5f;

    enum State { Idle, Running, Success, Error }
    State _state = State.Idle;
    IntPtr _runner = IntPtr.Zero;
    GCHandle _modelPin;
    NativeArray<Color32> _pixels;
    readonly NativeBox[] _native = new NativeBox[50];
    string[] _labels;
    int _texW, _texH;

    public bool IsModelLoaded { get; private set; }
    public List<Box> CurrentFrameBoxes { get; } = new List<Box>();
    public byte[] TargetMask { get; } = new byte[160 * 160];      // prob > thr && PixelInBoundingBox, texture row order

    void Start()
    {
        _labels = _labelsAsset.text.Split(new[] { '\n', '\r' }, StringSplitOptions.RemoveEmptyEntries);
        byte[] model = _sentisBytes.bytes;
        _modelPin = GCHandle.Alloc(model, GCHandleType.Pinned);
        var cfg = new Config
        {
            structSize = (uint)Marshal.SizeOf<Config>(), device = 0, maxBatch = 1, modelScale = 'n',
            weights = _modelPin.AddrOfPinnedObject(), weightsBytes = (UIntPtr)model.Length,
            maskThreshold = _confidenceThreshold, useCudaGraph = 1, reserved = new int[7]   // iou / score 0 = the asset's own 0.43 / 0.301
        };
        if (xrseg_create(ref cfg, out _runner) < 0)
        {
            Debug.LogError("xrseg_create: " + Marshal.PtrToStringAnsi(xrseg_last_error(IntPtr.Zero)));
            return;
        }
        IsModelLoaded = true;                           // the library warms itself up on the first schedule
    }

    public bool IsRunning() => _state == State.Running;

    public void RunInference(WebCamTexture tex)
    {
        if (!IsModelLoaded || _state == State.Running) return;
        if (!_pixels.IsCreated || _pixels.Length != tex.width * tex.height)
        {
            if (_pixels.IsCreated) _pixels.Dispose();
            _pixels = new NativeArray<Color32>(tex.width * tex.height, Allocator.Persistent);
        }
        // GetPixels32 returns rows BOTTOM-UP (texture origin bottom-left); XRSEG_FMT_BOTTOM_UP makes the library read image
        // row y from memory row h-1-y, which is what TextureConverter.ToTensor does internally.  RGBA8, stretched to 640x640
        // on the GPU like ToTensor.
        _pixels.CopyFrom(tex.GetPixels32());
        _texW = tex.width; _texH = tex.height;
        unsafe
        {
            int rc = xrseg_schedule(_runner, (IntPtr)_pixels.GetUnsafeReadOnlyPtr(), _texW, _texH, _texW * 4, FmtRgba8 | FmtBottomUp, 1);
            _state = rc < 0 ? State.Error : State.Running;
        }
    }

    void Update()
    {
        if (_state == State.Running)
        {
            int st = xrseg_poll(_runner);               // never blocks the frame loop
            if (st == 0) return;
            if (st == ErrCapacity) Debug.LogWarning("xrseg: " + Marshal.PtrToStringAnsi(xrseg_last_error(_runner)));   // truncated, still usable
            _state = st < 0 && st != ErrCapacity ? State.Error : State.Success;
        }
        if (_state == State.Success) ProcessResult();
        if (_state == State.Error) _state = State.Idle; // retry on the next trigger, like CleanupResources
    }

    void ProcessResult()
    {
        CurrentFrameBoxes.Clear();
        if (xrseg_decode(_runner, Screen.width, Screen.height, /*ParseBoxes*/ 0, _native, _native.Length, out int n) < 0 || n == 0)
        {
            _state = State.Error;                       // N == 0 is the sample's Error state
            return;
        }
        for (int i = 0; i < n; i++)
        {
            int id = _native[i].labelId;
            string name = id >= 0 && id < _labels.Length ? _labels[id].Replace(" ", "_") : "unknown";
            CurrentFrameBoxes.Add(new Box { CenterX = _native[i].centerX, CenterY = _native[i].centerY, Width = _native[i].width, Height = _native[i].height, ClassName = name });
        }
        _state = State.Idle;
    }

    // IEMasker.DrawSingleMask's pixel loop for detection `index`, computed on the GPU
    public unsafe bool FetchMask(int index)
    {
        var mp = new MaskParams { structSize = (uint)Marshal.SizeOf<MaskParams>(), mode = 0, boxConvention = 0, screenW = Screen.width, screenH = Screen.height, imageW = _texW, imageH = _texH, first = index, count = 1, threshold = 0f /* the runner's _confidenceThreshold */ };
        fixed (byte* dst = TargetMask) return xrseg_masks(_runner, ref mp, (IntPtr)dst, (UIntPtr)TargetMask.Length) == 1;
    }

    void OnDestroy()
    {
        if (_runner != IntPtr.Zero) xrseg_destroy(_runner);
        if (_modelPin.IsAllocated) _modelPin.Free();
        if (_pixels.IsCreated) _pixels.Dispose();
    }
}
