// CpuVoxB200.cs — P/Invoke binding of libcpuvox_b200.so (include/cpuvox_b200.h) for the reference's C# host.
// NOT compiled or run in the build environment (no dotnet/mono/csc in the image); it is the stub a maintainer of
// pipliz/cpuvox adds next to Assets/Code/RenderManager.cs. Struct layouts mirror the header field for field; the
// managed types they shadow are cited on each declaration.
using System;
using System.Runtime.InteropServices;

public static unsafe class CpuVoxB200
{
	const string LIB = "cpuvox_b200"; // libcpuvox_b200.so / cpuvox_b200.dll on the loader path

	public const int LOD_LEVELS = 6; // UnityManager.LOD_LEVELS, Assets/Code/UnityManager.cs:42

	[StructLayout(LayoutKind.Sequential)]
	public struct Segment // RenderManager.SegmentData, Assets/Code/RenderManager.cs:503-510 — identical layout, can be blitted
	{
		public float MinScreenX, MinScreenY;
		public float MaxScreenX, MaxScreenY;
		public float CamLocalPlaneRayMinX, CamLocalPlaneRayMinY;
		public float CamLocalPlaneRayMaxX, CamLocalPlaneRayMaxY;
		public int RayCount;
	}

	[StructLayout(LayoutKind.Sequential)]
	public struct Camera // CameraData, Assets/Code/Utils/CameraData.cs:11-36
	{
		public fixed float WorldToScreen[16]; // float4x4 stored c0, c1, c2, c3 (Unity.Mathematics column order)
		public float PositionX, PositionZ;
		public float PositionY;
		public int InverseElementIterationDirection;
		public float FarClip;
		public fixed float LODDistances[LOD_LEVELS];
	}

	[StructLayout(LayoutKind.Sequential)]
	public struct FrameSetup
	{
		public Segment Segment0, Segment1, Segment2, Segment3;
		public Camera Camera;
		public float VanishingPointX, VanishingPointY;
	}

	[StructLayout(LayoutKind.Sequential)]
	public struct Counters
	{
		public ulong DdaSteps, ColumnsNonEmpty, RunsVisited, PxVoxel, PxSky, Rays;
	}

	[StructLayout(LayoutKind.Sequential)]
	public struct Config { public int Device; public int Flags; }

	// Ray queries against the resident world (cvx_raycast; no reference analogue). 32 bytes each.
	[StructLayout(LayoutKind.Sequential)]
	public struct Ray
	{
		public float OriginX, OriginY, OriginZ;
		public float MaxDistance; // float.PositiveInfinity = unbounded
		public float DirectionX, DirectionY, DirectionZ; // need not be normalised
		public int Reserved;
	}

	[StructLayout(LayoutKind.Sequential)]
	public struct RayHit
	{
		public int Hit;  // 1 hit, 0 miss, -1 invalid ray
		public int Face; // entry face: 0 -X, 1 +X, 2 -Y, 3 +Y, 4 -Z, 5 +Z; 6 = origin inside the voxel
		public int CellX, CellY, CellZ; // LOD cell
		public float Distance; // world units along the normalised direction
		public uint Color; // ColorARGB32
		public int Steps;
	}
	[DllImport(LIB)] public static extern int cvx_create(ref Config config, out IntPtr ctx);
	[DllImport(LIB)] public static extern int cvx_destroy(IntPtr ctx);
	[DllImport(LIB)] public static extern IntPtr cvx_last_error(IntPtr ctx);
	[DllImport(LIB)] public static extern int cvx_world_upload(IntPtr ctx, int lod, int dimX, int dimY, int dimZ, void* blob, long bytes, int columnCount);
	[DllImport(LIB)] public static extern int cvx_world_free(IntPtr ctx);
	[DllImport(LIB)] public static extern int cvx_set_resolution(IntPtr ctx, int width, int height);
	[DllImport(LIB)] public static extern int cvx_draw(IntPtr ctx, ref FrameSetup setup);
	[DllImport(LIB)] public static extern int cvx_draw_batch(IntPtr ctx, FrameSetup* setups, int nViews, void* dstFrames);
	[DllImport(LIB)] public static extern int cvx_draw_batch_async(IntPtr ctx, FrameSetup* setups, int nViews, void* dstFrames, out long batch); // returns once enqueued
	[DllImport(LIB)] public static extern int cvx_batch_wait(IntPtr ctx, long batch);                                                       // that batch's frames are in dstFrames
	[DllImport(LIB)] public static extern int cvx_sync(IntPtr ctx);
	[DllImport(LIB)] public static extern int cvx_read_frame(IntPtr ctx, void* dstArgb, long bytes);
	[DllImport(LIB)] public static extern int cvx_read_raybuffer(IntPtr ctx, int which, void* dstArgb, long bytes);
	[DllImport(LIB)] public static extern int cvx_get_counters(IntPtr ctx, out Counters counters, int reset);
	[DllImport(LIB)] public static extern int cvx_device_frame(IntPtr ctx, out IntPtr devicePtr, out long bytes);
	[DllImport(LIB)] public static extern int cvx_clear_raybuffers(IntPtr ctx, uint argb);
	[DllImport(LIB)] public static extern int cvx_set_option(IntPtr ctx, int option, int value); // 1 lanes per ray, 2 counters, 3 general path, 4 views in flight
	// onDevice 0: host arrays, returns with the hits; onDevice 1: device pointers, ordered on the context's stream
	[DllImport(LIB)] public static extern int cvx_raycast(IntPtr ctx, Ray* rays, int n, int lod, RayHit* hits, int onDevice);
	// world production on the GPU (VoxelizerHelper + WorldBuilder.ToFinalColumn + World.DownSample as CUDA kernels); positions = n x float3
	// already in mesh space, colors32 = n x Color32; flips = int[3]. The first returns a builder handle (read its LOD blobs with
	// cvx_builder_lod, free with cvx_builder_free), the second installs the result as the context's world without a host copy.
	[DllImport(LIB)] public static extern int cvx_gpu_builder_from_mesh(IntPtr ctx, float* positions, byte* colors32, int nVertices, int maxDimension, int* flips, int nLods, out IntPtr builder);
	[DllImport(LIB)] public static extern int cvx_world_build_from_mesh(IntPtr ctx, float* positions, byte* colors32, int nVertices, int maxDimension, int* flips, int nLods, int* outDims, long* outVoxelCounts);
	[DllImport(LIB)] public static extern int cvx_builder_lod(IntPtr builder, int lod, out IntPtr blob, out long bytes, out int columnCount, out long voxelCount);
	[DllImport(LIB)] public static extern void cvx_builder_free(IntPtr builder);
	[DllImport(LIB)] public static extern int cvx_blit_raybuffer(IntPtr ctx, int which); // ERenderMode.RayBufferTopDown (0) / RayBufferLeftRight (1), UnityManager.cs:471-483
	[DllImport(LIB)] public static extern int cvx_present(IntPtr ctx, int format, int topDown, void* dst, int dstIsDevice); // 0 = RGBA8, 1 = BGRA8, 2 = packed RGB8
	[DllImport(LIB)] public static extern int cvx_present_jpeg(IntPtr ctx, int quality, int subsampling, void* dst, long dstCapacity, out long outBytes); // 0 = 4:4:4, 1 = 4:2:0; dstCapacity 0 = size query

	public static void Check (int code, IntPtr ctx)
	{
		if (code < 0) {
			throw new InvalidOperationException("cpuvox_b200 error " + code + ": " + Marshal.PtrToStringAnsi(cvx_last_error(ctx)));
		}
	}

	/// <summary>World hand-off: WorldAllocator.GetStartPointer/GetByteLength (Assets/Code/World.cs:273-283), once per LOD.</summary>
	public static void UploadWorlds (IntPtr ctx, World[] worldLODs)
	{
		for (int lod = 0; lod < worldLODs.Length; lod++) {
			if (!worldLODs[lod].Exists) { continue; }
			// World.Dimensions is the LOD-0 size at EVERY LOD (World.DownSample: `new World(dimensions, lod + extraLods)`, World.cs:47;
			// columns are indexed with `>> lod`, World.cs:145-149): pass it as is.
			Unity.Mathematics.int3 d = worldLODs[lod].Dimensions;
			Check(cvx_world_upload(ctx, lod, d.x, d.y, d.z,
				worldLODs[lod].Storage.GetStartPointer(), worldLODs[lod].Storage.GetByteLength(), worldLODs[lod].ColumnCount), ctx);
		}
	}

	/// <summary>Replaces the body of RenderManager.DrawSegments + ApplyPartials + BlitSegments (RenderManager.cs:156-189).</summary>
	public static void Draw (IntPtr ctx, Unity.Collections.NativeArray<RenderManager.SegmentData> segments, ref CameraData camData, Unity.Mathematics.float2 vanishingPointScreenSpace)
	{
		FrameSetup s = default;
		Segment* dst = &s.Segment0;
		for (int i = 0; i < 4; i++) {
			RenderManager.SegmentData sd = segments[i];
			dst[i] = *(Segment*)&sd; // same sequential layout
		}
		fixed (CameraData* cam = &camData) {
			// CameraData (CameraData.cs:11-16) in memory: float4x4 WorldToScreenMatrix (private; 64 bytes, c0..c3) at 0, float2 PositionXZ
			// at 64, float PositionY at 72, bool InverseElementIterationDirection at 76 (ONE byte + 3 bytes of padding whose content is
			// undefined), float FarClip at 80, fixed float LODDistances[6] at 84. Copied field by field; the bool becomes an explicit
			// 0 / 1 int. (Cleaner, if CameraData may be touched: add `public float4x4 WorldToScreen => WorldToScreenMatrix;`.)
			float* f = (float*)cam;
			for (int i = 0; i < 16; i++) { s.Camera.WorldToScreen[i] = f[i]; }
			s.Camera.PositionX = camData.PositionXZ.x;
			s.Camera.PositionZ = camData.PositionXZ.y;
			s.Camera.PositionY = camData.PositionY;
			s.Camera.InverseElementIterationDirection = camData.InverseElementIterationDirection ? 1 : 0;
			s.Camera.FarClip = camData.FarClip;
			for (int i = 0; i < LOD_LEVELS; i++) { s.Camera.LODDistances[i] = camData.LODDistances[i]; }
		}
		s.VanishingPointX = vanishingPointScreenSpace.x;
		s.VanishingPointY = vanishingPointScreenSpace.y;
		Check(cvx_draw(ctx, ref s), ctx);
	}
}
