// CoreSlamNative.cs — P/Invoke bindings for libcoreslam_b200 (include/coreslam_b200.h).
// NOT COMPILED IN THIS REPOSITORY: the build image has no .NET SDK.  It is the binding a SLAM.NET
// maintainer adds to CoreSLAM/CoreSLAM.csproj; struct layouts mirror the C header field for field.
using System;
using System.Runtime.InteropServices;

namespace CoreSLAM.B200
{
    public enum CsStatus : int
    {
        Ok = 0, InvalidArgument = 1, NoDevice = 2, Cuda = 3, OutOfMemory = 4, Capacity = 5, State = 6, Nccl = 7
    }

    [Flags]
    public enum CsFlags : uint
    {
        None = 0, RowMajorMap = 0x1, Timing = 0x2, KeepDistances = 0x4, NoHostSpin = 0x8, L2Persist = 0x10, DebugRays = 0x20,
        SearchWarp = 0x40, SearchSlab = 0x80,
        DebugBoundedSpin = 0x100   // device-side polls give up after 2 s: CS_ERR_CUDA instead of a hang (MPS, time-slicing, debuggers)
    }

    [StructLayout(LayoutKind.Sequential)]
    public unsafe struct CsConfig          // cs_config, 72 bytes
    {
        public float PhysicalMapSize;
        public int HoleMapSize;
        public fixed float StartPose[3];
        public float SigmaXY;
        public float SigmaTheta;
        public int IterationsPerThread;
        public int NumSearchThreads;
        public int Device;
        public int MaxPoints;
        public ulong Seed;
        public IntPtr Stream;
        public uint Flags;
        public int ObstacleMapSize;        // 0: no ObstacleMap on the device
    }

    [StructLayout(LayoutKind.Sequential)]
    public unsafe struct CsResult          // cs_result, 32 bytes
    {
        public fixed float Pose[3];
        public int Distance;
        public int Index;
        public int Searched;
        public long Visits;
    }

    [StructLayout(LayoutKind.Sequential)]
    public unsafe struct CsLattice         // cs_lattice, 36 bytes
    {
        public fixed float Origin[3];      // pose of lattice point (0,0,0): x, y (m), theta (rad)
        public fixed float Step[3];        // spacing along x, y (m), theta (rad)
        public fixed int Count[3];         // points along x, y, theta; each >= 1
    }

    [StructLayout(LayoutKind.Sequential)]
    public unsafe struct CsLatticeHit      // cs_lattice_hit, 20 bytes
    {
        public fixed float Pose[3];        // the lattice pose as evaluated (theta not normalised)
        public int Distance;               // CalculateDistanceSISD at that pose
        public int Index;                  // flat lattice index
    }

    [StructLayout(LayoutKind.Sequential)]
    public struct CsRelocalizeStats        // cs_relocalize_stats, 40 bytes
    {
        public long Poses;                 // count[0]*count[1]*count[2]
        public long Evaluated;             // poses whose exact distance was computed, summed over the passes
        public long Bounded;               // (node, level) bounds computed, summed over the passes
        public int Levels;                 // levels of the descent
        public int Passes;                 // 1, or more when the upper bound had to be raised
        public int UpperBound;             // U of the last pass
        public int Reserved;
    }

    internal static unsafe class Native
    {
        public const int LatticeMaxPoses = 1 << 28;   // CS_LATTICE_MAX_POSES
        public const int LatticeMaxHits = 64;         // CS_LATTICE_MAX_HITS
        public const int LatticeMaxPosesBounded = 2147483647;  // CS_LATTICE_MAX_POSES_BOUNDED
        public const int LatticeBoundedMaxNodes = 1 << 20;     // CS_LATTICE_BOUNDED_MAX_NODES
        public const int SequenceMaxScans = 32;                 // CS_SEQUENCE_MAX_SCANS

        private const string Lib = "coreslam_b200";   // libcoreslam_b200.so / coreslam_b200.dll

        [DllImport(Lib)] public static extern int cs_abi_version();
        [DllImport(Lib)] public static extern IntPtr cs_last_error(IntPtr h);
        [DllImport(Lib)] public static extern int cs_device_count();
        [DllImport(Lib)] public static extern CsStatus cs_create(ref CsConfig cfg, out IntPtr handle);
        [DllImport(Lib)] public static extern CsStatus cs_destroy(IntPtr h);
        [DllImport(Lib)] public static extern CsStatus cs_reset(IntPtr h);
        [DllImport(Lib)] public static extern CsStatus cs_set_quality(IntPtr h, int quality);
        [DllImport(Lib)] public static extern CsStatus cs_set_hole_width(IntPtr h, float metres);
        [DllImport(Lib)] public static extern CsStatus cs_set_position_search_beginning(IntPtr h, int scans);
        [DllImport(Lib)] public static extern CsStatus cs_get_pose(IntPtr h, float* pose3);
        [DllImport(Lib)] public static extern CsStatus cs_set_pose(IntPtr h, float* pose3, float* lastOdometry3, int scanCount);
        [DllImport(Lib)] public static extern CsStatus cs_update(IntPtr h, float* pointsXY, int nPoints, float* odometryPose3,
                                                                 float* candOffsets /* T*I*3 or null */, out CsResult result);
        [DllImport(Lib)] public static extern CsStatus cs_update_segments(IntPtr h, float* raysAngleRadius, int* segFirst, float* segPoses3,
                                                                          int nRays, int nSegments, float* candOffsets, out CsResult result);
        [DllImport(Lib)] public static extern CsStatus cs_segments_to_cloud(IntPtr h, float* raysAngleRadius, int* segFirst, float* segPoses3,
                                                                            int nRays, int nSegments, float* odometryPose3, float* pointsOut);
        [DllImport(Lib)] public static extern CsStatus cs_search(IntPtr h, float* pointsXY, int nPoints, float* searchPose3,
                                                                 float* candPoses, float* candCosSin, int nCand, uint scanIndex,
                                                                 out CsResult best, int* distances);
        // relocalisation on the current HoleMap (no reference counterpart): the k best window minima of the distance over a
        // pose lattice; distances (optional) receives Count[0]*Count[1]*Count[2] values in flat order
        [DllImport(Lib)] public static extern CsStatus cs_relocalize(IntPtr h, float* pointsXY, int nPoints, ref CsLattice lattice, int window,
                                                                     int k, CsLatticeHit* hits, out int nHits, int* distances);
        // the same hits by branch and bound, on lattices of up to LatticeMaxPosesBounded poses; stats optional (null)
        [DllImport(Lib)] public static extern CsStatus cs_relocalize_bounded(IntPtr h, float* pointsXY, int nPoints, ref CsLattice lattice,
                                                                             int window, int k, CsLatticeHit* hits, out int nHits,
                                                                             CsRelocalizeStats* stats);
        // the same two searches scoring each pose with nScans scans (points back to back, scan k owning
        // [scanFirst[k], scanFirst[k+1])) placed by their odometry (3 floats each) relative to the last scan's
        [DllImport(Lib)] public static extern CsStatus cs_relocalize_sequence(IntPtr h, float* pointsXY, int* scanFirst, float* odometry3,
                                                                              int nScans, ref CsLattice lattice, int window, int k,
                                                                              CsLatticeHit* hits, out int nHits, int* distances);
        [DllImport(Lib)] public static extern CsStatus cs_relocalize_sequence_bounded(IntPtr h, float* pointsXY, int* scanFirst, float* odometry3,
                                                                                      int nScans, ref CsLattice lattice, int window, int k,
                                                                                      CsLatticeHit* hits, out int nHits, CsRelocalizeStats* stats);
        [DllImport(Lib)] public static extern CsStatus cs_integrate(IntPtr h, float* pointsXY, int nPoints, float* pose3,
                                                                    float* poseCosSin, long* visits);
        [DllImport(Lib)] public static extern CsStatus cs_sync(IntPtr h);
        [DllImport(Lib)] public static extern CsStatus cs_map_download(IntPtr h, ushort* pixels);
        [DllImport(Lib)] public static extern CsStatus cs_map_upload(IntPtr h, ushort* pixels);
        [DllImport(Lib)] public static extern CsStatus cs_map_packed(IntPtr h, byte* packed);
        [DllImport(Lib)] public static extern CsStatus cs_set_unmapped_obstacle_hits(IntPtr h, int hits);
        [DllImport(Lib)] public static extern CsStatus cs_set_max_obstacle_hits(IntPtr h, int hits);
        [DllImport(Lib)] public static extern CsStatus cs_obstacle_map_download(IntPtr h, sbyte* pixels);
        [DllImport(Lib)] public static extern CsStatus cs_pinned_alloc(out IntPtr ptr, ulong bytes);
        [DllImport(Lib)] public static extern CsStatus cs_pinned_free(IntPtr ptr);

        [DllImport(Lib)] public static extern int cs_rings_hint(int sizePixels, float sizeMeters, float holeWidth, float* pointsXY, int nPoints);

        // ---- batches of independent sessions on one GPU (parameter sweeps, scan-log replays); no reference counterpart:
        // the reference would loop over CoreSLAMProcessor instances.  cfgs = nSessions CsConfig records.
        [DllImport(Lib)] public static extern CsStatus cs_batch_create(CsConfig* cfgs, int nSessions, out IntPtr batch);
        [DllImport(Lib)] public static extern CsStatus cs_batch_destroy(IntPtr batch);
        [DllImport(Lib)] public static extern IntPtr cs_batch_last_error(IntPtr batch);
        [DllImport(Lib)] public static extern CsStatus cs_batch_set_params(IntPtr batch, int session, int quality, float holeWidth);
        [DllImport(Lib)] public static extern CsStatus cs_batch_update(IntPtr batch, float* pointsXY, int* nPoints, float* odometry3,
                                                                       float* candOffsets, CsResult* results);
        // pipelined form: Submit(k+1) before Collect(k) overlaps the host staging with the device's work on step k
        [DllImport(Lib)] public static extern CsStatus cs_batch_submit(IntPtr batch, float* pointsXY, int* nPoints, float* odometry3,
                                                                       float* candOffsets);
        [DllImport(Lib)] public static extern CsStatus cs_batch_collect(IntPtr batch, CsResult* results);
        [DllImport(Lib)] public static extern CsStatus cs_batch_sync(IntPtr batch);
        [DllImport(Lib)] public static extern CsStatus cs_batch_get_poses(IntPtr batch, float* poses3);
        [DllImport(Lib)] public static extern CsStatus cs_batch_map_download(IntPtr batch, int session, ushort* pixels);
        // Reset() of every session at once; refused while submitted steps wait for cs_batch_collect
        [DllImport(Lib)] public static extern CsStatus cs_batch_reset(IntPtr batch);
        // per-session ObstacleMaps (CsConfig.ObstacleMapSize > 0, equal in all cfgs); session < 0: all sessions.
        // unmappedHits applies at the next cs_batch_reset, maxHits from the next step
        [DllImport(Lib)] public static extern CsStatus cs_batch_set_obstacle_params(IntPtr batch, int session, int unmappedHits, int maxHits);
        [DllImport(Lib)] public static extern CsStatus cs_batch_obstacle_map_download(IntPtr batch, int session, sbyte* pixels);
        [DllImport(Lib)] public static extern CsStatus cs_batch_obstacle_checksums(IntPtr batch, ulong* checksums);
        [DllImport(Lib)] public static extern CsStatus cs_batch_get_obstacle_visits(IntPtr batch, long* touched);
        [DllImport(Lib)] public static extern ulong cs_host_obstacle_checksum(sbyte* pixels, int size);

        // Candidate split over the GPUs of a node (BASELINE cfg4): one process per GPU exports the 64-byte handle of its exchange
        // table, the handles travel between the processes by any means (a pipe, a file, MPI), every process attaches all of them;
        // from then on Update on this handle evaluates this rank's slice of the candidates and the 8-byte arg-min is exchanged
        // inside the search kernels over NVLink peer memory.  cs_group_attach_local: the handles of one process (one per GPU).
        [StructLayout(LayoutKind.Sequential)] public unsafe struct CsIpcHandle { public fixed byte Bytes[64]; }
        [DllImport(Lib)] public static extern CsStatus cs_group_export(IntPtr h, out CsIpcHandle handle);
        [DllImport(Lib)] public static extern CsStatus cs_group_attach(IntPtr h, int rank, int world, CsIpcHandle* handles);
        [DllImport(Lib)] public static extern CsStatus cs_group_attach_local(IntPtr h, int rank, int world, IntPtr* peers);
        [DllImport(Lib)] public static extern CsStatus cs_group_detach(IntPtr h);

        public static void Check(CsStatus st, IntPtr h)
        {
            if (st != CsStatus.Ok)
                throw new InvalidOperationException($"{st}: {Marshal.PtrToStringAnsi(cs_last_error(h))}");
        }
    }
}
