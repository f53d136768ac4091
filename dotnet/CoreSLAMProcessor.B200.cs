// CoreSLAMProcessor.B200.cs — drop-in for CoreSLAM/CoreSLAMProcessor.cs with the whole of Update (ScanSegmentsToCloud,
// search, HoleMap and ObstacleMap integration) running on a B200 through libcoreslam_b200.  Public surface identical
// to the reference (ctor :119-120, Reset :167, Update :717, Dispose :757, properties :40-106).
// NOT COMPILED IN THIS REPOSITORY (no .NET SDK in the image).
using System;
using System.Collections.Generic;
using System.Linq;
using System.Numerics;
using BaseSLAM;

namespace CoreSLAM.B200
{
    public sealed unsafe class HoleMap
    {
        private readonly IntPtr handle;
        internal HoleMap(IntPtr handle, int sizePixels, float sizeMeters)
        {
            this.handle = handle;
            Size = sizePixels;
            Scale = sizePixels / sizeMeters;                 // HoleMap.cs:20
            Pixels = new ushort[sizePixels * sizePixels];    // host copy, refreshed by SyncToHost()
        }
        public readonly ushort[] Pixels;                      // HoleMap.cs:27 (public field, kept)
        public int Size { get; }
        public float Scale { get; }

        /// Pull the device-resident map into Pixels (waits for the pending integration).
        public void SyncToHost()
        {
            fixed (ushort* p = Pixels) Native.Check(Native.cs_map_download(handle, p), handle);
        }

        public byte[] GetPackedPixels()                       // HoleMap.cs:44-55, packed on the device
        {
            var packed = new byte[Pixels.Length / 2];
            fixed (byte* p = packed) Native.Check(Native.cs_map_packed(handle, p), handle);
            return packed;
        }
    }

    public sealed unsafe class ObstacleMap                     // CoreSLAM/ObstacleMap.cs:11-44
    {
        private readonly IntPtr handle;
        internal ObstacleMap(IntPtr handle, int sizePixels, float sizeMeters)
        {
            this.handle = handle;
            Size = sizePixels;
            Scale = sizePixels / sizeMeters;                  // ObstacleMap.cs:20
            Pixels = new sbyte[sizePixels, sizePixels];       // [y, x], host copy refreshed by SyncToHost()
        }
        public readonly sbyte[,] Pixels;                      // ObstacleMap.cs:27 (public field, kept)
        public int Size { get; }
        public float Scale { get; }
        public void SyncToHost()
        {
            fixed (sbyte* p = Pixels) Native.Check(Native.cs_obstacle_map_download(handle, p), handle);
        }
    }

    public sealed unsafe class CoreSLAMProcessor : IDisposable
    {
        private IntPtr handle;
        private readonly IntPtr staging;      // pinned: raw rays, segment poses and first-ray indices of the current Update
        private readonly int maxPoints;
        private byte quality = 50;
        private float holeWidth = 0.6f;
        private int positionSearchBeginning = 5;

        public float PhysicalMapSize { get; }
        public HoleMap HoleMap { get; }
        public ObstacleMap ObstacleMap { get; }
        public float SigmaXY { get; }
        public float SigmaTheta { get; }
        public int SearchIterationsPerThread { get; }
        public int NumSearchThreads { get; }
        public Vector3 Pose { get; private set; }
        /// true: HoleMap.Pixels is refreshed after every Update (reference semantics, costs a D2H copy)
        public bool SyncMapAfterUpdate { get; set; } = false;

        public byte Quality { get => quality; set { Native.Check(Native.cs_set_quality(handle, value), handle); quality = value; } }
        public float HoleWidth { get => holeWidth; set { Native.Check(Native.cs_set_hole_width(handle, value), handle); holeWidth = value; } }
        public int PositionSearchBeginning
        {
            get => positionSearchBeginning;
            set { Native.Check(Native.cs_set_position_search_beginning(handle, value), handle); positionSearchBeginning = value; }
        }

        private sbyte unmappedObstacleHits = -5, maxObstacleHits = 10;
        public sbyte UnmappedObstacleHits   // :98 — takes effect at the next Reset(), as in the reference
        {
            get => unmappedObstacleHits;
            set { Native.Check(Native.cs_set_unmapped_obstacle_hits(handle, value), handle); unmappedObstacleHits = value; }
        }
        public sbyte MaxObstacleHits        // :103
        {
            get => maxObstacleHits;
            set { Native.Check(Native.cs_set_max_obstacle_hits(handle, value), handle); maxObstacleHits = value; }
        }

        public CoreSLAMProcessor(float physicalMapSize, int holeMapSize, int obstacleMapSize, Vector3 startPose,
            float sigmaXY, float sigmaTheta, int iterationsPerThread, int numSearchThreads,
            int device = 0, ulong seed = 0x5EED, int maxPoints = 16384)
        {
            PhysicalMapSize = physicalMapSize; SigmaXY = sigmaXY; SigmaTheta = sigmaTheta;
            SearchIterationsPerThread = iterationsPerThread; NumSearchThreads = numSearchThreads;
            this.maxPoints = maxPoints;
            var cfg = new CsConfig
            {
                PhysicalMapSize = physicalMapSize, HoleMapSize = holeMapSize, SigmaXY = sigmaXY, SigmaTheta = sigmaTheta,
                IterationsPerThread = iterationsPerThread, NumSearchThreads = numSearchThreads,
                Device = device, MaxPoints = maxPoints, Seed = seed, ObstacleMapSize = obstacleMapSize
            };
            cfg.StartPose[0] = startPose.X; cfg.StartPose[1] = startPose.Y; cfg.StartPose[2] = startPose.Z;
            Native.Check(Native.cs_create(ref cfg, out handle), IntPtr.Zero);
            Native.Check(Native.cs_pinned_alloc(out staging, (ulong)maxPoints * (8 + 12 + 4) + 4), handle);  // rays, segment poses, first-ray indices
            HoleMap = new HoleMap(handle, holeMapSize, physicalMapSize);
            ObstacleMap = new ObstacleMap(handle, obstacleMapSize, physicalMapSize);
            Pose = startPose;
        }

        public void Reset()
        {
            Native.Check(Native.cs_reset(handle), handle);
            float* p = stackalloc float[3];
            Native.Check(Native.cs_get_pose(handle, p), handle);
            Pose = new Vector3(p[0], p[1], p[2]);
        }

        /// CoreSLAMProcessor.Update (:717-752), whole: the raw rays and segment poses are written straight into the
        /// pinned staging block and uploaded; ScanSegmentsToCloud (:187-207), search, NormalizeAngle and both map
        /// integrations run on the device.  Returns when the pose is known; the integration overlaps the caller.
        public void Update(List<ScanSegment> segments) => Update(segments, null);

        /// Distance and flat candidate index (0 = searchPose, 1 + t*I + i = thread t's i-th candidate) of the pose the last
        /// search chose; (int.MaxValue, 0) when the scan was integrated without a search.
        public int LastDistance { get; private set; } = int.MaxValue;
        public int LastIndex { get; private set; }

        /// Verification mode: the same Update with the candidate offsets given (T*I x (dX, dY, dTheta), thread t iteration i at
        /// (t*I + i)*3) instead of drawn on the device — what dotnet/reference_verification_hook.patch adds to the reference as
        /// CoreSLAMProcessor.CandidateTable, so that both implementations search the very same poses.
        public void Update(List<ScanSegment> segments, float[] candidateOffsets)
        {
            if (candidateOffsets != null && candidateOffsets.Length != 3 * SearchIterationsPerThread * Math.Max(NumSearchThreads, 1))
                throw new ArgumentException("candidateOffsets needs T*I*3 floats");
            if (segments.Count == 0) throw new InvalidOperationException("Sequence contains no elements");  // segments.Last(), :719
            float* rays = (float*)staging;                       // maxPoints * (angle, radius)
            float* poses = rays + 2 * maxPoints;                 // maxPoints * (x, y, theta)   (at most one segment per ray)
            int* first = (int*)(poses + 3 * maxPoints);          // maxPoints + 1
            int n = 0, s = 0;
            foreach (ScanSegment segment in segments)
            {
                if (s >= maxPoints) throw new InvalidOperationException("more segments than maxPoints");
                first[s] = n;
                poses[3 * s] = segment.Pose.X; poses[3 * s + 1] = segment.Pose.Y; poses[3 * s + 2] = segment.Pose.Z;
                s++;
                foreach (Ray r in segment.Rays)
                {
                    if (n >= maxPoints) throw new InvalidOperationException("scan larger than maxPoints");
                    rays[2 * n] = r.Angle;
                    rays[2 * n + 1] = r.Radius;
                    n++;
                }
            }
            first[s] = n;
            CsResult res;
            fixed (float* off = candidateOffsets)  // (null stays null: on-device Philox candidates)
                Native.Check(Native.cs_update_segments(handle, rays, first, poses, n, s, off, out res), handle);
            Pose = new Vector3(res.Pose[0], res.Pose[1], res.Pose[2]);
            LastDistance = res.Searched != 0 ? res.Distance : int.MaxValue;
            LastIndex = res.Searched != 0 ? res.Index : 0;
            if (SyncMapAfterUpdate) HoleMap.SyncToHost();
            // UpdateObstacleMap (:751) ran on the device too when the handle was created with obstacle_map_size > 0
        }

        // ---- relocalisation (no counterpart in the reference: its simulator only offers Reset).  After a restart, or when the
        // robot was carried elsewhere, find where a scan lies on the current HoleMap, then resume tracking there.
        /// <summary>The k best poses of the lattice origin + (ix, iy, it) * step (count poses per axis) that are strict local
        /// minima of (distance, flat index) within +-window steps; best first.  points: ScanCloud.Points of one scan.
        /// distances (optional): Count[0]*Count[1]*Count[2] values in flat order.  Changes nothing; adopt a hit with ResumeAt.</summary>
        public CsLatticeHit[] Relocalize(Vector2[] points, Vector3 origin, Vector3 step, int countX, int countY, int countTheta,
                                         int window, int k, int[] distances = null)
        {
            var lattice = new CsLattice();
            lattice.Origin[0] = origin.X; lattice.Origin[1] = origin.Y; lattice.Origin[2] = origin.Z;
            lattice.Step[0] = step.X; lattice.Step[1] = step.Y; lattice.Step[2] = step.Z;
            lattice.Count[0] = countX; lattice.Count[1] = countY; lattice.Count[2] = countTheta;
            if (distances != null && distances.LongLength != (long)countX * countY * countTheta)
                throw new ArgumentException("distances needs countX*countY*countTheta entries");
            var hits = new CsLatticeHit[Native.LatticeMaxHits];
            int n;
            fixed (Vector2* p = points)
            fixed (CsLatticeHit* h = hits)
            fixed (int* d = distances)
                Native.Check(Native.cs_relocalize(handle, (float*)p, points.Length, ref lattice, window, k, h, out n, d), handle);
            return hits.Take(n).ToArray();
        }

        /// <summary>Relocalize's hits for the same lattice, window and k, by branch and bound: most poses of a fine lattice over
        /// the whole map are never evaluated, and a lattice may hold up to 2^31 - 1 poses.  stats: what the search did.
        /// Changes nothing; adopt a hit with ResumeAt.</summary>
        public CsLatticeHit[] RelocalizeBounded(Vector2[] points, Vector3 origin, Vector3 step, int countX, int countY, int countTheta,
                                                int window, int k, out CsRelocalizeStats stats)
        {
            var lattice = new CsLattice();
            lattice.Origin[0] = origin.X; lattice.Origin[1] = origin.Y; lattice.Origin[2] = origin.Z;
            lattice.Step[0] = step.X; lattice.Step[1] = step.Y; lattice.Step[2] = step.Z;
            lattice.Count[0] = countX; lattice.Count[1] = countY; lattice.Count[2] = countTheta;
            var hits = new CsLatticeHit[Native.LatticeMaxHits];
            int n;
            CsRelocalizeStats st;
            fixed (Vector2* p = points)
            fixed (CsLatticeHit* h = hits)
                Native.Check(Native.cs_relocalize_bounded(handle, (float*)p, points.Length, ref lattice, window, k, h, out n, &st), handle);
            stats = st;
            return hits.Take(n).ToArray();
        }

        /// <summary>Relocalize with the last few scans: scans[k] is ScanCloud.Points of scan k (oldest first, at most
        /// Native.SequenceMaxScans), odometry[k] the odometry pose it came with.  The lattice pose is the pose of the last scan;
        /// the others are placed by their odometry relative to it, and a pose's distance is the sum of the scans' distances.
        /// Places one scan cannot tell apart (repeated doors, identical rooms) are told apart.  Adopt a hit with
        /// ResumeAt(hit pose, odometry[last]).  Changes nothing.</summary>
        public CsLatticeHit[] RelocalizeSequence(Vector2[][] scans, Vector3[] odometry, Vector3 origin, Vector3 step, int countX, int countY,
                                                 int countTheta, int window, int k, int[] distances = null)
        {
            var lattice = SequenceLattice(scans, odometry, origin, step, countX, countY, countTheta, out var points, out var first, out var odo);
            if (distances != null && distances.LongLength != (long)countX * countY * countTheta)
                throw new ArgumentException("distances needs countX*countY*countTheta entries");
            var hits = new CsLatticeHit[Native.LatticeMaxHits];
            int n;
            fixed (Vector2* p = points)
            fixed (int* f = first)
            fixed (float* o = odo)
            fixed (CsLatticeHit* h = hits)
            fixed (int* d = distances)
                Native.Check(Native.cs_relocalize_sequence(handle, (float*)p, f, o, scans.Length, ref lattice, window, k, h, out n, d), handle);
            return hits.Take(n).ToArray();
        }

        /// <summary>RelocalizeSequence's hits by branch and bound, for fine lattices over the whole map.</summary>
        public CsLatticeHit[] RelocalizeSequenceBounded(Vector2[][] scans, Vector3[] odometry, Vector3 origin, Vector3 step, int countX,
                                                        int countY, int countTheta, int window, int k, out CsRelocalizeStats stats)
        {
            var lattice = SequenceLattice(scans, odometry, origin, step, countX, countY, countTheta, out var points, out var first, out var odo);
            var hits = new CsLatticeHit[Native.LatticeMaxHits];
            int n;
            CsRelocalizeStats st;
            fixed (Vector2* p = points)
            fixed (int* f = first)
            fixed (float* o = odo)
            fixed (CsLatticeHit* h = hits)
                Native.Check(Native.cs_relocalize_sequence_bounded(handle, (float*)p, f, o, scans.Length, ref lattice, window, k, h, out n, &st),
                             handle);
            stats = st;
            return hits.Take(n).ToArray();
        }

        // the lattice, and the scans back to back with their first points and odometry as cs_relocalize_sequence* take them
        private static CsLattice SequenceLattice(Vector2[][] scans, Vector3[] odometry, Vector3 origin, Vector3 step, int countX, int countY,
                                                 int countTheta, out Vector2[] points, out int[] first, out float[] odo)
        {
            if (odometry.Length != scans.Length) throw new ArgumentException("odometry needs one pose per scan");
            first = new int[scans.Length + 1];
            for (int s = 0; s < scans.Length; s++) first[s + 1] = first[s] + scans[s].Length;
            points = scans.SelectMany(x => x).ToArray();
            odo = new float[3 * scans.Length];
            for (int s = 0; s < scans.Length; s++) { odo[3 * s] = odometry[s].X; odo[3 * s + 1] = odometry[s].Y; odo[3 * s + 2] = odometry[s].Z; }
            var lattice = new CsLattice();
            lattice.Origin[0] = origin.X; lattice.Origin[1] = origin.Y; lattice.Origin[2] = origin.Z;
            lattice.Step[0] = step.X; lattice.Step[1] = step.Y; lattice.Step[2] = step.Z;
            lattice.Count[0] = countX; lattice.Count[1] = countY; lattice.Count[2] = countTheta;
            return lattice;
        }

        /// <summary>Continue tracking from `pose` (e.g. the best Relocalize hit, refined): odometryPose is the odometry of the
        /// scan that pose belongs to.  The next Update searches around pose + (odometry - odometryPose).</summary>
        public void ResumeAt(Vector3 pose, Vector3 odometryPose)
        {
            float* p = stackalloc float[3];
            float* o = stackalloc float[3];
            p[0] = pose.X; p[1] = pose.Y; p[2] = pose.Z;
            o[0] = odometryPose.X; o[1] = odometryPose.Y; o[2] = odometryPose.Z;
            Native.Check(Native.cs_set_pose(handle, p, o, positionSearchBeginning), handle);
            Pose = pose;
        }

        // ---- candidate split over the GPUs of a node (no counterpart in the reference: its split is over CPU threads,
        // ParallelMonteCarloSearch :674-710).  One CoreSLAMProcessor per GPU, all fed the same scans in the same order; after
        // AttachGroup every Update evaluates this rank's slice of the candidates and ends on the group's winner.
        /// <summary>64-byte handle of this processor's exchange table, to be passed to the other processes of the group.</summary>
        public byte[] ExportGroupHandle()
        {
            Native.Check(Native.cs_group_export(handle, out Native.CsIpcHandle h), handle);
            var bytes = new byte[64];
            for (int i = 0; i < 64; i++) bytes[i] = h.Bytes[i];
            return bytes;
        }

        /// <summary>One process per GPU: attach the handles of all ranks (this rank's own entry is ignored).</summary>
        public void AttachGroup(int rank, byte[][] handlesOfAllRanks)
        {
            var hs = new Native.CsIpcHandle[handlesOfAllRanks.Length];
            for (int r = 0; r < hs.Length; r++)
                for (int i = 0; i < 64; i++) hs[r].Bytes[i] = handlesOfAllRanks[r][i];
            fixed (Native.CsIpcHandle* p = hs) Native.Check(Native.cs_group_attach(handle, rank, hs.Length, p), handle);
        }

        /// <summary>One process driving several GPUs: the processors of the group, this one at index rank.</summary>
        public void AttachGroup(int rank, CoreSLAMProcessor[] group)
        {
            var hs = new IntPtr[group.Length];
            for (int r = 0; r < hs.Length; r++) hs[r] = group[r].handle;
            fixed (IntPtr* p = hs) Native.Check(Native.cs_group_attach_local(handle, rank, hs.Length, p), handle);
        }

        public void DetachGroup() => Native.Check(Native.cs_group_detach(handle), handle);

        public void Dispose()
        {
            if (handle == IntPtr.Zero) return;
            Native.cs_pinned_free(staging);
            Native.cs_destroy(handle);
            handle = IntPtr.Zero;
            GC.SuppressFinalize(this);
        }
    }
}
