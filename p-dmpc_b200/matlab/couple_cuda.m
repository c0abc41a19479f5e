function [adjacency, overlap_area] = couple_cuda(handle, iter, mpa)
% COUPLE_CUDA  The reachable-set coupling of ALL vehicles of a time step in ONE call on the GPU (pdmpc_couple).
%
%   Replaces ReachableSetCoupler.couple (hlc/controller/coupling/ReachableSetCoupler.m:5-54): vehicles i and j are
%   coupled iff their reachable sets of the last horizon step, iter.reachable_sets{i, end} and {j, end}, overlap by more
%   than 1e-3 (:39-42, area(intersect(...))).  The sets are mpa.local_reachable_sets_conv{trim, Hp} placed at the
%   measured poses, as mpa.reachable_sets_at_pose places them (MotionPrimitiveAutomaton.m:649-687); the overlap is a
%   convex clipping in FP64 (DESIGN.md §4.12), not polyshape's.  The prioritizer classes stay MATLAB's.
%   Not done here: HighLevelController.m:241-246 clips a reachable set by the predicted lanelets (polyshape
%   intersection); keep ReachableSetCoupler if a scenario depends on it.
%
%   handle       : planner handle of pdmpc_b200_mex (GraphSearchCuda.handle), MPA uploaded
%   iter         : IterationData of the time step (x0 [N x 4], trim_indices [N]), N <= 64
%   adjacency    : N x N, 1 where coupled                  -> what ReachableSetCoupler.couple returns
%   overlap_area : N x N overlap areas, 0 on the diagonal

    UPLOAD_REACHABLE_SETS = 10; COUPLE = 12;
    persistent uploaded_for
    if isempty(uploaded_for) || uploaded_for ~= handle
        % closed 2 x m polygons, as HighLevelController.m:258-264 turns polyshapes into plain arrays
        sets = cellfun(@(c) [c.Vertices(:, 1)', c.Vertices(1, 1); c.Vertices(:, 2)', c.Vertices(1, 2)], ...
            mpa.local_reachable_sets_conv, UniformOutput = false);
        pdmpc_b200_mex(UPLOAD_REACHABLE_SETS, handle, sets);
        uploaded_for = handle;
    end

    [adjacency, overlap_area] = pdmpc_b200_mex(COUPLE, handle, iter.x0(:, 1:3), iter.trim_indices(:));

end
